// opn_kernels.cu -- the single CUDA translation unit of libopusb200 (sm_100a, -fmad=false).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "imdct.cuh"
#include "imdct_warp.cuh"
#include "frame_warp.cuh"
#include "mathops.cuh"
#include "opn_tables.h"
#include "softclip.cuh"
#include "symbols.cuh"
#include "silk.cuh"

namespace opn {


static std::mutex g_tab_mutex;
static int g_sm_count = 148;
constexpr int W_CARVEOUT_PCT = 100;
static bool g_tab_done[64];
static uint16_t g_fblob_bytes[4][2];  // FBlobHdr::total per (LM, channels): the launchers size shared memory with it

template <int LM, int C> static cudaError_t set_carveout()
{
    // percent of the SM's unified 256 KB used as shared memory; the rest is L1 (history taps, per-stream state)
    const int smem = (int)frame_smem_bytes(LM, C, g_fblob_bytes[LM][C - 1]);
    cudaError_t e = cudaFuncSetAttribute(k_frame_w<LM, C, FRAME_SYNTH1>, cudaFuncAttributePreferredSharedMemoryCarveout, W_CARVEOUT_PCT);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_frame_w<LM, C, FRAME_SYNTH1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_frame_w<LM, C, FRAME_SYNTH2>, cudaFuncAttributePreferredSharedMemoryCarveout, W_CARVEOUT_PCT);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_frame_w<LM, C, FRAME_SYNTH2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    return e;
}
template <int LM, int C, int CS> static cudaError_t set_carveout_cross()
{
    const int smem = (int)frame_smem_bytes(LM, 2, g_fblob_bytes[LM][CS - 1]);
    cudaError_t e = cudaFuncSetAttribute(k_frame_w<LM, C, FRAME_SYNTH1, CS>, cudaFuncAttributePreferredSharedMemoryCarveout, W_CARVEOUT_PCT);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_frame_w<LM, C, FRAME_SYNTH1, CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_frame_w<LM, C, FRAME_SYNTH2, CS>, cudaFuncAttributePreferredSharedMemoryCarveout, W_CARVEOUT_PCT);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_frame_w<LM, C, FRAME_SYNTH2, CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    return e;
}
static size_t mix_smem_bytes(int C)
{
    size_t m = 0;
    for (int lm = 0; lm < 4; lm++) m = std::max(m, frame_smem_bytes(lm, C, g_fblob_bytes[lm][C - 1]));
    return m;
}
template <int C> static cudaError_t set_carveout_mix()
{
    const int smem = (int)mix_smem_bytes(C);
    cudaError_t e = cudaFuncSetAttribute(k_frame_mix<C, FRAME_SYNTH1>, cudaFuncAttributePreferredSharedMemoryCarveout, W_CARVEOUT_PCT);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_frame_mix<C, FRAME_SYNTH1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_frame_mix<C, FRAME_SYNTH2>, cudaFuncAttributePreferredSharedMemoryCarveout, W_CARVEOUT_PCT);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_frame_mix<C, FRAME_SYNTH2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    return e;
}
static cudaError_t set_warp_kernel_attributes()
{
    cudaError_t e = set_carveout<0, 1>();
    if (e == cudaSuccess) e = set_carveout_cross<0, 1, 2>();
    if (e == cudaSuccess) e = set_carveout_cross<0, 2, 1>();
    if (e == cudaSuccess) e = set_carveout_cross<1, 1, 2>();
    if (e == cudaSuccess) e = set_carveout_cross<1, 2, 1>();
    if (e == cudaSuccess) e = set_carveout_cross<2, 1, 2>();
    if (e == cudaSuccess) e = set_carveout_cross<2, 2, 1>();
    if (e == cudaSuccess) e = set_carveout_cross<3, 1, 2>();
    if (e == cudaSuccess) e = set_carveout_cross<3, 2, 1>();
    if (e == cudaSuccess) e = set_carveout_mix<1>();
    if (e == cudaSuccess) e = set_carveout_mix<2>();
    if (e == cudaSuccess) e = set_carveout<0, 2>();
    if (e == cudaSuccess) e = set_carveout<1, 1>();
    if (e == cudaSuccess) e = set_carveout<1, 2>();
    if (e == cudaSuccess) e = set_carveout<2, 1>();
    if (e == cudaSuccess) e = set_carveout<2, 2>();
    if (e == cudaSuccess) e = set_carveout<3, 1>();
    if (e == cudaSuccess) e = set_carveout<3, 2>();
    return e;
}

cudaError_t upload_tables(int device)
{
    std::lock_guard<std::mutex> lock(g_tab_mutex);
    if (device < 0 || device >= 64) return cudaErrorInvalidDevice;
    if (g_tab_done[device]) return cudaSuccess;
    static DevTables h;  // ~19 KB: keep it off the stack
    for (int i = 0; i < 1800; i++) h.trig[i] = OPN_TRIG[i];
    for (int i = 0; i < 120; i++) {
        h.window[i] = OPN_WINDOW[i];
        h.window_sq[i] = OPN_WINDOW[i] * OPN_WINDOW[i];  // host f32 product, single rounding
    }
    for (int i = 0; i < 480; i++) h.twiddles[i] = make_float2(OPN_TWIDDLES[2 * i], OPN_TWIDDLES[2 * i + 1]);
    for (int s = 0, trigp = 0, nn = 1920; s < 4; s++) {
        const int n4 = 480 >> s;
        for (int i = 0; i < n4; i++) h.trig_pair[trig_pair_off(s) + i] = make_float2(OPN_TRIG[trigp + i], OPN_TRIG[trigp + n4 + i]);
        nn >>= 1;
        trigp += nn;
    }
    for (int i = 0; i < 480; i++) h.bitrev[0][i] = OPN_BITREV_480[i];
    for (int i = 0; i < 240; i++) h.bitrev[1][i] = OPN_BITREV_240[i];
    for (int i = 0; i < 120; i++) h.bitrev[2][i] = OPN_BITREV_120[i];
    for (int i = 0; i < 60; i++) h.bitrev[3][i] = OPN_BITREV_60[i];
    for (int i = 0; i < 1272; i++) h.pvq_u_data[i] = OPN_PVQ_U_DATA[i];
    for (int i = 0; i < 15; i++) h.pvq_u_row[i] = OPN_PVQ_U_ROW[i];
    for (int k = 0; k < 15; k++) {  // row k holds columns k .. last(k); the rows are stored back to back
        const int first = OPN_PVQ_U_ROW[k] + k, end = k < 14 ? OPN_PVQ_U_ROW[k + 1] + k + 1 : 1272;
        const int next_end = k < 13 ? OPN_PVQ_U_ROW[k + 2] + k + 2 : 1272;  // end of row k+1
        uint32_t acc = 0;
        for (int i = first; i < end; i++) {
            const int m = i - OPN_PVQ_U_ROW[k];
            h.pvq_cw_data[i].x = acc;
            acc += OPN_PVQ_U_DATA[i];
            const int up = k < 14 ? OPN_PVQ_U_ROW[k + 1] + m : 1272;
            h.pvq_cw_data[i].y = (m >= k + 1 && up < next_end) ? OPN_PVQ_U_DATA[up] - OPN_PVQ_U_DATA[i] : 0u;
        }
    }
    for (int k = 0; k < 16; k++) {
        h.pvq_ev_nmax[k] = 0;
        if (k > 13) continue;  // the k < n regime reads U(k+1,.): rows 1..14
        auto last_col = [](int r) { return (r < 14 ? OPN_PVQ_U_ROW[r + 1] + r : 1271) - OPN_PVQ_U_ROW[r]; };  // rows are stored back to back
        const int last = std::min(last_col(k), last_col(k + 1));
        uint64_t rowsum = 0;  // sum_{j=k..n} U(k,j)
        for (int n = k; n <= last && n < 256; n++) {
            rowsum += OPN_PVQ_U_DATA[OPN_PVQ_U_ROW[k] + n];
            if (n > k && rowsum + OPN_PVQ_U_DATA[OPN_PVQ_U_ROW[k + 1] + n] < (1ull << 32)) h.pvq_ev_nmax[k] = (uint8_t)n;
            else if (n > k) break;
        }
    }
    for (int i = 0; i < 22; i++) h.e_bands[i] = OPN_E_BANDS[i];
    for (int l = 0; l < 4; l++)
        for (int b = 0; b < 21; b++)
            for (int k = 0; k < 3; k++) h.synth_sched[l][b][k] = OPN_SYNTH_SCHED[l][b][k];
    for (int lm = 0; lm < 4; lm++)
        for (int C = 1; C <= 2; C++) {
            int ne = 0;
            const int nf = 120 << lm;
            for (int b = 0; b < 21; b++)
                for (int c = 0; c < C; c++) {
                    const uint32_t n = OPN_SYNTH_SCHED[lm][b][0], parts = OPN_SYNTH_SCHED[lm][b][1], k = OPN_SYNTH_SCHED[lm][b][2];
                    for (uint32_t p = 0; p < parts; p++) {
                        SynthEntry &e = h.synth_entries[lm][C - 1][ne++];
                        e.base = (uint16_t)(c * nf + ((int)OPN_E_BANDS[b] << lm) + (int)(p * n));
                        e.n = (uint8_t)n;
                        e.k = (uint8_t)k;
                        e.ft_minus1 = 0; e.magic = 0; e.ft1 = 0; e.ftb = 0; e.sh = 0;
                        if (n > 64 || k > 6) return cudaErrorInvalidValue;  // w_expand keeps a part's pulses as six 10-bit records
                        if (n == 1) continue;
                        if (n > 2 && k < n) {
                            // k_synth_expand bisects on 32-bit sums: the whole row sum plus U(k+1,n) must not wrap
                            uint64_t rowsum = 0;
                            for (uint32_t j = k; j <= n; j++) rowsum += OPN_PVQ_U_DATA[OPN_PVQ_U_ROW[k] + j];
                            if (k >= 14 || rowsum + OPN_PVQ_U_DATA[OPN_PVQ_U_ROW[k + 1] + n] >= (1ull << 32)) return cudaErrorInvalidValue;
                            if (n > h.pvq_ev_nmax[k]) return cudaErrorInvalidValue;  // the schedule's parts all take the event path
                        }
                        auto U = [](uint32_t a, uint32_t bb) { return OPN_PVQ_U_DATA[OPN_PVQ_U_ROW[a < bb ? a : bb] + (a < bb ? bb : a)]; };
                        const uint32_t ft = U(n, k) + U(n, k + 1);   // pvq_v, pvc.rs:289-291
                        e.ft_minus1 = ft - 1;
                        uint32_t ftb = 32u - (uint32_t)__builtin_clz(ft - 1);  // ilog(ft-1), decoder.rs:247-248
                        uint32_t ft1;
                        if (ftb > 8) { ftb -= 8; ft1 = ((ft - 1) >> ftb) + 1; } else { ftb = 0; ft1 = ft; }
                        e.ftb = (uint8_t)ftb;
                        e.ft1 = (uint16_t)ft1;
                        uint32_t sh = 0;
                        while ((1ull << sh) < ft1) sh++;
                        e.sh = (uint8_t)sh;
                        e.magic = (uint32_t)((((1ull << sh) - ft1) << 32) / ft1 + 1);
                    }
                }
            h.synth_n_entries[lm][C - 1] = (uint8_t)ne;
            // bin -> part map for the coefficient write of k_synth_expand
            uint8_t *eo = h.synth_entry_of[lm][C - 1];
            for (int i = 0; i < 2 * 960; i++) eo[i] = SYNTH_MAX_ENTRIES;
            for (int e = 0; e < ne; e++) {
                const SynthEntry &E = h.synth_entries[lm][C - 1][e];
                for (int j = 0; j < (int)E.n; j++) eo[E.base + j] = (uint8_t)e;
            }
            // k_synth_expand: parts sorted by the number of dimensions cwrsi has to walk (descending), 32 per slot,
            // so that the lanes of a slot have walks of similar length.  Sign-only bands (n == 1) and
            // single-pulse parts (k == 1, closed form) walk nothing.
            {
                auto walk = [&](int e) {
                    const SynthEntry &E = h.synth_entries[lm][C - 1][e];
                    return (E.n == 1 || E.k == 1) ? 0 : (int)E.n;
                };
                int order[SYNTH_MAX_ENTRIES];
                for (int e = 0; e < ne; e++) order[e] = e;
                for (int a = 1; a < ne; a++) {  // insertion sort, stable
                    const int v = order[a];
                    int b2 = a - 1;
                    while (b2 >= 0 && walk(order[b2]) < walk(v)) {
                        order[b2 + 1] = order[b2];
                        b2--;
                    }
                    order[b2 + 1] = v;
                }
                const int nslots = (ne + 31) / 32;
                if (nslots > SYNTH_SLOTS) return cudaErrorInvalidValue;
                h.synth_n_slots[lm][C - 1] = (uint8_t)nslots;
                for (int sl = 0; sl < SYNTH_SLOTS; sl++) {
                    h.synth_slot_maxn[lm][C - 1][sl] = 0;
                    for (int l = 0; l < 32; l++) {
                        const int r = sl * 32 + l;
                        h.synth_slot_entries[lm][C - 1][sl][l] = r < ne ? (uint8_t)order[r] : 0xFF;
                        if (r < ne && walk(order[r]) > h.synth_slot_maxn[lm][C - 1][sl]) h.synth_slot_maxn[lm][C - 1][sl] = (uint8_t)walk(order[r]);
                    }
                }
            }
        }
    for (int i = 0; i < 21; i++) h.log_n[i] = OPN_LOG_N[i];
    for (int i = 0; i < 231; i++) h.alloc_vectors[i] = OPN_ALLOC_VECTORS[i];
    for (int i = 0; i < 105; i++) h.cache_index[i] = OPN_CACHE_INDEX[i];
    for (int i = 0; i < 392; i++) h.cache_bits[i] = OPN_CACHE_BITS[i];
    for (int i = 0; i < 168; i++) h.cache_caps[i] = OPN_CACHE_CAPS[i];
    for (int i = 0; i < 24; i++) h.log2_frac[i] = OPN_LOG2_FRAC_TABLE[i];
    h.tapset_icdf[0] = 2; h.tapset_icdf[1] = 1; h.tapset_icdf[2] = 0; h.tapset_icdf[3] = 0;
    for (int i = 0; i < 9; i++) h.comb_gains[i] = OPN_COMB_GAINS[i];
    // ---- the frame kernel's table blobs (FBlobHdr), one per (LM, channels)
    static uint8_t blobs[4][2][FBLOB_MAX_BYTES];
    for (int lm = 0; lm < 4; lm++)
        for (int C = 1; C <= 2; C++) {
            uint8_t *bl = blobs[lm][C - 1];
            std::memset(bl, 0, FBLOB_MAX_BYTES);
            FBlobHdr &H = h.fblob_hdr[lm][C - 1];
            size_t at = 0;
            auto put = [&](const void *src, size_t bytes) {
                const size_t off = at;
                if (off + bytes > FBLOB_MAX_BYTES) return (size_t)0xFFFF;
                if (src) std::memcpy(bl + off, src, bytes);
                at = (off + bytes + 15) & ~(size_t)15;
                return off;
            };
            const int shift = 3 - lm;
            H.tp_long = (uint16_t)put(h.trig_pair + trig_pair_off(shift), (size_t)(480 >> shift) * sizeof(float2));
            H.tp_short = (uint16_t)put(h.trig_pair + trig_pair_off(3), 60 * sizeof(float2));
            H.tw = (uint16_t)put(h.twiddles, 480 * sizeof(float2));
            H.win = (uint16_t)put(h.window, 120 * sizeof(float));
            H.win_sq = (uint16_t)put(h.window_sq, 120 * sizeof(float));
            // rectangular slice of the PVQ tables that covers the schedule's parts: rows 0 .. kmax+1, columns 0 .. nmax
            const int ne = h.synth_n_entries[lm][C - 1];
            int kmax = 1, nmax = 2;
            for (int e2 = 0; e2 < ne; e2++) {
                kmax = std::max(kmax, (int)h.synth_entries[lm][C - 1][e2].k);
                nmax = std::max(nmax, (int)h.synth_entries[lm][C - 1][e2].n);
            }
            nmax = std::max(nmax, kmax + 1);
            const int rows = kmax + 2, cols = nmax + 1;
            if (rows > 15) return cudaErrorInvalidValue;
            std::vector<uint32_t> cu((size_t)rows * cols, 0u);
            std::vector<uint2> ccw((size_t)rows * cols, make_uint2(0u, 0u));
            auto last_col = [](int r) { return (r < 14 ? OPN_PVQ_U_ROW[r + 1] + r : 1271) - OPN_PVQ_U_ROW[r]; };
            for (int k = 0; k < rows; k++)
                for (int n = 0; n < cols; n++) {
                    const int lo = std::min(k, n), hi = std::max(k, n);
                    if (hi > last_col(lo)) return cudaErrorInvalidValue;
                    cu[(size_t)k * cols + n] = OPN_PVQ_U_DATA[OPN_PVQ_U_ROW[lo] + hi];
                    if (n >= k) ccw[(size_t)k * cols + n] = h.pvq_cw_data[OPN_PVQ_U_ROW[k] + n];
                }
            H.pvq_u = (uint16_t)put(cu.data(), cu.size() * sizeof(uint32_t));
            H.pvq_cw = (uint16_t)put(ccw.data(), ccw.size() * sizeof(uint2));
            uint16_t row16[16];
            for (int k = 0; k < 16; k++) row16[k] = (uint16_t)(std::min(k, rows - 1) * cols);
            H.pvq_row = (uint16_t)put(row16, sizeof(row16));
            H.pvq_nmax = (uint16_t)put(h.pvq_ev_nmax, 16);
            H.ent = (uint16_t)put(h.synth_entries[lm][C - 1], (size_t)ne * sizeof(SynthEntry));
            H.slots = (uint16_t)put(h.synth_slot_entries[lm][C - 1], SYNTH_SLOTS * 32);
            if (at > FBLOB_MAX_BYTES || at > 0xFFF0) return cudaErrorInvalidValue;
            H.total = (uint16_t)at;
            H.n_slots = h.synth_n_slots[lm][C - 1];
            H.n_entries = (uint16_t)ne;
            H.cols = (uint16_t)cols;
            H.pad = 0;
            g_fblob_bytes[lm][C - 1] = H.total;
        }
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess) return e;
    e = cudaMemcpyToSymbol(g_tab, &h, sizeof(h));
    if (e != cudaSuccess) return e;
    e = cudaMemcpyToSymbol(g_fblob, blobs, sizeof(blobs));
    if (e != cudaSuccess) return e;
    e = cudaMemcpyToSymbol(g_exp2_q9, OPN_EXP2_Q9, sizeof(float) * 512);
    if (e == cudaSuccess) {
        static SilkTables sk;
        std::memset(&sk, 0, sizeof(sk));
        for (int i = 0; i < 64; i++) sk.gain_q10[i] = OPN_SILK_GAIN_Q10[i];
        for (int i = 0; i < 40; i++) sk.ltp_q14[i] = OPN_SILK_LTP_Q14[i];
        for (int i = 0; i < 3; i++) sk.type_icdf[i] = OPN_SILK_TYPE_ICDF[i];
        for (int i = 0; i < 9; i++) sk.delta_icdf[i] = OPN_SILK_DELTA_GAIN_ICDF[i];
        for (int i = 0; i < 4; i++) sk.contour_icdf[i] = OPN_SILK_CONTOUR_ICDF[i];
        for (int i = 0; i < 8; i++) sk.ltp_icdf[i] = OPN_SILK_LTP_ICDF[i];
        for (int i = 0; i < 18; i++) sk.pulses_icdf[i] = OPN_SILK_PULSES_ICDF[i];
        static float up[3][48];
        std::memset(up, 0, sizeof(up));
        for (int i = 0; i < 48; i++) up[0][i] = OPN_SILK_UP6[i];
        for (int i = 0; i < 32; i++) up[1][i] = OPN_SILK_UP4[i];
        for (int i = 0; i < 24; i++) up[2][i] = OPN_SILK_UP3[i];
        e = cudaMemcpyToSymbol(g_silk, &sk, sizeof(sk));
        if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_silk_up, up, sizeof(up));
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_silk_frame<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)silk_frame_smem());
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_silk_frame<1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)silk_frame_smem());
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_silk_frame<2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)silk_frame_smem());
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_silk_frame<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)silk_frame_smem());
    }
    if (e != cudaSuccess) return e;
    e = set_warp_kernel_attributes();
    if (e != cudaSuccess) return e;
    // kernel 1 needs more than the 48 KB default only if ever re-tiled; set the limits once here
    e = cudaFuncSetAttribute(k_rangedec_script, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_synth_expand, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)synth_expand_smem());
    if (e != cudaSuccess) return e;
    g_tab_done[device] = true;
    return cudaSuccess;
}

template <int LM, int C> static cudaError_t launch_frame_w(const FrameArgs &a, cudaStream_t st)
{
    const size_t smem = frame_smem_bytes(LM, C, g_fblob_bytes[LM][C - 1]);
    const uint32_t grid = (a.item_end - a.item0 + FRAME_WARPS - 1) / FRAME_WARPS;
    if (a.parts) k_frame_w<LM, C, FRAME_SYNTH2><<<grid, 32 * FRAME_WARPS, smem, st>>>(a);
    else k_frame_w<LM, C, FRAME_SYNTH1><<<grid, 32 * FRAME_WARPS, smem, st>>>(a);
    return cudaGetLastError();
}

// packets of CS channels into a decoder of C != CS channels (mono <-> stereo mapping inside the frame kernel)
template <int LM, int C, int CS> static cudaError_t launch_frame_cross(const FrameArgs &a, cudaStream_t st)
{
    const size_t smem = frame_smem_bytes(LM, 2, g_fblob_bytes[LM][CS - 1]);
    const uint32_t grid = (a.item_end - a.item0 + FRAME_WARPS - 1) / FRAME_WARPS;
    if (a.parts) k_frame_w<LM, C, FRAME_SYNTH2, CS><<<grid, 32 * FRAME_WARPS, smem, st>>>(a);
    else k_frame_w<LM, C, FRAME_SYNTH1, CS><<<grid, 32 * FRAME_WARPS, smem, st>>>(a);
    return cudaGetLastError();
}

static size_t symbols_smem(uint32_t pkt_cap)
{
    return 3 * PVQ_TABLE_WORDS * 4 + 32 + 16 + (size_t)SYM_WARPS_PER_CTA * Y_STAGE * 4 + (size_t)SYM_WARPS_PER_CTA * pkt_cap;
}

cudaError_t launch_rangedec_script(const uint8_t *arena, const uint32_t *offsets, const uint32_t *lens, uint32_t n_packets,
                                   const opn_op *ops, uint32_t n_ops, const uint8_t *icdf_pool, opn_op_out *out,
                                   int32_t *y_out, uint32_t y_stride, uint32_t pkt_cap, cudaStream_t st)
{
    if (n_packets == 0) return cudaSuccess;
    const uint32_t grid = (n_packets + SYM_WARPS_PER_CTA - 1) / SYM_WARPS_PER_CTA;
    k_rangedec_script<<<grid, SYM_WARPS_PER_CTA * 32, symbols_smem(pkt_cap), st>>>(arena, offsets, lens, n_packets, ops, n_ops,
                                                                                 icdf_pool, out, y_out, y_stride, pkt_cap);
    return cudaGetLastError();
}

cudaError_t launch_synth_rangedec(const SymbolArgs &a, cudaStream_t st)
{
    if (a.n_items == 0) return cudaSuccess;
    if (!a.idx) return cudaErrorInvalidValue;
    constexpr uint32_t per_cta = RANGEDEC_WARPS_PER_CTA * 32u;
    k_synth_rangedec<<<(a.n_items + per_cta - 1u) / per_cta, per_cta, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_synth_expand(const SymbolArgs &a, cudaStream_t st)
{
    if (a.n_items == 0) return cudaSuccess;
    if (!a.idx) return cudaErrorInvalidValue;
    const uint32_t grid = (a.n_items + EXPAND_WARPS_PER_CTA - 1) / EXPAND_WARPS_PER_CTA;
    k_synth_expand<<<grid, EXPAND_WARPS_PER_CTA * 32, synth_expand_smem(), st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_celt2_rangedec(const SymbolArgs &a, cudaStream_t st)
{
    if (a.n_items == 0) return cudaSuccess;
    if (!a.parts || !a.hdr || !a.bande) return cudaErrorInvalidValue;
    k_celt2_rangedec<<<(a.n_items + C2_RD_ITEMS_PER_CTA - 1u) / C2_RD_ITEMS_PER_CTA, RANGEDEC_WARPS_PER_CTA * 32u, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_celt2_expand(const SymbolArgs &a, cudaStream_t st)
{
    if (a.n_items == 0) return cudaSuccess;
    k_celt2_expand<<<(a.n_items + 3u) / 4u, 128, 4 * 2 * 960 * sizeof(float), st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_synth_symbols(const SymbolArgs &a, cudaStream_t st)
{
    cudaError_t e = launch_synth_rangedec(a, st);
    if (e != cudaSuccess) return e;
    return launch_synth_expand(a, st);
}

cudaError_t launch_frame(const FrameArgs &a, cudaStream_t st)
{
    if (a.item_end <= a.item0) return cudaSuccess;
    if (!a.idx && !a.parts) return cudaErrorInvalidValue;
    if (a.stream_channels != 0 && a.stream_channels != a.channels) {
        switch (a.lm * 2 + (a.channels - 1)) {
        case 0: return launch_frame_cross<0, 1, 2>(a, st);
        case 1: return launch_frame_cross<0, 2, 1>(a, st);
        case 2: return launch_frame_cross<1, 1, 2>(a, st);
        case 3: return launch_frame_cross<1, 2, 1>(a, st);
        case 4: return launch_frame_cross<2, 1, 2>(a, st);
        case 5: return launch_frame_cross<2, 2, 1>(a, st);
        case 6: return launch_frame_cross<3, 1, 2>(a, st);
        case 7: return launch_frame_cross<3, 2, 1>(a, st);
        default: return cudaErrorInvalidValue;
        }
    }
    switch (a.lm * 2 + (a.channels - 1)) {
    case 0: return launch_frame_w<0, 1>(a, st);
    case 1: return launch_frame_w<0, 2>(a, st);
    case 2: return launch_frame_w<1, 1>(a, st);
    case 3: return launch_frame_w<1, 2>(a, st);
    case 4: return launch_frame_w<2, 1>(a, st);
    case 5: return launch_frame_w<2, 2>(a, st);
    case 6: return launch_frame_w<3, 1>(a, st);
    case 7: return launch_frame_w<3, 2>(a, st);
    default: return cudaErrorInvalidValue;
    }
}

int kernels_frame_groups() { return OPN_FRAME_GROUPS; }

cudaError_t launch_mix_plan(const MixArgs &a, cudaStream_t st)
{
    if (a.n_streams == 0) return cudaSuccess;
    if (!a.plan || !a.key || !a.rank || !a.last_lm || !a.item_lm || !a.item_offsets || !a.item_lens || !a.item_stream) return cudaErrorInvalidValue;
    if (a.n_groups != 1 && a.n_groups != MIX_GROUPS) return cudaErrorInvalidValue;
    cudaError_t e = cudaMemsetAsync(a.plan, 0, sizeof(MixPlan), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(a.item_lm, MIX_NO_ITEM, mix_item_cap(a.n_streams), st);
    if (e != cudaSuccess) return e;
    const uint32_t grid = (a.n_streams + 255u) / 256u;
    k_mix_key<<<grid, 256, 0, st>>>(a);
    k_mix_place<<<grid, 256, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_frame_mix(const FrameArgs &a, uint32_t n_streams_in_group, cudaStream_t st)
{
    if (n_streams_in_group == 0) return cudaSuccess;
    if (!a.plan || a.group < 0 || a.group >= MIX_GROUPS || (!a.idx && !a.parts) || !a.stream_idx) return cudaErrorInvalidValue;
    const uint32_t grid = (n_streams_in_group + FRAME_WARPS - 1) / FRAME_WARPS + 4u;  // each of the four buckets rounds up
    const size_t smem = mix_smem_bytes(a.channels);
    if (a.channels == 2) {
        if (a.parts) k_frame_mix<2, FRAME_SYNTH2><<<grid, 32 * FRAME_WARPS, smem, st>>>(a);
        else k_frame_mix<2, FRAME_SYNTH1><<<grid, 32 * FRAME_WARPS, smem, st>>>(a);
    } else if (a.channels == 1) {
        if (a.parts) k_frame_mix<1, FRAME_SYNTH2><<<grid, 32 * FRAME_WARPS, smem, st>>>(a);
        else k_frame_mix<1, FRAME_SYNTH1><<<grid, 32 * FRAME_WARPS, smem, st>>>(a);
    } else {
        return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t launch_op_imdct(const float *in, size_t in_stride, float *out, size_t out_stride, uint32_t n_rows, int shift,
                            int nblk, cudaStream_t st)
{
    if (n_rows == 0) return cudaSuccess;
    const size_t smem = (size_t)((960 >> shift) * nblk + 60) * 4;
    if (nblk == 1) {
        switch (shift) {
        case 0: k_op_imdct_w<0, 1><<<n_rows, 32, smem, st>>>(in, in_stride, out, out_stride); break;
        case 1: k_op_imdct_w<1, 1><<<n_rows, 32, smem, st>>>(in, in_stride, out, out_stride); break;
        case 2: k_op_imdct_w<2, 1><<<n_rows, 32, smem, st>>>(in, in_stride, out, out_stride); break;
        default: k_op_imdct_w<3, 1><<<n_rows, 32, smem, st>>>(in, in_stride, out, out_stride); break;
        }
    } else {
        if (shift != 3) return cudaErrorInvalidValue;  // short blocks are always 120-bin MDCTs
        switch (nblk) {
        case 2: k_op_imdct_w<3, 2><<<n_rows, 32, smem, st>>>(in, in_stride, out, out_stride); break;
        case 4: k_op_imdct_w<3, 4><<<n_rows, 32, smem, st>>>(in, in_stride, out, out_stride); break;
        case 8: k_op_imdct_w<3, 8><<<n_rows, 32, smem, st>>>(in, in_stride, out, out_stride); break;
        default: return cudaErrorInvalidValue;
        }
    }
    return cudaGetLastError();
}

cudaError_t launch_op_comb_inplace(float *y, size_t row_stride, int y_offset, int n, uint32_t n_rows, const int32_t *params4,
                                   const float *gains2, int overlap, cudaStream_t st)
{
    if (n_rows == 0) return cudaSuccess;
    const size_t smem = ((size_t)n * 4 + 15) & ~(size_t)15;
    if (smem > 48 * 1024) return cudaErrorInvalidValue;
    k_op_comb_inplace_w<<<n_rows, 32, smem, st>>>(y, row_stride, y_offset, n, params4, gains2, overlap);
    return cudaGetLastError();
}

cudaError_t launch_op_comb(float *y, const float *x, size_t row_stride, int offset, int n, uint32_t n_rows,
                           const int32_t *params4, const float *gains2, int overlap, cudaStream_t st)
{
    if (n_rows == 0) return cudaSuccess;
    k_op_comb<<<n_rows, IM_TPC, 0, st>>>(y, x, row_stride, offset, n, params4, gains2, overlap);
    return cudaGetLastError();
}

cudaError_t launch_op_bitexact_trig(const int16_t *x, int16_t *out_cos, uint32_t n_cos, const int32_t *isin, const int32_t *icos,
                                    int32_t *out_l2t, uint32_t n_l2t, cudaStream_t st)
{
    const uint32_t n = n_cos > n_l2t ? n_cos : n_l2t;
    if (n == 0) return cudaSuccess;
    k_op_bitexact_trig<<<(n + 255) / 256, 256, 0, st>>>(x, out_cos, n_cos, isin, icos, out_l2t, n_l2t);
    return cudaGetLastError();
}

template <typename T>
static cudaError_t launch_softclip_convert_t(const float *dense, size_t dense_stride, const int32_t *clip_len, int channels,
                                             uint32_t row_floats, uint32_t first_row, uint32_t n_rows, float *mem, void *out,
                                             size_t out_stride, cudaStream_t st)
{
    // the row is staged in shared memory: frame sizes beyond 120 ms (a larger buffer than any packet can fill) need more
    // than the 48 KB default
    const size_t smem = (size_t)row_floats * sizeof(float);
    if (smem > 200 * 1024) return cudaErrorInvalidValue;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k_softclip_convert<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
    }
    k_softclip_convert<T><<<n_rows, 32, smem, st>>>(dense, dense_stride, clip_len, channels, row_floats,
                                                                                   first_row, mem, static_cast<T *>(out), out_stride);
    return cudaGetLastError();
}

cudaError_t launch_softclip_convert(int sample_format, const float *dense, size_t dense_stride, const int32_t *clip_len, int channels,
                                    uint32_t row_floats, uint32_t first_row, uint32_t n_rows, float *mem, void *out, size_t out_stride,
                                    cudaStream_t st)
{
    if (n_rows == 0) return cudaSuccess;
    if (row_floats % 8u || (dense_stride & 3) || (out_stride & 7)) return cudaErrorInvalidValue;
    switch (sample_format) {
    case OPN_SAMPLE_F32: return launch_softclip_convert_t<float>(dense, dense_stride, clip_len, channels, row_floats, first_row, n_rows, mem, out, out_stride, st);
    case OPN_SAMPLE_I16: return launch_softclip_convert_t<int16_t>(dense, dense_stride, clip_len, channels, row_floats, first_row, n_rows, mem, out, out_stride, st);
    case OPN_SAMPLE_I32: return launch_softclip_convert_t<int32_t>(dense, dense_stride, clip_len, channels, row_floats, first_row, n_rows, mem, out, out_stride, st);
    case OPN_SAMPLE_U16: return launch_softclip_convert_t<uint16_t>(dense, dense_stride, clip_len, channels, row_floats, first_row, n_rows, mem, out, out_stride, st);
    case OPN_SAMPLE_U32: return launch_softclip_convert_t<uint32_t>(dense, dense_stride, clip_len, channels, row_floats, first_row, n_rows, mem, out, out_stride, st);
    case OPN_SAMPLE_F64: return launch_softclip_convert_t<double>(dense, dense_stride, clip_len, channels, row_floats, first_row, n_rows, mem, out, out_stride, st);
    default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_op_soft_clip(float *pcm, size_t row_stride, size_t row_len, int channels, uint32_t n_rows, float *mem,
                                cudaStream_t st)
{
    if (n_rows == 0 || channels <= 0) return cudaSuccess;
    const uint32_t total = n_rows * (uint32_t)channels;
    k_op_soft_clip<<<(total + 63) / 64, 64, 0, st>>>(pcm, row_stride, row_len, channels, n_rows, mem);
    return cudaGetLastError();
}

cudaError_t launch_op_smooth_fade(const float *in1, const float *in2, float *out, size_t row_stride, int overlap, int channels, int fs,
                                  uint32_t n_rows, cudaStream_t st)
{
    if (n_rows == 0 || overlap <= 0) return cudaSuccess;
    if (channels < 1 || fs <= 0 || 48000 % fs != 0 || (overlap - 1) * (48000 / fs) >= 120) return cudaErrorInvalidValue;
    const dim3 grid((uint32_t)(overlap * channels + 127) / 128, n_rows);
    k_op_smooth_fade<<<grid, 128, 0, st>>>(in1, in2, out, row_stride, overlap, channels, 48000 / fs);
    return cudaGetLastError();
}

cudaError_t launch_silk_rangedec(const SilkArgs &a, cudaStream_t st)
{
    if (a.n_items == 0) return cudaSuccess;
    k_silk_rangedec<<<(a.n_items + 31u) / 32u, 32, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_silk_frame(const SilkArgs &a0, cudaStream_t st)
{
    if (a0.n_items == 0) return cudaSuccess;
    SilkArgs a = a0;
    static unsigned long long *clk = [] {  // OPN_SILK_CLK=1: per-phase cycle counters, printed when the process exits
        unsigned long long *p = nullptr;
        const char *e = std::getenv("OPN_SILK_CLK");
        if (e && e[0] == '1' && cudaMallocManaged(&p, 4 * sizeof(unsigned long long)) == cudaSuccess) {
            std::memset(p, 0, 4 * sizeof(unsigned long long));
            static unsigned long long *keep = p;
            std::atexit([] {
                if (keep[3]) fprintf(stderr, "k_silk_frame cycles per CTA: A %.0f  B %.0f  C %.0f  (%llu CTAs)\n", (double)keep[0] / keep[3],
                                     (double)keep[1] / keep[3], (double)keep[2] / keep[3], keep[3]);
            });
        }
        return p;
    }();
    a.phase_clk = clk;
    const int cs = a.stream_channels, c = a.channels;
    if (cs < 1 || cs > 2 || c < 1 || c > 2 || (a.frame_ms != 10 && a.frame_ms != 20)) return cudaErrorInvalidValue;
    if (a.item_end == 0) a.item_end = a.n_items;
    if (a.item_end <= a.item0) return cudaSuccess;
    const uint32_t items_per_cta = (uint32_t)(SILK_ROWS / cs), grid = (a.item_end - a.item0 + items_per_cta - 1u) / items_per_cta;
    const size_t smem = silk_frame_smem();
    if (cs == 1 && c == 1) k_silk_frame<1, 1><<<grid, 32 * SILK_WARPS, smem, st>>>(a);
    else if (cs == 1) k_silk_frame<1, 2><<<grid, 32 * SILK_WARPS, smem, st>>>(a);
    else if (c == 1) k_silk_frame<2, 1><<<grid, 32 * SILK_WARPS, smem, st>>>(a);
    else k_silk_frame<2, 2><<<grid, 32 * SILK_WARPS, smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_transition_fade(float *dense, size_t dense_stride, const uint32_t *d_streams, uint32_t n_streams, uint32_t n_rows, int channels,
                                   cudaStream_t st)
{
    if (n_streams == 0) return cudaSuccess;
    k_transition_fade<<<n_streams, 128, 0, st>>>(dense, dense_stride, d_streams, n_rows, channels);
    return cudaGetLastError();
}

}  // namespace opn
