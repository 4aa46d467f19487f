// silk.cuh -- SYNTH-SILK/1 frames on the device (DESIGN.md section 3c): north_star's src/silk part -- "LPC synthesis across
// streams and the polyphase resampler to 48 kHz".  The reference's SilkDecoder::decode is unimplemented!()
// (src/silk/decoder.rs:71-80; caller src/decoder.rs:552-624, merge src/decoder.rs:722-729), so the frame layout is this
// repo's own (oracle/silk.c states it; parity unpinned): range-coder operations the crate implements around long-term
// prediction, the integer short-term synthesis recursion of SURVEY.md appendix B and a polyphase interpolator.
//
// One step = two launches, like the CELT path:
//   k_silk_rangedec   one LANE per packet (LaneDec): symbols -> one 144-byte record per coded channel
//   k_silk_frame      one CTA per 32 coded channels ("rows"; a stereo packet is two rows), 8 warps, three phases:
//     A  warp per row:  PVQ shell blocks -> excitation (one lane per 16-sample block, cwrsi_events), sign dither, long-term
//                       prediction in spans of lag-2 samples (a sample's taps lie at least lag-2 samples back), reflection
//                       coefficients -> A_Q12 with one lane per coefficient; rows land TRANSPOSED in shared memory
//                       ([sample][row], row stride 33 words: conflict-free for both access patterns)
//     B  lane per row:  the LPC recursion is strictly serial per channel (sat32 makes it non-linear: no scan), so it runs
//                       ACROSS streams: 32 channels per warp, the 16-sample window and the 16 coefficients in registers
//     C  warp per item: mid/side -> left/right, polyphase interpolation to 48 kHz, x 1/32768, coalesced stores into the PCM
//                       ring and the dense rows
#pragma once
#include "opn_device.cuh"
#include "rangedec.cuh"
#include "symbols.cuh"

namespace opn {

struct SilkTables {
    int32_t gain_q10[64];
    int16_t ltp_q14[40];
    uint8_t type_icdf[4], delta_icdf[12], contour_icdf[4], ltp_icdf[8], pulses_icdf[20];
};
__device__ SilkTables g_silk;
// resampler taps [0] x6 (8 kHz), [1] x4 (12 kHz), [2] x3 (16 kHz), [phase][tap]: constant memory, so that the fully unrolled
// interpolation reads them as instruction operands
__constant__ float c_silk_up[3][48];

__device__ __forceinline__ int32_t silk_smulwb(int32_t a, int32_t b16) { return (int32_t)(((int64_t)a * (int64_t)b16) >> 16); }
// the same with the 16-bit factor pre-shifted: (a * (b << 16)) >> 32 == (a * b) >> 16, one IMAD.HI
#ifdef OPN_SILK_EXP_FAKE_MUL  // timing experiment only (wrong results): what the multiply-high costs
__device__ __forceinline__ int32_t silk_smulwb_sh(int32_t a, int32_t b16_shl16) { return a * b16_shl16; }
#else
__device__ __forceinline__ int32_t silk_smulwb_sh(int32_t a, int32_t b16_shl16) { return __mulhi(a, b16_shl16); }
#endif
__device__ __forceinline__ int32_t silk_smulww(int32_t a, int32_t b) { return (int32_t)(((int64_t)a * (int64_t)b) >> 16); }
__device__ __forceinline__ int32_t silk_sat16(int32_t x) { return max(-32768, min(32767, x)); }

// ------------------------------------------------------------------------------------------------- range decode
__global__ void __launch_bounds__(32) k_silk_rangedec(SilkArgs A)
{
    __shared__ uint8_t s_icdf[48];  // type 0..3 | delta 4..15 | contour 16..19 | ltp 20..27 | pulses 28..47
    const uint32_t lane = threadIdx.x;
    if (lane < 4u) s_icdf[lane] = g_silk.type_icdf[lane];
    if (lane < 12u) s_icdf[4u + lane] = g_silk.delta_icdf[lane];
    if (lane < 4u) s_icdf[16u + lane] = g_silk.contour_icdf[lane];
    if (lane < 8u) s_icdf[20u + lane] = g_silk.ltp_icdf[lane];
    if (lane < 20u) s_icdf[28u + lane] = g_silk.pulses_icdf[lane];
    __syncwarp();
    const uint32_t item = blockIdx.x * 32u + lane;
    if (item >= A.n_items) return;
    int frame_ms = A.frame_ms;
    if (A.item_ms) {  // mixed-mode step: padding items between the buckets
        frame_ms = A.item_ms[item];
        if (frame_ms == MIX_NO_ITEM) return;
    }
    const uint32_t stream = A.stream_idx ? A.stream_idx[item] : item;
    uint32_t len = A.lens[item];
    const uint8_t *src = A.arena + A.offsets[item];
    const uint32_t dtx = (A.has_toc ? len > 0u : A.offsets[item] != 0u) ? HDR_DTX : 0u;  // a lost item of a packet: PLC/DTX
    int32_t status = len == 0u ? ITEM_LOST : ITEM_OK;
    int bandwidth = A.bandwidth;
    if (A.has_toc && len > 0u) {
        // what a host caller checks with query_packet_* (src/lib.rs:219-325) before decode_frame
        const uint32_t toc = __ldg(src), config = toc >> 3;
        if (config >= 12u) status = OPN_ERR_UNIMPLEMENTED;                                  // hybrid / CELT: not this launch
        else if ((toc & 0x3u) != 0u) status = OPN_ERR_UNIMPLEMENTED;                        // multi-frame: host path only
        else if ((config & 3u) > 1u) status = OPN_ERR_UNIMPLEMENTED;                        // 40 / 60 ms: several SILK frames
        else if ((int)((config & 3u) ? 20 : 10) != frame_ms) status = OPN_ERR_FRAME_SIZE_TOO_SMALL;
        else if (((toc & 0x4u) ? 2 : 1) != A.stream_channels) status = OPN_ERR_UNIMPLEMENTED;
        bandwidth = (int)(config >> 2);
        src += 1;
        len -= 1u;
    }
    if (status == ITEM_OK && len <= 1u) status = ITEM_LOST;  // decoder.rs:467
    A.status[stream] = status;
    if (status != ITEM_OK) {
        if (status == ITEM_LOST) A.hdr[stream] = make_uint4(dtx, 0u, 0u, 0u);
        return;
    }
    const int fs_khz = bandwidth == 0 ? 8 : bandwidth == 1 ? 12 : 16;
    const int nb_subfr = frame_ms / 5, order = fs_khz == 16 ? 16 : 10, nblk = (nb_subfr * 5 * fs_khz + 15) / 16;
    const int min_lag = 2 * fs_khz, max_lag = 18 * fs_khz;
    const PvqTable T{g_tab.pvq_u_data, g_tab.pvq_u_row};
    LaneDec d;
    d.init(src, len);
    // lbrr: a redundant copy of the PREVIOUS frame (same syntax) comes before the regular frame -- the in-band FEC behind
    // Decoder::decode(.., decode_fec = true) (decoder.rs:343-386; LostFlag::DecodeFec, silk/decoder.rs:6-14).  Decoding the regular frame
    // walks through the copy first (its values are overwritten by the second pass); decoding the copy stops after it.
    const uint32_t lbrr = d.bit_logp(1u);
    if (A.fec && !lbrr) {  // FEC asked of a packet that has none: conceal
        A.status[stream] = ITEM_LOST;
        A.hdr[stream] = make_uint4(HDR_DTX, 0u, 0u, 0u);
        if (A.side) A.side[stream].lbrr = 0;
        return;
    }
    const int npass = (!A.fec && lbrr) ? 2 : 1;
    for (int pass = 0; pass < npass; pass++)
    for (int c = 0; c < A.stream_channels; c++) {
        SilkRec *r = A.rec + (size_t)stream * 2 + c;
        opn_silk_chan_side *sd = A.side ? &A.side[stream].ch[c] : nullptr;
        const uint32_t type = d.icdf(s_icdf, 8u);
        uint32_t g = d.uint_small(64u);
        r->type = (uint8_t)type;
        r->gidx[0] = (uint8_t)g;
        if (sd) {
            sd->type = (int32_t)type;
            sd->gidx[0] = (int32_t)g;
        }
        for (int f = 1; f < 4; f++) {
            if (f < nb_subfr) {
                const int v = (int)g + (int)d.icdf(s_icdf + 4, 8u) - 4;
                g = (uint32_t)max(0, min(63, v));
            }
            r->gidx[f] = (uint8_t)g;
            if (sd) sd->gidx[f] = f < nb_subfr ? (int32_t)g : 0;
        }
        for (int k = 0; k < 16; k++) {
            const uint32_t v = k < order ? d.bits(k < 2 ? 5u : 4u) : 0u;
            r->rc[k] = (uint8_t)v;
            if (sd) sd->rc_idx[k] = (int32_t)v;
        }
        if (type == 2u) {
            const int lag0 = min_lag + (int)d.uint_any((uint32_t)(max_lag - min_lag + 1));
            for (int f = 0; f < 4; f++) {
                int l = 0;
                if (f < nb_subfr) l = max(min_lag, min(max_lag, lag0 + (int)d.icdf(s_icdf + 16, 8u) - 1));
                r->lag[f] = (uint16_t)l;
                if (sd) sd->lag[f] = l;
            }
            for (int f = 0; f < 4; f++) {
                const uint32_t v = f < nb_subfr ? d.icdf(s_icdf + 20, 8u) : 0u;
                r->ltp[f] = (uint8_t)v;
                if (sd) sd->ltp_idx[f] = (int32_t)v;
            }
        } else {
            for (int f = 0; f < 4; f++) {
                r->lag[f] = 0;
                r->ltp[f] = 0;
                if (sd) sd->lag[f] = sd->ltp_idx[f] = 0;
            }
        }
        const uint32_t seed = d.bits(2u);
        r->seed = (uint8_t)seed;
        if (sd) sd->seed = (int32_t)seed;
        const uint8_t *pt = s_icdf + 28 + (type != 0u ? 9 : 0);
        for (int b = 0; b < 20; b++) {
            uint32_t k = 0u, idx = 0u;
            if (b < nblk) {
                k = d.icdf(pt, 8u);
                if (k) idx = d.uint_any(T.v(16u, k));
            }
            r->pulses[b] = (uint8_t)k;
            r->index[b] = idx;
            if (sd) {
                sd->pulses[b] = (int32_t)k;
                sd->index[b] = idx;
            }
        }
    }
    const uint32_t tf = d.tell_frac();
    if (A.side) {
        A.side[stream].final_rng = d.rng;
        A.side[stream].tell_frac = tf;
        A.side[stream].lbrr = (int32_t)lbrr;
    }
    A.hdr[stream] = make_uint4((uint32_t)fs_khz, d.rng, tf, 0u);
}

// ------------------------------------------------------------------------------------------------- frame kernel
// t / up and t % up for up in {3, 4, 6} without a runtime division
__device__ __forceinline__ void silk_divmod(int t, int up, int &q, int &r)
{
    q = up == 3 ? t / 3 : up == 4 ? t >> 2 : t / 6;
    r = t - q * up;
}

constexpr int SILK_LEAD = 8;  // rows before sample 0: the resampler's history (x[-7..-1]) sits in front of the frame
constexpr size_t silk_frame_smem() { return (size_t)((SILK_MAX_FRAME + SILK_LEAD) * SILK_RS + 16 * SILK_RS + 16 * SILK_RS + 4 * SILK_RS) * 4 + 8 * SILK_ROWS; }

// Polyphase interpolation by UP of one item's NCH channels (x[i * SILK_RS + c], floats, history at i = -7..-1) and the PCM
// stores: y[UP i + p] = sum_j h[p][j] x[i - j] summed in tap order, then the merge of decoder.rs:722-729 onto a zero CELT part.
// One lane per INPUT sample: its eight-sample window is loaded once for the UP outputs it produces.
template <int UP, int NCH, int C>
__device__ __forceinline__ void silk_resample_store(const float *x, int L, uint32_t lane, float *ring, uint32_t pos, float *dense, float gain,
                                                    const float *rs1 /* C == 2 from one channel: history of output channel 1 */)
{
    constexpr int T = UP == 6 ? 0 : UP == 4 ? 1 : 2;
    for (int i0 = 0; i0 < L; i0 += 32) {
        const int i = i0 + (int)lane;
        if (i >= L) continue;
        float xv[2][8];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            xv[0][j] = x[(i - j) * SILK_RS];
            xv[1][j] = NCH == 2 ? x[(i - j) * SILK_RS + 1] : xv[0][j];
            if (NCH == 1 && C == 2 && rs1 && i - j < 0) xv[1][j] = rs1[-1 - (i - j)];
        }
#pragma unroll
        for (int p = 0; p < UP; p++) {
            float o[2];
#pragma unroll
            for (int c = 0; c < 2; c++) {
                if (c == 1 && C == 1) continue;
                float acc = c_silk_up[T][8 * p] * xv[c][0];
#pragma unroll
                for (int j = 1; j < 8; j++) acc = acc + c_silk_up[T][8 * p + j] * xv[c][j];
                o[c] = 0.0f + (1.0f / 32768.0f) * acc;
            }
            const int t = UP * i + p;
            uint32_t rp = pos + (uint32_t)t;
            if (rp >= (uint32_t)RING_SAMPLES) rp -= RING_SAMPLES;
            if (C == 2) {
                *reinterpret_cast<float2 *>(ring + (size_t)rp * 2) = make_float2(o[0], o[1]);
                if (dense) *reinterpret_cast<float2 *>(dense + (size_t)t * 2) = make_float2(o[0] * gain, o[1] * gain);
            } else {
                ring[rp] = o[0];
                if (dense) dense[t] = o[0] * gain;
            }
        }
    }
}

// MIX: a mixed-mode step's launch (A.plan); a separate instance, so that the uniform and host-path launches keep their registers
template <int CS, int C, bool MIX = false> __global__ void __launch_bounds__(32 * SILK_WARPS, 4) k_silk_frame(SilkArgs A)
{
    extern __shared__ __align__(16) uint8_t silk_smem[];
    // [SILK_LEAD + SILK_MAX_FRAME][SILK_RS]: excitation, then internal-rate samples (as floats); s_res points at sample 0
    int32_t *s_res = reinterpret_cast<int32_t *>(silk_smem) + SILK_LEAD * SILK_RS;
    int32_t *s_a = s_res + SILK_MAX_FRAME * SILK_RS;          // [16][SILK_RS] A_Q12
    int32_t *s_lpc = s_a + 16 * SILK_RS;                      // [16][SILK_RS] sLPC_Q14 window, [15] newest
    int32_t *s_gain = s_lpc + 16 * SILK_RS;                   // [4][SILK_RS]
    // per row: [0] fs_khz (0 = the row does nothing), [1] lost, [2] state was reset, [3] silent (lost before any frame)
    uint8_t *s_meta = reinterpret_cast<uint8_t *>(s_gain + 4 * SILK_RS);  // [SILK_ROWS][8]
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const long long clk0 = A.phase_clk ? clock64() : 0;
    constexpr uint32_t ITEMS = SILK_ROWS / CS;
    uint32_t item0 = A.item0 + blockIdx.x * ITEMS, item_end = A.item_end;
    int frame_ms = A.frame_ms;
    if constexpr (MIX) {  // mixed-mode step: the CTA's bucket (20 ms first); the grid is an upper bound, CTAs past the last bucket retire
        const MixPlan &P = *A.plan;
        const int g = A.group;
        const uint32_t c = blockIdx.x;
        if (c >= P.scta0[g][2]) return;
        const int j = c >= P.scta0[g][1], k = 1 - j;
        frame_ms = k ? 20 : 10;
        item0 = P.sstart[g][k] + (c - P.scta0[g][j]) * ITEMS;
        item_end = P.sstart[g][k] + P.scount[g][k];
    }
    const int nb_subfr = frame_ms / 5;

    // ---- phase A0: one thread per row: what the row is (frame parameters, where its state lives)
    __shared__ uint32_t s_chs[SILK_ROWS];  // stream * 2 + coded channel
    if (threadIdx.x < (uint32_t)SILK_ROWS) {
        const uint32_t row = threadIdx.x, item = item0 + row / CS, c = row % CS;
        uint8_t *meta = s_meta + row * 8;
        meta[0] = 0;
        meta[3] = 3;  // no item
        if (item < item_end) {
            const uint32_t stream = A.stream_idx ? A.stream_idx[item] : item;
            const int32_t status = A.status[stream];
            const uint32_t fs_prev = A.st.fs[2 * stream], cs_prev = A.st.fs[2 * stream + 1];
            const bool lost = status == ITEM_LOST;
            const uint32_t fs_khz = lost ? fs_prev : A.hdr[stream].x;
            const bool silent = status < 0 || (lost && (fs_prev == 0u || c >= cs_prev));  // errors and losses before any frame: no work
            meta[0] = silent ? 0 : (uint8_t)fs_khz;
            meta[1] = lost;
            meta[2] = !lost && fs_khz != fs_prev;  // first frame or a new internal rate: every filter starts from rest
            meta[3] = status < 0 ? 2 : (lost && fs_prev == 0u) ? 1 : 0;
            s_chs[row] = stream * 2u + c;
        }
    }
    __syncthreads();

    // ---- phase A1: excitation, one LANE per 16-sample shell block: task (row, b), the rows of a warp's 32 tasks all different
    // (conflict-free stores into the transposed rows); the codeword walk is the product's cwrsi_events (pvc.rs:182-284)
    for (uint32_t t = threadIdx.x; t < (uint32_t)SILK_ROWS * 20u; t += 32u * SILK_WARPS) {
        const uint32_t row = t & 31u, blk = t >> 5;
        const int fs_khz = s_meta[row * 8];
        const int L = nb_subfr * 5 * fs_khz;
        if (16 * (int)blk >= L) continue;  // also rows that do nothing (fs_khz == 0)
        int32_t *res = s_res + row;
        if (s_meta[row * 8 + 1]) {  // lost: no excitation
#pragma unroll
            for (int j = 0; j < 16; j++)
                if (16 * (int)blk + j < L) res[(16 * blk + j) * SILK_RS] = 0;
            continue;
        }
        const SilkRec *r = A.rec + s_chs[row];
        const uint32_t type = r->type, seed = r->seed, k = r->pulses[blk], idx = r->index[blk];
        uint64_t lo = 0ull, hi = 0ull;  // y[j] as a signed byte, j < 8 in lo, the rest in hi
        if (k) {
            cwrsi_events(g_tab.pvq_u_data, g_tab.pvq_cw_data, g_tab.pvq_u_row, g_tab.pvq_ev_nmax, 16u, k, idx, [&](uint32_t pos, int32_t val) {
                const uint64_t v = (uint64_t)(uint8_t)(int8_t)val << (8u * (pos & 7u));
                if (pos < 8u) lo |= v;
                else hi |= v;
            });
        }
        const int32_t offs = type == 1u ? (100 << 4) : (32 << 4);
        uint32_t rr = (seed + 1u) * 2654435761u + blk * 2246822519u;
#pragma unroll
        for (int j = 0; j < 16; j++) {
            const int32_t y = (int32_t)(int8_t)(uint8_t)((j < 8 ? lo : hi) >> (8 * (j & 7)));
            int32_t e = y * 16384;
            e += y > 0 ? -(80 << 4) : y < 0 ? (80 << 4) : 0;
            e += offs;
            rr = rr * 196314165u + 907633515u;
            if (rr & 0x80000000u) e = -e;
            rr += (uint32_t)y;
            const int i = 16 * (int)blk + j;
            if (i < L) res[i * SILK_RS] = e;
        }
    }
    __syncthreads();

    // ---- phase A2: one warp per row: long-term prediction, filter coefficients, state
    for (uint32_t row = warp; row < (uint32_t)SILK_ROWS; row += SILK_WARPS) {
        const int fs_khz = s_meta[row * 8];
        if (fs_khz == 0) continue;
        const bool lost = s_meta[row * 8 + 1], reset = s_meta[row * 8 + 2];
        const int order = fs_khz == 16 ? 16 : 10, sub = 5 * fs_khz, L = nb_subfr * sub;
        const size_t chs = s_chs[row];
        int32_t *hist = A.st.hist + chs * SILK_HIST;
        int32_t *res = s_res + row;  // sample i at res[i * SILK_RS]
        // previous window of the LPC recursion, coefficient and gain state
        if (lane < 16u) s_lpc[lane * SILK_RS + row] = reset ? 0 : A.st.slpc[chs * 16 + lane];
        if (lost) {
            if (lane < 16u) s_a[lane * SILK_RS + row] = (int32_t)A.st.a_q12[chs * 16 + lane] << 16;
            if (lane < 4u) s_gain[lane * SILK_RS + row] = A.st.gain[chs];
        } else {
            const SilkRec *r = A.rec + chs;
            const uint32_t type = r->type;
            __syncwarp();
            if (type == 2u) {
                // long-term prediction: pres[i] = exc[i] + ((2 + sum_k smulwb(pres[i - lag + 2 - k], B[k])) << 2); the newest tap lies
                // lag - 2 samples back, so spans of min(32, lag - 2) samples are independent
                for (int f = 0; f < nb_subfr; f++) {
                    const int lag = (int)r->lag[f];
                    const int16_t *B = g_silk.ltp_q14 + 5 * r->ltp[f];
                    const int32_t b0 = (int32_t)B[0] << 16, b1 = (int32_t)B[1] << 16, b2 = (int32_t)B[2] << 16, b3 = (int32_t)B[3] << 16, b4 = (int32_t)B[4] << 16;
                    const int span = min(32, lag - 2), end = (f + 1) * sub;
                    for (int i0 = f * sub; i0 < end; i0 += span) {
                        const int i = i0 + (int)lane;
                        if ((int)lane < span && i < end) {
                            const int top = i - lag + 2;  // index of tap 0; taps run downwards
                            int32_t pred = 2;
                            const int32_t bk[5] = {b0, b1, b2, b3, b4};
#pragma unroll
                            for (int k = 0; k < 5; k++) {
                                const int q = top - k;
                                const int32_t v = q >= 0 ? res[q * SILK_RS] : (reset ? 0 : hist[SILK_HIST + q]);
                                pred += silk_smulwb_sh(v, bk[k]);
                            }
                            res[i * SILK_RS] += (int32_t)((uint32_t)pred << 2);
                        }
                        __syncwarp();
                    }
                }
            }
            // reflection coefficients -> A_Q12: lane n holds c[n] (Q24); step k adds rc_k * c[k-1-n] to every n < k at once
            {
                int32_t cn = 0;
                for (int k = 0; k < order; k++) {
                    const int32_t idx = (int32_t)r->rc[k];
                    const int32_t rc = k < 2 ? (idx - 16) * 3600 : (idx - 8) * (k < 6 ? 4800 : 2400);
                    const int32_t partner = __shfl_sync(0xffffffffu, cn, (k - 1 - (int)lane) & 31);
                    if ((int)lane < k) cn += silk_smulww(partner, rc);
                    else if ((int)lane == k) cn = rc * 256;
                }
                if (lane < 16u) {
                    const int32_t x = (int)lane < order ? (int32_t)(0u - (uint32_t)cn) : 0;
                    const int32_t aq = silk_sat16(((x >> 11) + 1) >> 1);
                    s_a[lane * SILK_RS + row] = aq << 16;  // pre-shifted: smulwb becomes one multiply-high in phase B
                    A.st.a_q12[chs * 16 + lane] = (int16_t)aq;
                }
                if (lane < 4u) s_gain[lane * SILK_RS + row] = g_silk.gain_q10[r->gidx[min((int)lane, nb_subfr - 1)]];
            }
        }
        __syncwarp();
        if (A.exc_out)
            for (int i = (int)lane; i < L; i += 32) A.exc_out[chs * SILK_MAX_FRAME + i] = res[i * SILK_RS];
        // excitation history: the last SILK_HIST samples of (old history ++ this frame)
        {
            int32_t keep[8];  // old samples that stay (L < SILK_HIST): read before anything is overwritten
            const int stay = SILK_HIST - L;
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int j = (int)lane + 32 * u;
                keep[u] = (j < stay && !reset) ? hist[j + L] : 0;
            }
            __syncwarp();
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int j = (int)lane + 32 * u;
                if (j < stay) hist[j] = keep[u];
            }
            for (int j = max(stay, 0) + (int)lane; j < SILK_HIST; j += 32) hist[j] = res[(j - stay) * SILK_RS];
        }
        if (reset && CS == 1) {  // a mono frame at a new rate: the second channel's filters start from rest as well
            for (int j = (int)lane; j < SILK_HIST; j += 32) hist[SILK_HIST + j] = 0;
            if (lane < 16u) {
                A.st.slpc[(chs + 1) * 16 + lane] = 0;
                A.st.a_q12[(chs + 1) * 16 + lane] = 0;
            }
            if (lane == 0) A.st.gain[chs + 1] = 0;
        }
    }
    __syncthreads();

    // ---- phase B: warp 0, one lane per row (the hardware spreads the warp slots of co-resident CTAs over the four schedulers: picking
    // the warp by hardware slot measured the same, picking it by blockIdx measured 5-25 % slower).  SURVEY.md appendix B:
    //   pred_Q10 = order/2 + sum_k smulwb(sLPC_Q14[i-1-k], A_Q12[k]); sLPC_Q14[i] = sat32(res_Q14[i] + (pred_Q10 << 4));
    //   out[i] = sat16(rshift_round(smulww(sLPC_Q14[i], gain_Q10), 8))
    const long long clk1 = A.phase_clk ? clock64() : 0;
    if (warp == 0) {
        const uint32_t row = lane;
        const int fs_khz = s_meta[row * 8];
        const int sub = 5 * fs_khz, L = nb_subfr * sub;
        int Lmax = L;
#pragma unroll
        for (int o = 16; o; o >>= 1) Lmax = max(Lmax, __shfl_xor_sync(0xffffffffu, Lmax, o));
        // a: A_Q12 << 16 (smulwb is then one multiply-high).  s[0..15]: the window sLPC[i0-16 .. i0-1], oldest first; four samples
        // per iteration land in s[16..19], then the window slides by four.  (Sixteen samples per iteration with the window as a
        // ring needed no moves but made the loop 11 KB of code: the four co-resident CTAs' serial warps then ran 25 % slower on
        // four schedulers than on one -- instruction fetch, not arithmetic, was the limit.)
        int32_t a[16], s[20];
#pragma unroll
        for (int k = 0; k < 16; k++) {
            a[k] = s_a[k * SILK_RS + row];
            s[k] = s_lpc[k * SILK_RS + row];
        }
        const int32_t rnd = fs_khz == 16 ? 8 : 5;
        const int32_t g0 = s_gain[row], g1 = s_gain[SILK_RS + row], g2 = s_gain[2 * SILK_RS + row], g3 = s_gain[3 * SILK_RS + row];
        const int e1 = sub, e2 = 2 * sub, e3 = 3 * sub;
        int32_t *rp = s_res + row;
        // one sample of the recursion; the window slides after every four
        auto lpc4 = [&](int i0, int32_t g, bool act) {
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int i = i0 + u;
                // four partial sums; the tap on the previous sample comes last, so that only one product and one sum wait for it
                int32_t p0 = rnd, p1 = 0, p2 = 0, p3 = 0;
#pragma unroll
                for (int k = 15; k >= 3; k -= 4) {
                    p0 += silk_smulwb_sh(s[15 + u - k], a[k]);
                    p1 += silk_smulwb_sh(s[16 + u - k], a[k - 1]);
                    p2 += silk_smulwb_sh(s[17 + u - k], a[k - 2]);
                    p3 += silk_smulwb_sh(s[18 + u - k], a[k - 3]);
                }
                const int32_t pred = (p0 + p1) + (p2 + p3);
                const int64_t v = (int64_t)pred * 16 + (int64_t)rp[i * SILK_RS];          // one IMAD.WIDE
                const int32_t lo = (int32_t)v, hi = (int32_t)(v >> 32);
                const int32_t v32 = hi == (lo >> 31) ? lo : (0x7fffffff ^ (hi >> 31));      // sat32
                s[16 + u] = v32;
                const int64_t wg = (int64_t)v32 * (int64_t)g;                               // smulww: one IMAD.WIDE and a funnel shift
                const int32_t w = (int32_t)__funnelshift_r((uint32_t)wg, (uint32_t)(wg >> 32), 16);
                const int32_t o = __float_as_int((float)silk_sat16(((w >> 7) + 1) >> 1));  // exact: |x| <= 2^15
                if (act) rp[i * SILK_RS] = o;
            }
        };
        if (__all_sync(0xffffffffu, L == Lmax)) {  // every row of the CTA has the same frame length (the usual case): no predication
#pragma unroll 1
            for (int i0 = 0; i0 < L; i0 += 4) {
                lpc4(i0, i0 < e1 ? g0 : i0 < e2 ? g1 : i0 < e3 ? g2 : g3, true);  // subframes are multiples of 8 samples
#pragma unroll
                for (int k = 0; k < 16; k++) s[k] = s[k + 4];
            }
        } else {  // mixed bandwidths in one CTA: rows of a shorter frame idle through the tail (L is a multiple of 8)
#pragma unroll 1
            for (int i0 = 0; i0 < Lmax; i0 += 4) {
                const bool act = i0 < L;
                lpc4(i0, i0 < e1 ? g0 : i0 < e2 ? g1 : i0 < e3 ? g2 : g3, act);
#pragma unroll
                for (int k = 0; k < 16; k++) s[k] = act ? s[k + 4] : s[k];
            }
        }
        if (fs_khz) {
            const uint32_t item = item0 + row / CS, c = row % CS;
            const uint32_t stream = A.stream_idx ? A.stream_idx[item] : item;
            const size_t chs = (size_t)stream * 2 + c;
#pragma unroll
            for (int k = 0; k < 16; k++) A.st.slpc[chs * 16 + k] = s[k];
            A.st.gain[chs] = nb_subfr == 4 ? g3 : g1;
        }
    }
    __syncthreads();

    const long long clk2 = A.phase_clk ? clock64() : 0;
    // ---- phase C: one warp per item
    for (uint32_t it = warp; it < ITEMS; it += SILK_WARPS) {
        const uint32_t item = item0 + it;
        if (item >= item_end) continue;
        const uint32_t row0 = it * CS;
        const uint32_t stream = A.stream_idx ? A.stream_idx[item] : item;
        const int n48 = frame_ms * 48;
        const uint32_t flag = s_meta[row0 * 8 + 3];
        const uint32_t dense_off = (A.dense && A.dense_off) ? A.dense_off[item] : 0u;
        float *dense = A.dense ? A.dense + (size_t)stream * A.dense_stride + dense_off : nullptr;
        if (flag == 2u) {  // rejected packet: state untouched, the error is the result
            if (lane == 0 && A.result) A.result[stream] = A.status[stream];
            continue;
        }
        if (flag == 1u) {  // lost before anything was decoded: silence, state untouched
            if (dense)
                for (int t = (int)lane; t < n48 * C; t += 32) dense[t] = 0.0f;
            if (lane == 0) {
                if (A.result) A.result[stream] = n48;
                if (A.final_range) A.final_range[stream] = 0u;
                // a PLC/DTX packet still sets the stream's codec and size (the mode record of mixed-mode steps)
                if (A.pf && (A.hdr[stream].x & HDR_DTX)) A.pf[stream].lm1 = (nb_subfr == 4 ? 4 : 3) | PF_SILK;
            }
            continue;
        }
        const int fs_khz = s_meta[row0 * 8];
        const bool lost = s_meta[row0 * 8 + 1], reset = s_meta[row0 * 8 + 2];
        const int L = nb_subfr * 5 * fs_khz, up = 48 / fs_khz;
        const uint32_t pos = A.ring_pos[stream];
        float *ring = A.ring + (size_t)stream * RING_SAMPLES * C;
        float *rs = A.st.rs + (size_t)stream * 16;
        float *x = reinterpret_cast<float *>(s_res) + row0;  // sample i of coded channel c at x[i * SILK_RS + c]
        constexpr int NCH = (CS == 2 && C == 2) ? 2 : 1;      // channels that go through the interpolator
        // stream_channels -> channels (decoder.rs:332): mid/side -> left/right in place; a mono packet feeds both outputs; a mono
        // decoder takes the mid channel of a stereo packet
        if (NCH == 2) {
            for (int i = (int)lane; i < L; i += 32) {
                const float m = x[i * SILK_RS], sd = x[i * SILK_RS + 1];
                x[i * SILK_RS] = fminf(fmaxf(m + sd, -32768.0f), 32767.0f);  // sat16 of an exact integer sum
                x[i * SILK_RS + 1] = fminf(fmaxf(m - sd, -32768.0f), 32767.0f);
            }
        }
        if (lane < 7u) {  // resampler history in front of the frame: x[-1-j] = rs[c][j]
#pragma unroll
            for (int c = 0; c < NCH; c++) x[-(1 + (int)lane) * SILK_RS + c] = reset ? 0.0f : rs[c * 8 + lane];
        }
        float rs1[8];  // a mono packet in a stereo decoder: output channel 1 keeps its own history (it differs after a stereo packet)
        if (NCH == 1 && C == 2) {
#pragma unroll
            for (int j = 0; j < 8; j++) rs1[j] = (reset || j == 7) ? 0.0f : rs[8 + j];
        }
        __syncwarp();
        const float *r1 = (NCH == 1 && C == 2) ? rs1 : nullptr;
        if (up == 3) silk_resample_store<3, NCH, C>(x, L, lane, ring, pos, dense, A.gain, r1);
        else if (up == 4) silk_resample_store<4, NCH, C>(x, L, lane, ring, pos, dense, A.gain, r1);
        else silk_resample_store<6, NCH, C>(x, L, lane, ring, pos, dense, A.gain, r1);
        if (lane < 7u) {
#pragma unroll
            for (int c = 0; c < C; c++) rs[c * 8 + lane] = x[(L - 1 - (int)lane) * SILK_RS + (NCH == 2 ? c : 0)];
        }
        if (lane == 0) {
            uint32_t np = pos + (uint32_t)n48;
            if (np >= (uint32_t)RING_SAMPLES) np -= RING_SAMPLES;
            A.ring_pos[stream] = np;
            if (!lost) {
                A.st.fs[2 * stream] = (uint8_t)fs_khz;
                A.st.fs[2 * stream + 1] = (uint8_t)CS;
            }
            if (A.pf && (!lost || (A.hdr[stream].x & HDR_DTX))) A.pf[stream].lm1 = (nb_subfr == 4 ? 4 : 3) | PF_SILK;
            if (A.result) A.result[stream] = n48;
            if (A.final_range) A.final_range[stream] = lost ? 0u : A.hdr[stream].y;
            if (A.softclip_reset && !lost) *reinterpret_cast<float2 *>(A.softclip_reset + 2 * (size_t)stream) = make_float2(0.f, 0.f);
        }
        if (A.out16)
            for (int i = (int)lane; i < L; i += 32)
                for (int c = 0; c < C; c++) A.out16[((size_t)stream * 2 + c) * SILK_MAX_FRAME + i] = (int16_t)x[i * SILK_RS + (NCH == 2 ? c : 0)];
    }
    if (A.phase_clk) {  // measurement only (OPN_SILK_CLK=1): cycles per phase summed over the CTAs
        __syncthreads();
        if (threadIdx.x == 0) {
            const long long clk3 = clock64();
            atomicAdd(A.phase_clk + 0, (unsigned long long)(clk1 - clk0));
            atomicAdd(A.phase_clk + 1, (unsigned long long)(clk2 - clk1));
            atomicAdd(A.phase_clk + 2, (unsigned long long)(clk3 - clk2));
            atomicAdd(A.phase_clk + 3, 1ull);
        }
    }
}

}  // namespace opn
