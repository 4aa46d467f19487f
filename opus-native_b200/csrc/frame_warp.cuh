// frame_warp.cuh -- the frame kernel: one WARP turns one stream's decoded symbols into PCM.
//
//   codeword indices --w_expand--> coefficient rows (shared memory) --w_imdct--> out[0 .. nf+60) (same rows)
//   --w_comb_ring--> post-filtered frame (same rows) --> interleaved float4 PCM in the ring (+ dense rows)
//
// Nothing between the range decoder's 288 bytes of indices and the PCM leaves the SM: the coefficient rows are
// produced in the very shared-memory rows Mdct::backward transforms in place, and the pitch comb post-filter
// (comb_filter_inplace, src/celt/comb_filter/mod.rs:130-193, scalar kernel fallback.rs:32-53) runs on those rows
// before the only PCM store.  The post-filter's history -- the previous max(T0,T1)+2 output samples -- is the PCM ring
// itself: taps that fall before the frame are read from the ring through L1/L2 (one float2 = both channels of a
// sample), taps inside the frame from the rows.  Shared memory per stream: C rows of nf+60 floats and a small stash
// (8 KB for a stereo 20 ms frame), as for the IMDCT alone.
#pragma once
#include "imdct_warp.cuh"
#include "symbols.cuh"

namespace opn {

// ---- post-filter -------------------------------------------------------------------------------
// One sample of the C channels of a stream.  For stereo the two channels of a sample travel as a float2 and every sum
// of the filter is ONE packed add (p_add, imdct.cuh) for both; the products stay scalar (see p_add).
template <int C> struct WSmp;
template <> struct WSmp<1> {
    float a;
    __device__ __forceinline__ static WSmp ld(const float *p) { return WSmp{*p}; }  // interleaved layout (the PCM ring)
    __device__ __forceinline__ WSmp operator+(WSmp o) const { return WSmp{a + o.a}; }
    __device__ __forceinline__ WSmp scaled(float g) const { return WSmp{g * a}; }
};
template <> struct WSmp<2> {
    float a, b;
    __device__ __forceinline__ static WSmp ld(const float *p)
    {
        const float2 v = *reinterpret_cast<const float2 *>(p);
        return WSmp{v.x, v.y};
    }
    __device__ __forceinline__ WSmp operator+(WSmp o) const
    {
        const float2 r = p_add(make_float2(a, b), make_float2(o.a, o.b));
        return WSmp{r.x, r.y};
    }
    __device__ __forceinline__ WSmp scaled(float g) const { return WSmp{g * a, g * b}; }
};
// comb_filter_const_inplace term order (fallback.rs:46-51): y + g0*x2 + g1*(x1+x3) + g2*(x0+x4)
template <int C>
__device__ __forceinline__ WSmp<C> w_comb5(WSmp<C> y, WSmp<C> x0, WSmp<C> x1, WSmp<C> x2, WSmp<C> x3, WSmp<C> x4, float g0, float g1,
                                           float g2)
{
    return y + x2.scaled(g0) + (x1 + x3).scaled(g1) + (x0 + x4).scaled(g2);
}
// cross-fade accumulation order of comb_filter_inplace (mod.rs:166-177); a* = y[i-t0-2 .. i-t0+2],
// b* = y[i-t1-2 .. i-t1+2]
template <int C>
__device__ __forceinline__ WSmp<C> w_xfade(WSmp<C> y, const WSmp<C> *a, const WSmp<C> *b, bool has0, bool has1, float f, float g00,
                                           float g01, float g02, float g10, float g11, float g12)
{
    WSmp<C> v = y;
    if (has0) {
        v = v + a[2].scaled((1.0f - f) * g00);
        v = v + (a[3] + a[1]).scaled((1.0f - f) * g01);
        v = v + (a[4] + a[0]).scaled((1.0f - f) * g02);
    }
    if (has1) {
        v = v + b[2].scaled(f * g10);
        v = v + (b[3] + b[1]).scaled(f * g11);
        v = v + (b[4] + b[0]).scaled(f * g12);
    }
    return v;
}

// tap gains of the old and the new filter (comb_filter/mod.rs:45-55, 146-151)
struct CombGains {
    float g00, g01, g02, g10, g11, g12;
};
__device__ __forceinline__ CombGains w_comb_gains(float g0, float g1, int tap0, int tap1)
{
    CombGains k;
    k.g00 = g0 * g_tab.comb_gains[tap0 * 3];
    k.g01 = g0 * g_tab.comb_gains[tap0 * 3 + 1];
    k.g02 = g0 * g_tab.comb_gains[tap0 * 3 + 2];
    k.g10 = g1 * g_tab.comb_gains[tap1 * 3];
    k.g11 = g1 * g_tab.comb_gains[tap1 * 3 + 1];
    k.g12 = g1 * g_tab.comb_gains[tap1 * 3 + 2];
    return k;
}

// Where the samples of one stream live while its frame is filtered: sample i >= 0 of channel c is rows[c*CHF + i]
// (shared memory, planar), sample i < 0 (history) is ring[((pos + i) mod RING_SAMPLES)*C + c] (global memory, interleaved).
template <int C, int CHF> struct FrameView {
    using S = WSmp<C>;
    float *rows;
    const float *ring;
    int pos;  // ring position of sample 0
    __device__ __forceinline__ S ld_row(int i) const
    {
        S r;
        r.a = rows[i];
        if constexpr (C == 2) r.b = rows[CHF + i];
        return r;
    }
    __device__ __forceinline__ void st_row(int i, S v) const
    {
        rows[i] = v.a;
        if constexpr (C == 2) rows[CHF + i] = v.b;
    }
    __device__ __forceinline__ S ld_hist(int i) const
    {
        int j = pos + i;
        if (j < 0) j += RING_SAMPLES;
        return S::ld(ring + (size_t)j * C);
    }
    __device__ __forceinline__ S ld(int i) const { return i >= 0 ? ld_row(i) : ld_hist(i); }
};

// comb_filter_inplace (comb_filter/mod.rs:130-193) on the frame in V.  The filter is recursive, y[i] depends on the
// already filtered y[i-T-2 .. i-T+2]; samples whose taps all lie before the span being processed are independent and are
// filtered in parallel, one per lane, consecutive lanes on consecutive samples (conflict-free in shared memory,
// coalesced in the ring); the frame is swept in spans no longer than T-2.  A tap set whose gain is exactly zero
// contributes +-0 to every sum and is skipped.
template <int C, int CHF, bool TS = false>
__device__ __forceinline__ void w_comb_ring(const FrameView<C, CHF> &V, int t0, int t1, int n, float g0, float g1, int tap0, int tap1,
                                            int overlap, int lane, const float *win_sq, const CombGains &kg)
{
    using S = WSmp<C>;
    if (g0 == 0.0f && g1 == 0.0f) return;
    t0 = max(t0, 15);
    t1 = max(t1, 15);
    const float g00 = kg.g00, g01 = kg.g01, g02 = kg.g02, g10 = kg.g10, g11 = kg.g11, g12 = kg.g12;
    if (fabsf(g0 - g1) < 1.1920929e-7f && t0 == t1 && tap0 == tap1) overlap = 0;
    const bool has0 = g0 != 0.0f, has1 = g1 != 0.0f;

    // ---- cross-fade part (mod.rs:162-179): samples [0, overlap), spans of min(T)-2 (at most 32) samples
    if (overlap > 0) {
        const int tmin = min(has0 ? t0 : 1 << 20, has1 ? t1 : 1 << 20);
        const int W = min(tmin - 2, 32);
        for (int base = 0; base < overlap; base += W) {
            const int i = base + lane;
            if (lane < W && i < overlap) {
                const float f = tab_ld<TS>(win_sq + i);
                S a[5], b[5];
#pragma unroll
                for (int k = 0; k < 5; k++) {
                    a[k] = has0 ? V.ld(i - t0 - 2 + k) : S{};
                    b[k] = has1 ? V.ld(i - t1 - 2 + k) : S{};
                }
                V.st_row(i, w_xfade<C>(V.ld_row(i), a, b, has0, has1, f, g00, g01, g02, g10, g11, g12));
            }
            __syncwarp();
        }
    }
    if (!has1) return;

    // ---- constant part (fallback.rs:32-53): samples [overlap, n)
    // (1) [overlap, hend): every tap is history -> no recursion, 128 samples per step straight from the ring
    int at = overlap;
    {
        const int hend = max(at, min(n, t1 - 2));
        for (int base = at; base < hend; base += 128) {
#pragma unroll
            for (int e = 0; e < 4; e++) {
                const int i = base + lane + 32 * e;
                if (i < hend) {
                    int j = V.pos + i - t1 - 2;  // ring index of the lowest tap, y[i-T-2]
                    if (j < 0) j += RING_SAMPLES;
                    if (j + 4 < RING_SAMPLES) {  // the five taps are contiguous in the ring (all but <= 4 samples per frame)
                        const float *hp = V.ring + (size_t)j * C;
                        V.st_row(i, w_comb5<C>(V.ld_row(i), S::ld(hp + 4 * C), S::ld(hp + 3 * C), S::ld(hp + 2 * C), S::ld(hp + C), S::ld(hp), g10, g11, g12));
                    } else {
                        const int p = i - t1;
                        V.st_row(i, w_comb5<C>(V.ld_row(i), V.ld_hist(p + 2), V.ld_hist(p + 1), V.ld_hist(p), V.ld_hist(p - 1), V.ld_hist(p - 2),
                                               g10, g11, g12));
                    }
                }
            }
        }
        at = hend;
        __syncwarp();
    }
    // (2) recursive remainder [at, n): spans of min(T1-2, 128) samples; inside a span every tap lies before the span.
    //     Only the first span can still reach below the frame start.
    const int W2 = min(t1 - 2, 128);
    const int rounds = (W2 + 31) >> 5;
    for (int base = at; base < n; base += W2) {
        const bool mixed = base - t1 - 2 < 0;
        for (int e = 0; e < rounds; e++) {
            const int l = lane + 32 * e, i = base + l;
            if (l < W2 && i < n) {
                const int p = i - t1;
                if (mixed)
                    V.st_row(i, w_comb5<C>(V.ld_row(i), V.ld(p + 2), V.ld(p + 1), V.ld(p), V.ld(p - 1), V.ld(p - 2), g10, g11, g12));
                else
                    V.st_row(i, w_comb5<C>(V.ld_row(i), V.ld_row(p + 2), V.ld_row(p + 1), V.ld_row(p), V.ld_row(p - 1), V.ld_row(p - 2), g10,
                                           g11, g12));
            }
        }
        __syncwarp();
    }
}

__device__ __forceinline__ void prefetch_l1(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ---------------------------------------------------------------------------------------------
// The frame kernel: one warp = one stream (item), FRAME_WARPS warps per CTA.  The warps of a CTA are independent (all
// hand-offs inside a stream are __syncwarp); what they share is one copy of the read-only tables (trig pairs, twiddles,
// window, the schedule's slice of the PVQ tables, part entries: FBlobHdr), staged in shared memory by ONE TMA bulk copy
// per CTA that is in flight while the warps load their streams' state and clear their rows.
// Shared memory: [mbarrier 16 B | table blob | FRAME_WARPS x (C rows of nf+60 floats + 16 B)].
#ifndef OPN_FRAME_WARPS
#define OPN_FRAME_WARPS 5
#endif
#ifndef OPN_FRAME_CTAS
#define OPN_FRAME_CTAS 4
#endif
constexpr int FRAME_WARPS = OPN_FRAME_WARPS, FRAME_CTAS = OPN_FRAME_CTAS;
#ifndef OPN_STORE_UNROLL
#define OPN_STORE_UNROLL 3  // 15 (the whole loop) measured 1-2 % slower per step: the kernel is sensitive to its code size
#endif
constexpr int STORE_UNROLL = OPN_STORE_UNROLL;  // iterations of the PCM store loop in flight
// per warp: the rows, 16 bytes of padding (the layout the kernel was tuned with) and a 48-byte stash (frame header, previous
// post-filter parameters, ring position: read once in the prologue, used again after the transform)
__host__ __device__ constexpr size_t frame_warp_bytes(int lm, int channels) { return (size_t)channels * w_ch_floats(lm) * 4 + 16 + 48; }
__host__ __device__ constexpr size_t frame_smem_bytes(int lm, int channels, size_t blob_bytes)
{
    return 16 + blob_bytes + (size_t)FRAME_WARPS * frame_warp_bytes(lm, channels);
}

// MODE: where the coefficient rows come from.  FRAME_SYNTH1: expanded from the codeword indices of the static SYNTH-CELT/1
// schedule; FRAME_SYNTH2: expanded from the per-frame part list of SYNTH-CELT/2.
enum { FRAME_SYNTH1 = 1, FRAME_SYNTH2 = 2 };
// One CTA of the frame kernel: its FRAME_WARPS warps take the items first_item .. first_item + FRAME_WARPS - 1 (< item_end).
// CS: channels of the PACKETS (the crate's stream_channels, decoder.rs:332,376,395), C: channels of the decoder.  They
// differ when a mono packet reaches a stereo decoder or the reverse; the frame is then expanded with the packet's layout
// into max(C, CS) rows and mapped onto the decoder's channels before the transform, as libopus' celt_synthesis does:
// mono -> stereo copies the spectrum (each output channel keeps its own overlap and post-filter history), stereo ->
// mono averages the two spectra, 0.5 * (l + r).
template <int LM, int C, int MODE, int CS = C>
__device__ __forceinline__ void frame_cta(const FrameArgs &A, uint32_t first_item, uint32_t item_end)
{
    constexpr int R = C > CS ? C : CS;  // rows of shared memory per stream
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr int NF = 120 << LM;
    constexpr int CHF = w_ch_floats(LM);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t *tbar = reinterpret_cast<uint64_t *>(smem);
    const uint8_t *blob = smem + 16;
    const FBlobHdr H = g_tab.fblob_hdr[LM][CS - 1];  // the schedule's tables are the packet layout's; the transform's are the same in both
    float *o = reinterpret_cast<float *>(smem + 16 + H.total + (size_t)warp * frame_warp_bytes(LM, R));
    uint4 *stash = reinterpret_cast<uint4 *>(o + R * CHF + 4);  // [0] frame header, [1] previous PfState, [2].x ring position

    if (threadIdx.x == 0) {
        mbar_init(tbar, 1);
        mbar_expect_tx(tbar, H.total);
        bulk_g2s(smem + 16, g_fblob[LM][CS - 1], H.total, tbar);
    }
    const uint32_t item = first_item + warp;
    const bool in_range = item < item_end;
    const uint32_t stream = in_range ? (A.stream_idx ? A.stream_idx[item] : item) : 0u;
    // What the transform needs is loaded now; the rest of the post-filter state is read after the transform, so that it
    // does not occupy registers across it (its cache lines are already here by then).
    const int32_t status = in_range ? A.status[stream] : -1;
    // Lanes 0-2 fetch the frame header, the previous post-filter parameters and the ring position (one round trip through
    // L2, together with everything else the prologue asks for) and park them in shared memory for the post-filter.
    {
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (in_range) {
            if (lane == 0) v = A.hdr[stream];
            else if (lane == 1) v = *reinterpret_cast<const uint4 *>(A.pf + stream);
            else if (lane == 2) v.x = A.ring_pos[stream];
        }
        if (lane < 3) stash[lane] = v;
    }
    __syncwarp();
    const uint32_t hdr_x = stash[0].x;
    // SYNTH-CELT/1: the stream's codeword indices, three coalesced words per lane, requested with the rest of the prologue;
    // a lane later picks its parts' indices out of them with shuffles (the dealing table is in the blob, still in flight)
    [[maybe_unused]] uint32_t ix0 = 0u, ix1 = 0u, ix2 = 0u;
    if constexpr (MODE == FRAME_SYNTH1) {
        if (in_range) {
            const uint32_t *ip = A.idx + (size_t)stream * SYNTH_MAX_ENTRIES;
            ix0 = __ldg(ip + lane);
            ix1 = __ldg(ip + 32 + lane);
            if (lane < SYNTH_MAX_ENTRIES - 64) ix2 = __ldg(ip + 64 + lane);
        }
    }
    float *carry_g = A.carry + (size_t)stream * C * 60;
    float4 carry = make_float4(0.f, 0.f, 0.f, 0.f);
    if (in_range && lane < 15 * C) carry = *reinterpret_cast<const float4 *>(carry_g + 4 * lane);  // [C][60] = 15 float4 per channel
    float *ring = A.ring + (size_t)stream * RING_SAMPLES * C;
    if (in_range && status >= 0 && A.postfilter) {
        // The post-filter will read the last max(T_old, T_new)+2 samples before this frame from the ring: ask for those
        // lines now (HBM -> L2), a whole transform ahead of their use.
        const int t_old = (int)stash[1].x, t_new = (hdr_x >> 1) & 1u ? (int)(hdr_x >> 16) : 0;
        const int pos0 = (int)stash[2].x;
        const int need = max(max(t_old, t_new), 15) + 2;
        for (int l = lane * (128 / (4 * C)); l < need + 128 / (4 * C); l += 32 * (128 / (4 * C))) {  // one 128-byte line per lane and round
            int j = pos0 - need + l;
            if (j >= pos0) j = pos0 - 1;
            if (j < 0) j += RING_SAMPLES;
            prefetch_l2(ring + (size_t)j * C);
        }
    }
    // the coefficient rows start out zero: w_expand only writes the pulses
#pragma unroll
    for (int c = 0; c < R; c++)
        for (int i = lane; i < NF / 4; i += 32) reinterpret_cast<float4 *>(o + c * CHF)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();  // the table barrier is initialised
    mbar_wait(tbar, 0);
    if (status < 0) {  // out of range, or a rejected packet: state untouched (decoder.rs:397)
        if (in_range && lane == 0 && A.result) A.result[stream] = status;
        return;
    }
    const float2 *t_long = reinterpret_cast<const float2 *>(blob + H.tp_long), *t_short = reinterpret_cast<const float2 *>(blob + H.tp_short);
    const float2 *t_tw = reinterpret_cast<const float2 *>(blob + H.tw);
    const float *t_win = reinterpret_cast<const float *>(blob + H.win), *t_winsq = reinterpret_cast<const float *>(blob + H.win_sq);
    const bool lost = status == ITEM_LOST;
    // a transient frame's coefficients go to block-major positions (w_imdct's BM), a long frame's stay where they are
    const int lmt = (LM > 0 && ((hdr_x >> 2) & 1u)) ? LM : 0;
    if constexpr (MODE == FRAME_SYNTH1) {
        if (!lost && !(hdr_x & 1u)) {  // not silence
            const ExpandTables T{reinterpret_cast<const uint32_t *>(blob + H.pvq_u), reinterpret_cast<const uint2 *>(blob + H.pvq_cw),
                                 reinterpret_cast<const uint16_t *>(blob + H.pvq_row), blob + H.pvq_nmax,
                                 reinterpret_cast<const SynthEntry *>(blob + H.ent), blob + H.slots, (int)H.n_slots};
            w_expand<CS>(T, LM, (uint32_t)lane, [&](uint32_t e) {  // every lane calls it: e = 0xFF for "no part"
                const int src = (int)(e & 31u);
                const uint32_t a = __shfl_sync(0xFFFFFFFFu, ix0, src), b2 = __shfl_sync(0xFFFFFFFFu, ix1, src), c2 = __shfl_sync(0xFFFFFFFFu, ix2, src);
                return e == 0xFFu ? 0u : e < 32u ? a : e < 64u ? b2 : c2;
            }, o, CHF, nullptr, lmt);
        }
        __syncwarp();
    } else if constexpr (MODE == FRAME_SYNTH2) {
        if (!lost && !(hdr_x & 1u)) {
            // part shapes are only known per frame: the walk uses the full PVQ tables in global memory (L1/L2 resident)
            const ExpandTables T{g_tab.pvq_u_data, g_tab.pvq_cw_data, g_tab.pvq_u_row, g_tab.pvq_ev_nmax, nullptr, nullptr, 0};
            w_expand2<CS>(T, LM, (uint32_t)lane, A.parts + (size_t)stream * CELT2_MAX_PARTS, stash[0].w, A.bande + (size_t)stream * 42, o, CHF, nullptr, lmt);
        }
        __syncwarp();
    }
    if constexpr (CS == 1 && C == 2) {  // mono packet, stereo decoder: both channels transform the same spectrum
        for (int i = lane; i < NF / 4; i += 32) reinterpret_cast<float4 *>(o + CHF)[i] = reinterpret_cast<const float4 *>(o)[i];
        __syncwarp();
    } else if constexpr (CS == 2 && C == 1) {  // stereo packet, mono decoder: 0.5 * (l + r)
        for (int i = lane; i < NF / 4; i += 32) {
            const float4 a = reinterpret_cast<const float4 *>(o)[i], b = reinterpret_cast<const float4 *>(o + CHF)[i];
            reinterpret_cast<float4 *>(o)[i] = make_float4(0.5f * (a.x + b.x), 0.5f * (a.y + b.y), 0.5f * (a.z + b.z), 0.5f * (a.w + b.w));
        }
        __syncwarp();
    }
    if constexpr (LM > 0) {
        if ((hdr_x >> 2) & 1u) w_imdct<3, (1 << LM), C, true, true>(o, lane, carry, t_short, t_tw, t_win);  // expanded rows are block-major
        else w_imdct<3 - LM, 1, C, true>(o, lane, carry, t_long, t_tw, t_win);
    } else {
        w_imdct<3, 1, C, true>(o, lane, carry, t_long, t_tw, t_win);
    }

    // post-filter parameters: previous frame -> this frame
    const uint4 hdr = stash[0];
    PfState old;
    {
        const uint4 q = stash[1];
        old.period = (int32_t)q.x;
        old.tapset = (int32_t)q.y;
        old.gain = __uint_as_float(q.z);
        old.pad = 0;
    }
    const uint32_t pos = stash[2].x;
    const int s_on = (hdr.x >> 1) & 1u, s_tapset = (hdr.x >> 4) & 15u, s_gain = (hdr.x >> 8) & 15u, s_period = hdr.x >> 16;
    int t1 = old.period, tap1 = old.tapset;
    float g1 = old.gain;
    if (!lost) {
        t1 = s_on ? s_period : 0;
        g1 = s_on ? 0.09375f * (float)(s_gain + 1) : 0.0f;
        tap1 = s_on ? s_tapset : 0;
    }
    const bool comb_on = A.postfilter && (old.gain != 0.0f || g1 != 0.0f);

    // tail of this frame -> carry
    if (lane < 15 * C) {
        const int ch = (C == 2 && lane >= 15) ? 1 : 0;
        *reinterpret_cast<float4 *>(carry_g + 4 * lane) = *reinterpret_cast<const float4 *>(o + ch * CHF + NF + 4 * (lane - 15 * ch));
    }
    // pitch comb post-filter, previous parameters -> this frame's over the first 120 samples
    if (comb_on) {
        const FrameView<C, CHF> V{o, ring, (int)pos};
        w_comb_ring<C, CHF, true>(V, old.period, t1, NF, old.gain, g1, old.tapset, tap1, 120, lane, t_winsq,
                                  w_comb_gains(old.gain, g1, old.tapset, tap1));
        __syncwarp();
        if (A.hist_samples && lane == 0) atomicAdd(A.hist_samples, (unsigned long long)(C * (max(max(old.period, t1), 15) + 2)));
    }
    // interleaved PCM -> ring (history of the next frames + device-resident output) and dense rows (host-path output).
    // The frame is contiguous in the ring except when it wraps (pos is a multiple of 120).
    const uint32_t dense_off = (A.dense && A.dense_off) ? A.dense_off[item] : 0u;
    float *dense = A.dense ? A.dense + (size_t)stream * A.dense_stride + dense_off : nullptr;
    const float gain = A.gain;
    constexpr int VEC = C == 2 ? NF / 2 : NF / 4;         // float4 per frame
    constexpr int SPV = C == 2 ? 2 : 4;                   // samples per float4
    const int wrap_at = (int)(RING_SAMPLES - pos) / SPV;  // first float4 that lands at the ring start
    float4 *r0 = reinterpret_cast<float4 *>(ring + (size_t)pos * C);
    float4 *r1 = reinterpret_cast<float4 *>(ring) - wrap_at;
#pragma unroll STORE_UNROLL
    for (int i = lane; i < VEC; i += 32) {
        float4 v;
        if (C == 2) {
            const float2 a = *reinterpret_cast<const float2 *>(o + 2 * i), b = *reinterpret_cast<const float2 *>(o + CHF + 2 * i);
            v = make_float4(a.x, b.x, a.y, b.y);
        } else {
            v = *reinterpret_cast<const float4 *>(o + 4 * i);
        }
        (i < wrap_at ? r0 : r1)[i] = v;
        if (dense) {
            if (gain != 1.0f) { v.x *= gain; v.y *= gain; v.z *= gain; v.w *= gain; }
            reinterpret_cast<float4 *>(dense)[i] = v;
        }
    }
    if (lane == 0) {
        uint32_t np = pos + (uint32_t)NF;
        if (np >= RING_SAMPLES) np -= RING_SAMPLES;
        A.ring_pos[stream] = np;
        PfState nw;
        nw.period = t1;
        nw.tapset = tap1;
        nw.gain = g1;
        nw.pad = 0;
        A.pf[stream] = nw;
        if (A.result) A.result[stream] = NF;
        if (A.final_range) A.final_range[stream] = lost ? 0u : hdr.y;
        if (A.softclip_reset && !lost) *reinterpret_cast<float2 *>(A.softclip_reset + 2 * (size_t)stream) = make_float2(0.f, 0.f);
    }
}

template <int LM, int C, int MODE, int CS = C> __global__ void __launch_bounds__(32 * FRAME_WARPS, FRAME_CTAS) k_frame_w(FrameArgs A)
{
    frame_cta<LM, C, MODE, CS>(A, A.item0 + blockIdx.x * FRAME_WARPS, A.item_end);
}

// The frame kernel of a step whose streams have different frame sizes: one launch per group of the step's MixPlan; a
// CTA looks up which bucket (frame size) it belongs to and runs that size's frame_cta.  The grid is the caller's upper
// bound; CTAs past the last bucket retire at once.  Shared memory is sized for the largest frame.
template <int C, int MODE> __global__ void __launch_bounds__(32 * FRAME_WARPS, FRAME_CTAS) k_frame_mix(FrameArgs A)
{
    const MixPlan &P = *A.plan;
    const int g = A.group;
    const uint32_t c = blockIdx.x;
    if (c >= P.cta0[g][4]) return;
    // the buckets take their CTAs longest frames first (cta0[g][j] belongs to lm = 3 - j): the short ones fill the tail
    const int j = (c >= P.cta0[g][1]) + (c >= P.cta0[g][2]) + (c >= P.cta0[g][3]), lm = 3 - j;
    const uint32_t first = P.start[g][lm] + (c - P.cta0[g][j]) * FRAME_WARPS, end = P.start[g][lm] + P.count[g][lm];
    switch (lm) {
    case 0: frame_cta<0, C, MODE>(A, first, end); break;
    case 1: frame_cta<1, C, MODE>(A, first, end); break;
    case 2: frame_cta<2, C, MODE>(A, first, end); break;
    default: frame_cta<3, C, MODE>(A, first, end); break;
    }
}

// ---- bucketing of a mixed-frame step (MixPlan, opn_internal.h)
// k_mix_key: one thread per stream reads its packet's TOC (the checks a host caller makes with query_packet_*,
// src/lib.rs:219-325), picks the bucket and takes a position in it.  Streams of a warp that fall into the same bucket
// take their positions with one atomic.  A lost packet (len 0) conceals one frame of the stream's previous size.
__global__ void __launch_bounds__(256) k_mix_key(MixArgs A)
{
    const uint32_t s = blockIdx.x * 256u + threadIdx.x;
    const bool on = s < A.n_streams;
    uint32_t key = MIX_NO_ITEM;
    int32_t err = 0;
    if (on) {
        const uint32_t len = A.lens[s];
        int lm = -1;
        if (len == 0u) {
            const uint32_t l = A.last_lm[s];
            // nothing decoded yet: zeros for the caller's frame size (decoder.rs:473-484); the frame kernel produces
            // them from an empty spectrum and an empty overlap
            lm = l != MIX_NO_ITEM ? (int)l : (A.capacity >= 960u ? 3 : A.capacity >= 480u ? 2 : A.capacity >= 240u ? 1 : 0);
        } else {
            const uint32_t toc = A.arena[A.offsets[s]];
            if ((toc & 0x80u) == 0u) err = OPN_ERR_UNIMPLEMENTED;                  // SILK / hybrid
            else if ((toc & 0x3u) != 0u) err = OPN_ERR_UNIMPLEMENTED;              // multi-frame packets: host path only
            else if (((toc & 0x4u) ? 2 : 1) != A.channels) err = OPN_ERR_UNIMPLEMENTED;  // mono<->stereo mapping
            else lm = (int)((toc >> 3) & 0x3u);
        }
        if (lm >= 0 && (120u << lm) > A.capacity) {
            err = OPN_ERR_FRAME_SIZE_TOO_SMALL;  // decoder.rs:388-390
            lm = -1;
        }
        if (lm >= 0) {
            uint32_t g = 0u;  // group g holds the streams [floor(n g / G), floor(n (g+1) / G)), as a uniform bucket's launches do
            if (A.n_groups > 1) {
                const uint32_t G = (uint32_t)A.n_groups;
                g = (uint32_t)(((uint64_t)s * G) / A.n_streams);
                if (g + 1u < G && (uint32_t)(((uint64_t)A.n_streams * (g + 1u)) / G) <= s) g += 1u;
            }
            key = g * 4u + (uint32_t)lm;
            if (len > 1u) A.last_lm[s] = (uint8_t)lm;  // len <= 1 is PLC/DTX (decoder.rs:467): the size is not taken from it
        }
    }
    const uint32_t peers = __match_any_sync(0xFFFFFFFFu, key);
    uint32_t rank = 0u;
    if (key != MIX_NO_ITEM) {
        const int leader = __ffs(peers) - 1;
        uint32_t base = 0u;
        if ((int)(threadIdx.x & 31u) == leader) base = atomicAdd(&A.plan->count[key >> 2][key & 3u], (uint32_t)__popc(peers));
        base = __shfl_sync(peers, base, leader);
        rank = base + (uint32_t)__popc(peers & ((1u << (threadIdx.x & 31u)) - 1u));
    }
    if (on) {
        A.key[s] = (uint8_t)key;
        A.rank[s] = rank;
        if (key == MIX_NO_ITEM && A.result) A.result[s] = err;
    }
}
// k_mix_place: bucket starts from the counts (every CTA recomputes the dozen sums), then each stream's item record.
__global__ void __launch_bounds__(256) k_mix_place(MixArgs A)
{
    __shared__ uint32_t s_start[MIX_GROUPS * 4];
    if (threadIdx.x == 0) {
        uint32_t at = 0u;
        MixPlan &P = *A.plan;
        for (int g = 0; g < MIX_GROUPS; g++) {
            uint32_t cta = 0u;
            for (int j = 0; j < 4; j++) {  // longest frames first, in the item table and in the frame kernel's CTA order
                const int lm = 3 - j;
                const uint32_t n = P.count[g][lm];
                s_start[g * 4 + lm] = at;
                if (blockIdx.x == 0) {
                    P.start[g][lm] = at;
                    P.cta0[g][j] = cta;
                }
                at += (n + MIX_PAD - 1u) / MIX_PAD * MIX_PAD;
                cta += (n + FRAME_WARPS - 1u) / FRAME_WARPS;
            }
            if (blockIdx.x == 0) P.cta0[g][4] = cta;
        }
        if (blockIdx.x == 0) P.items_padded = at;
    }
    __syncthreads();
    const uint32_t s = blockIdx.x * 256u + threadIdx.x;
    if (s >= A.n_streams) return;
    const uint32_t key = A.key[s];
    if (key == MIX_NO_ITEM) return;
    const uint32_t item = s_start[key] + A.rank[s];
    A.item_offsets[item] = A.offsets[s];
    A.item_lens[item] = A.lens[s];
    A.item_stream[item] = s;
    A.item_lm[item] = (uint8_t)(key & 3u);
}

// Operator-level Mdct::backward on independent rows (tests; opn_op_imdct_tdac): one warp per row.
template <int SHIFT, int NBLK>
__global__ void __launch_bounds__(32)
k_op_imdct_w(const float *__restrict__ input, size_t in_stride, float *__restrict__ output, size_t out_stride)
{
    extern __shared__ __align__(16) float sm[];
    constexpr int N2 = 960 >> SHIFT, NF = N2 * NBLK;
    const int lane = threadIdx.x;
    const float *in = input + (size_t)blockIdx.x * in_stride;
    float *out = output + (size_t)blockIdx.x * out_stride;
    for (int i = lane; i < NF; i += 32) sm[i] = in[i];
    float4 carry = make_float4(0.f, 0.f, 0.f, 0.f);
    if (lane < 15) carry = make_float4(out[4 * lane], out[4 * lane + 1], out[4 * lane + 2], out[4 * lane + 3]);
    __syncwarp();
    w_imdct<SHIFT, NBLK, 1>(sm, lane, carry, g_tab.trig_pair + trig_pair_off(SHIFT), g_tab.twiddles, g_tab.window);
    for (int i = lane; i < NF + 60; i += 32) out[i] = sm[i];
}

// Operator-level comb_filter_inplace on rows (tests; opn_op_comb_filter_inplace): one warp per row runs the frame
// kernel's w_comb_ring; the n samples from y_offset on are the frame (shared memory), the row's own prefix in global
// memory plays the role of the PCM ring (history).
__global__ void __launch_bounds__(32)
k_op_comb_inplace_w(float *__restrict__ y, size_t row_stride, int y_offset, int n, const int32_t *__restrict__ params4,
                    const float *__restrict__ gains2, int overlap)
{
    extern __shared__ __align__(16) float sm[];
    const int lane = threadIdx.x;
    float *row = y + (size_t)blockIdx.x * row_stride;
    const int t0 = params4[4 * blockIdx.x], t1 = params4[4 * blockIdx.x + 1];
    const int tap0 = params4[4 * blockIdx.x + 2], tap1 = params4[4 * blockIdx.x + 3];
    const float g0 = gains2[2 * blockIdx.x], g1 = gains2[2 * blockIdx.x + 1];
    for (int i = lane; i < n; i += 32) sm[i] = row[y_offset + i];
    __syncwarp();
    const FrameView<1, 0> V{sm, row, y_offset};  // max(t0, t1) + 2 <= y_offset (checked by the caller): the view never wraps
    w_comb_ring<1, 0>(V, t0, t1, n, g0, g1, tap0, tap1, overlap, lane, g_tab.window_sq, w_comb_gains(g0, g1, tap0, tap1));
    __syncwarp();
    for (int i = lane; i < n; i += 32) row[y_offset + i] = sm[i];
}

}  // namespace opn
