// symbols.cuh -- kernel 0: warp-per-packet symbol decode (range decoder + PVQ expansion).
//
//   k_rangedec_script : replays an arbitrary list of RangeDecoder calls (operator-level parity
//                       with src/range_coder/decoder.rs and src/celt/pvc.rs).
//   k_synth_symbols   : decodes one SYNTH-CELT/1 frame per warp (DESIGN.md "frame layout"):
//                       flags, post-filter parameters, Laplace coarse energies, raw fine bits,
//                       PVQ pulse vectors -> unit-norm coefficients for the IMDCT kernel.
#pragma once
#include <type_traits>
#include "opn_device.cuh"
#include "opn_internal.h"
#include "rangedec.cuh"
#include "celt2.cuh"
#include "celt2_lane.cuh"

namespace opn {

constexpr int PVQ_TABLE_WORDS = 1272;
constexpr int Y_STAGE = 192;  // >= 176, the largest PVQ part (pvc.rs:309-313)

__device__ __forceinline__ void stage_bytes(uint8_t *dst, const uint8_t *src, uint32_t len, uint32_t lane)
{
    if ((reinterpret_cast<uintptr_t>(src) & 3u) == 0u) {
        uint32_t words = len >> 2;
        const uint32_t *s4 = reinterpret_cast<const uint32_t *>(src);
        uint32_t *d4 = reinterpret_cast<uint32_t *>(dst);
        for (uint32_t w = lane; w < words; w += 32u) d4[w] = __ldg(s4 + w);
        for (uint32_t i = (words << 2) + lane; i < len; i += 32u) dst[i] = __ldg(src + i);
    } else {
        for (uint32_t i = lane; i < len; i += 32u) dst[i] = __ldg(src + i);
    }
    __syncwarp();
}

__device__ __forceinline__ void load_pvq_table(uint32_t *s_data, uint16_t *s_row)
{
    for (int i = threadIdx.x; i < PVQ_TABLE_WORDS; i += blockDim.x) s_data[i] = g_tab.pvq_u_data[i];
    if (threadIdx.x < 15) s_row[threadIdx.x] = g_tab.pvq_u_row[threadIdx.x];
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// cwrsi (pvc.rs:182-284) walked by ONE LANE in EVENTS, not dimensions; `y` (zero-initialised by the caller, only nonzero
// pulses are stored) receives the pulse vector, the return value is yy = sum y^2.  n <= 2 on entry skips the walk
// (n == 0: nothing to do, the lane idles through its slot).
//
// While k < n (pvc.rs:232-258) a dimension is empty iff U(k,n) <= i < U(k+1,n), and stepping over it subtracts U(k,n);
// after t empty dimensions i has lost A(t) = C(k,n) - C(k,n-t) (C = running row sum of U), so "dimension n-t is empty
// given all before it were" reads A(t) + U(k,n-t) <= i < A(t) + U(k+1,n-t), or as one unsigned comparison
// i - C(k,n) + C(k,n-t-1) < U(k+1,n-t) - U(k,n-t).  That predicate is monotone in t (once a dimension is occupied the
// sequential loop stops there), so the length of the run of empty dimensions is found by bisection over t in [0, T],
// T = n - max(k,2) being where the regime ends (k >= n, or the closed-form tail n == 2).  One event = one run + the
// occupied dimension after it: a part with k pulses takes at most k+1 events instead of n-2 steps.
// The single comparison is only valid while the 32-bit sums cannot wrap: C(k,n) + U(k+1,n) < 2^32.  `ev_nmax[k]` is the
// largest n for which that holds (built next to the tables in upload_tables); above it the walk takes the reference's
// one-dimension step until n has come down.  The k >= n regime keeps the reference's per-dimension code.
// Every nonzero pulse is handed to `put(position, value)`; zero dimensions are never visited.
template <class Sink>
__device__ __forceinline__ int32_t cwrsi_events(const uint32_t *U, const uint2 *CW, const uint16_t *row, const uint8_t *ev_nmax,
                                                uint32_t n, uint32_t k, uint32_t i, Sink &&put)
{
    int32_t yy = 0;
    uint32_t y = 0u;  // position inside the part
    uint32_t rk = row[min(k, 14u)], rk1 = row[min(k + 1u, 14u)];  // row offsets of U(k,.) and U(k+1,.): only read when k < n
#pragma unroll 1
    while (n > 2u) {
        if (k >= n) {  // lots of pulses, pvc.rs:196-231: one dimension per event
            const uint32_t rn = row[n];
            uint32_t p = U[rn + k + 1u];
            const int32_t sg = i >= p ? -1 : 0;
            i -= (uint32_t)((int32_t)p & sg);
            const uint32_t k0 = k;
            const uint32_t q = U[rn + n];
            if (q > i) {
                k = n;
                do {
                    k -= 1u;
                    p = U[row[k] + n];
                } while (p > i);
            } else {
                p = U[rn + k];
                while (p > i) {
                    k -= 1u;
                    p = U[rn + k];
                }
            }
            i -= p;
            const int32_t val = ((int32_t)k0 - (int32_t)k + sg) ^ sg;
            if (val) put(y, val);
            yy += val * val;
            rk = row[min(k, 14u)];
            rk1 = row[min(k + 1u, 14u)];
            y++;
            n -= 1u;
        } else {  // lots of dimensions, pvc.rs:232-258
            uint32_t T, lo = 0u;
            if (n <= (uint32_t)ev_nmax[k]) {
                T = n - max(k, 2u);
                const uint2 *pw = CW + rk + n;                  // pw[-t] = (C(k,n-t-1), V(n-t-1,k))
                const uint32_t ic = i - (pw[0].x + U[rk + n]);  // i - C(k,n)
                uint32_t hi = T;
                while (lo < hi) {
                    const uint32_t mid = (lo + hi) >> 1;
                    const uint2 cw = pw[-(int32_t)mid];
                    // i - A(mid) - U(k,n-mid) as one unsigned number: below V(n-mid-1,k) iff dimension n-mid is empty
                    const bool empty = ic + cw.x < cw.y;
                    lo = empty ? mid + 1u : lo;
                    hi = empty ? hi : mid;
                }
                if (lo) i = ic + pw[1 - (int32_t)lo].x;  // i - A(lo)
            } else {  // the sums could wrap for this (n, k): the reference's test of one dimension
                T = 1u;
                const uint32_t p = U[rk + n];
                if (p <= i && i < U[rk1 + n]) {
                    i -= p;
                    lo = 1u;
                }
            }
            y += lo;
            n -= lo;
            if (lo < T) {  // dimension n holds pulses
                const uint32_t q = U[rk1 + n];
                const int32_t sg = i >= q ? -1 : 0;
                i -= (uint32_t)((int32_t)q & sg);
                const uint32_t k0 = k;
                uint32_t p;
                do {
                    k -= 1u;
                    p = U[row[k] + n];
                } while (p > i);
                i -= p;
                const int32_t val = ((int32_t)k0 - (int32_t)k + sg) ^ sg;
                put(y, val);  // never zero here: k dropped by at least one
                yy += val * val;
                rk = row[k];
                rk1 = row[k + 1u];
                y++;
                n -= 1u;
            }
        }
    }
    if (n == 2u) {
        // n == 2 (pvc.rs:262-275)
        uint32_t p = 2u * k + 1u;
        int32_t sg = i >= p ? -1 : 0;
        i -= (uint32_t)((int32_t)p & sg);
        const uint32_t k0 = k;
        k = (i + 1u) >> 1;
        if (k != 0u) i -= 2u * k - 1u;
        int32_t val = ((int32_t)k0 - (int32_t)k + sg) ^ sg;
        if (val) put(y, val);
        yy += val * val;
        // n == 1 (pvc.rs:277-281)
        sg = -(int32_t)i;
        val = ((int32_t)k + sg) ^ sg;
        if (val) put(y + 1u, val);
        yy += val * val;
    }
    return yy;
}

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SYM_WARPS_PER_CTA * 32)
k_rangedec_script(const uint8_t *__restrict__ arena, const uint32_t *__restrict__ offsets,
                  const uint32_t *__restrict__ lens, uint32_t n_packets, const opn_op *__restrict__ ops,
                  uint32_t n_ops, const uint8_t *__restrict__ icdf_pool, opn_op_out *__restrict__ out,
                  int32_t *__restrict__ y_out, uint32_t y_stride, uint32_t pkt_cap)
{
    extern __shared__ __align__(16) uint8_t smem[];
    uint32_t *s_pvq = reinterpret_cast<uint32_t *>(smem);
    uint2 *s_cw = reinterpret_cast<uint2 *>(s_pvq + PVQ_TABLE_WORDS);
    uint16_t *s_row = reinterpret_cast<uint16_t *>(s_cw + PVQ_TABLE_WORDS);
    uint8_t *s_nmax = reinterpret_cast<uint8_t *>(s_row + 16);
    int32_t *s_y = reinterpret_cast<int32_t *>(s_nmax + 16) + (threadIdx.x >> 5) * Y_STAGE;
    uint8_t *s_pkt = reinterpret_cast<uint8_t *>(reinterpret_cast<int32_t *>(s_nmax + 16) + SYM_WARPS_PER_CTA * Y_STAGE) +
                     (threadIdx.x >> 5) * pkt_cap;
    for (int i = threadIdx.x; i < PVQ_TABLE_WORDS; i += blockDim.x) s_cw[i] = g_tab.pvq_cw_data[i];
    if (threadIdx.x < 16) s_nmax[threadIdx.x] = g_tab.pvq_ev_nmax[threadIdx.x];
    load_pvq_table(s_pvq, s_row);
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t pkt = blockIdx.x * SYM_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (pkt >= n_packets) return;
    const uint32_t len = lens[pkt];
    // Packets that fit are staged in shared memory; oversized test streams (the reference's
    // test_simple_uint_bits stream is ~0.5 MB) are read in place from global memory.
    const uint8_t *bytes = arena + offsets[pkt];
    if (len <= pkt_cap) {
        stage_bytes(s_pkt, bytes, len, lane);
        bytes = s_pkt;
    }
    PvqTable T{s_pvq, s_row};
    RangeDec d;
    d.init(bytes, len);
    uint32_t ny = 0u;
    for (uint32_t i = 0; i < n_ops; i++) {
        const uint32_t op = ops[i].op, a = ops[i].a, b = ops[i].b;
        uint32_t v = 0u;
        switch (op) {
        case OPN_OP_UINT: v = d.uint(a); break;
        case OPN_OP_BITS: v = d.bits(a); break;
        case OPN_OP_BIT_LOGP: v = d.bit_logp(a); break;
        case OPN_OP_ICDF: v = d.icdf(icdf_pool + a, b); break;
        case OPN_OP_LAPLACE: v = (uint32_t)d.laplace(a, b); break;
        case OPN_OP_BIT_VIA_DECODE: {  // src/range_coder/mod.rs:446-454
            uint32_t fs = d.decode(1u << a);
            uint32_t s = fs >= (1u << a) - 1u ? 1u : 0u;
            d.update(s ? (1u << a) - 1u : 0u, (1u << a) - (s ? 0u : 1u), 1u << a);
            v = s;
            break;
        }
        case OPN_OP_BIT_VIA_DECODE_BIN: {  // src/range_coder/mod.rs:455-463
            uint32_t fs = d.decode_bin(a);
            uint32_t s = fs >= (1u << a) - 1u ? 1u : 0u;
            d.update(s ? (1u << a) - 1u : 0u, (1u << a) - (s ? 0u : 1u), 1u << a);
            v = s;
            break;
        }
        case OPN_OP_PULSES: {
            float yy = decode_pulses_warp(d, T, s_y, a, b, lane);
            v = __float_as_uint(yy);
            if (y_out)
                for (uint32_t j = lane; j < a; j += 32u) y_out[(size_t)pkt * y_stride + ny + j] = s_y[j];
            ny += a;
            __syncwarp();
            break;
        }
        case OPN_OP_PULSES_EVENTS: {
            // decode_pulses (pvc.rs:156-160) with the product path's cwrsi: the event walk of k_synth_expand, run by lane 0
            const uint32_t ci = d.uint(T.v(a, b));
            for (uint32_t j = lane; j < a; j += 32u) s_y[j] = 0;
            __syncwarp();
            int32_t yy = 0;
            if (lane == 0u) yy = cwrsi_events(s_pvq, s_cw, s_row, s_nmax, a, b, ci, [&](uint32_t at, int32_t val) { s_y[at] = val; });
            yy = __shfl_sync(0xFFFFFFFFu, yy, 0);
            __syncwarp();
            v = __float_as_uint((float)yy);
            if (y_out)
                for (uint32_t j = lane; j < a; j += 32u) y_out[(size_t)pkt * y_stride + ny + j] = s_y[j];
            ny += a;
            __syncwarp();
            break;
        }
        case OPN_OP_SHRINK: d.shrink_storage(a); break;
        case OPN_OP_TELL: v = d.tell(); break;
        default: break;
        }
        if (lane == 0u) {
            opn_op_out o;
            o.value = v;
            o.tell_frac = d.tell_frac();
            o.rng = d.rng;
            out[(size_t)pkt * n_ops + i] = o;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// SYNTH-CELT/1 symbol decode, two kernels:
//
//   k_synth_rangedec  ONE LANE decodes one packet.  The entropy decoder is a strictly serial
//      dependency chain per packet (two divisions and a byte refill per symbol); a warp that
//      shares one chain between its 32 lanes issues ~60 warp-instructions per symbol for one
//      packet, a warp whose lanes each own a chain issues about the same for 32 packets.  The chain
//      only produces what depends on it: flags, post-filter parameters, energies and, for every PVQ
//      part, the codeword INDEX (decode_uint with the host-precomputed alphabet split and
//      reciprocal).  Packet bytes are read in place through L1 (each lane walks its own packet
//      front-to-back and back-to-front, so every 128-byte line is fetched once).
//   k_synth_expand    ONE WARP expands one packet's indices into pulse vectors (cwrsi never feeds
//      back into the range decoder): the parts are dealt to the 32 lanes by a host-computed
//      longest-first schedule, one part per lane and slot; a lane walks its part in events (one run of
//      empty dimensions, found by bisection, plus the occupied dimension after it), then the warp writes
//      pulses x gain as coalesced float4 coefficient rows.
//
// Shared memory of k_synth_expand (per CTA of EXPAND_WARPS_PER_CTA warps):
//   PVQ U(n,k) table 5088 B + bisection table 10176 B (both by TMA) + row offsets 32 B + mbarrier 16 B |
//   entry table 72 x 16 B | per warp: codeword indices 72 x 4 B, gains 76 x 4 B (slot 72 = 0 for bins without a part), 16-bit pulses 2 x 960 x 2 B.
constexpr size_t SYM_EXPAND_WARP_BYTES = 2 * 960 * 4;  // coefficient rows of one packet
__host__ __device__ constexpr size_t synth_expand_smem()
{
    return 3 * PVQ_TABLE_WORDS * 4 + 32 + 16 + 16 + SYNTH_MAX_ENTRIES * sizeof(SynthEntry) + (size_t)EXPAND_WARPS_PER_CTA * SYM_EXPAND_WARP_BYTES;
}

__global__ void __launch_bounds__(RANGEDEC_WARPS_PER_CTA * 32) k_synth_rangedec(SymbolArgs A)
{
    __shared__ SynthEntry s_ent[SYNTH_MAX_ENTRIES];
    __shared__ uint32_t s_lfl[21][LAP_N + 1], s_lfs[21][LAP_N + 1];  // decode_laplace states per band (laplace_table)
    const uint32_t lane = threadIdx.x;  // index inside the CTA: one packet per thread
    const int C = A.channels;
    int lm = A.lm;
    if (A.item_lm) {  // mixed-frame step: buckets start on CTA boundaries, the CTA's first item tells its frame size
        const uint32_t l = A.item_lm[blockIdx.x * (RANGEDEC_WARPS_PER_CTA * 32u)];
        if (l == MIX_NO_ITEM) return;
        lm = (int)l;
    }
    if (lane < 21u) {
        const uint32_t decay = 6000u + 400u * lane;
        const uint32_t fs0 = ((32768u - 33u) * (16384u - decay)) / (16384u + decay) + 1u;  // get_start_freq, src/range_coder/mod.rs:530-534
        laplace_table(fs0, decay, s_lfl[lane], s_lfs[lane]);
    }
    const int ne = g_tab.synth_n_entries[lm][C - 1];
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(g_tab.synth_entries[lm][C - 1]);
        uint4 *dst = reinterpret_cast<uint4 *>(s_ent);
        for (int i = lane; i < ne; i += RANGEDEC_WARPS_PER_CTA * 32) dst[i] = src[i];
    }
    __syncthreads();
    const uint32_t item = blockIdx.x * (RANGEDEC_WARPS_PER_CTA * 32u) + lane;
    if (item >= A.n_items) return;
    if (A.item_lm && A.item_lm[item] == MIX_NO_ITEM) return;
    const uint32_t stream = A.stream_idx ? A.stream_idx[item] : item;
    uint32_t len = A.lens[item];
    const uint8_t *src = A.arena + A.offsets[item];

    int32_t status = len == 0u ? ITEM_LOST : ITEM_OK;
    if (A.has_toc && len > 0u) {
        // TOC checks a host caller does with query_packet_* (src/lib.rs:219-325) before decode_frame
        const uint32_t toc = __ldg(src);
        if ((toc & 0x80u) == 0u) status = OPN_ERR_UNIMPLEMENTED;                         // SILK / hybrid
        else if ((toc & 0x3u) != 0u) status = OPN_ERR_UNIMPLEMENTED;                     // multi-frame: host path only
        else if ((int)((toc >> 3) & 0x3u) != lm) status = OPN_ERR_FRAME_SIZE_TOO_SMALL;  // frame size != call's
        else if (((toc & 0x4u) ? 2 : 1) != C) status = OPN_ERR_UNIMPLEMENTED;            // mono<->stereo mapping
        src += 1;
        len -= 1u;
    }
    if (status == ITEM_OK && len <= 1u) status = ITEM_LOST;  // decoder.rs:467: len <= 1 means PLC/DTX
    A.status[stream] = status;
    if (status < 0) return;

    // What the frame kernel needs travels in one 16-byte header; the full side record (energies included) is only
    // written when the caller asked for it (operator entry / tests).
    opn_synth_side *sd = A.side ? A.side + stream : nullptr;
    uint32_t *sw = reinterpret_cast<uint32_t *>(sd);
    constexpr uint32_t SIDE_WORDS = sizeof(opn_synth_side) / 4u;
    if (status == ITEM_LOST) {
        if (sd)
            for (uint32_t i = 0; i < SIDE_WORDS; i++) sw[i] = 0u;
        A.hdr[stream] = make_uint4(0u, 0u, 0u, 0u);
        return;
    }
    LaneDec d;
    d.init(src, len);
    const uint32_t silence = d.bit_logp(15u);
    if (silence) {
        if (sd) {
            for (uint32_t i = 0; i < SIDE_WORDS; i++) sw[i] = 0u;
            sd->silence = 1;
            sd->final_rng = d.rng;
            sd->tell_frac = d.tell_frac();
        }
        A.hdr[stream] = make_uint4(1u, d.rng, d.tell_frac(), 0u);
        return;
    }
    const uint32_t postfilter = d.bit_logp(1u);
    uint32_t octave = 0u, period = 0u, gain_idx = 0u, tapset = 0u;
    if (postfilter) {
        octave = d.uint_small(6u);
        period = (16u << octave) + d.bits(4u + octave) - 1u;
        gain_idx = d.bits(3u);
        tapset = d.icdf(g_tab.tapset_icdf, 2u);
    }
    const uint32_t transient = d.bit_logp(3u);
    const uint32_t intra = d.bit_logp(3u);
    if (sd) {
        sd->silence = 0;
        sd->postfilter = (int32_t)postfilter;
        sd->octave = (int32_t)octave;
        sd->period = (int32_t)period;
        sd->gain_idx = (int32_t)gain_idx;
        sd->tapset = (int32_t)tapset;
        sd->transient = (int32_t)transient;
        sd->intra = (int32_t)intra;
    }
    for (int b = 0; b < 21; b++) {
        const uint32_t decay = 6000u + 400u * (uint32_t)b;
        for (int c = 0; c < C; c++) {
            const int32_t v = d.laplace(s_lfl[b], s_lfs[b], decay);
            if (sd) sd->coarse[c][b] = v;
        }
        if (sd && C == 1) sd->coarse[1][b] = 0;
    }
    // fine energy: 21*C two-bit fields, band-major.  decode_bits is a plain LSB-first bit window (decoder.rs:279-303), so
    // twelve consecutive 2-bit reads are one 24-bit read cut into fields.
    for (int f0 = 0; f0 < 21 * C; f0 += 12) {
        const int nfld = min(12, 21 * C - f0);
        uint32_t w = d.bits(2u * (uint32_t)nfld);
        if (sd)
            for (int f = f0; f < f0 + nfld; f++, w >>= 2) sd->fine[f % C][f / C] = (int32_t)(w & 3u);
    }
    if (sd && C == 1)
        for (int b = 0; b < 21; b++) sd->fine[1][b] = 0;
    uint32_t *idx = A.idx + (size_t)stream * SYNTH_MAX_ENTRIES;
    uint32_t n_pulses = 0u;
    for (int e = 0; e < ne; e++) {
        const SynthEntry E = s_ent[e];
        uint32_t v;
        if (E.n == 1) {
            v = d.bits(1u);
            n_pulses += 1u;
        } else {
            v = d.uint_precomputed(E.ft_minus1, E.ft1, E.ftb, E.magic, E.sh);
            n_pulses += E.k;
        }
        idx[e] = v;
    }
    const uint32_t tf = d.tell_frac();
    if (sd) {
        sd->final_rng = d.rng;
        sd->tell_frac = tf;
        sd->n_pulses = n_pulses;
    }
    A.hdr[stream] = make_uint4(hdr_pack(0u, postfilter, transient, intra, tapset, gain_idx, octave, period), d.rng, tf, n_pulses);
}

// PVQ expansion of one packet by one warp: codeword indices -> coefficient rows (SYNTH-CELT/1: unit-norm parts scaled by
// 2^-5, DESIGN.md).  `rows` holds C channels of `chs` floats each and must be ZERO on entry: only the nonzero pulses are
// written.  The parts are dealt to the lanes by the host-built slot tables (sorted by size, 32 per slot); a lane walks its
// part with cwrsi_events and keeps the (position, value) pairs of the at most 6 nonzero pulses in one 64-bit register
// (10 bits each: the schedule has n <= 64 and k <= 6, checked in upload_tables) until the part's norm is known.
// Tables may live in shared or global memory.
struct ExpandTables {
    const uint32_t *U;
    const uint2 *CW;
    const uint16_t *row;
    const uint8_t *nmax;
    const SynthEntry *ent;  // [n_entries]
    const uint8_t *slots;   // [n_slots][32]: lane -> entry, 0xFF = none
    int n_slots;
};
// lmt > 0: the frame is transient with 2^lmt short blocks and the rows are wanted block-major (bin j of a channel at
// (j mod 2^lmt) * (nf >> lmt) + (j >> lmt), see w_imdct); 0: bins stay in the bitstream's order.  y_out is never remapped.
__device__ __forceinline__ uint32_t block_major(uint32_t j, int lmt, int nf) { return (j & ((1u << lmt) - 1u)) * (uint32_t)(nf >> lmt) + (j >> lmt); }
// get_idx(e): the codeword index of part e (0xFF: none); called by every lane of the warp for every slot.
template <int C, class IdxFn>
__device__ __forceinline__ void w_expand(const ExpandTables &T, int lm, uint32_t lane, IdxFn get_idx, float *rows, int chs,
                                         int32_t *__restrict__ y_out, int lmt = 0)
{
    const int nf = 120 << lm;
    const int nslots = T.n_slots;
    // everything a lane needs for its (at most SYNTH_SLOTS) parts is requested before the first walk starts
    uint32_t ee[SYNTH_SLOTS], ii[SYNTH_SLOTS];
#pragma unroll
    for (int slot = 0; slot < SYNTH_SLOTS; slot++) {
        ee[slot] = slot < nslots ? T.slots[slot * 32 + lane] : 0xFFu;
        ii[slot] = get_idx(ee[slot]);
    }
#pragma unroll 1
    for (int slot = 0; slot < nslots; slot++) {
        uint32_t e = ee[0], i = ii[0];
#pragma unroll
        for (int q = 1; q < SYNTH_SLOTS; q++)
            if (slot == q) { e = ee[q]; i = ii[q]; }
        const bool has = e != 0xFFu;
        const SynthEntry E = T.ent[has ? e : 0u];
        uint32_t n = has ? E.n : 0u;
        const uint32_t k = E.k;
        uint64_t rec = 0ull;  // nonzero pulses, 10 bits each: position << 4 | (value & 15)
        uint32_t cnt = 0u;
        auto put = [&](uint32_t at, int32_t val) {
            rec |= (uint64_t)((at << 4) | ((uint32_t)val & 15u)) << (10u * cnt);
            cnt += 1u;
        };
        int32_t yy = 0;
        if (has && n == 1u) {  // sign-only band
            put(0u, i ? -1 : 1);
            yy = 1;
        } else if (has && k == 1u) {
            // one pulse: cwrsi reduces to a closed form, y[i] = +1 for i < n, y[2n-1-i] = -1 otherwise
            // (checked against the oracle for every band size in tests/test_oracle_kat.py::test_cwrsi_single_pulse_closed_form)
            if (i < n) put(i, 1);
            else put(2u * n - 1u - i, -1);
            yy = 1;
            n = 0u;  // done: takes no part in the walk below
        }
        yy += cwrsi_events(T.U, T.CW, T.row, T.nmax, n, k, i, put);
        if (has) {
            const float gain = 0.03125f / sqrtf((float)yy);
            const uint32_t ch = E.base >= (uint32_t)nf ? 1u : 0u;
            const uint32_t bin0 = E.base - ch * (uint32_t)nf;  // first bin of the part inside its channel
            float *dst = rows + ch * (uint32_t)chs;
            auto store = [&](auto remap) {  // the frame is all long or all short blocks: one uniform branch, two plain loops
#pragma unroll
                for (uint32_t j = 0; j < 6u; j++) {
                    if (j < cnt) {
                        const uint32_t r = (uint32_t)(rec >> (10u * j)) & 1023u;
                        const int32_t val = ((int32_t)(r << 28)) >> 28;
                        const uint32_t at = bin0 + (r >> 4);
                        dst[decltype(remap)::value ? block_major(at, lmt, nf) : at] = (float)val * gain;
                        if (y_out) y_out[E.base + (r >> 4)] = val;
                    }
                }
            };
            if (lmt) store(std::true_type{});
            else store(std::false_type{});
        }
    }
}

// Stand-alone expansion kernel (operator entry opn_op_synth_symbols): the same w_expand the frame kernel runs, with the PVQ
// tables staged in shared memory by TMA; the coefficient rows leave as float4.
__global__ void __launch_bounds__(EXPAND_WARPS_PER_CTA * 32) k_synth_expand(SymbolArgs A)
{
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    uint32_t *s_pvq = reinterpret_cast<uint32_t *>(smem);
    uint2 *s_cw = reinterpret_cast<uint2 *>(s_pvq + PVQ_TABLE_WORDS);
    uint16_t *s_row = reinterpret_cast<uint16_t *>(s_cw + PVQ_TABLE_WORDS);
    uint8_t *s_nmax = reinterpret_cast<uint8_t *>(s_row + 16);  // 16 bytes: ev_nmax[k] of cwrsi_events
    uint64_t *bar = reinterpret_cast<uint64_t *>(s_nmax + 16);
    SynthEntry *s_ent = reinterpret_cast<SynthEntry *>(bar + 2);
    float *s_rows = reinterpret_cast<float *>(reinterpret_cast<uint8_t *>(s_ent + SYNTH_MAX_ENTRIES) + (size_t)warp * SYM_EXPAND_WARP_BYTES);

    const int lm = A.lm, C = A.channels, nf = 120 << lm;
    const int ne = g_tab.synth_n_entries[lm][C - 1];
    // the two PVQ tables (15 KB) arrive by TMA while the warps clear their rows
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        mbar_expect_tx(bar, 3 * PVQ_TABLE_WORDS * 4);
        bulk_g2s(s_pvq, g_tab.pvq_u_data, PVQ_TABLE_WORDS * 4, bar);
        bulk_g2s(s_cw, g_tab.pvq_cw_data, 2 * PVQ_TABLE_WORDS * 4, bar);
    }
    if (threadIdx.x < 15) s_row[threadIdx.x] = g_tab.pvq_u_row[threadIdx.x];
    if (threadIdx.x < 16) s_nmax[threadIdx.x] = g_tab.pvq_ev_nmax[threadIdx.x];
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(g_tab.synth_entries[lm][C - 1]);
        uint4 *dst = reinterpret_cast<uint4 *>(s_ent);
        for (int i = threadIdx.x; i < ne; i += blockDim.x) dst[i] = src[i];
    }
    const uint32_t item = blockIdx.x * EXPAND_WARPS_PER_CTA + warp;
    const bool in_range = item < A.n_items;
    const uint32_t stream = in_range ? (A.stream_idx ? A.stream_idx[item] : item) : 0u;
    const int32_t status = in_range ? A.status[stream] : -1;
    const int32_t silence = in_range ? (int32_t)(A.hdr[stream].x & 1u) : 0;
    const bool zero_frame = status == ITEM_LOST || (status >= 0 && silence != 0);
    const int nvec = C * nf / 4;
    for (int i = lane; i < nvec; i += 32) reinterpret_cast<float4 *>(s_rows)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();  // entry table, row offsets and the mbarrier are set up
    mbar_wait(bar, 0);
    if (status < 0) return;
    float4 *coef4 = A.coef ? reinterpret_cast<float4 *>(A.coef + (size_t)stream * C * nf) : nullptr;
    int32_t *yo = A.y_out ? A.y_out + (size_t)stream * C * nf : nullptr;
    if (yo)
        for (int i = lane; i < nvec; i += 32) reinterpret_cast<int4 *>(yo)[i] = make_int4(0, 0, 0, 0);
    __syncwarp();
    if (!zero_frame) {
        const ExpandTables T{s_pvq, s_cw, s_row, s_nmax, s_ent, &g_tab.synth_slot_entries[lm][C - 1][0][0], g_tab.synth_n_slots[lm][C - 1]};
        const uint32_t *ip = A.idx + (size_t)stream * SYNTH_MAX_ENTRIES;
        auto get_idx = [&](uint32_t e) { return e != 0xFFu ? __ldg(ip + e) : 0u; };
        if (C == 2) w_expand<2>(T, lm, lane, get_idx, s_rows, nf, yo);
        else w_expand<1>(T, lm, lane, get_idx, s_rows, nf, yo);
    }
    __syncwarp();
    if (coef4)
        for (int i = lane; i < nvec; i += 32) coef4[i] = reinterpret_cast<const float4 *>(s_rows)[i];
}

// ---------------------------------------------------------------------------------------------
// SYNTH-CELT/2 (celt2.cuh): allocation-driven frames.  ONE LANE decodes one packet: the whole frame logic is a serial
// function of the range decoder's state (every budget decision reads tell_frac).  It leaves the frame header and the list
// of PVQ leaves (position, size, pulses, codeword index, gain) for the frame kernel, whose warps expand them.
__device__ __forceinline__ Celt2Tabs device_celt2_tabs()
{
    return Celt2Tabs{g_tab.e_bands, g_tab.log_n, g_tab.alloc_vectors, g_tab.cache_bits, g_tab.cache_caps, g_tab.log2_frac, g_tab.cache_index,
                     g_tab.pvq_u_data, g_tab.pvq_u_row};
}

// The frame logic of SYNTH-CELT/2 branches on the packet's content at every band (allocation searches, split recursion): the
// lanes of a warp each follow their own path and the warp executes the union of them.  C2_RD_LANES packets per warp
// (lanes 0 .. C2_RD_LANES-1; the others idle) trades idle lanes -- the kernel is latency-bound on a few hundred warps, the
// SMs have the room -- for a shorter union.  128 registers (16 warps per SM) so that its warps fit beside resident frame-kernel CTAs.
#ifndef OPN_C2_RD_MIN_CTAS
#define OPN_C2_RD_MIN_CTAS 16
#endif
#ifndef OPN_C2_RD_LANES
#define OPN_C2_RD_LANES 32
#endif
constexpr uint32_t C2_RD_LANES = OPN_C2_RD_LANES;
constexpr uint32_t C2_RD_ITEMS_PER_CTA = RANGEDEC_WARPS_PER_CTA * C2_RD_LANES;
static_assert(32u % C2_RD_LANES == 0u, "a mixed-frame bucket starts on a multiple of MIX_PAD items: a CTA must not span two");
__global__ void __launch_bounds__(RANGEDEC_WARPS_PER_CTA * 32, OPN_C2_RD_MIN_CTAS) k_celt2_rangedec(SymbolArgs A)
{
    __shared__ uint32_t s_lfl[21][LAP_N + 1], s_lfs[21][LAP_N + 1];
    __shared__ int16_t s_e9[2 * 21][RANGEDEC_WARPS_PER_CTA * 32];  // band energies, one column per packet
    const uint32_t lane = threadIdx.x;
    const int C = A.channels;
    int lm = A.lm;
    if (A.item_lm) {  // mixed-frame step, as in k_synth_rangedec
        const uint32_t l = A.item_lm[blockIdx.x * C2_RD_ITEMS_PER_CTA];
        if (l == MIX_NO_ITEM) return;
        lm = (int)l;
    }
    if (lane < 21u) {
        const uint32_t decay = 6000u + 400u * lane;
        const uint32_t fs0 = ((32768u - 33u) * (16384u - decay)) / (16384u + decay) + 1u;
        laplace_table(fs0, decay, s_lfl[lane], s_lfs[lane]);
    }
    __syncthreads();
    if ((lane & 31u) >= C2_RD_LANES) return;
    const uint32_t item = blockIdx.x * C2_RD_ITEMS_PER_CTA + (lane >> 5) * C2_RD_LANES + (lane & 31u);
    if (item >= A.n_items) return;
    if (A.item_lm && A.item_lm[item] == MIX_NO_ITEM) return;
    const uint32_t stream = A.stream_idx ? A.stream_idx[item] : item;
    uint32_t len = A.lens[item];
    const uint8_t *src = A.arena + A.offsets[item];
    int32_t status = len == 0u ? ITEM_LOST : ITEM_OK;
    if (A.has_toc && len > 0u) {
        const uint32_t toc = __ldg(src);
        if ((toc & 0x80u) == 0u) status = OPN_ERR_UNIMPLEMENTED;
        else if ((toc & 0x3u) != 0u) status = OPN_ERR_UNIMPLEMENTED;
        else if ((int)((toc >> 3) & 0x3u) != lm) status = OPN_ERR_FRAME_SIZE_TOO_SMALL;
        else if (((toc & 0x4u) ? 2 : 1) != C) status = OPN_ERR_UNIMPLEMENTED;
        src += 1;
        len -= 1u;
    }
    if (status == ITEM_OK && len <= 1u) status = ITEM_LOST;
    Celt2Side *sd = A.side2 ? A.side2 + stream : nullptr;
    if (sd) {
        uint32_t *sw = reinterpret_cast<uint32_t *>(sd);
        for (uint32_t i = 0; i < sizeof(Celt2Side) / 4u; i++) sw[i] = 0u;
    }
    if (status != ITEM_OK) {
        A.status[stream] = status;
        if (status == ITEM_LOST) A.hdr[stream] = make_uint4(0u, 0u, 0u, 0u);
        return;
    }
    LaneCoder ec;
    ec.lfl = s_lfl;
    ec.lfs = s_lfs;
    ec.d.init(src, len);
    LanePartSink sink{A.parts + (size_t)stream * CELT2_MAX_PARTS, 0u, 0u, 0u, &s_e9[0][lane], RANGEDEC_WARPS_PER_CTA * 32u};
    for (int i = 0; i < 2 * 21; i++) s_e9[i][lane] = 0;
    uint32_t flags = 0u, n_pulses = 0u;
    celt2_frame(ec, device_celt2_tabs(), len, lm, C, sd, sink, flags, n_pulses);
    if (A.bande) {
        uint32_t *be = reinterpret_cast<uint32_t *>(A.bande + (size_t)stream * 42);
        for (int i = 0; i < 21; i++) be[i] = (uint32_t)(uint16_t)s_e9[2 * i][lane] | (uint32_t)(uint16_t)s_e9[2 * i + 1][lane] << 16;
    }
    const uint32_t tf = ec.d.tell_frac();
    if (sd) {
        sd->n_parts = sink.n - sink.nsign;  // PVQ leaves (the list also holds the one-bin bands)
        sd->n_pulses = n_pulses;
        sd->final_rng = ec.d.rng;
        sd->tell_frac = tf;
    }
    if (sink.n > (uint32_t)CELT2_MAX_PARTS) status = OPN_ERR_INTERNAL;  // more leaves than the list holds: reject the packet, state untouched
    A.status[stream] = status;
    A.hdr[stream] = make_uint4(flags, ec.d.rng, tf, sink.n);
}

// Expansion of a SYNTH-CELT/2 part list by one warp: the leaves are dealt to the lanes round-robin; a lane walks its leaf
// with cwrsi_events (any (n, K): the walk itself falls back where its 32-bit sums could wrap), writes the pulses as
// floats and scales the leaf by gain / sqrt(yy) once the norm is known.  `rows` must be zero on entry.
// `bande`: the packet's band energies (Q9, [2][21]).  denormalise_bands: the decoded band has unit norm (times the split
// gains), its energy gives it its level -- every coefficient of band b, channel c is then multiplied by 2^(bande[c][b]/512).
template <int C>
__device__ __forceinline__ void w_expand2(const ExpandTables &T, int lm, uint32_t lane, const Celt2Part *__restrict__ parts, uint32_t n_parts,
                                          const int16_t *__restrict__ bande, float *rows, int chs, int32_t *__restrict__ y_out, int lmt = 0)
{
    const int nf = 120 << lm;
    for (uint32_t p = lane; p < n_parts; p += 32u) {
        const Celt2Part P = parts[p];
        const uint32_t pos = P.base & (uint32_t)C2_POS_MASK, band = P.base >> C2_BAND_SHIFT;
        const uint32_t ch = pos >= (uint32_t)nf ? 1u : 0u;
        const uint32_t bin0 = pos - ch * (uint32_t)nf;  // first bin of the leaf inside its channel
        float *dst = rows + ch * (uint32_t)chs;         // bin j of the channel lives at dst[block_major(j)]
        int32_t *yo = y_out ? y_out + pos : nullptr;
        const float bg = c2_band_gain(g_exp2_q9, (int)bande[ch * 21u + band]);
        if (P.n == 1u) {  // sign-only band
            dst[block_major(bin0, lmt, nf)] = (P.index ? -P.gain : P.gain) * bg;
            if (yo) yo[0] = P.index ? -1 : 1;
            continue;
        }
        const int32_t yy = cwrsi_events(T.U, T.CW, T.row, T.nmax, (uint32_t)P.n, (uint32_t)P.k, P.index, [&](uint32_t at, int32_t val) {
            dst[block_major(bin0 + at, lmt, nf)] = (float)val;
            if (yo) yo[at] = val;
        });
        const float g = P.gain / sqrtf((float)yy);
        for (uint32_t j = 0; j < P.n; j++) {
            float *q = dst + block_major(bin0 + j, lmt, nf);
            const float v = *q;
            if (v != 0.0f) *q = (v * g) * bg;  // normalised coefficient, then the band's gain
        }
    }
}

// Stand-alone expansion of part lists (operator entry opn_op_celt2_symbols): coefficient rows and pulses to global memory.
__global__ void __launch_bounds__(128) k_celt2_expand(SymbolArgs A)
{
    extern __shared__ __align__(16) float s_rows_all[];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const int lm = A.lm, C = A.channels, nf = 120 << lm;
    float *rows = s_rows_all + (size_t)warp * 2 * 960;
    const uint32_t item = blockIdx.x * 4u + warp;
    if (item >= A.n_items) return;
    const uint32_t stream = A.stream_idx ? A.stream_idx[item] : item;
    const int32_t status = A.status[stream];
    if (status < 0) return;
    const uint4 hdr = A.hdr[stream];
    const int nvec = C * nf / 4;
    for (int i = lane; i < nvec; i += 32) reinterpret_cast<float4 *>(rows)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    int32_t *yo = A.y_out ? A.y_out + (size_t)stream * C * nf : nullptr;
    if (yo)
        for (int i = lane; i < nvec; i += 32) reinterpret_cast<int4 *>(yo)[i] = make_int4(0, 0, 0, 0);
    __syncwarp();
    if (status == ITEM_OK && !(hdr.x & 1u)) {
        const ExpandTables T{g_tab.pvq_u_data, g_tab.pvq_cw_data, g_tab.pvq_u_row, g_tab.pvq_ev_nmax, nullptr, nullptr, 0};
        if (C == 2) w_expand2<2>(T, lm, lane, A.parts + (size_t)stream * CELT2_MAX_PARTS, hdr.w, A.bande + (size_t)stream * 42, rows, nf, yo);
        else w_expand2<1>(T, lm, lane, A.parts + (size_t)stream * CELT2_MAX_PARTS, hdr.w, A.bande + (size_t)stream * 42, rows, nf, yo);
    }
    __syncwarp();
    if (A.coef) {
        float4 *coef4 = reinterpret_cast<float4 *>(A.coef + (size_t)stream * C * nf);
        for (int i = lane; i < nvec; i += 32) coef4[i] = reinterpret_cast<const float4 *>(rows)[i];
    }
}

}  // namespace opn
