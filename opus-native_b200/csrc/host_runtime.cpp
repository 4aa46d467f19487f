// host_runtime.cpp -- C-ABI entry points and the host runtime of libopusb200.
//
// Mirrors the reference's decode-path surface (src/decoder.rs): `opn_decoder` stands in for
// `Decoder` (decode_native / decode_frame orchestration stays on the host, exactly as in the
// crate: it is control flow over 1-3 header bytes), and `opn_batch` is the batch-of-streams
// entry point: per-GPU context, per-stream state arenas in HBM (structure of arrays), pinned
// staging and two kernels per step.  There is no CPU decode path in this library.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>  // header-only: ranges cost a predicted branch unless a profiler has attached

#include "opn_internal.h"
#include "celt2.cuh"

using namespace opn;

namespace {

thread_local std::string g_cuda_err;

int cuda_fail(cudaError_t e, const char *what)
{
    char buf[256];
    std::snprintf(buf, sizeof(buf), "%s: %s", what, cudaGetErrorString(e));
    g_cuda_err = buf;
    return OPN_ERR_CUDA;
}

#define CU(call)                                          \
    do {                                                  \
        cudaError_t e_ = (call);                          \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call); \
    } while (0)

int lm_of_frame(size_t nf)
{
    switch (nf) {
    case 120: return 0;
    case 240: return 1;
    case 480: return 2;
    case 960: return 3;
    default: return -1;
    }
}

int select_device(int device)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount");
    if (n == 0 || device < 0 || device >= n) return cuda_fail(cudaErrorInvalidDevice, "no such CUDA device");
    CU(cudaSetDevice(device));
    cudaDeviceProp p;
    CU(cudaGetDeviceProperties(&p, device));
    if (p.major < 10) {
        g_cuda_err = std::string("device '") + p.name + "' is not sm_100-class; libopusb200 ships sm_100a code only";
        return OPN_ERR_CUDA;
    }
    CU(upload_tables(device));
    return OPN_OK;
}

struct EventRing {
    static constexpr int N = 512;
    cudaEvent_t a[N], b[N];
    int used = 0;
    bool made = false;
    double ms = 0.0;
    uint64_t launches = 0;
    int make()
    {
        if (made) return OPN_OK;
        for (int i = 0; i < N; i++) {
            CU(cudaEventCreate(&a[i]));
            CU(cudaEventCreate(&b[i]));
        }
        made = true;
        return OPN_OK;
    }
    int resolve()
    {
        for (int i = 0; i < used; i++) {
            CU(cudaEventSynchronize(b[i]));
            float t = 0;
            CU(cudaEventElapsedTime(&t, a[i], b[i]));
            ms += t;
        }
        used = 0;
        return OPN_OK;
    }
    void destroy()
    {
        if (!made) return;
        for (int i = 0; i < N; i++) {
            cudaEventDestroy(a[i]);
            cudaEventDestroy(b[i]);
        }
        made = false;
    }
};

struct Item {
    uint32_t stream, offset, len, dense_off;
    int lm, wave;
    int cs;  // channels of the packet (stream_channels, decoder.rs:332); concealed frames: the decoder's
};

}  // namespace

struct opn_batch {
    int device = 0;
    uint32_t n = 0;
    opn_config cfg{};
    float gain = 1.0f;
    cudaStream_t stream = nullptr;
    // One step = two launches: the range decode (k_synth_rangedec: one lane per packet, a latency-bound serial chain on a
    // few hundred warps) and the frame kernel (k_frame_w: PVQ expansion + IMDCT + post-filter + PCM store, one warp per
    // stream).  The range decode runs on its own streams and may run up to NSETS-1 steps ahead of the frame kernel: its
    // outputs (frame header, status, codeword indices: 308 bytes per stream) live in NSETS buffer sets handed over with
    // events.
#ifndef OPN_NSETS
#define OPN_NSETS 8
#endif
#ifndef OPN_NRD
#define OPN_NRD 8
#endif
    static constexpr int NSETS = OPN_NSETS, NRD = OPN_NRD;
    cudaStream_t stream_rd[NRD] = {};     // set p decodes on stream_rd[p % NRD]: entropy stages of NRD steps overlap each other
    cudaStream_t stream_mix = nullptr;    // bucketing of mixed-frame steps (k_mix_key / k_mix_place), ahead of their range decodes
    // A large bucket's frame kernel is cut into NGROUPS launches over contiguous stream ranges, group g on stream_fr[g]
    // (stream_fr[0] is `stream`).  A stream's frames stay in order (its group's stream), but the tail of one group's launch
    // overlaps the body of the other's, and step n+1 of a group may start while step n of the other is still running:
    // the SMs never drain between steps.  Measured at 4096 stereo 20 ms streams (tools/experiments/variants.sh, us per
    // step): 1 group 71-72, 2 groups 46.3, 3 groups 44.1-44.8, 4 groups 49.
#ifndef OPN_FRAME_GROUPS
#define OPN_FRAME_GROUPS 3
#endif
    static constexpr int NGROUPS = OPN_FRAME_GROUPS;
    static constexpr uint32_t GROUP_MIN_ITEMS = 2048;  // smaller batches run the frame kernel as one launch on `stream`
    cudaStream_t stream_fr[NGROUPS] = {};
    cudaEvent_t ev_fr[NSETS][NGROUPS] = {};  // frame kernel of set p, group g finished
    cudaEvent_t ev_sw = nullptr;             // mode switch: everything enqueued on `stream` so far
    bool fr_pending[NGROUPS] = {};           // group g >= 1 has work that `stream` has not been ordered after yet
    int fr_last_set[NGROUPS] = {};
    cudaEvent_t ev_k1[NSETS] = {};        // frame kernel(s) of set p finished on `stream` (group 0 / ungrouped): the set is free again
    bool k1_recorded[NSETS] = {};
    bool k1_grouped[NSETS] = {};          // set p was last used by a grouped launch: ev_fr[p][1..] are part of "set p is free"
    cudaEvent_t ev_rd[NSETS] = {};        // range decode of set p finished
    cudaEvent_t ev_in = nullptr;          // inputs ordered on `stream` / `stream_up` are complete
    static constexpr int MAX_CHUNKS = 8;
    cudaStream_t stream_up = nullptr, stream_dn = nullptr;  // host path: item/packet upload, PCM download
    cudaEvent_t ev_chunk[MAX_CHUNKS] = {};                  // frame kernels (and epilogue) of a chunk finished
    int set = 0;
    // per-stream state (device, SoA)
    float *d_carry = nullptr, *d_ring = nullptr;
    uint32_t *d_ring_pos = nullptr, *d_final = nullptr, *d_idx[NSETS] = {};
    PfState *d_pf = nullptr;
    uint4 *d_hdr[NSETS] = {};
    int32_t *d_status[NSETS] = {};
    Celt2Part *d_parts[NSETS] = {};  // SYNTH-CELT/2 batches only: PVQ leaves per stream
    int16_t *d_bande[NSETS] = {};    // SYNTH-CELT/2 batches only: band energies per stream, Q9 [2][21]
    // host-path staging (device + pinned host)
    // Two staging slots, so a host-buffer call can be submitted while the previous one is still downloading.
    struct Staging {
        uint8_t *d_arena = nullptr;
        size_t arena_cap = 0;
        uint32_t *d_items = nullptr, *h_items = nullptr;  // per chunk: [offsets | lens | stream ids | dense offsets]
        size_t items_cap = 0;
        float *d_dense = nullptr;
        size_t dense_cap = 0;          // floats per stream
        void *d_conv = nullptr;        // converted rows (decode::<S> calls), conv_cap samples of conv_esize bytes per stream
        size_t conv_cap = 0, conv_esize = 0;
        int32_t *d_cliplen = nullptr, *h_cliplen = nullptr;  // [n] soft-clip slice length per stream
        uint32_t *d_trans = nullptr, *h_trans = nullptr;       // [n] streams that switch from CELT to SILK in this call
        cudaEvent_t done = nullptr;    // everything that uses this slot has finished (incl. the PCM download)
        bool pending = false;
    } stg[2];
    int stg_next = 0;
    float *d_softclip = nullptr;
    // mixed-frame steps (OPN_FLAG_MIXED_FRAMES), allocated on first use: the step's buckets are built on the device
    // (k_mix_key / k_mix_place on stream_mix, in step order) into one item table + plan per buffer set
    uint8_t *d_last_lm = nullptr, *d_mix_key = nullptr;  // [n] state: LM of the last decoded packet; scratch: bucket of the stream
    uint32_t *d_mix_rank = nullptr;                      // [n] scratch
    uint32_t *d_mix_items[NSETS] = {};                   // [3][mix_item_cap(n)]: offsets | lens | stream ids, by item
    uint8_t *d_mix_lm[NSETS] = {};                       // [mix_item_cap(n)]
    MixPlan *d_mix_plan[NSETS] = {};
    cudaEvent_t ev_mix[NSETS] = {};                      // buckets of set p are built
    // SYNTH-SILK/1 (OPN_BITSTREAM_SYNTH_SILK_1): per-stream filter state and one record set per range decode in flight
    bool silk = false;
    SilkState d_silk{};
    SilkRec *d_silk_rec[NSETS] = {};
    std::vector<uint8_t> silk_cs;  // host mirror: coded channels of the stream's last SILK frame (0 = none)
    unsigned long long *d_hist_samples = nullptr;  // measurement: history samples the post-filter needed (timed passes only)
    // host mirrors of DecoderInner fields (decoder.rs:236-258), per stream
    std::vector<int32_t> last_nf, bandwidth, last_duration, have_mode;
    // measurement
    bool timing = false;
    EventRing ev[3];
    uint64_t launches[3] = {0, 0, 0};
};

namespace {

// NVTX range for the host-side stages of a call (visible in Nsight Systems timelines next to the kernels)
struct Range {
    explicit Range(const char *name) { nvtxRangePushA(name); }
    ~Range() { nvtxRangePop(); }
    Range(const Range &) = delete;
    Range &operator=(const Range &) = delete;
};

int batch_alloc_staging(opn_batch *b, opn_batch::Staging &g, size_t arena_bytes, size_t n_items, size_t dense_floats, size_t conv_esize)
{
    if (!g.done) CU(cudaEventCreateWithFlags(&g.done, cudaEventDisableTiming));
    if (arena_bytes > g.arena_cap) {
        if (g.d_arena) cudaFree(g.d_arena);
        g.arena_cap = arena_bytes + arena_bytes / 4 + 256;
        CU(cudaMalloc(&g.d_arena, g.arena_cap));
    }
    if (n_items > g.items_cap) {
        if (g.d_items) cudaFree(g.d_items);
        if (g.h_items) cudaFreeHost(g.h_items);
        g.items_cap = n_items + n_items / 4 + 64;
        CU(cudaMalloc(&g.d_items, g.items_cap * 4 * sizeof(uint32_t)));
        CU(cudaMallocHost(&g.h_items, g.items_cap * 4 * sizeof(uint32_t)));
    }
    if (dense_floats > g.dense_cap) {
        if (g.d_dense) cudaFree(g.d_dense);
        g.dense_cap = dense_floats;
        // a SILK-capable batch keeps 5 ms per stream BEHIND the rows (at n * dense_cap + 240 C i): the transition buffer of a
        // CELT -> SILK switch (decoder.rs:519-543); the rows themselves stay contiguous for the PCM download
        CU(cudaMalloc(&g.d_dense, (size_t)b->n * (g.dense_cap + (b->silk ? 240 * (size_t)b->cfg.channels : 0)) * sizeof(float)));
    }
    if (conv_esize && (g.dense_cap > g.conv_cap || conv_esize > g.conv_esize)) {
        if (g.d_conv) cudaFree(g.d_conv);
        g.d_conv = nullptr;
        g.conv_cap = g.dense_cap;
        g.conv_esize = std::max(conv_esize, g.conv_esize);
        CU(cudaMalloc(&g.d_conv, (size_t)b->n * g.conv_cap * g.conv_esize));
    }
    if (conv_esize && !g.d_cliplen) {
        CU(cudaMalloc(&g.d_cliplen, (size_t)b->n * sizeof(int32_t)));
        CU(cudaMallocHost(&g.h_cliplen, (size_t)b->n * sizeof(int32_t)));
    }
    return OPN_OK;
}

// Runs `launch`, which enqueues one stage of a step.  In a timed pass the stage sits between two events on `stream`, so
// whatever it enqueues on other streams must be joined back onto `stream` before it returns.
template <class F> int timed_launch(opn_batch *b, int kind, F &&launch)
{
    EventRing &r = b->ev[kind];
    if (b->timing) {
        if (r.used == EventRing::N) {
            int rc = r.resolve();
            if (rc) return rc;
        }
        CU(cudaEventRecord(r.a[r.used], b->stream));
    }
    int rc = launch();
    if (rc) return rc;
    if (b->timing) {
        CU(cudaEventRecord(r.b[r.used], b->stream));
        r.used++;
        r.launches++;
    }
    return OPN_OK;
}

// Orders `stream` after everything the other frame groups have been given so far.
int join_groups(opn_batch *b)
{
    for (int g = 1; g < opn_batch::NGROUPS; g++)
        if (b->fr_pending[g]) {
            CU(cudaStreamWaitEvent(b->stream, b->ev_fr[b->fr_last_set[g]][g], 0));
            b->fr_pending[g] = false;
        }
    return OPN_OK;
}

int sync_pipeline(opn_batch *b)
{
    for (int q = 0; q < opn_batch::NRD; q++) CU(cudaStreamSynchronize(b->stream_rd[q]));
    CU(cudaStreamSynchronize(b->stream_mix));
    for (int g = 1; g < opn_batch::NGROUPS; g++) {
        CU(cudaStreamSynchronize(b->stream_fr[g]));
        b->fr_pending[g] = false;
    }
    CU(cudaStreamSynchronize(b->stream_up));
    CU(cudaStreamSynchronize(b->stream));
    CU(cudaStreamSynchronize(b->stream_dn));
    return OPN_OK;
}

// A timed pass runs every stage of a step in order on `stream`.
cudaStream_t rd_stream(const opn_batch *b, int p) { return b->timing ? b->stream : b->stream_rd[p % opn_batch::NRD]; }
cudaStream_t mix_stream(const opn_batch *b) { return b->timing ? b->stream : b->stream_mix; }

// Makes `to` wait for everything enqueued on `from` so far.
int order_after(cudaEvent_t ev, cudaStream_t from, cudaStream_t to)
{
    if (from == to) return OPN_OK;
    CU(cudaEventRecord(ev, from));
    CU(cudaStreamWaitEvent(to, ev, 0));
    return OPN_OK;
}

// Start of a step: claims buffer set p and returns it (or an error).  The stream of the step's first kernel -- the
// bucketing stream of a mixed-frame step, else the range-decode stream of set p -- is ordered after the step's inputs and
// waits until set p is free again: the frame kernels of the step that used it last have finished.
// inputs_on: 0 = the packets are already complete in device memory (the step may start at once),
//            1 = they are ordered on b->stream, 2 = they are ordered on b->stream_up (host path).
int begin_step(opn_batch *b, bool mixed, int inputs_on)
{
    const int p = b->set;
    b->set = (p + 1) % opn_batch::NSETS;
    const cudaStream_t first = mixed ? mix_stream(b) : rd_stream(b, p);
    if (inputs_on) {
        const int rc = order_after(b->ev_in, inputs_on == 1 ? b->stream : b->stream_up, first);
        if (rc) return rc;
    }
    if (b->k1_recorded[p] && first != b->stream) {  // ev_k1[p] and the groups it joined are behind `stream` already
        CU(cudaStreamWaitEvent(first, b->ev_k1[p], 0));
        if (b->k1_grouped[p])
            for (int g = 1; g < opn_batch::NGROUPS; g++) CU(cudaStreamWaitEvent(first, b->ev_fr[p][g], 0));
    }
    return p;
}

// The range decode of a step on buffer set p: launch(st) enqueues it on st; ev_rd[p] marks its end.
template <class F> int range_decode(opn_batch *b, int p, F &&launch)
{
    const cudaStream_t srd = rd_stream(b, p);
    const int rc = timed_launch(b, 0, [&]() -> int {
        CU(launch(srd));
        return OPN_OK;
    });
    if (rc) return rc;
    CU(cudaEventRecord(b->ev_rd[p], srd));
    b->launches[0]++;
    return OPN_OK;
}

// streams [group_first(n, g, G), group_first(n, g + 1, G)) of n are group g of G
uint32_t group_first(uint32_t n, int g, int G) { return (uint32_t)((uint64_t)n * (uint32_t)g / (uint32_t)G); }

// The number of launches a step's frame kernel is cut into.  A device-resident step (item k = stream k) of a large batch
// runs as NGROUPS launches, group g over items [group_first(n, g, G), group_first(n, g + 1, G)); a host-path bucket (any
// subset of the streams, in any order) runs as one.
int frame_groups(const opn_batch *b, bool device_step)
{
    return device_step && b->n >= opn_batch::GROUP_MIN_ITEMS ? opn_batch::NGROUPS : 1;
}

// The frame kernel of a step on buffer set p, after its range decode: launch(g, st) enqueues group g of G on st.  One group
// runs on `stream` after whatever the other groups' streams hold.  G groups: group 0 on `stream`, the others on their
// own streams, each after its own previous frames (stream order), this step's range decode and whatever `stream` held
// when the groups were last joined.  A timed pass joins them again before its end event.
template <class F> int frame_launches(opn_batch *b, int p, int G, F &&launch)
{
    const int rc = timed_launch(b, 1, [&]() -> int {
        if (G == 1) {
            const int rc = join_groups(b);  // streams of the other groups' ranges may be in this bucket
            if (rc) return rc;
            CU(cudaStreamWaitEvent(b->stream, b->ev_rd[p], 0));
            CU(launch(0, b->stream));
            b->launches[1]++;
            return OPN_OK;
        }
        CU(cudaEventRecord(b->ev_sw, b->stream));
        for (int g = 0; g < G; g++) {
            const cudaStream_t st = g == 0 ? b->stream : b->stream_fr[g];
            if (g > 0 && !b->fr_pending[g]) CU(cudaStreamWaitEvent(st, b->ev_sw, 0));
            CU(cudaStreamWaitEvent(st, b->ev_rd[p], 0));
            CU(launch(g, st));
            b->launches[1]++;
            if (g > 0) {
                CU(cudaEventRecord(b->ev_fr[p][g], st));
                b->fr_pending[g] = true;
                b->fr_last_set[g] = p;
            }
        }
        return b->timing ? join_groups(b) : OPN_OK;
    });
    if (rc) return rc;
    CU(cudaEventRecord(b->ev_k1[p], b->stream));
    b->k1_recorded[p] = true;
    b->k1_grouped[p] = G > 1;
    return OPN_OK;
}

// One bucket = items of equal frame size that may run concurrently.
// softclip_reset: a float call clears the soft-clip memory of every stream that decodes a packet (decoder.rs:420-423).
int run_bucket(opn_batch *b, const uint8_t *d_arena, const uint32_t *d_offsets, const uint32_t *d_lens,
               const uint32_t *d_stream_idx, const uint32_t *d_dense_off, uint32_t n_items, int lm, int has_toc,
               uint32_t pkt_cap, float *dense, size_t dense_stride, int32_t *d_result, int inputs_on, bool softclip_reset,
               int stream_channels = 0)
{
    Range nv("opn: step (range decode + frame kernel)");
    if (stream_channels == 0) stream_channels = b->cfg.channels;
    const int p = begin_step(b, false, inputs_on);
    if (p < 0) return p;
    SymbolArgs s{};
    s.arena = d_arena;
    s.offsets = d_offsets;
    s.lens = d_lens;
    s.stream_idx = d_stream_idx;
    s.n_items = n_items;
    s.lm = lm;
    s.channels = stream_channels;  // the range decode follows the packets' layout
    s.has_toc = has_toc;
    s.hdr = b->d_hdr[p];
    s.status = b->d_status[p];
    s.idx = b->d_idx[p];
    s.pkt_cap = pkt_cap;
    s.parts = b->d_parts[p];
    s.bande = b->d_bande[p];
    const bool celt2 = b->cfg.bitstream == OPN_BITSTREAM_SYNTH_CELT_2;
    int rc = range_decode(b, p, [&](cudaStream_t st) { return celt2 ? launch_celt2_rangedec(s, st) : launch_synth_rangedec(s, st); });
    if (rc) return rc;
    FrameArgs m{};
    m.idx = celt2 ? nullptr : b->d_idx[p];
    m.parts = celt2 ? b->d_parts[p] : nullptr;
    m.bande = b->d_bande[p];
    m.hdr = b->d_hdr[p];
    m.status = b->d_status[p];
    m.stream_idx = d_stream_idx;
    m.dense_off = d_dense_off;
    m.n_items = n_items;
    m.lm = lm;
    m.channels = b->cfg.channels;
    m.stream_channels = stream_channels;
    m.postfilter = b->cfg.postfilter;
    m.carry = b->d_carry;
    m.ring = b->d_ring;
    m.ring_pos = b->d_ring_pos;
    m.pf = b->d_pf;
    m.dense = dense;
    m.dense_stride = dense_stride;
    m.gain = b->gain;
    m.result = d_result;
    m.final_range = b->d_final;
    m.softclip_reset = softclip_reset ? b->d_softclip : nullptr;
    m.hist_samples = b->timing ? b->d_hist_samples : nullptr;
    const int G = frame_groups(b, !d_stream_idx);
    return frame_launches(b, p, G, [&](int g, cudaStream_t st) {
        m.item0 = group_first(n_items, g, G);
        m.item_end = group_first(n_items, g + 1, G);
        return launch_frame(m, st);
    });
}

// One bucket of SILK-only frames (SYNTH-SILK/1) of one duration and one coded channel count: the range decode on an entropy
// stream (it may run ahead like the CELT one), the frame kernel on the batch stream (it owns the streams' filter state and
// the PCM ring).  bandwidth < 0: read from each packet's TOC (has_toc).
int run_silk_bucket(opn_batch *b, const uint8_t *d_arena, const uint32_t *d_offsets, const uint32_t *d_lens, const uint32_t *d_stream_idx,
                    const uint32_t *d_dense_off, uint32_t n_items, int frame_ms, int has_toc, int bandwidth, int stream_channels,
                    float *dense, size_t dense_stride, int32_t *d_result, int inputs_on, bool softclip_reset, int fec = 0)
{
    Range nv("opn: SILK step (range decode + frame kernel)");
    if (!b->silk) return OPN_ERR_UNIMPLEMENTED;  // silk/decoder.rs:79
    const int p = begin_step(b, false, inputs_on);
    if (p < 0) return p;
    SilkArgs a{};
    a.arena = d_arena;
    a.offsets = d_offsets;
    a.lens = d_lens;
    a.stream_idx = d_stream_idx;
    a.n_items = n_items;
    a.frame_ms = frame_ms;
    a.stream_channels = stream_channels;
    a.channels = b->cfg.channels;
    a.has_toc = has_toc;
    a.bandwidth = bandwidth;
    a.fec = fec;
    a.rec = b->d_silk_rec[p];
    a.hdr = b->d_hdr[p];
    a.status = b->d_status[p];
    a.st = b->d_silk;
    a.ring = b->d_ring;
    a.ring_pos = b->d_ring_pos;
    a.dense = dense;
    a.dense_stride = dense_stride;
    a.dense_off = d_dense_off;
    a.gain = b->gain;
    a.result = d_result;
    a.final_range = b->d_final;
    a.softclip_reset = softclip_reset ? b->d_softclip : nullptr;
    int rc = range_decode(b, p, [&](cudaStream_t st) { return launch_silk_rangedec(a, st); });
    if (rc) return rc;
    // Groups as for the CELT frame kernel: the serial LPC phase of one group's CTAs then overlaps the parallel phases of the
    // others'.  A timed pass launches the SILK frame kernel once.
    const int G = b->timing ? 1 : frame_groups(b, !d_stream_idx);
    return frame_launches(b, p, G, [&](int g, cudaStream_t st) {
        a.item0 = group_first(n_items, g, G);
        a.item_end = group_first(n_items, g + 1, G);
        return launch_silk_frame(a, st);
    });
}

int mix_alloc(opn_batch *b)
{
    if (b->d_last_lm) return OPN_OK;
    const size_t n = b->n, cap = mix_item_cap(b->n);
    CU(cudaMalloc(&b->d_mix_key, n));
    CU(cudaMalloc(&b->d_mix_rank, n * sizeof(uint32_t)));
    for (int q = 0; q < opn_batch::NSETS; q++) {
        CU(cudaMalloc(&b->d_mix_items[q], 3 * cap * sizeof(uint32_t)));
        CU(cudaMalloc(&b->d_mix_lm[q], cap));
        CU(cudaMalloc(&b->d_mix_plan[q], sizeof(MixPlan)));
        CU(cudaEventCreateWithFlags(&b->ev_mix[q], cudaEventDisableTiming));
    }
    uint8_t *p = nullptr;
    CU(cudaMalloc(&p, n));
    CU(cudaMemsetAsync(p, MIX_NO_ITEM, n, b->stream_mix));
    CU(cudaStreamSynchronize(b->stream_mix));  // a timed pass buckets on `stream`
    b->d_last_lm = p;
    return OPN_OK;
}

// One step whose streams may have different frame sizes (device-resident: one single-frame packet or a loss per stream).
// The step's buckets are built on the device, so the host never learns the sizes: the range decode is ONE launch over the
// padded item table, the frame kernel one k_frame_mix launch per group, each sized by its upper bound.
int run_mixed(opn_batch *b, const uint8_t *d_arena, const uint32_t *d_offsets, const uint32_t *d_lens, size_t capacity, float *dense,
              size_t dense_stride, int32_t *d_result, int inputs_on, bool softclip_reset)
{
    Range nv("opn: mixed-frame step (bucketing + range decode + frame kernel)");
    int rc = mix_alloc(b);
    if (rc) return rc;
    const int p = begin_step(b, true, inputs_on);
    if (p < 0) return p;
    const uint32_t cap = mix_item_cap(b->n);
    const int G = frame_groups(b, true);
    MixArgs x{};
    x.arena = d_arena;
    x.offsets = d_offsets;
    x.lens = d_lens;
    x.n_streams = b->n;
    x.channels = b->cfg.channels;
    x.n_groups = G;
    x.capacity = (uint32_t)std::min<size_t>(capacity, 1u << 20);
    x.last_lm = b->d_last_lm;
    x.key = b->d_mix_key;
    x.rank = b->d_mix_rank;
    x.plan = b->d_mix_plan[p];
    x.item_offsets = b->d_mix_items[p];
    x.item_lens = b->d_mix_items[p] + cap;
    x.item_stream = b->d_mix_items[p] + 2 * (size_t)cap;
    x.item_lm = b->d_mix_lm[p];
    x.result = d_result;
    SymbolArgs s{};
    s.arena = d_arena;
    s.offsets = x.item_offsets;
    s.lens = x.item_lens;
    s.stream_idx = x.item_stream;
    s.item_lm = x.item_lm;
    s.n_items = cap;
    s.lm = 0;
    s.channels = b->cfg.channels;
    s.has_toc = 1;
    s.hdr = b->d_hdr[p];
    s.status = b->d_status[p];
    s.idx = b->d_idx[p];
    s.pkt_cap = 1280u;
    s.parts = b->d_parts[p];
    s.bande = b->d_bande[p];
    const bool celt2 = b->cfg.bitstream == OPN_BITSTREAM_SYNTH_CELT_2;
    FrameArgs m{};
    m.idx = celt2 ? nullptr : b->d_idx[p];
    m.parts = celt2 ? b->d_parts[p] : nullptr;
    m.bande = b->d_bande[p];
    m.hdr = b->d_hdr[p];
    m.status = b->d_status[p];
    m.stream_idx = x.item_stream;
    m.n_items = cap;
    m.channels = b->cfg.channels;
    m.postfilter = b->cfg.postfilter;
    m.carry = b->d_carry;
    m.ring = b->d_ring;
    m.ring_pos = b->d_ring_pos;
    m.pf = b->d_pf;
    m.dense = dense;
    m.dense_stride = dense_stride;
    m.gain = b->gain;
    m.result = d_result;
    m.final_range = b->d_final;
    m.softclip_reset = softclip_reset ? b->d_softclip : nullptr;
    m.hist_samples = b->timing ? b->d_hist_samples : nullptr;
    m.plan = b->d_mix_plan[p];
    CU(launch_mix_plan(x, mix_stream(b)));
    b->launches[2] += 2;
    rc = order_after(b->ev_mix[p], mix_stream(b), rd_stream(b, p));
    if (rc) return rc;
    rc = range_decode(b, p, [&](cudaStream_t st) { return celt2 ? launch_celt2_rangedec(s, st) : launch_synth_rangedec(s, st); });
    if (rc) return rc;
    return frame_launches(b, p, G, [&](int g, cudaStream_t st) {
        m.group = g;
        return launch_frame_mix(m, group_first(b->n, g + 1, G) - group_first(b->n, g, G), st);
    });
}

// PLC sizing of decode_native(None)/decode_frame(None), src/decoder.rs:427-441 and 467-513.
void plc_frames(size_t frame_size, int32_t last_nf, std::vector<uint32_t> &out)
{
    size_t done = 0;
    while (done < frame_size) {
        size_t a = std::min(frame_size - done, (size_t)last_nf);
        if (a > 960) a = 960;
        else if (a < 960) {
            if (a > 480) a = 480;
            else if (a > 240 && a < 480) a = 240;
        }
        out.push_back((uint32_t)a);
        done += a;
    }
}

}  // namespace

extern "C" {

const char *opn_strerror(int code)
{
    switch (code) {
    case OPN_OK: return "ok";
    case OPN_ERR_BAD_ARG: return "bad arguments";
    case OPN_ERR_BUFFER_TOO_SMALL: return "buffer is too small";
    case OPN_ERR_INTERNAL: return "internal error";
    case OPN_ERR_INVALID_PACKET: return "invalid packet";
    case OPN_ERR_FRAME_SIZE_TOO_SMALL: return "the frame size is too small for the packet";
    case OPN_ERR_UNIMPLEMENTED: return "not implemented (the reference crate stubs this path too)";
    case OPN_ERR_CUDA: return "CUDA error";
    default: return "unknown error";
    }
}

const char *opn_last_cuda_error(void) { return g_cuda_err.c_str(); }

int opn_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

// ------------------------------------------------------------------------------------ host memory
// The host-buffer entry points copy straight between the caller's buffers and the device.  With page-locked buffers
// those copies are asynchronous DMA at PCIe speed; with ordinary (pageable) memory -- what a Rust Vec or slice is --
// the CUDA runtime stages them through its own pinned bounce buffer, synchronously.  Both work; these helpers give a
// caller the fast kind.
void *opn_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (bytes == 0 || cudaMallocHost(&p, bytes) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void opn_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

int opn_host_register(void *p, size_t bytes)
{
    if (!p || bytes == 0) return OPN_ERR_BAD_ARG;
    CU(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return OPN_OK;
}

int opn_host_unregister(void *p)
{
    if (!p) return OPN_ERR_BAD_ARG;
    CU(cudaHostUnregister(p));
    return OPN_OK;
}

// ------------------------------------------------------------------------------------ batch
int opn_batch_create(int device, uint32_t n_streams, const opn_config *cfg, opn_batch **out)
{
    if (!out || !cfg || n_streams == 0) return OPN_ERR_BAD_ARG;
    if (cfg->channels < 1 || cfg->channels > 2) return OPN_ERR_BAD_ARG;
    if (cfg->bitstream & ~(OPN_BITSTREAM_CELT_MASK | OPN_BITSTREAM_SYNTH_SILK_1)) return OPN_ERR_BAD_ARG;
    const int32_t celt_bitstream = cfg->bitstream & OPN_BITSTREAM_CELT_MASK;
    if (celt_bitstream != OPN_BITSTREAM_OPUS && celt_bitstream != OPN_BITSTREAM_SYNTH_CELT_1 && celt_bitstream != OPN_BITSTREAM_SYNTH_CELT_2)
        return OPN_ERR_BAD_ARG;
    switch (cfg->fs_hz) {
    case 48000: break;
    case 8000: case 12000: case 16000: case 24000: return OPN_ERR_UNIMPLEMENTED;  // celt/decoder.rs:23 "TODO ... downsample"
    default: return OPN_ERR_BAD_ARG;
    }
    int rc = select_device(device);
    if (rc) return rc;
    if (kernels_frame_groups() != OPN_FRAME_GROUPS) return OPN_ERR_INTERNAL;  // kernels and runtime of different builds
    opn_batch *b = new (std::nothrow) opn_batch();
    if (!b) return OPN_ERR_INTERNAL;
    b->device = device;
    b->n = n_streams;
    b->cfg = *cfg;
    b->cfg.bitstream = celt_bitstream;  // how CELT frames are laid out; the SILK opt-in is b->silk
    b->silk = (cfg->bitstream & OPN_BITSTREAM_SYNTH_SILK_1) != 0;
    b->gain = host_gain_from_q8(cfg->gain_q8);
    const size_t n = n_streams, C = (size_t)cfg->channels;
    cudaError_t e = cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking);
    // All pipeline streams have the same priority (measured in round 1, tools/experiments/priorities.sh: raising the
    // entropy streams gave slow stretches, raising the frame stream serialised the pipeline).
    {
        // SYNTH-CELT/2: the range decode is the long pole (333 us per launch, 128 registers per thread): its streams run at
        // the highest priority, so that its CTAs are placed first whenever a frame-kernel CTA retires (125 -> 116 us per
        // step).  SYNTH-CELT/1: no difference in steady state (44.3 us either way), but a short burst loses 2-3 us per step
        // (20 steps after a drained pipeline: 47.9-49.2 us at equal priority, 50.2-52.5 with the range decodes of eight
        // steps placed ahead of the first frame kernels), so those keep the default.
        const bool high = celt_bitstream == OPN_BITSTREAM_SYNTH_CELT_2;
        int lo_p = 0, hi_p = 0;
        if (high) cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p);
        for (int q = 0; q < opn_batch::NRD && e == cudaSuccess; q++)
            e = cudaStreamCreateWithPriority(&b->stream_rd[q], cudaStreamNonBlocking, high ? hi_p : 0);
    }
    for (int q = 0; q < opn_batch::NSETS && e == cudaSuccess; q++) {
        e = cudaEventCreateWithFlags(&b->ev_rd[q], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ev_k1[q], cudaEventDisableTiming);
        for (int g = 1; g < opn_batch::NGROUPS && e == cudaSuccess; g++) e = cudaEventCreateWithFlags(&b->ev_fr[q][g], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaMalloc(&b->d_idx[q], n * 72 * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaMalloc(&b->d_hdr[q], n * sizeof(uint4));
        if (e == cudaSuccess && celt_bitstream == OPN_BITSTREAM_SYNTH_CELT_2) e = cudaMalloc(&b->d_parts[q], n * CELT2_MAX_PARTS * sizeof(Celt2Part));
        if (e == cudaSuccess && b->silk) e = cudaMalloc(&b->d_silk_rec[q], n * 2 * sizeof(SilkRec));
        if (e == cudaSuccess && celt_bitstream == OPN_BITSTREAM_SYNTH_CELT_2) e = cudaMalloc(&b->d_bande[q], n * 42 * sizeof(int16_t));
        if (e == cudaSuccess) e = cudaMalloc(&b->d_status[q], n * sizeof(int32_t));
    }
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&b->stream_mix, cudaStreamNonBlocking);
    for (int g = 1; g < opn_batch::NGROUPS && e == cudaSuccess; g++) e = cudaStreamCreateWithFlags(&b->stream_fr[g], cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ev_sw, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ev_in, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&b->stream_up, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&b->stream_dn, cudaStreamNonBlocking);
    for (int q = 0; q < opn_batch::MAX_CHUNKS && e == cudaSuccess; q++) e = cudaEventCreateWithFlags(&b->ev_chunk[q], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc(&b->d_carry, n * C * 60 * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&b->d_ring, n * C * RING_SAMPLES * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&b->d_ring_pos, n * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc(&b->d_final, n * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc(&b->d_pf, n * sizeof(PfState));
    if (e == cudaSuccess) e = cudaMalloc(&b->d_softclip, n * 2 * sizeof(float));
    if (b->silk) {
        if (e == cudaSuccess) e = cudaMalloc(&b->d_silk.slpc, n * 2 * 16 * sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMalloc(&b->d_silk.hist, n * 2 * SILK_HIST * sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMalloc(&b->d_silk.a_q12, n * 2 * 16 * sizeof(int16_t));
        if (e == cudaSuccess) e = cudaMalloc(&b->d_silk.gain, n * 2 * sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMalloc(&b->d_silk.rs, n * 2 * 8 * sizeof(float));
        if (e == cudaSuccess) e = cudaMalloc(&b->d_silk.fs, n * 2);
    }
    if (e == cudaSuccess) e = cudaMalloc(&b->d_hist_samples, sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemset(b->d_hist_samples, 0, sizeof(unsigned long long));
    if (e != cudaSuccess) {
        opn_batch_destroy(b);
        return cuda_fail(e, "opn_batch_create: allocation");
    }
    b->last_nf.assign(n, 120);  // DecoderInner::frame_size starts at fs/400 (decoder.rs:273)
    b->bandwidth.assign(n, -1);
    b->last_duration.assign(n, -1);
    b->have_mode.assign(n, 0);
    b->silk_cs.assign(n, 0);
    *out = b;
    rc = opn_batch_reset(b);
    if (rc) {
        opn_batch_destroy(b);
        *out = nullptr;
    }
    return rc;
}

void opn_batch_destroy(opn_batch *b)
{
    if (!b) return;
    cudaSetDevice(b->device);
    for (int q = 0; q < opn_batch::NRD; q++)
        if (b->stream_rd[q]) cudaStreamSynchronize(b->stream_rd[q]);
    for (cudaStream_t st : {b->stream_mix, b->stream_up, b->stream, b->stream_dn})
        if (st) cudaStreamSynchronize(st);
    for (int g = 1; g < opn_batch::NGROUPS; g++)
        if (b->stream_fr[g]) {
            cudaStreamSynchronize(b->stream_fr[g]);
            cudaStreamDestroy(b->stream_fr[g]);
        }
    if (b->ev_sw) cudaEventDestroy(b->ev_sw);
    for (int q = 0; q < opn_batch::NSETS; q++) {
        for (int g = 1; g < opn_batch::NGROUPS; g++)
            if (b->ev_fr[q][g]) cudaEventDestroy(b->ev_fr[q][g]);
        if (b->ev_rd[q]) cudaEventDestroy(b->ev_rd[q]);
        if (b->ev_k1[q]) cudaEventDestroy(b->ev_k1[q]);
        cudaFree(b->d_idx[q]);
        cudaFree(b->d_hdr[q]);
        cudaFree(b->d_parts[q]);
        cudaFree(b->d_bande[q]);
        cudaFree(b->d_status[q]);
        cudaFree(b->d_silk_rec[q]);
    }
    cudaFree(b->d_silk.slpc);
    cudaFree(b->d_silk.hist);
    cudaFree(b->d_silk.a_q12);
    cudaFree(b->d_silk.gain);
    cudaFree(b->d_silk.rs);
    cudaFree(b->d_silk.fs);
    if (b->ev_in) cudaEventDestroy(b->ev_in);
    for (int q = 0; q < opn_batch::MAX_CHUNKS; q++)
        if (b->ev_chunk[q]) cudaEventDestroy(b->ev_chunk[q]);
    for (cudaStream_t st : {b->stream_mix, b->stream_up, b->stream_dn})
        if (st) cudaStreamDestroy(st);
    for (int q = 0; q < opn_batch::NRD; q++)
        if (b->stream_rd[q]) cudaStreamDestroy(b->stream_rd[q]);
    for (int k = 0; k < 3; k++) b->ev[k].destroy();
    cudaFree(b->d_carry);
    cudaFree(b->d_ring);
    cudaFree(b->d_ring_pos);
    cudaFree(b->d_final);
    cudaFree(b->d_pf);
    cudaFree(b->d_softclip);
    cudaFree(b->d_last_lm);
    cudaFree(b->d_mix_key);
    cudaFree(b->d_mix_rank);
    for (int q = 0; q < opn_batch::NSETS; q++) {
        cudaFree(b->d_mix_items[q]);
        cudaFree(b->d_mix_lm[q]);
        cudaFree(b->d_mix_plan[q]);
        if (b->ev_mix[q]) cudaEventDestroy(b->ev_mix[q]);
    }
    cudaFree(b->d_hist_samples);
    for (auto &g : b->stg) {
        cudaFree(g.d_arena);
        cudaFree(g.d_items);
        cudaFree(g.d_dense);
        cudaFree(g.d_conv);
        cudaFree(g.d_cliplen);
        cudaFree(g.d_trans);
        if (g.h_trans) cudaFreeHost(g.h_trans);
        if (g.h_cliplen) cudaFreeHost(g.h_cliplen);
        if (g.h_items) cudaFreeHost(g.h_items);
        if (g.done) cudaEventDestroy(g.done);
    }
    if (b->stream) cudaStreamDestroy(b->stream);
    delete b;
}

int opn_batch_reset(opn_batch *b)  // DecoderInner::reset, decoder.rs:286-303, for every stream
{
    if (!b) return OPN_ERR_BAD_ARG;
    CU(cudaSetDevice(b->device));
    // Steps may still be in flight on any of the pipeline's streams (a frame kernel writing the ring, a range decode
    // writing a buffer set, a download reading staging): nothing is cleared before all of them have drained.
    int rc = sync_pipeline(b);
    if (rc) return rc;
    for (auto &g : b->stg) g.pending = false;
    const size_t n = b->n, C = (size_t)b->cfg.channels;
    CU(cudaMemsetAsync(b->d_carry, 0, n * C * 60 * sizeof(float), b->stream));
    CU(cudaMemsetAsync(b->d_ring, 0, n * C * RING_SAMPLES * sizeof(float), b->stream));
    CU(cudaMemsetAsync(b->d_ring_pos, 0, n * sizeof(uint32_t), b->stream));
    CU(cudaMemsetAsync(b->d_final, 0, n * sizeof(uint32_t), b->stream));
    CU(cudaMemsetAsync(b->d_pf, 0, n * sizeof(PfState), b->stream));
    for (int q = 0; q < opn_batch::NSETS; q++) {
        CU(cudaMemsetAsync(b->d_hdr[q], 0, n * sizeof(uint4), b->stream));
        CU(cudaMemsetAsync(b->d_status[q], 0, n * sizeof(int32_t), b->stream));
        b->k1_recorded[q] = false;
    }
    b->set = 0;
    CU(cudaMemsetAsync(b->d_softclip, 0, n * 2 * sizeof(float), b->stream));
    if (b->d_last_lm) CU(cudaMemsetAsync(b->d_last_lm, MIX_NO_ITEM, n, b->stream));
    if (b->silk) {
        CU(cudaMemsetAsync(b->d_silk.slpc, 0, n * 2 * 16 * sizeof(int32_t), b->stream));
        CU(cudaMemsetAsync(b->d_silk.hist, 0, n * 2 * SILK_HIST * sizeof(int32_t), b->stream));
        CU(cudaMemsetAsync(b->d_silk.a_q12, 0, n * 2 * 16 * sizeof(int16_t), b->stream));
        CU(cudaMemsetAsync(b->d_silk.gain, 0, n * 2 * sizeof(int32_t), b->stream));
        CU(cudaMemsetAsync(b->d_silk.rs, 0, n * 2 * 8 * sizeof(float), b->stream));
        CU(cudaMemsetAsync(b->d_silk.fs, 0, n * 2, b->stream));
    }
    CU(cudaStreamSynchronize(b->stream));
    std::fill(b->last_nf.begin(), b->last_nf.end(), 120);
    std::fill(b->bandwidth.begin(), b->bandwidth.end(), -1);
    std::fill(b->last_duration.begin(), b->last_duration.end(), -1);
    std::fill(b->have_mode.begin(), b->have_mode.end(), 0);
    std::fill(b->silk_cs.begin(), b->silk_cs.end(), 0);
    return OPN_OK;
}

// Host-buffer path.  The streams are cut into chunks that flow through a five-stage pipeline:
// host parse (decode_native's TOC/frame split) -> item upload -> entropy stage -> PVQ/IMDCT stage -> PCM
// download, so that parsing, kernels and the PCIe copy of different chunks overlap.  The download is
// the long pole (31.5 MB per 4096 stereo 20 ms frames); everything else hides behind it.
static int batch_decode_host(opn_batch *b, const uint8_t *arena, const uint32_t *offsets, const uint32_t *lens, float *pcm,
                             size_t pcm_stride, size_t frame_size, int32_t *results, uint32_t flags,
                             void *pcm_conv = nullptr, int sample_format = OPN_SAMPLE_F32)
{
    Range nv_call("opn: host-buffer call (parse, upload, decode, download)");
    const uint32_t n = b->n;
    const int C = b->cfg.channels;
    // pre-pass: bytes to upload and an upper bound of the number of frames (items)
    size_t arena_end = 0, items_ub = 0;
    for (uint32_t i = 0; i < n; i++) {
        if (lens[i] == 0) {
            items_ub += frame_size / 120;
            continue;
        }
        arena_end = std::max(arena_end, (size_t)offsets[i] + lens[i]);
        const int fc = opn_packet_frame_count(arena + offsets[i], lens[i]);
        items_ub += (fc > 0 ? (size_t)fc : 1) + (b->silk ? 1 : 0);  // + the concealed frame of a CELT -> SILK transition
    }
    const size_t dense_stride = (frame_size * (size_t)C + 3) & ~(size_t)3;
    const int slot = b->stg_next;
    b->stg_next ^= 1;
    opn_batch::Staging &g = b->stg[slot];
    if (g.pending) {  // the call that used this slot two submissions ago must be completely finished
        CU(cudaEventSynchronize(g.done));
        g.pending = false;
    }
    const size_t esize = pcm_conv ? opn_sample_size(sample_format) : 0;
    if (pcm_conv && esize == 0) return OPN_ERR_BAD_ARG;
    int rc = batch_alloc_staging(b, g, arena_end, items_ub, dense_stride, esize);
    if (rc) return rc;
    const bool want_pcm = (pcm != nullptr || pcm_conv != nullptr) && !(flags & OPN_FLAG_NO_PCM_COPY);
    if (arena_end) CU(cudaMemcpyAsync(g.d_arena, arena, arena_end, cudaMemcpyHostToDevice, b->stream_up));

    const uint32_t n_chunks = std::min<uint32_t>(opn_batch::MAX_CHUNKS, std::max<uint32_t>(1u, n / 1024u));
    const size_t cap = g.items_cap;
    std::vector<Item> items;
    items.reserve(items_ub / n_chunks + 64);
    std::vector<int32_t> res(n, 0);
    std::vector<uint32_t> plc;
    std::vector<uint32_t> silk_resets, celt_resets;  // streams whose codec mode changes in this chunk
    size_t kbase = 0;  // items of earlier chunks
    for (uint32_t ch = 0; ch < n_chunks; ch++) {
        const uint32_t s0 = (uint32_t)((uint64_t)n * ch / n_chunks), s1 = (uint32_t)((uint64_t)n * (ch + 1) / n_chunks);
        Range nv_chunk("opn: chunk (host parse -> enqueue)");
        items.clear();
        silk_resets.clear();
        celt_resets.clear();
        bool any_gap = false;  // some stream of the chunk leaves part of its dense row unwritten
        uint32_t max_len = 8;
        for (uint32_t i = s0; i < s1; i++) {
            const uint32_t len = lens[i];
            // decode_native(None, n) (decoder.rs:427-441): conceal n samples from sample `at0` of the row; the concealed frames take
            // waves w0, w0+1, ...  Returns the number of frames pushed, -1 when nothing was decoded yet (zeros, state untouched,
            // decoder.rs:478-487), -2 when this kind of concealment is not built.
            auto conceal = [&](uint32_t i, size_t n_samples, uint32_t at0, int w0) -> int {
                if (!b->have_mode[i]) return -1;
                plc.clear();
                plc_frames(n_samples, b->last_nf[i], plc);
                uint32_t at = at0;
                int w = w0;
                if (b->have_mode[i] == 1 + OPN_MODE_SILK) {
                    // the stream's last packet was SILK: concealed by the SILK path (10 and 20 ms frames only)
                    bool ok = b->silk;
                    for (uint32_t a : plc) ok = ok && (a == 480 || a == 960);
                    if (!ok) return -2;
                    for (uint32_t a : plc) {
                        items.push_back(Item{i, 0u, 0u, at * (uint32_t)C, 8 + (a == 960 ? 1 : 0), w++, (int)b->silk_cs[i]});
                        at += a;
                    }
                } else {
                    for (uint32_t a : plc) {
                        items.push_back(Item{i, 0u, 0u, at * (uint32_t)C, lm_of_frame(a), w++, C});
                        at += a;
                    }
                }
                return w - w0;
            };
            if (len == 0) {  // lost packet
                const int k = conceal(i, frame_size, 0u, 0);
                if (k < 0) any_gap = true;
                res[i] = k == -2 ? OPN_ERR_UNIMPLEMENTED : (int32_t)frame_size;
                if (k != -2) b->last_duration[i] = (int32_t)frame_size;
                continue;
            }
            const uint8_t *pkt = arena + offsets[i];
            // decode_native, decoder.rs:322-341
            const int mode = opn_packet_mode(pkt);
            const int pfs = opn_packet_samples_per_frame(pkt, 48000);
            uint32_t fr[48], sz[48];
            const int count = opn_parse_packet(pkt, len, 0, fr, sz, nullptr, nullptr);
            if (count < 0) {
                res[i] = count;
                any_gap = true;
                continue;
            }
            if (flags & OPN_FLAG_DECODE_FEC) {  // decode_native(Some(packet), decode_fec = true), decoder.rs:343-386
                // no FEC can be present in a CELT packet or for a CELT stream, nor fit a row shorter than a packet frame: conceal it all
                if (frame_size < (size_t)pfs || mode == OPN_MODE_CELT || b->have_mode[i] == 1 + OPN_MODE_CELT) {
                    const int k = conceal(i, frame_size, 0u, 0);
                    if (k < 0) any_gap = true;
                    res[i] = k == -2 ? OPN_ERR_UNIMPLEMENTED : (int32_t)frame_size;
                    if (k != -2) b->last_duration[i] = (int32_t)frame_size;
                    continue;
                }
                if (mode != OPN_MODE_SILK || !b->silk || (pfs != 480 && pfs != 960) || opn_packet_bandwidth(pkt) > OPN_BW_WIDE) {
                    res[i] = OPN_ERR_UNIMPLEMENTED;  // hybrid frames, 40 / 60 ms SILK frames
                    any_gap = true;
                    continue;
                }
                // conceal everything but the one frame the packet may hold a redundant copy of, then decode that copy
                int k = 0;
                if (frame_size > (size_t)pfs) {
                    k = conceal(i, frame_size - (size_t)pfs, 0u, 0);
                    if (k == -2) {
                        res[i] = OPN_ERR_UNIMPLEMENTED;
                        any_gap = true;
                        continue;
                    }
                    if (k < 0) {
                        any_gap = true;
                        k = 0;
                    }
                }
                const int cs = opn_packet_channels(pkt);
                const int code = 8 + 2 * opn_packet_bandwidth(pkt) + (pfs == 960 ? 1 : 0) + 16;  // + 16: the redundant copy
                items.push_back(Item{i, offsets[i] + fr[0], sz[0], (uint32_t)((frame_size - (size_t)pfs) * C), code, k, cs});
                max_len = std::max(max_len, sz[0]);
                res[i] = (int32_t)frame_size;
                b->have_mode[i] = 1 + OPN_MODE_SILK;
                b->silk_cs[i] = (uint8_t)cs;
                b->last_nf[i] = pfs;
                b->bandwidth[i] = opn_packet_bandwidth(pkt);
                b->last_duration[i] = (int32_t)frame_size;
                continue;
            }
            if ((size_t)count * (size_t)pfs > frame_size) {  // decoder.rs:388-390
                res[i] = OPN_ERR_FRAME_SIZE_TOO_SMALL;
                any_gap = true;
                continue;
            }
            if (mode == OPN_MODE_SILK && b->silk && (pfs == 480 || pfs == 960) && opn_packet_bandwidth(pkt) <= OPN_BW_WIDE) {
                // SYNTH-SILK/1 (DESIGN.md 3c): bucket code 8 + 2 * bandwidth + (20 ms)
                const int code = 8 + 2 * opn_packet_bandwidth(pkt) + (pfs == 960 ? 1 : 0);
                const int cs = opn_packet_channels(pkt);
                for (int w = 0; w < count; w++) {
                    items.push_back(Item{i, offsets[i] + fr[w], sz[w], (uint32_t)(w * pfs * C), code, w, cs});
                    max_len = std::max(max_len, sz[w]);
                }
                if (b->have_mode[i] == 1 + OPN_MODE_CELT) {
                    silk_resets.push_back(i);  // decoder.rs:555-557: silk_dec.reset()
                    // decoder.rs:519-543, 674-676: the CELT decoder conceals 5 ms into the transition buffer (the tail of the row)
                    // (its "row offset" reaches from the stream's row to its slot in the tail area behind all rows)
                    items.push_back(Item{i, 0u, 0u, (uint32_t)((size_t)(n - i) * g.dense_cap + (size_t)i * 240 * C), 1, -1, C});
                }
                if ((size_t)count * (size_t)pfs < frame_size) any_gap = true;
                res[i] = count * pfs;
                b->have_mode[i] = 1 + OPN_MODE_SILK;
                b->silk_cs[i] = (uint8_t)cs;
                b->last_nf[i] = pfs;
                b->bandwidth[i] = opn_packet_bandwidth(pkt);
                b->last_duration[i] = count * pfs;
                continue;
            }
            if (mode != OPN_MODE_CELT || b->cfg.bitstream == OPN_BITSTREAM_OPUS) {
                // SilkDecoder::decode is unimplemented!() in the reference (silk/decoder.rs:79); CeltDecoder::decode itself
                // is todo!() (celt/decoder.rs:47-56): CELT frames decode only when the batch was created for one of the
                // SYNTH-CELT layouts.  A packet whose channel count differs from the decoder's is decoded with its own
                // layout and mapped in the frame kernel (stream_channels, decoder.rs:332,376,395).
                res[i] = OPN_ERR_UNIMPLEMENTED;
                any_gap = true;
                continue;
            }
            const int lm = lm_of_frame((size_t)pfs);
            const int cs = opn_packet_channels(pkt);
            for (int w = 0; w < count; w++) {
                items.push_back(Item{i, offsets[i] + fr[w], sz[w], (uint32_t)(w * pfs * C), lm, w, cs});
                max_len = std::max(max_len, sz[w]);
            }
            if ((size_t)count * (size_t)pfs < frame_size) any_gap = true;
            if (b->have_mode[i] == 1 + OPN_MODE_SILK) celt_resets.push_back(i);  // decoder.rs:703-705: celt_dec.reset() on a mode change
            res[i] = count * pfs;
            b->have_mode[i] = 1 + OPN_MODE_CELT;
            b->last_nf[i] = pfs;
            b->bandwidth[i] = opn_packet_bandwidth(pkt);
            b->last_duration[i] = count * pfs;
        }
        if (kbase + items.size() > cap) return OPN_ERR_INTERNAL;  // the pre-pass bound covers every frame
        if (want_pcm && any_gap)
            CU(cudaMemsetAsync(g.d_dense + (size_t)s0 * g.dense_cap, 0, (size_t)(s1 - s0) * g.dense_cap * sizeof(float), b->stream));
        if (!items.empty()) {
            // order: wave-major, then frame size, then the packets' channel count, so each bucket is contiguous
            std::stable_sort(items.begin(), items.end(), [](const Item &x, const Item &y) {
                return x.wave != y.wave ? x.wave < y.wave : x.lm != y.lm ? x.lm < y.lm : x.cs < y.cs;
            });
            // one upload per chunk: [offsets | lens | stream ids | dense offsets], each cnt words, at 4*kbase
            const size_t cnt = items.size();
            uint32_t *hi = g.h_items + 4 * kbase, *di = g.d_items + 4 * kbase;
            for (size_t k = 0; k < cnt; k++) {
                hi[k] = items[k].offset;
                hi[cnt + k] = items[k].len;
                hi[2 * cnt + k] = items[k].stream;
                hi[3 * cnt + k] = items[k].dense_off;
            }
            CU(cudaMemcpyAsync(di, hi, 4 * cnt * sizeof(uint32_t), cudaMemcpyHostToDevice, b->stream_up));
            // mode changes: the decoder that takes over starts from rest (ordered before this chunk's range decodes, which
            // wait for stream_up; the stream's earlier frames ran in earlier calls)
            for (uint32_t i : silk_resets) CU(cudaMemsetAsync(b->d_silk.fs + 2 * (size_t)i, 0, 2, b->stream_up));
            for (uint32_t i : celt_resets) {
                CU(cudaMemsetAsync(b->d_carry + (size_t)i * C * 60, 0, (size_t)C * 60 * sizeof(float), b->stream_up));
                CU(cudaMemsetAsync(b->d_pf + i, 0, sizeof(PfState), b->stream_up));
                // CeltDecoder::reset clears its decode memory: the post-filter must not see SILK output as history
                CU(cudaMemsetAsync(b->d_ring + (size_t)i * C * RING_SAMPLES, 0, (size_t)C * RING_SAMPLES * sizeof(float), b->stream_up));
            }
            const uint32_t pkt_cap = (max_len + 15u) & ~15u;
            size_t k0 = 0;
            while (k0 < cnt) {
                size_t k1 = k0;
                while (k1 < cnt && items[k1].wave == items[k0].wave && items[k1].lm == items[k0].lm && items[k1].cs == items[k0].cs) k1++;
                if (items[k0].lm >= 8) {
                    const int fec = (items[k0].lm - 8) >> 4, code = (items[k0].lm - 8) & 15;
                    rc = run_silk_bucket(b, g.d_arena, di + k0, di + cnt + k0, di + 2 * cnt + k0, di + 3 * cnt + k0, (uint32_t)(k1 - k0),
                                         (code & 1) ? 20 : 10, 0, code >> 1, items[k0].cs, want_pcm ? g.d_dense : nullptr, g.dense_cap, nullptr, 2,
                                         pcm_conv == nullptr, fec);
                    if (rc) return rc;
                    k0 = k1;
                    continue;
                }
                rc = run_bucket(b, g.d_arena, di + k0, di + cnt + k0, di + 2 * cnt + k0, di + 3 * cnt + k0, (uint32_t)(k1 - k0),
                                items[k0].lm, 0, pkt_cap, want_pcm ? g.d_dense : nullptr, g.dense_cap, nullptr, 2, pcm_conv == nullptr,
                                items[k0].cs);
                if (rc) return rc;
                k0 = k1;
            }
            kbase += items.size();
            if (want_pcm && !silk_resets.empty()) {
                // decoder.rs:765-788: first 2.5 ms = the concealed CELT audio, next 2.5 ms = smooth_fade_into_in2(transition, samples)
                if (!g.d_trans) {
                    CU(cudaMalloc(&g.d_trans, (size_t)b->n * sizeof(uint32_t)));
                    CU(cudaMallocHost(&g.h_trans, (size_t)b->n * sizeof(uint32_t)));
                }
                std::memcpy(g.h_trans + s0, silk_resets.data(), silk_resets.size() * sizeof(uint32_t));
                CU(cudaMemcpyAsync(g.d_trans + s0, g.h_trans + s0, silk_resets.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, b->stream_up));
                CU(cudaEventRecord(b->ev_in, b->stream_up));
                CU(cudaStreamWaitEvent(b->stream, b->ev_in, 0));
                CU(launch_transition_fade(g.d_dense, g.dense_cap, g.d_trans + s0, (uint32_t)silk_resets.size(), n, C, b->stream));
            }
        }
        if (want_pcm && pcm_conv) {
            // decode::<S>: soft clip + Sample::from_f32 on the device; for the 16-bit types half the bytes go home.
            // The epilogue kernel follows the chunk's frame kernels on the batch stream.  Concealed frames are not
            // clipped and leave the soft-clip memory alone (decode_native's None branch, decoder.rs:427-441).
            for (uint32_t i = s0; i < s1; i++) g.h_cliplen[i] = (lens[i] != 0 && res[i] > 0) ? res[i] : 0;
            CU(cudaMemcpyAsync(g.d_cliplen + s0, g.h_cliplen + s0, (size_t)(s1 - s0) * sizeof(int32_t), cudaMemcpyHostToDevice, b->stream_up));
            CU(cudaEventRecord(b->ev_in, b->stream_up));
            CU(cudaStreamWaitEvent(b->stream, b->ev_in, 0));
            CU(launch_softclip_convert(sample_format, g.d_dense, g.dense_cap, g.d_cliplen, C, (uint32_t)(frame_size * (size_t)C), s0, s1 - s0,
                                       b->d_softclip, g.d_conv, g.conv_cap, b->stream));
            CU(cudaEventRecord(b->ev_chunk[ch], b->stream));
            CU(cudaStreamWaitEvent(b->stream_dn, b->ev_chunk[ch], 0));
            const size_t row_bytes = frame_size * (size_t)C * esize;
            uint8_t *dst = static_cast<uint8_t *>(pcm_conv) + (size_t)s0 * pcm_stride * esize;
            const uint8_t *srcp = static_cast<const uint8_t *>(g.d_conv) + (size_t)s0 * g.conv_cap * esize;
            if (pcm_stride == g.conv_cap && pcm_stride * esize == row_bytes)
                CU(cudaMemcpyAsync(dst, srcp, (size_t)(s1 - s0) * row_bytes, cudaMemcpyDeviceToHost, b->stream_dn));
            else
                CU(cudaMemcpy2DAsync(dst, pcm_stride * esize, srcp, g.conv_cap * esize, row_bytes, s1 - s0, cudaMemcpyDeviceToHost, b->stream_dn));
        } else if (want_pcm) {
            // this chunk's PCM rows go home while the next chunk is decoded
            CU(cudaEventRecord(b->ev_chunk[ch], b->stream));
            CU(cudaStreamWaitEvent(b->stream_dn, b->ev_chunk[ch], 0));
            const size_t row_bytes = frame_size * (size_t)C * sizeof(float);
            if (pcm_stride == g.dense_cap && pcm_stride * sizeof(float) == row_bytes)
                CU(cudaMemcpyAsync(pcm + (size_t)s0 * pcm_stride, g.d_dense + (size_t)s0 * g.dense_cap, (size_t)(s1 - s0) * row_bytes,
                                   cudaMemcpyDeviceToHost, b->stream_dn));
            else
                CU(cudaMemcpy2DAsync(pcm + (size_t)s0 * pcm_stride, pcm_stride * sizeof(float), g.d_dense + (size_t)s0 * g.dense_cap,
                                     g.dense_cap * sizeof(float), row_bytes, s1 - s0, cudaMemcpyDeviceToHost, b->stream_dn));
        }
    }
    // completion of this call = the batch stream and the download stream have drained
    CU(cudaEventRecord(b->ev_in, b->stream));
    CU(cudaStreamWaitEvent(b->stream_dn, b->ev_in, 0));
    CU(cudaEventRecord(g.done, b->stream_dn));
    g.pending = true;
    if (results) std::memcpy(results, res.data(), n * sizeof(int32_t));
    if (!(flags & OPN_FLAG_SUBMIT_ONLY)) {
        CU(cudaEventSynchronize(g.done));
        g.pending = false;
    }
    return slot;
}

int opn_batch_decode_float(opn_batch *b, const uint8_t *arena, const uint32_t *offsets, const uint32_t *lens, float *pcm,
                           size_t pcm_stride_floats, size_t frame_size, int32_t *result_per_stream, uint32_t flags)
{
    if (!b || !offsets || !lens) return OPN_ERR_BAD_ARG;
    if (frame_size == 0 || frame_size % 120 != 0) return OPN_ERR_BAD_ARG;  // decoder.rs:316-320
    const int C = b->cfg.channels;
    CU(cudaSetDevice(b->device));
    if (!(flags & OPN_FLAG_DEVICE_PTRS)) {
        if (!arena) return OPN_ERR_BAD_ARG;
        if (pcm && pcm_stride_floats < frame_size * (size_t)C) return OPN_ERR_BUFFER_TOO_SMALL;
        const int rc = batch_decode_host(b, arena, offsets, lens, pcm, pcm_stride_floats, frame_size, result_per_stream, flags);
        if (rc < 0) return rc;
        return (flags & OPN_FLAG_SUBMIT_ONLY) ? rc : OPN_OK;  // submit-only: the ticket for opn_batch_wait
    }
    // Device-resident step: one single-frame CELT packet per stream; the TOC is validated on the device and reported per
    // stream.  Asynchronous on the batch's streams.  Without OPN_FLAG_MIXED_FRAMES every packet must hold exactly
    // frame_size samples; with it frame_size is the capacity of a stream's row, as in decode_float, and each stream
    // decodes whatever single frame its packet holds.
    if (!arena) return OPN_ERR_BAD_ARG;
    if (b->cfg.bitstream == OPN_BITSTREAM_OPUS && !(flags & OPN_FLAG_SILK_FRAMES)) return OPN_ERR_UNIMPLEMENTED;  // celt/decoder.rs:47-56 is todo!()
    float *dense = (flags & OPN_FLAG_NO_PCM_COPY) ? nullptr : pcm;
    if (dense && (pcm_stride_floats < std::min<size_t>(frame_size, 960) * (size_t)C || (pcm_stride_floats & 3) ||
                  (reinterpret_cast<uintptr_t>(dense) & 15)))
        return OPN_ERR_BAD_ARG;
    if (flags & OPN_FLAG_SILK_FRAMES) {
        if (!b->silk || (flags & OPN_FLAG_MIXED_FRAMES) || (frame_size != 480 && frame_size != 960)) return OPN_ERR_BAD_ARG;
        if (dense && pcm_stride_floats < frame_size * (size_t)C) return OPN_ERR_BAD_ARG;
        return run_silk_bucket(b, arena, offsets, lens, nullptr, nullptr, b->n, frame_size == 960 ? 20 : 10, 1, -1, C, dense, pcm_stride_floats,
                               result_per_stream, (flags & OPN_FLAG_INPUTS_READY) ? 0 : 1, true);
    }
    if (flags & OPN_FLAG_MIXED_FRAMES)
        return run_mixed(b, arena, offsets, lens, frame_size, dense, pcm_stride_floats, result_per_stream,
                         (flags & OPN_FLAG_INPUTS_READY) ? 0 : 1, true);
    const int lm = lm_of_frame(frame_size);
    if (lm < 0) return OPN_ERR_BAD_ARG;
    if (dense && pcm_stride_floats < frame_size * (size_t)C) return OPN_ERR_BAD_ARG;
    return run_bucket(b, arena, offsets, lens, nullptr, nullptr, b->n, lm, 1, 1280u, dense, pcm_stride_floats, result_per_stream,
                      (flags & OPN_FLAG_INPUTS_READY) ? 0 : 1, true);
}

size_t opn_sample_size(int sample_format)
{
    switch (sample_format) {
    case OPN_SAMPLE_F32: return sizeof(float);
    case OPN_SAMPLE_I16: return sizeof(int16_t);
    case OPN_SAMPLE_I32: return sizeof(int32_t);
    case OPN_SAMPLE_U16: return sizeof(uint16_t);
    case OPN_SAMPLE_U32: return sizeof(uint32_t);
    case OPN_SAMPLE_F64: return sizeof(double);
    default: return 0;
    }
}

int opn_batch_decode_pcm(opn_batch *b, const uint8_t *arena, const uint32_t *offsets, const uint32_t *lens, void *pcm,
                         size_t pcm_stride_samples, int sample_format, size_t frame_size, int32_t *result_per_stream, uint32_t flags)
{
    if (!b || !arena || !offsets || !lens || !pcm) return OPN_ERR_BAD_ARG;
    if (opn_sample_size(sample_format) == 0) return OPN_ERR_BAD_ARG;
    if (frame_size == 0 || frame_size % 120 != 0) return OPN_ERR_BAD_ARG;  // decoder.rs:316-320
    if (flags & (OPN_FLAG_DEVICE_PTRS | OPN_FLAG_NO_PCM_COPY)) return OPN_ERR_BAD_ARG;
    if (pcm_stride_samples < frame_size * (size_t)b->cfg.channels) return OPN_ERR_BUFFER_TOO_SMALL;
    if (frame_size * (size_t)b->cfg.channels * sizeof(float) > 200 * 1024) return OPN_ERR_BAD_ARG;  // the clip epilogue stages a row on chip
    CU(cudaSetDevice(b->device));
    const int rc = batch_decode_host(b, arena, offsets, lens, nullptr, pcm_stride_samples, frame_size, result_per_stream, flags, pcm,
                                     sample_format);
    if (rc < 0) return rc;
    return (flags & OPN_FLAG_SUBMIT_ONLY) ? rc : OPN_OK;
}

int opn_batch_decode_i16(opn_batch *b, const uint8_t *arena, const uint32_t *offsets, const uint32_t *lens, int16_t *pcm,
                         size_t pcm_stride_samples, size_t frame_size, int32_t *result_per_stream, uint32_t flags)
{
    return opn_batch_decode_pcm(b, arena, offsets, lens, pcm, pcm_stride_samples, OPN_SAMPLE_I16, frame_size, result_per_stream, flags);
}

int opn_batch_synchronize(opn_batch *b)
{
    if (!b) return OPN_ERR_BAD_ARG;
    CU(cudaSetDevice(b->device));
    int rc = sync_pipeline(b);
    if (rc) return rc;
    for (auto &g : b->stg) g.pending = false;
    return OPN_OK;
}

int opn_batch_join(opn_batch *b)
{
    if (!b) return OPN_ERR_BAD_ARG;
    CU(cudaSetDevice(b->device));
    // every step ends with frame kernels: group 0 on the batch stream, the other groups on their own streams
    return join_groups(b);
}

int opn_batch_wait(opn_batch *b, int ticket)
{
    if (!b || ticket < 0 || ticket > 1) return OPN_ERR_BAD_ARG;
    CU(cudaSetDevice(b->device));
    opn_batch::Staging &g = b->stg[ticket];
    if (g.pending) {
        CU(cudaEventSynchronize(g.done));
        g.pending = false;
    }
    return OPN_OK;
}

int opn_batch_final_ranges(opn_batch *b, uint32_t *out)
{
    if (!b || !out) return OPN_ERR_BAD_ARG;
    CU(cudaSetDevice(b->device));
    int rc = join_groups(b);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out, b->d_final, b->n * sizeof(uint32_t), cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    return OPN_OK;
}

int opn_batch_ring(opn_batch *b, float **ring, uint32_t *ring_samples, uint32_t **ring_pos_dev)
{
    if (!b) return OPN_ERR_BAD_ARG;
    if (ring) *ring = b->d_ring;
    if (ring_samples) *ring_samples = RING_SAMPLES;
    if (ring_pos_dev) *ring_pos_dev = b->d_ring_pos;
    return OPN_OK;
}

int opn_batch_enable_timing(opn_batch *b, int on)
{
    if (!b) return OPN_ERR_BAD_ARG;
    CU(cudaSetDevice(b->device));
    if (on) {
        for (int k = 0; k < 3; k++) {
            int rc = b->ev[k].make();
            if (rc) return rc;
        }
    }
    if (b->timing != (on != 0)) {
        // the two modes order their kernels differently (events across streams / one stream): drain before switching
        int rc = sync_pipeline(b);
        if (rc) return rc;
    }
    b->timing = on != 0;
    return OPN_OK;
}

int opn_batch_stats(opn_batch *b, uint64_t kernel_launches[3], double kernel_ms[3], int reset)
{
    if (!b) return OPN_ERR_BAD_ARG;
    CU(cudaSetDevice(b->device));
    CU(cudaStreamSynchronize(b->stream));
    for (int k = 0; k < 3; k++) {
        int rc = b->ev[k].resolve();
        if (rc) return rc;
        if (kernel_launches) kernel_launches[k] = b->launches[k];
        if (kernel_ms) kernel_ms[k] = b->ev[k].ms;
        if (reset) {
            b->launches[k] = 0;
            b->ev[k].ms = 0.0;
            b->ev[k].launches = 0;
        }
    }
    return OPN_OK;
}

int opn_batch_history_samples(opn_batch *b, uint64_t *out, int reset)
{
    if (!b || !out) return OPN_ERR_BAD_ARG;
    CU(cudaSetDevice(b->device));
    CU(cudaStreamSynchronize(b->stream));
    unsigned long long v = 0;
    CU(cudaMemcpy(&v, b->d_hist_samples, sizeof(v), cudaMemcpyDeviceToHost));
    if (reset) CU(cudaMemset(b->d_hist_samples, 0, sizeof(v)));
    *out = v;
    return OPN_OK;
}

void *opn_batch_cuda_stream(opn_batch *b) { return b ? (void *)b->stream : nullptr; }

// ------------------------------------------------------------------------------------ decoder
}  // extern "C"

struct opn_decoder {
    opn_batch *batch = nullptr;  // a batch of one stream
    int32_t fs = 48000, channels = 2;
    int16_t gain_q8 = 0;
    uint32_t final_range = 0;
    void *h_pcm = nullptr;  // pinned staging of decode::<S> (converted samples)
    size_t h_cap = 0;       // bytes
};

extern "C" {

int opn_decoder_create(int device, int32_t fs_hz, int32_t channels, int16_t gain_q8, int32_t bitstream, opn_decoder **out)
{
    if (!out) return OPN_ERR_BAD_ARG;
    opn_config cfg{fs_hz, channels, gain_q8, 1, bitstream};
    opn_batch *b = nullptr;
    int rc = opn_batch_create(device, 1, &cfg, &b);
    if (rc) return rc;
    opn_decoder *d = new (std::nothrow) opn_decoder();
    if (!d) {
        opn_batch_destroy(b);
        return OPN_ERR_INTERNAL;
    }
    d->batch = b;
    d->fs = fs_hz;
    d->channels = channels;
    d->gain_q8 = gain_q8;
    *out = d;
    return OPN_OK;
}

void opn_decoder_destroy(opn_decoder *d)
{
    if (!d) return;
    if (d->h_pcm) cudaFreeHost(d->h_pcm);
    opn_batch_destroy(d->batch);
    delete d;
}

int opn_decoder_reset(opn_decoder *d)
{
    if (!d) return OPN_ERR_BAD_ARG;
    d->final_range = 0;
    return opn_batch_reset(d->batch);
}

static int decoder_decode(opn_decoder *d, const uint8_t *packet, size_t len, float *pcm, size_t frame_size, int decode_fec,
                          void *pcm_conv = nullptr, int sample_format = OPN_SAMPLE_F32)
{
    if (!d || (!pcm && !pcm_conv)) return OPN_ERR_BAD_ARG;
    if (frame_size == 0 || frame_size % (size_t)(d->fs / 400) != 0) return OPN_ERR_BAD_ARG;  // decoder.rs:316-320
    if (packet && len == 0) return OPN_ERR_BAD_ARG;                                           // decoder.rs:323-325
    if (packet && len > 0xFFFFFFFFull) return OPN_ERR_BAD_ARG;
    uint32_t off = 0, l = packet ? (uint32_t)len : 0u;
    // decoder.rs:343-386: FEC only exists in SILK frames; for a CELT-only packet (or stream) the reference conceals the whole gap
    // instead, otherwise it conceals all but one packet frame and decodes the packet's redundant copy of the previous frame:
    // batch_decode_host does both under OPN_FLAG_DECODE_FEC
    static const uint8_t dummy = 0;
    int32_t res = 0;
    int rc = batch_decode_host(d->batch, packet ? packet : &dummy, &off, &l, pcm, frame_size * (size_t)d->channels, frame_size,
                               &res, (packet && decode_fec) ? OPN_FLAG_DECODE_FEC : 0u, pcm_conv, sample_format);
    if (rc < 0) return rc;
    if (res >= 0) {
        uint32_t fr = 0;
        rc = opn_batch_final_ranges(d->batch, &fr);
        if (rc) return rc;
        d->final_range = l ? fr : 0u;  // decoder.rs:799-803
    }
    return res;
}

int opn_decode_float(opn_decoder *d, const uint8_t *packet, size_t len, float *pcm, size_t frame_size, int decode_fec)
{
    return decoder_decode(d, packet, len, pcm, frame_size, decode_fec);
}

int opn_decode_pcm(opn_decoder *d, const uint8_t *packet, size_t len, void *pcm, size_t pcm_capacity, int sample_format,
                   size_t frame_size, int decode_fec)
{
    if (!d || !pcm) return OPN_ERR_BAD_ARG;
    const size_t esize = opn_sample_size(sample_format);
    if (esize == 0) return OPN_ERR_BAD_ARG;
    // Decoder::decode<S>, decoder.rs:148-193
    if (!decode_fec && packet) {
        if (len == 0) return OPN_ERR_BAD_ARG;
        const int sc = opn_packet_sample_count(packet, len, d->fs);
        if (sc < 0) return sc;
        if (sc == 0) return OPN_ERR_INVALID_PACKET;
        frame_size = std::min(frame_size, (size_t)sc);
    }
    const size_t need = frame_size * (size_t)d->channels * esize;
    if (need > d->h_cap) {
        if (d->h_pcm) cudaFreeHost(d->h_pcm);
        d->h_pcm = nullptr;
        d->h_cap = 0;
        CU(cudaMallocHost(&d->h_pcm, need));
        d->h_cap = need;
    }
    // soft clip and S::from_f32 run on the device (k_softclip_convert); the converted samples land in the decoder's
    // own buffer first, as in the crate (self.buffer), and reach the caller's slice only if it is long enough
    const int n = decoder_decode(d, packet, len, nullptr, frame_size, decode_fec, d->h_pcm, sample_format);
    if (n <= 0) return n;
    if ((size_t)n > pcm_capacity) return OPN_ERR_BUFFER_TOO_SMALL;  // decoder.rs:181 (per-channel count vs slice length)
    if ((size_t)n * (size_t)d->channels > pcm_capacity) return OPN_ERR_BUFFER_TOO_SMALL;  // Rust would panic on the index
    std::memcpy(pcm, d->h_pcm, (size_t)n * (size_t)d->channels * esize);
    return n;
}

int opn_decode_i16(opn_decoder *d, const uint8_t *packet, size_t len, int16_t *pcm, size_t pcm_capacity, size_t frame_size,
                   int decode_fec)
{
    return opn_decode_pcm(d, packet, len, pcm, pcm_capacity, OPN_SAMPLE_I16, frame_size, decode_fec);
}

int32_t opn_decoder_sampling_rate(const opn_decoder *d) { return d ? d->fs : 0; }
int32_t opn_decoder_channels(const opn_decoder *d) { return d ? d->channels : 0; }
int32_t opn_decoder_gain(const opn_decoder *d) { return d ? d->gain_q8 : 0; }
int32_t opn_decoder_bandwidth(const opn_decoder *d) { return d ? d->batch->bandwidth[0] : -1; }
int32_t opn_decoder_last_packet_duration(const opn_decoder *d) { return d ? d->batch->last_duration[0] : -1; }
uint32_t opn_decoder_final_range(const opn_decoder *d) { return d ? d->final_range : 0u; }

int32_t opn_decoder_pitch(const opn_decoder *d)
{
    // Decoder::pitch (decoder.rs:100-109) forwards to CeltDecoder::pitch, a todo!() in the reference;
    // libopus reports the post-filter period of the last frame, so do that.
    if (!d || !d->batch->have_mode[0]) return -1;
    PfState pf{};
    if (cudaSetDevice(d->batch->device) != cudaSuccess) return -1;
    if (cudaMemcpy(&pf, d->batch->d_pf, sizeof(pf), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    return pf.period;
}

// ------------------------------------------------------------------------------------ operators
}  // extern "C"
namespace {
struct DevBuf {
    void *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 16); }
    template <class T> T *as() { return static_cast<T *>(p); }
};
}  // namespace
extern "C" {

int opn_op_rangedec_script(int device, const uint8_t *arena, const uint32_t *offsets, const uint32_t *lens, uint32_t n_packets,
                           const opn_op *ops, uint32_t n_ops, const uint8_t *icdf_pool, uint32_t icdf_pool_len, opn_op_out *out,
                           int32_t *y_out, uint32_t y_stride)
{
    if (!arena || !offsets || !lens || !ops || !out || n_packets == 0) return OPN_ERR_BAD_ARG;
    int rc = select_device(device);
    if (rc) return rc;
    size_t arena_end = 0;
    uint32_t max_len = 8;
    for (uint32_t i = 0; i < n_packets; i++) {
        arena_end = std::max(arena_end, (size_t)offsets[i] + lens[i]);
        max_len = std::max(max_len, lens[i]);
    }
    const uint32_t pkt_cap = std::min((max_len + 15u) & ~15u, 4096u);  // larger packets are read from global memory
    DevBuf dA, dO, dL, dOps, dPool, dOut, dY;
    CU(dA.alloc(arena_end));
    CU(dO.alloc(n_packets * 4));
    CU(dL.alloc(n_packets * 4));
    CU(dOps.alloc((size_t)n_ops * sizeof(opn_op)));
    CU(dPool.alloc(icdf_pool_len));
    CU(dOut.alloc((size_t)n_packets * n_ops * sizeof(opn_op_out)));
    CU(dY.alloc((size_t)n_packets * y_stride * 4));
    CU(cudaMemcpy(dA.p, arena, arena_end, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dO.p, offsets, n_packets * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dL.p, lens, n_packets * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dOps.p, ops, (size_t)n_ops * sizeof(opn_op), cudaMemcpyHostToDevice));
    if (icdf_pool && icdf_pool_len) CU(cudaMemcpy(dPool.p, icdf_pool, icdf_pool_len, cudaMemcpyHostToDevice));
    CU(cudaMemset(dY.p, 0, (size_t)n_packets * y_stride * 4 + (y_stride ? 0 : 16)));
    CU(launch_rangedec_script(dA.as<uint8_t>(), dO.as<uint32_t>(), dL.as<uint32_t>(), n_packets, dOps.as<opn_op>(), n_ops,
                              dPool.as<uint8_t>(), dOut.as<opn_op_out>(), y_out ? dY.as<int32_t>() : nullptr, y_stride, pkt_cap,
                              nullptr));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(out, dOut.p, (size_t)n_packets * n_ops * sizeof(opn_op_out), cudaMemcpyDeviceToHost));
    if (y_out && y_stride) CU(cudaMemcpy(y_out, dY.p, (size_t)n_packets * y_stride * 4, cudaMemcpyDeviceToHost));
    return OPN_OK;
}

int opn_op_imdct_tdac(int device, const float *input, size_t in_stride, float *output, size_t out_stride, uint32_t n_rows,
                      int shift, int stride, int blocks)
{
    if (!input || !output || n_rows == 0 || shift < 0 || shift > 3 || blocks < 1 || stride != blocks) return OPN_ERR_BAD_ARG;
    const size_t n2 = 960u >> shift;
    if (n2 * (size_t)blocks > 960 || in_stride < n2 * (size_t)blocks || out_stride < n2 * (size_t)blocks + 60) return OPN_ERR_BAD_ARG;
    int rc = select_device(device);
    if (rc) return rc;
    DevBuf dI, dO;
    CU(dI.alloc((size_t)n_rows * in_stride * 4));
    CU(dO.alloc((size_t)n_rows * out_stride * 4));
    CU(cudaMemcpy(dI.p, input, (size_t)n_rows * in_stride * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dO.p, output, (size_t)n_rows * out_stride * 4, cudaMemcpyHostToDevice));
    CU(launch_op_imdct(dI.as<float>(), in_stride, dO.as<float>(), out_stride, n_rows, shift, blocks, nullptr));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(output, dO.p, (size_t)n_rows * out_stride * 4, cudaMemcpyDeviceToHost));
    return OPN_OK;
}

static int comb_args_ok(size_t offset, size_t n, uint32_t n_rows, const int32_t *p, const float *g, size_t row_stride,
                        size_t overlap)
{
    if (!p || !g || n_rows == 0 || offset + n > row_stride || overlap > 120 || overlap > n) return 0;
    for (uint32_t r = 0; r < n_rows; r++) {
        const int32_t t0 = std::max(p[4 * r], 15), t1 = std::max(p[4 * r + 1], 15);
        if (t0 > 1022 || t1 > 1022 || p[4 * r + 2] < 0 || p[4 * r + 2] > 2 || p[4 * r + 3] < 0 || p[4 * r + 3] > 2) return 0;
        if ((size_t)std::max(t0, t1) + 2 > offset) return 0;  // history must exist (the Rust slice would panic)
    }
    return 1;
}

int opn_op_comb_filter_inplace(int device, float *y, size_t row_stride, size_t y_offset, size_t n, uint32_t n_rows,
                               const int32_t *params4, const float *gains2, size_t overlap)
{
    if (!y || !comb_args_ok(y_offset, n, n_rows, params4, gains2, row_stride, overlap)) return OPN_ERR_BAD_ARG;
    int rc = select_device(device);
    if (rc) return rc;
    DevBuf dY, dP, dG;
    CU(dY.alloc((size_t)n_rows * row_stride * 4));
    CU(dP.alloc((size_t)n_rows * 16));
    CU(dG.alloc((size_t)n_rows * 8));
    CU(cudaMemcpy(dY.p, y, (size_t)n_rows * row_stride * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dP.p, params4, (size_t)n_rows * 16, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dG.p, gains2, (size_t)n_rows * 8, cudaMemcpyHostToDevice));
    CU(launch_op_comb_inplace(dY.as<float>(), row_stride, (int)y_offset, (int)n, n_rows, dP.as<int32_t>(), dG.as<float>(),
                              (int)overlap, nullptr));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(y, dY.p, (size_t)n_rows * row_stride * 4, cudaMemcpyDeviceToHost));
    return OPN_OK;
}

int opn_op_comb_filter(int device, float *y, const float *x, size_t row_stride, size_t offset, size_t n, uint32_t n_rows,
                       const int32_t *params4, const float *gains2, size_t overlap)
{
    if (!y || !x || !comb_args_ok(offset, n, n_rows, params4, gains2, row_stride, overlap)) return OPN_ERR_BAD_ARG;
    int rc = select_device(device);
    if (rc) return rc;
    DevBuf dY, dX, dP, dG;
    CU(dY.alloc((size_t)n_rows * row_stride * 4));
    CU(dX.alloc((size_t)n_rows * row_stride * 4));
    CU(dP.alloc((size_t)n_rows * 16));
    CU(dG.alloc((size_t)n_rows * 8));
    CU(cudaMemcpy(dY.p, y, (size_t)n_rows * row_stride * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dX.p, x, (size_t)n_rows * row_stride * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dP.p, params4, (size_t)n_rows * 16, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dG.p, gains2, (size_t)n_rows * 8, cudaMemcpyHostToDevice));
    CU(launch_op_comb(dY.as<float>(), dX.as<float>(), row_stride, (int)offset, (int)n, n_rows, dP.as<int32_t>(), dG.as<float>(),
                      (int)overlap, nullptr));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(y, dY.p, (size_t)n_rows * row_stride * 4, cudaMemcpyDeviceToHost));
    return OPN_OK;
}

int opn_op_pcm_soft_clip(int device, float *pcm, size_t row_stride, size_t row_len, int channels, uint32_t n_rows,
                         float *softclip_mem)
{
    if (!pcm || !softclip_mem || n_rows == 0 || channels < 1 || row_len > row_stride) return OPN_ERR_BAD_ARG;
    int rc = select_device(device);
    if (rc) return rc;
    DevBuf dP, dM;
    CU(dP.alloc((size_t)n_rows * row_stride * 4));
    CU(dM.alloc((size_t)n_rows * channels * 4));
    CU(cudaMemcpy(dP.p, pcm, (size_t)n_rows * row_stride * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dM.p, softclip_mem, (size_t)n_rows * channels * 4, cudaMemcpyHostToDevice));
    CU(launch_op_soft_clip(dP.as<float>(), row_stride, row_len, channels, n_rows, dM.as<float>(), nullptr));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(pcm, dP.p, (size_t)n_rows * row_stride * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(softclip_mem, dM.p, (size_t)n_rows * channels * 4, cudaMemcpyDeviceToHost));
    return OPN_OK;
}

int opn_op_smooth_fade(int device, const float *in1, const float *in2, float *out, size_t row_stride, size_t overlap, int channels,
                       int32_t fs_hz, uint32_t n_rows)
{
    if (!in1 || !in2 || !out || n_rows == 0 || channels < 1 || channels > 2 || overlap * (size_t)channels > row_stride) return OPN_ERR_BAD_ARG;
    if (fs_hz <= 0 || 48000 % fs_hz != 0 || (overlap > 0 && (overlap - 1) * (size_t)(48000 / fs_hz) >= 120)) return OPN_ERR_BAD_ARG;
    int rc = select_device(device);
    if (rc) return rc;
    const size_t bytes = (size_t)n_rows * row_stride * 4;
    DevBuf d1, d2;
    CU(d1.alloc(bytes));
    CU(d2.alloc(bytes));
    CU(cudaMemcpy(d1.p, in1, bytes, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d2.p, in2, bytes, cudaMemcpyHostToDevice));
    // the result goes into in1's copy (smooth_fade_into_in1); the caller's `out` may be either input or a third buffer
    CU(launch_op_smooth_fade(d1.as<float>(), d2.as<float>(), d1.as<float>(), row_stride, (int)overlap, channels, fs_hz, n_rows, nullptr));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(out, d1.p, bytes, cudaMemcpyDeviceToHost));
    return OPN_OK;
}

int opn_op_bitexact_trig(int device, const int16_t *x, int16_t *cos_out, uint32_t n_cos, const int32_t *isin, const int32_t *icos,
                         int32_t *log2tan_out, uint32_t n_log2tan)
{
    if ((n_cos && (!x || !cos_out)) || (n_log2tan && (!isin || !icos || !log2tan_out))) return OPN_ERR_BAD_ARG;
    int rc = select_device(device);
    if (rc) return rc;
    DevBuf dX, dC, dS, dK, dL;
    CU(dX.alloc((size_t)n_cos * 2));
    CU(dC.alloc((size_t)n_cos * 2));
    CU(dS.alloc((size_t)n_log2tan * 4));
    CU(dK.alloc((size_t)n_log2tan * 4));
    CU(dL.alloc((size_t)n_log2tan * 4));
    if (n_cos) CU(cudaMemcpy(dX.p, x, (size_t)n_cos * 2, cudaMemcpyHostToDevice));
    if (n_log2tan) {
        CU(cudaMemcpy(dS.p, isin, (size_t)n_log2tan * 4, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(dK.p, icos, (size_t)n_log2tan * 4, cudaMemcpyHostToDevice));
    }
    CU(launch_op_bitexact_trig(dX.as<int16_t>(), dC.as<int16_t>(), n_cos, dS.as<int32_t>(), dK.as<int32_t>(), dL.as<int32_t>(),
                               n_log2tan, nullptr));
    CU(cudaDeviceSynchronize());
    if (n_cos) CU(cudaMemcpy(cos_out, dC.p, (size_t)n_cos * 2, cudaMemcpyDeviceToHost));
    if (n_log2tan) CU(cudaMemcpy(log2tan_out, dL.p, (size_t)n_log2tan * 4, cudaMemcpyDeviceToHost));
    return OPN_OK;
}

int opn_op_synth_symbols(int device, const uint8_t *arena, const uint32_t *offsets, const uint32_t *lens, uint32_t n_packets,
                         int lm, int channels, opn_synth_side *side_out, int32_t *y_out, float *coef_out)
{
    if (!arena || !offsets || !lens || n_packets == 0 || lm < 0 || lm > 3 || channels < 1 || channels > 2) return OPN_ERR_BAD_ARG;
    int rc = select_device(device);
    if (rc) return rc;
    size_t arena_end = 0;
    uint32_t max_len = 8;
    for (uint32_t i = 0; i < n_packets; i++) {
        arena_end = std::max(arena_end, (size_t)offsets[i] + lens[i]);
        max_len = std::max(max_len, lens[i]);
    }
    const size_t row = (size_t)channels * (120u << lm);
    DevBuf dA, dO, dL, dS, dSt, dY, dC, dI, dH;
    CU(dA.alloc(arena_end));
    CU(dO.alloc(n_packets * 4));
    CU(dL.alloc(n_packets * 4));
    CU(dS.alloc((size_t)n_packets * sizeof(opn_synth_side)));
    CU(dSt.alloc(n_packets * 4));
    CU(dH.alloc((size_t)n_packets * sizeof(uint4)));
    CU(dY.alloc((size_t)n_packets * row * 4));
    CU(dC.alloc((size_t)n_packets * row * 4));
    CU(dI.alloc((size_t)n_packets * 72 * 4));
    CU(cudaMemcpy(dA.p, arena, arena_end, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dO.p, offsets, n_packets * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dL.p, lens, n_packets * 4, cudaMemcpyHostToDevice));
    CU(cudaMemset(dS.p, 0, (size_t)n_packets * sizeof(opn_synth_side)));
    SymbolArgs s{};
    s.arena = dA.as<uint8_t>();
    s.offsets = dO.as<uint32_t>();
    s.lens = dL.as<uint32_t>();
    s.n_items = n_packets;
    s.lm = lm;
    s.channels = channels;
    s.has_toc = 0;
    s.side = dS.as<opn_synth_side>();
    s.hdr = dH.as<uint4>();
    s.status = dSt.as<int32_t>();
    s.coef = dC.as<float>();
    s.y_out = dY.as<int32_t>();
    s.idx = dI.as<uint32_t>();
    s.pkt_cap = (max_len + 15u) & ~15u;
    CU(launch_synth_symbols(s, nullptr));
    CU(cudaDeviceSynchronize());
    if (side_out) CU(cudaMemcpy(side_out, dS.p, (size_t)n_packets * sizeof(opn_synth_side), cudaMemcpyDeviceToHost));
    if (y_out) CU(cudaMemcpy(y_out, dY.p, (size_t)n_packets * row * 4, cudaMemcpyDeviceToHost));
    if (coef_out) CU(cudaMemcpy(coef_out, dC.p, (size_t)n_packets * row * 4, cudaMemcpyDeviceToHost));
    return OPN_OK;
}

int opn_op_celt2_symbols(int device, const uint8_t *arena, const uint32_t *offsets, const uint32_t *lens, uint32_t n_packets,
                         int lm, int channels, opn_celt2_side *side_out, int32_t *y_out, float *coef_out)
{
    if (!arena || !offsets || !lens || n_packets == 0 || lm < 0 || lm > 3 || channels < 1 || channels > 2) return OPN_ERR_BAD_ARG;
    int rc = select_device(device);
    if (rc) return rc;
    size_t arena_end = 0;
    for (uint32_t i = 0; i < n_packets; i++) arena_end = std::max(arena_end, (size_t)offsets[i] + lens[i]);
    const size_t row = (size_t)channels * (120u << lm);
    DevBuf dA, dO, dL, dS, dSt, dY, dC, dH, dP, dE;
    CU(dE.alloc((size_t)n_packets * 42 * sizeof(int16_t)));
    CU(dA.alloc(arena_end + 8));
    CU(dO.alloc(n_packets * 4));
    CU(dL.alloc(n_packets * 4));
    CU(dS.alloc((size_t)n_packets * sizeof(Celt2Side)));
    CU(dSt.alloc(n_packets * 4));
    CU(dH.alloc((size_t)n_packets * sizeof(uint4)));
    CU(dP.alloc((size_t)n_packets * CELT2_MAX_PARTS * sizeof(Celt2Part)));
    CU(dY.alloc((size_t)n_packets * row * 4));
    CU(dC.alloc((size_t)n_packets * row * 4));
    CU(cudaMemcpy(dA.p, arena, arena_end, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dO.p, offsets, n_packets * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dL.p, lens, n_packets * 4, cudaMemcpyHostToDevice));
    CU(cudaMemset(dY.p, 0, (size_t)n_packets * row * 4));
    CU(cudaMemset(dC.p, 0, (size_t)n_packets * row * 4));
    SymbolArgs s{};
    s.arena = dA.as<uint8_t>();
    s.offsets = dO.as<uint32_t>();
    s.lens = dL.as<uint32_t>();
    s.n_items = n_packets;
    s.lm = lm;
    s.channels = channels;
    s.has_toc = 0;
    s.hdr = dH.as<uint4>();
    s.status = dSt.as<int32_t>();
    s.coef = dC.as<float>();
    s.y_out = dY.as<int32_t>();
    s.parts = dP.as<Celt2Part>();
    s.side2 = dS.as<Celt2Side>();
    s.bande = dE.as<int16_t>();
    CU(launch_celt2_rangedec(s, nullptr));
    CU(launch_celt2_expand(s, nullptr));
    CU(cudaDeviceSynchronize());
    if (side_out) CU(cudaMemcpy(side_out, dS.p, (size_t)n_packets * sizeof(Celt2Side), cudaMemcpyDeviceToHost));
    if (y_out) CU(cudaMemcpy(y_out, dY.p, (size_t)n_packets * row * 4, cudaMemcpyDeviceToHost));
    if (coef_out) CU(cudaMemcpy(coef_out, dC.p, (size_t)n_packets * row * 4, cudaMemcpyDeviceToHost));
    return OPN_OK;
}

// SYNTH-SILK/1 operator: every packet is decoded by a fresh decoder (zero state) through the product's two kernels.
int opn_op_silk_frames(int device, const uint8_t *arena, const uint32_t *offsets, const uint32_t *lens, uint32_t n_packets,
                       int stream_channels, int channels, size_t frame_size, int decode_fec, opn_silk_side *side_out, int32_t *exc_out,
                       int16_t *out16, float *pcm_out, int32_t *result)
{
    if (!arena || !offsets || !lens || n_packets == 0 || channels < 1 || channels > 2 || stream_channels < 1 || stream_channels > 2)
        return OPN_ERR_BAD_ARG;
    if (frame_size != 480 && frame_size != 960) return OPN_ERR_BAD_ARG;
    int rc = select_device(device);
    if (rc) return rc;
    size_t arena_end = 0;
    for (uint32_t i = 0; i < n_packets; i++) arena_end = std::max(arena_end, (size_t)offsets[i] + lens[i]);
    const size_t n = n_packets, row = frame_size * (size_t)channels;
    DevBuf dA, dO, dL, dS, dSt, dH, dR, dX, dY, dP, dRes, dRing, dPos, dFin;
    DevBuf sL, sH, sA, sG, sR, sF;
    CU(dA.alloc(arena_end + 8));
    CU(dO.alloc(n * 4));
    CU(dL.alloc(n * 4));
    CU(dS.alloc(n * sizeof(opn_silk_side)));
    CU(dSt.alloc(n * 4));
    CU(dH.alloc(n * sizeof(uint4)));
    CU(dR.alloc(n * 2 * sizeof(SilkRec)));
    CU(dX.alloc(n * 2 * SILK_MAX_FRAME * 4));
    CU(dY.alloc(n * 2 * SILK_MAX_FRAME * 2));
    CU(dP.alloc(n * row * 4));
    CU(dRes.alloc(n * 4));
    CU(dRing.alloc(n * (size_t)channels * RING_SAMPLES * 4));
    CU(dPos.alloc(n * 4));
    CU(dFin.alloc(n * 4));
    CU(sL.alloc(n * 2 * 16 * 4));
    CU(sH.alloc(n * 2 * SILK_HIST * 4));
    CU(sA.alloc(n * 2 * 16 * 2));
    CU(sG.alloc(n * 2 * 4));
    CU(sR.alloc(n * 2 * 8 * 4));
    CU(sF.alloc(n * 2));
    CU(cudaMemcpy(dA.p, arena, arena_end, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dO.p, offsets, n * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dL.p, lens, n * 4, cudaMemcpyHostToDevice));
    CU(cudaMemset(dS.p, 0, n * sizeof(opn_silk_side)));
    CU(cudaMemset(dX.p, 0, n * 2 * SILK_MAX_FRAME * 4));
    CU(cudaMemset(dY.p, 0, n * 2 * SILK_MAX_FRAME * 2));
    CU(cudaMemset(dP.p, 0, n * row * 4));
    CU(cudaMemset(dPos.p, 0, n * 4));
    CU(cudaMemset(sL.p, 0, n * 2 * 16 * 4));
    CU(cudaMemset(sH.p, 0, n * 2 * SILK_HIST * 4));
    CU(cudaMemset(sA.p, 0, n * 2 * 16 * 2));
    CU(cudaMemset(sG.p, 0, n * 2 * 4));
    CU(cudaMemset(sR.p, 0, n * 2 * 8 * 4));
    CU(cudaMemset(sF.p, 0, n * 2));
    SilkArgs a{};
    a.arena = dA.as<uint8_t>();
    a.offsets = dO.as<uint32_t>();
    a.lens = dL.as<uint32_t>();
    a.n_items = n_packets;
    a.frame_ms = frame_size == 960 ? 20 : 10;
    a.stream_channels = stream_channels;
    a.channels = channels;
    a.has_toc = 1;
    a.bandwidth = -1;
    a.fec = decode_fec ? 1 : 0;
    a.rec = dR.as<SilkRec>();
    a.hdr = dH.as<uint4>();
    a.status = dSt.as<int32_t>();
    a.st = SilkState{sL.as<int32_t>(), sH.as<int32_t>(), sA.as<int16_t>(), sG.as<int32_t>(), sR.as<float>(), sF.as<uint8_t>()};
    a.ring = dRing.as<float>();
    a.ring_pos = dPos.as<uint32_t>();
    a.dense = dP.as<float>();
    a.dense_stride = row;
    a.gain = 1.0f;
    a.result = dRes.as<int32_t>();
    a.final_range = dFin.as<uint32_t>();
    a.side = dS.as<opn_silk_side>();
    a.exc_out = dX.as<int32_t>();
    a.out16 = dY.as<int16_t>();
    CU(launch_silk_rangedec(a, nullptr));
    CU(launch_silk_frame(a, nullptr));
    CU(cudaDeviceSynchronize());
    if (side_out) CU(cudaMemcpy(side_out, dS.p, n * sizeof(opn_silk_side), cudaMemcpyDeviceToHost));
    if (exc_out) CU(cudaMemcpy(exc_out, dX.p, n * 2 * SILK_MAX_FRAME * 4, cudaMemcpyDeviceToHost));
    if (out16) CU(cudaMemcpy(out16, dY.p, n * 2 * SILK_MAX_FRAME * 2, cudaMemcpyDeviceToHost));
    if (pcm_out) CU(cudaMemcpy(pcm_out, dP.p, n * row * 4, cudaMemcpyDeviceToHost));
    if (result) CU(cudaMemcpy(result, dRes.p, n * 4, cudaMemcpyDeviceToHost));
    return OPN_OK;
}

}  // extern "C"
