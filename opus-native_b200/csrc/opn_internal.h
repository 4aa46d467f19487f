// opn_internal.h -- declarations shared by the CUDA translation unit and the C++ host runtime.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/opusb200.h"

namespace opn {

struct Celt2Part;
struct Celt2Side;

constexpr int SYM_WARPS_PER_CTA = 4;
#ifndef OPN_RD_WARPS
#define OPN_RD_WARPS 1
#endif
// k_synth_rangedec: one packet per thread.  1, 2, 4 and 8 warps per CTA measure the same (46.7-48 us per step):
// the SMs' 32 CTA slots are not what the long-running entropy launches take from the other kernels.
constexpr int RANGEDEC_WARPS_PER_CTA = OPN_RD_WARPS;
#ifndef OPN_EXPAND_WARPS
#define OPN_EXPAND_WARPS 4
#endif
constexpr int EXPAND_WARPS_PER_CTA = OPN_EXPAND_WARPS;  // stand-alone k_synth_expand: 47 KB per CTA (tables 16.5 KB + 7.5 KB of rows per warp)
constexpr int IM_TPC = 128;         // threads per row of the out-of-place comb operator kernel
// per-channel PCM ring (output + comb history): 3 x 960 = 6 x 480 = 12 x 240 = 24 x 120 samples.  A frame never overlaps
// the history it is filtered against: 960 + 1024 + 2 <= 2880.
constexpr int RING_SAMPLES = 2880;
constexpr int32_t ITEM_OK = 0, ITEM_LOST = 1;  // kernel-0 status; negative = OPN_ERR_* (state untouched)

struct PfState {  // post-filter parameters of the previous frame
    int32_t period, tapset;
    float gain;
    // 1 + LM of the frame size the stream conceals a loss with, 0 = no packet yet: the size of its last frame that came from
    // a packet, decoded or PLC/DTX (a TOC with a payload of at most one byte: libopus takes st->frame_size from the TOC
    // before it decodes the frames).  Written by every CELT frame kernel and by the SILK frame kernel (960 -> 4, 480 -> 3).
    int32_t lm1;
};

// Frame header, range decode -> frame kernel: one uint4 per stream.
//   .x = silence | postfilter << 1 | transient << 2 | intra << 3 | tapset << 4 | gain_idx << 8 | octave << 12 | period << 16
//   .y = final range (Decoder::final_range), .z = tell_frac, .w = number of pulses
// A lost item's header is zero but for HDR_DTX in .x: the item came from a packet (PLC/DTX), so it sets PfState::lm1.  On
// the host path an item came from a packet when its offset is not 0: a concealed frame has offset 0, a parsed frame starts
// after its packet's TOC.
constexpr uint32_t HDR_DTX = 1u << 15;
__host__ __device__ inline uint32_t hdr_pack(uint32_t silence, uint32_t postfilter, uint32_t transient, uint32_t intra, uint32_t tapset,
                                             uint32_t gain_idx, uint32_t octave, uint32_t period)
{
    return silence | postfilter << 1 | transient << 2 | intra << 3 | tapset << 4 | gain_idx << 8 | octave << 12 | period << 16;
}

// ---- steps whose streams have different frame sizes (OPN_FLAG_MIXED_FRAMES): device-side bucketing
// The streams of a batch are cut into MIX_GROUPS contiguous ranges (the frame kernel's concurrent launches: a stream stays
// on its group's CUDA stream for life) and, inside a group, sorted by frame size.  Bucket (g, lm) owns the items
// [start, start + count); every bucket starts on a multiple of MIX_PAD items so that a range-decode CTA never spans two
// frame sizes.  Written by k_mix_place, read by the range decode and frame kernels of the same step.
#ifndef OPN_FRAME_GROUPS
#define OPN_FRAME_GROUPS 3  // a library variant must be built with the same value in the kernels and in the host runtime
#endif
constexpr int MIX_GROUPS = OPN_FRAME_GROUPS > 1 ? OPN_FRAME_GROUPS : 1;
constexpr uint32_t MIX_PAD = 32u * OPN_RD_WARPS;
constexpr uint8_t MIX_NO_ITEM = 0xFF;
struct MixPlan {
    uint32_t count[MIX_GROUPS][4];
    uint32_t start[MIX_GROUPS][4];
    uint32_t cta0[MIX_GROUPS][5];  // frame kernel: first CTA of group g's j-th bucket (lm = 3 - j: longest frames first); [4] = CTAs in use
    uint32_t items_padded;         // items up to the end of the last bucket
};
__host__ __device__ constexpr uint32_t mix_item_cap(uint32_t n_streams) { return n_streams + MIX_GROUPS * 4u * MIX_PAD; }

struct SymbolArgs {
    const uint8_t *arena;
    const uint32_t *offsets;     // [n_items] byte offset of the packet (or of the payload if !has_toc)
    const uint32_t *lens;        // [n_items] bytes, 0 = lost
    const uint32_t *stream_idx;  // [n_items] or nullptr (item k = stream k)
    uint32_t n_items;
    int lm, channels, has_toc;
    opn_synth_side *side;        // [n_streams] or nullptr: full side record (tests)
    uint4 *hdr;                  // [n_streams] frame header for the frame kernel
    int32_t *status;             // [n_streams]
    float *coef;                 // [n_streams][channels][120<<lm] or nullptr
    int32_t *y_out;              // same shape or nullptr
    uint32_t *idx;               // [n_streams][72] scratch: PVQ codeword indices (range decode -> expansion)
    uint32_t pkt_cap;            // bytes of shared memory per warp for the packet
    struct Celt2Part *parts;     // SYNTH-CELT/2: [n_streams][CELT2_MAX_PARTS] PVQ leaves (range decode -> expansion)
    struct Celt2Side *side2;     // SYNTH-CELT/2: [n_streams] or nullptr: full side record (tests)
    int16_t *bande;              // SYNTH-CELT/2: [n_streams][2][21] band energies in Q9 (range decode -> expansion) or nullptr
    const uint8_t *item_lm;      // mixed-frame step: [n_items] LM of the item, MIX_NO_ITEM = padding (overrides lm); else nullptr
};

struct FrameArgs {
    const uint32_t *idx;          // [n_streams][72] PVQ codeword indices (range decode output, SYNTH-CELT/1)
    const struct Celt2Part *parts;  // [n_streams][CELT2_MAX_PARTS] PVQ leaves (range decode output, SYNTH-CELT/2) or nullptr
    const uint4 *hdr;             // [n_streams] frame headers (range decode output)
    const int32_t *status;        // [n_streams]  (range decode output)
    const uint32_t *stream_idx;   // [n_items] or nullptr
    uint32_t n_items;             // items of the bucket
    uint32_t item0, item_end;     // this launch covers items [item0, item_end) of them (a bucket may be cut into groups)
    int lm, channels, postfilter;
    int stream_channels;          // channels of the packets (decoder.rs:332 stream_channels); 0 = the decoder's
    float *carry;                 // [n_streams][C][60]
    float *ring;                  // [n_streams][RING_SAMPLES][C]
    uint32_t *ring_pos;           // [n_streams]
    PfState *pf;                  // [n_streams]
    float *dense;                 // [n_streams] rows of dense_stride floats, or nullptr
    size_t dense_stride;
    const uint32_t *dense_off;    // [n_items] float offset inside the row (frame w of a packet: w*nf*C) or nullptr
    float gain;                   // DecoderConfiguration::gain as a linear factor (decoder.rs:790-797); 1 = none
    int32_t *result;              // [n_streams] samples per channel or OPN_ERR_*; nullptr to skip
    uint32_t *final_range;        // [n_streams]
    float *softclip_reset;        // [n_streams][2] or nullptr: cleared for every stream that decodes a packet (decoder.rs:420-423)
    unsigned long long *hist_samples;  // measurement (or nullptr): += max(T0,T1)+2 per channel-frame the post-filter runs on
    const int16_t *bande;         // SYNTH-CELT/2: [n_streams][2][21] band energies in Q9 (range decode output)
    const MixPlan *plan;          // mixed-frame step (k_frame_mix): buckets of this step, else nullptr
    int group;                    // mixed-frame step: which group of the plan this launch covers
};

struct MixArgs {  // k_mix_key / k_mix_place
    const uint8_t *arena;
    const uint32_t *offsets, *lens;  // [n_streams] the caller's arrays
    uint32_t n_streams;
    int channels, n_groups;          // n_groups = 1 or MIX_GROUPS
    uint32_t capacity;               // samples per channel the caller's rows hold (frame_size argument)
    uint8_t *last_lm;                // [n_streams] LM of the stream's last packet (decoded or PLC/DTX), MIX_NO_ITEM = none yet (state)
    const PfState *pf;               // [n_streams] or nullptr: after other CELT steps, last_lm is first taken from PfState::lm1
    uint8_t *key;                    // [n_streams] scratch: g*4 + lm, or MIX_NO_ITEM
    uint32_t *rank;                  // [n_streams] scratch: position inside the bucket
    MixPlan *plan;                   // zeroed before k_mix_key
    uint32_t *item_offsets, *item_lens, *item_stream;  // [mix_item_cap] out
    uint8_t *item_lm;                // [mix_item_cap] out, preset to MIX_NO_ITEM
    int32_t *result;                 // [n_streams] or nullptr: OPN_ERR_* of the streams no bucket takes
};

// ---- SYNTH-SILK/1 (silk.cuh; DESIGN.md section 3c)
constexpr int SILK_MAX_FRAME = 320;  // 20 ms at 16 kHz
constexpr int SILK_HIST = 320;       // excitation history of the long-term predictor
constexpr int SILK_ROWS = 32;        // coded channels per CTA
constexpr int SILK_WARPS = 8;
constexpr int SILK_RS = 33;          // row stride of the transposed rows (words)

// range decode -> frame kernel, one per coded channel
struct alignas(16) SilkRec {
    uint32_t index[20];
    uint16_t lag[4];
    uint8_t pulses[20];
    uint8_t rc[16];
    uint8_t gidx[4], ltp[4];
    uint8_t type, seed, pad[2];
    uint32_t pad2[2];
};
static_assert(sizeof(SilkRec) == 144, "SilkRec layout");

struct SilkState {  // per stream (structure of arrays, device)
    int32_t *slpc;   // [n][2][16]  sLPC_Q14 of the last 16 samples, [15] newest
    int32_t *hist;   // [n][2][SILK_HIST] excitation after long-term prediction, newest last
    int16_t *a_q12;  // [n][2][16]
    int32_t *gain;   // [n][2]
    float *rs;       // [n][2][8] resampler history per output channel: rs[j] = x[-1-j]
    uint8_t *fs;     // [n][2]: internal rate of the previous SILK frame in kHz (0 = none), its coded channels
};

struct SilkArgs {
    const uint8_t *arena;
    const uint32_t *offsets, *lens, *stream_idx;  // per item; stream_idx may be nullptr
    uint32_t n_items;
    uint32_t item0, item_end;  // frame kernel: this launch covers items [item0, item_end) (a large bucket is cut into groups); 0, 0 = all
    int frame_ms;          // 10 or 20: every item of the launch
    int stream_channels;   // coded channels of every item
    int channels;          // the decoder's
    int has_toc;           // 1: offsets point at the TOC (device-resident steps); 0: at the frame payload, bandwidth below
    int bandwidth;         // host path: 0 NB, 1 MB, 2 WB of every item
    int fec;               // LostFlag::DecodeFec: decode each packet's redundant copy of the previous frame (none: conceal)
    SilkRec *rec;          // [n_streams][2]
    uint4 *hdr;            // [n_streams] .x = fs_khz of the frame, .y final range, .z tell_frac
    int32_t *status;       // [n_streams]
    SilkState st;
    float *ring;           // [n_streams][RING_SAMPLES][C]
    uint32_t *ring_pos;
    float *dense;          // rows of dense_stride floats or nullptr
    size_t dense_stride;
    const uint32_t *dense_off;
    float gain;
    int32_t *result;
    uint32_t *final_range;
    float *softclip_reset;
    PfState *pf;           // [n_streams] or nullptr: the frame kernel records the frame size in PfState::lm1
    // operator entry / tests (indexed by stream)
    opn_silk_side *side;   // or nullptr
    int32_t *exc_out;      // [n_streams][2][SILK_MAX_FRAME] or nullptr
    int16_t *out16;        // [n_streams][2][SILK_MAX_FRAME] or nullptr
    unsigned long long *phase_clk;  // measurement (OPN_SILK_CLK=1): [3] cycles in phases A, B, C summed over CTAs, [3] = CTAs; else nullptr
};

// ---- launchers (opn_kernels.cu).  All return a cudaError_t and never synchronise.
cudaError_t upload_tables(int device);  // idempotent per device
cudaError_t launch_rangedec_script(const uint8_t *arena, const uint32_t *offsets, const uint32_t *lens, uint32_t n_packets,
                                   const opn_op *ops, uint32_t n_ops, const uint8_t *icdf_pool, opn_op_out *out,
                                   int32_t *y_out, uint32_t y_stride, uint32_t pkt_cap, cudaStream_t st);
cudaError_t launch_synth_symbols(const SymbolArgs &a, cudaStream_t st);   // both stages on one stream
cudaError_t launch_synth_rangedec(const SymbolArgs &a, cudaStream_t st);  // stage 0a: one lane per packet
cudaError_t launch_synth_expand(const SymbolArgs &a, cudaStream_t st);    // stage 0b: one warp per packet
cudaError_t launch_celt2_rangedec(const SymbolArgs &a, cudaStream_t st);  // SYNTH-CELT/2: one lane per packet -> header + part list
cudaError_t launch_celt2_expand(const SymbolArgs &a, cudaStream_t st);    // SYNTH-CELT/2 operator: part lists -> coefficient rows
// the frame kernel: PVQ expansion + IMDCT + TDAC + comb post-filter + PCM store
cudaError_t launch_frame(const FrameArgs &a, cudaStream_t st);
// mixed-frame step: bucketing (two kernels on one stream) and the frame kernel of one group (a.plan, a.group; grid sized by the
// caller's upper bound n_streams_in_group)
cudaError_t launch_mix_plan(const MixArgs &a, cudaStream_t st);
cudaError_t launch_op_smooth_fade(const float *in1, const float *in2, float *out, size_t row_stride, int overlap, int channels, int fs,
                                  uint32_t n_rows, cudaStream_t st);
cudaError_t launch_silk_rangedec(const SilkArgs &a, cudaStream_t st);  // one lane per packet -> one record per coded channel
cudaError_t launch_silk_frame(const SilkArgs &a, cudaStream_t st);     // excitation + LTP + LPC synthesis + resampler + PCM store
cudaError_t launch_transition_fade(float *dense, size_t dense_stride, const uint32_t *d_streams, uint32_t n_streams, uint32_t n_rows, int channels,
                                   cudaStream_t st);  // CELT -> SILK: 2.5 ms of the old decoder's concealment, then a 2.5 ms cross-fade
int kernels_frame_groups();  // OPN_FRAME_GROUPS the kernels were built with
cudaError_t launch_frame_mix(const FrameArgs &a, uint32_t n_streams_in_group, cudaStream_t st);
cudaError_t launch_op_imdct(const float *in, size_t in_stride, float *out, size_t out_stride, uint32_t n_rows, int shift,
                            int nblk, cudaStream_t st);
cudaError_t launch_op_comb_inplace(float *y, size_t row_stride, int y_offset, int n, uint32_t n_rows, const int32_t *params4,
                                   const float *gains2, int overlap, cudaStream_t st);
cudaError_t launch_op_comb(float *y, const float *x, size_t row_stride, int offset, int n, uint32_t n_rows,
                           const int32_t *params4, const float *gains2, int overlap, cudaStream_t st);
cudaError_t launch_op_bitexact_trig(const int16_t *x, int16_t *out_cos, uint32_t n_cos, const int32_t *isin, const int32_t *icos,
                                    int32_t *out_l2t, uint32_t n_l2t, cudaStream_t st);
cudaError_t launch_softclip_convert(int sample_format, const float *dense, size_t dense_stride, const int32_t *clip_len, int channels,
                                    uint32_t row_floats, uint32_t first_row, uint32_t n_rows, float *mem, void *out, size_t out_stride,
                                    cudaStream_t st);
cudaError_t launch_op_soft_clip(float *pcm, size_t row_stride, size_t row_len, int channels, uint32_t n_rows, float *mem,
                                cudaStream_t st);

// ---- host-side pieces (host_*.cpp)
float host_gain_from_q8(int16_t gain_q8);  // decoder.rs:790-791

}  // namespace opn
