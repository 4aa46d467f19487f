/* opusb200.h -- C ABI of the B200-native batched Opus decode engine (libopusb200.so).
 *
 * Drop-in boundary for the decode path of the Rust crate hasenbanck/opus-native.  The crate
 * has no FFI of its own (SURVEY.md 8b); each entry point below names the crate item it
 * stands in for (paths relative to the crate root).  INTEGRATION.md shows the Rust
 * `extern "C"` block and the safe wrapper a maintainer would add on the crate side.
 *
 * Rules: plain pointers and sizes only; no exceptions cross the ABI; the library keeps no
 * caller pointer after a call returns (async device calls: after opn_batch_synchronize);
 * one in-flight call per handle; handles are bound to one CUDA device.  There is no CPU
 * fallback: every decode entry point fails with OPN_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef OPUSB200_H
#define OPUSB200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- errors: OpusError, src/error.rs:5-16 ------------------------------------------- */
#define OPN_OK 0
#define OPN_ERR_BAD_ARG (-1)              /* OpusError::BadArguments       */
#define OPN_ERR_BUFFER_TOO_SMALL (-2)     /* OpusError::BufferToSmall      */
#define OPN_ERR_INTERNAL (-3)             /* OpusError::InternalError      */
#define OPN_ERR_INVALID_PACKET (-4)       /* OpusError::InvalidPacket      */
#define OPN_ERR_FRAME_SIZE_TOO_SMALL (-5) /* OpusError::FrameSizeTooSmall  */
#define OPN_ERR_UNIMPLEMENTED (-6)        /* reference: todo!()/unimplemented!() (SILK, hybrid, PLC bodies) */
#define OPN_ERR_CUDA (-7)                 /* CUDA runtime failure or no usable device */
const char *opn_strerror(int code);       /* Display for OpusError, src/error.rs:18-38 */
const char *opn_last_cuda_error(void);    /* thread-local text of the last CUDA failure */
int opn_device_count(void);

/* ---- packet inspection: src/lib.rs:219-498 (host only) ------------------------------ */
enum { OPN_BW_NARROW = 0, OPN_BW_MEDIUM = 1, OPN_BW_WIDE = 2, OPN_BW_SUPERWIDE = 3, OPN_BW_FULL = 4 };
enum { OPN_MODE_SILK = 0, OPN_MODE_HYBRID = 1, OPN_MODE_CELT = 2 };
int opn_packet_bandwidth(const uint8_t *packet);                             /* query_packet_bandwidth         lib.rs:219 */
int opn_packet_channels(const uint8_t *packet);                              /* query_packet_channel_count     lib.rs:233 */
int opn_packet_frame_count(const uint8_t *packet, size_t len);               /* query_packet_frame_count       lib.rs:250 */
int opn_packet_samples_per_frame(const uint8_t *packet, int32_t fs_hz);      /* query_packet_samples_per_frame lib.rs:271 */
int opn_packet_sample_count(const uint8_t *packet, size_t len, int32_t fs_hz); /* query_packet_sample_count    lib.rs:299 */
int opn_packet_mode(const uint8_t *packet);                                  /* query_packet_codec_mode        lib.rs:317 */
/* parse_packet, lib.rs:345-498.  frames may be NULL.  Returns the frame count or an error. */
int opn_parse_packet(const uint8_t *packet, size_t len, int self_delimited, uint32_t frames[48],
                     uint32_t sizes[48], uint32_t *payload_offset, uint32_t *packet_offset);

/* ---- single-stream decoder: Decoder / DecoderConfiguration, src/decoder.rs:27-232 --- */
typedef struct opn_decoder opn_decoder;
/* Decoder::new (decoder.rs:61); fs_hz in {8000,12000,16000,24000,48000}, channels in {1,2}.
 * Only 48000 Hz is implemented (the crate never computes its `downsample`, celt/decoder.rs:23). */
int opn_decoder_create(int device, int32_t fs_hz, int32_t channels, int16_t gain_q8, int32_t bitstream /* OPN_BITSTREAM_* */,
                       opn_decoder **out);
void opn_decoder_destroy(opn_decoder *dec);
int opn_decoder_reset(opn_decoder *dec);                                     /* Decoder::reset decoder.rs:74 */
/* Decoder::decode_float (decoder.rs:216-232).  packet == NULL means a lost packet.  Returns
 * samples per channel (>= 0) or an error.  pcm holds frame_size*channels interleaved floats. */
int opn_decode_float(opn_decoder *dec, const uint8_t *packet, size_t len, float *pcm,
                     size_t frame_size, int decode_fec);
/* Decoder::decode::<i16> (decoder.rs:148-193): soft clip then Sample::from_f32 (lib.rs:76-82).
 * pcm_capacity is the slice length the Rust caller would pass (`samples.len()`). */
int opn_decode_i16(opn_decoder *dec, const uint8_t *packet, size_t len, int16_t *pcm,
                   size_t pcm_capacity, size_t frame_size, int decode_fec);
/* Decoder::decode::<S> (decoder.rs:148-193) for every S the crate implements `Sample` for (lib.rs:63-107):
 * pcm_soft_clip, then S::from_f32 on the device.  sample_format picks S; pcm points at pcm_capacity elements of
 * that type.  The crate's conversions are kept as written: i16/i32 clamp to the type's range (the i32 bound
 * 2147483647.0 rounds to 2^31 in f32 and the cast saturates), u16/u32 clamp to [0, 32768] / [0, 2^31] (upper
 * bound = midpoint + full scale, lib.rs:93-107), NaN converts to 0 like a Rust `as` cast. */
#define OPN_SAMPLE_F32 0 /* Sample for f32, lib.rs:63-68  */
#define OPN_SAMPLE_I16 1 /* Sample for i16, lib.rs:77-83  */
#define OPN_SAMPLE_I32 2 /* Sample for i32, lib.rs:85-91  */
#define OPN_SAMPLE_U16 3 /* Sample for u16, lib.rs:93-99  */
#define OPN_SAMPLE_U32 4 /* Sample for u32, lib.rs:101-107 */
#define OPN_SAMPLE_F64 5 /* Sample for f64, lib.rs:70-75  */
int opn_decode_pcm(opn_decoder *dec, const uint8_t *packet, size_t len, void *pcm, size_t pcm_capacity,
                   int sample_format, size_t frame_size, int decode_fec);
size_t opn_sample_size(int sample_format); /* bytes per sample, 0 for an unknown format */
int32_t opn_decoder_sampling_rate(const opn_decoder *dec);                   /* decoder.rs:80  */
int32_t opn_decoder_channels(const opn_decoder *dec);                        /* decoder.rs:85  */
int32_t opn_decoder_gain(const opn_decoder *dec);                            /* decoder.rs:90  */
int32_t opn_decoder_bandwidth(const opn_decoder *dec);                       /* decoder.rs:95, -1 = None */
int32_t opn_decoder_pitch(const opn_decoder *dec);                           /* decoder.rs:100, -1 = None */
int32_t opn_decoder_last_packet_duration(const opn_decoder *dec);            /* decoder.rs:112, -1 = None */
uint32_t opn_decoder_final_range(const opn_decoder *dec);                    /* decoder.rs:121 */

/* ---- host memory for the host-buffer entry points ------------------------------------- */
/* The decode calls below accept any host memory.  Page-locked buffers are copied by asynchronous DMA at PCIe speed
 * (and are what OPN_FLAG_SUBMIT_ONLY needs to overlap two calls); ordinary pageable memory -- a Rust Vec or slice --
 * is staged by the CUDA runtime through a bounce buffer, synchronously: correct, but slower (bench.py e2e_pageable).
 * A caller that owns its buffers gets the fast kind by allocating them here, or by registering (pinning in place)
 * memory it already has; registered memory must be unregistered before it is freed. */
void *opn_host_alloc(size_t bytes);          /* page-locked, NULL on failure */
void opn_host_free(void *p);
int opn_host_register(void *p, size_t bytes);
int opn_host_unregister(void *p);

/* ---- batch of independent streams (the entry point north_star adds) ------------------ */
typedef struct opn_batch opn_batch;
typedef struct {
    int32_t fs_hz;        /* 48000 */
    int32_t channels;     /* output channels, 1 or 2 */
    int16_t gain_q8;      /* DecoderConfiguration::gain */
    int16_t postfilter;   /* 1: run the comb post-filter epilogue (default), 0: IMDCT only */
    int32_t bitstream;    /* OPN_BITSTREAM_*: how CELT frame payloads are laid out */
} opn_config;
/* CeltDecoder::decode is todo!() in the crate (src/celt/decoder.rs:47-56): nothing defines how the symbols of a real
 * RFC 6716 CELT frame become MDCT coefficients, so with OPN_BITSTREAM_OPUS (the default a drop-in caller gets) every
 * CELT frame is reported as OPN_ERR_UNIMPLEMENTED -- exactly where the crate panics.  OPN_BITSTREAM_SYNTH_CELT_1 is an
 * explicit opt-in to the synthetic frame layout of DESIGN.md section 3 (flags, post-filter parameters, Laplace energies,
 * PVQ parts on a fixed schedule): built only from operations the crate implements, NOT interoperable with Opus. */
#define OPN_BITSTREAM_OPUS 0
#define OPN_BITSTREAM_SYNTH_CELT_1 1
/* OPN_BITSTREAM_SYNTH_CELT_2: the allocation-driven layout of DESIGN.md section 3b -- band boosts, allocation trim,
 * compute_allocation from the mode's tables (src/celt/mode.rs:13-28, 70-111) driven by the running tell_frac, fine-energy
 * bits, and per band a theta split (bitexact_cos / bitexact_log2tan, src/math.rs:51-75) down to PVQ leaves whose (n, K) are
 * computed per frame on the device; the band energies (coarse + fine + final bits) scale the decoded bands
 * (denormalise_bands).  A slice of a real CELT frame (no tf, spreading, folding, joint stereo, energy prediction):
 * closer to RFC 6716 section 4.3 than SYNTH-CELT/1, still NOT Opus-interoperable, and parity-unpinned like it. */
#define OPN_BITSTREAM_SYNTH_CELT_2 2

/* OPN_BITSTREAM_SYNTH_SILK_1 (a bit, OR-ed onto one of the values above): SILK-only frames (TOC configs 0..11, 10 or 20 ms) decode
 * with the synthetic layout of DESIGN.md section 3c -- range-coded side information and PVQ shell blocks around long-term
 * prediction, the integer LPC synthesis recursion and a polyphase resampler to 48 kHz -- instead of reporting
 * OPN_ERR_UNIMPLEMENTED.  SilkDecoder::decode is unimplemented!() in the crate (src/silk/decoder.rs:71-80): the layout is this
 * library's own, NOT Opus-interoperable, parity-unpinned.  Hybrid frames and 40/60 ms SILK frames stay unimplemented. */
#define OPN_BITSTREAM_SYNTH_SILK_1 0x100
#define OPN_BITSTREAM_CELT_MASK 0xFF

#define OPN_FLAG_DEVICE_PTRS 1u  /* arena/offsets/lens/pcm/results are device pointers; call is asynchronous */
#define OPN_FLAG_NO_PCM_COPY 2u  /* leave PCM in the device ring only (read it with opn_batch_ring) */
#define OPN_FLAG_INPUTS_READY 4u /* with DEVICE_PTRS: arena/offsets/lens are already complete in device memory and stay
                                  * untouched until opn_batch_synchronize, so the entropy stage of this call may overlap the
                                  * PVQ/IMDCT stage of the previous one (without the flag it is ordered after everything
                                  * enqueued on opn_batch_cuda_stream) */
#define OPN_FLAG_SUBMIT_ONLY 8u  /* host-buffer call: enqueue and return a ticket for opn_batch_wait */
#define OPN_FLAG_MIXED_FRAMES 16u /* with DEVICE_PTRS: the streams' packets may hold frames of different sizes (2.5, 5, 10 or
                                  * 20 ms, read from each packet's TOC on the device); frame_size is then the capacity of
                                  * a stream's PCM row in samples per channel, as for Decoder::decode_float, and
                                  * result_per_stream[i] the samples stream i decoded (OPN_ERR_FRAME_SIZE_TOO_SMALL if its
                                  * frame does not fit).  A lost packet (lens[i] == 0) conceals one frame of the size of
                                  * the stream's previous packet, whichever kind of call decoded it; a PLC/DTX packet (the
                                  * TOC alone or with one byte of payload) is concealed too, but sets that size from its
                                  * TOC, as any packet does.  The step's buckets are built on the device.  SILK packets are
                                  * OPN_ERR_UNIMPLEMENTED in this step; OPN_FLAG_MIXED_MODES takes them. */
#define OPN_FLAG_MIXED_MODES 128u /* with DEVICE_PTRS, on a batch created with OPN_BITSTREAM_SYNTH_SILK_1 (else OPN_ERR_BAD_ARG; not with
                                  * OPN_FLAG_SILK_FRAMES): OPN_FLAG_MIXED_FRAMES for CELT and SILK packets in one step.  Each stream
                                  * takes a single-frame CELT packet (2.5-20 ms), a single-frame SILK-only packet (NB/MB/WB, 10 or
                                  * 20 ms) or a loss; frame_size is the capacity of a row and result_per_stream[i] the samples stream
                                  * i decoded, as for OPN_FLAG_MIXED_FRAMES.  A stream switches codec as Decoder::decode does: SILK
                                  * after CELT resets the SILK decoder, the CELT decoder conceals 5 ms, which replace the first
                                  * 2.5 ms of the row and cross-fade into the next 2.5 ms (decoder.rs:519-557, 765-788); CELT after
                                  * SILK resets the CELT decoder (decoder.rs:703-705).  A loss conceals one frame of the stream's
                                  * last size with the codec of its last packet.  Per-stream errors, state untouched:
                                  * OPN_ERR_UNIMPLEMENTED for hybrid, 40/60 ms SILK, multi-frame packets, a foreign channel count and
                                  * CELT packets of OPN_BITSTREAM_OPUS; OPN_ERR_FRAME_SIZE_TOO_SMALL when the frame does not fit. */

#define OPN_FLAG_SILK_FRAMES 32u  /* with DEVICE_PTRS: every packet of the step is a single SILK-only frame of frame_size samples
                                  * (480 or 960 at 48 kHz) of the batch's channel count; the bandwidth (NB/MB/WB) is read from each
                                  * packet's TOC on the device.  Needs OPN_BITSTREAM_SYNTH_SILK_1. */

#define OPN_FLAG_DECODE_FEC 64u   /* host-buffer calls: Decoder::decode(.., decode_fec = true) for every stream (decoder.rs:343-386):
                                  * conceal frame_size minus one packet frame, then decode the packet's in-band redundant copy of the
                                  * previous frame (SILK LBRR); CELT packets, CELT streams and rows too short for a frame conceal
                                  * everything.  opn_decode_* take the same as their decode_fec argument. */

int opn_batch_create(int device, uint32_t n_streams, const opn_config *cfg, opn_batch **out);
void opn_batch_destroy(opn_batch *b);
int opn_batch_reset(opn_batch *b);
/* One packet per stream (lens[i] == 0: lost).  Every stream i decodes packet
 * arena[offsets[i] .. offsets[i]+lens[i]) into pcm[i*pcm_stride_floats ..] (interleaved).
 * result_per_stream[i] = samples per channel or a negative error for that stream only: a bad
 * packet never poisons its neighbours.  Semantics per stream = Decoder::decode_float.
 * Host-buffer calls take any mix of frame sizes, multi-frame packets and packets whose channel count differs from the
 * batch's (stream_channels, decoder.rs:332: a mono packet fills both channels of a stereo decoder, a stereo packet is
 * averaged into a mono decoder).  Device-resident calls (OPN_FLAG_DEVICE_PTRS) take single-frame packets of the batch's
 * channel count: all of frame_size samples, or of any size with OPN_FLAG_MIXED_FRAMES; CELT and SILK packets in one call,
 * with mode switches, take OPN_FLAG_MIXED_MODES. */
int opn_batch_decode_float(opn_batch *b, const uint8_t *arena, const uint32_t *offsets,
                           const uint32_t *lens, float *pcm, size_t pcm_stride_floats,
                           size_t frame_size, int32_t *result_per_stream, uint32_t flags);
/* Decoder::decode::<i16> (decoder.rs:148-193) for every stream: pcm_soft_clip (per-stream memory, the reference's
 * slice quirk kept, see opn_decode_i16) and Sample::from_f32 run on the device, so only 2 bytes per sample cross
 * PCIe.  Host buffers only; pcm_stride_samples must be a multiple of 8 when it differs from frame_size*channels.
 * OPN_FLAG_SUBMIT_ONLY / opn_batch_wait work as for opn_batch_decode_float. */
int opn_batch_decode_i16(opn_batch *b, const uint8_t *arena, const uint32_t *offsets,
                         const uint32_t *lens, int16_t *pcm, size_t pcm_stride_samples,
                         size_t frame_size, int32_t *result_per_stream, uint32_t flags);
/* The same for any sample type (OPN_SAMPLE_*): Decoder::decode::<S> for every stream. */
int opn_batch_decode_pcm(opn_batch *b, const uint8_t *arena, const uint32_t *offsets,
                         const uint32_t *lens, void *pcm, size_t pcm_stride_samples, int sample_format,
                         size_t frame_size, int32_t *result_per_stream, uint32_t flags);
int opn_batch_synchronize(opn_batch *b);
/* Host-buffer calls made with OPN_FLAG_SUBMIT_ONLY return a ticket (0 or 1) instead of waiting: at most two
 * calls are in flight, so the PCM download of one overlaps the decode of the next.  The call's host buffers
 * (arena, offsets, lens, pcm) belong to the library until opn_batch_wait(ticket) returns; result_per_stream is
 * final on return of the submitting call. */
int opn_batch_wait(opn_batch *b, int ticket);
/* Per-stream Decoder::final_range() of the last decoded frame (host buffer, n_streams words). */
int opn_batch_final_ranges(opn_batch *b, uint32_t *out);
/* Device-resident PCM ring (history + output): base pointer, samples per channel in the ring,
 * and the per-stream write position after the last call (device pointer, n_streams words).  The ring holds the PCM
 * before the decoder gain (opn_config.gain_q8): it is also the post-filter's history.  Only the dense PCM rows are
 * scaled; a caller of OPN_FLAG_NO_PCM_COPY applies the gain itself. */
int opn_batch_ring(opn_batch *b, float **ring, uint32_t *ring_samples, uint32_t **ring_pos_dev);
/* Counters for the measurement harness.  kernel_ms[k]/kernel_launches[k]: k = 0 range decode (k_synth_rangedec),
 * 1 frame kernel (k_frame_w: PVQ expansion + IMDCT + TDAC + comb post-filter + PCM store; a large batch runs it as three
 * concurrent launches over thirds of the streams, and kernel_ms[1] is the time from the first launch to the last
 * completion), 2 the two bucketing kernels of a mixed-frame step (k_mix_key, k_mix_place: counted, not timed; kernel_ms[2]
 * stays 0).  A mixed-mode step counts its CELT and SILK range decodes under 0, its CELT and SILK frame kernels under 1,
 * and its mode-switch launches (resets, fade) under 2; they run inside the frame stage's timed span.  Timing must be enabled first (the stages of a step then run one after the other, with cudaEvents around
 * each). */
int opn_batch_enable_timing(opn_batch *b, int on);
int opn_batch_stats(opn_batch *b, uint64_t kernel_launches[3], double kernel_ms[3], int reset);
/* Sum over the channel-frames the post-filter ran on, in timed passes, of max(T0,T1)+2: the history samples it had to
 * read (4 bytes each) -- the comb term of the frame kernel's algorithmic bytes. */
int opn_batch_history_samples(opn_batch *b, uint64_t *out, int reset);
void *opn_batch_cuda_stream(opn_batch *b);
/* The library runs its stages on several internal streams (range decode; the frame kernel of a large batch in three
 * groups of streams).  opn_batch_join makes everything enqueued so far an ancestor of whatever is enqueued next on
 * opn_batch_cuda_stream (e.g. the caller's end-of-region event or a consumer kernel reading the PCM ring); it does
 * not block the host. */
int opn_batch_join(opn_batch *b);

/* ---- operator-level entry points (host pointers in/out; mirror the pub(crate) operators) */
/* One record per range-coder call; replayed by one warp per packet.  RangeDecoder::*,
 * src/range_coder/decoder.rs:50-355; decode_pulses, src/celt/pvc.rs:156-160. */
enum { OPN_OP_UINT = 0, OPN_OP_BITS = 1, OPN_OP_BIT_LOGP = 2, OPN_OP_ICDF = 3, OPN_OP_LAPLACE = 4,
       OPN_OP_BIT_VIA_DECODE = 5, OPN_OP_BIT_VIA_DECODE_BIN = 6, OPN_OP_PULSES = 7,
       OPN_OP_SHRINK = 8, OPN_OP_TELL = 9,
       OPN_OP_PULSES_EVENTS = 10 /* decode_pulses through the product path's cwrsi (event walk, csrc/symbols.cuh) */ };
typedef struct { uint32_t op, a, b; } opn_op;
typedef struct { uint32_t value, tell_frac, rng; } opn_op_out;
/* n_packets packets share one script.  out: [n_packets][n_ops]; y_out: [n_packets][y_stride]. */
int opn_op_rangedec_script(int device, const uint8_t *arena, const uint32_t *offsets,
                           const uint32_t *lens, uint32_t n_packets, const opn_op *ops,
                           uint32_t n_ops, const uint8_t *icdf_pool, uint32_t icdf_pool_len,
                           opn_op_out *out, int32_t *y_out, uint32_t y_stride);
/* Mdct::backward, src/celt/mdct.rs:159-260, on n_rows independent rows with the standard
 * window (mode::WINDOW) and overlap 120.  input row: (960>>shift)*stride floats; output row:
 * out_stride floats whose first 60 hold the previous tail on entry; `blocks` (1 or `stride`)
 * consecutive interleaved short blocks are transformed per row (blocks = stride = B). */
int opn_op_imdct_tdac(int device, const float *input, size_t in_stride, float *output,
                      size_t out_stride, uint32_t n_rows, int shift, int stride, int blocks);
/* comb_filter_inplace / comb_filter, src/celt/comb_filter/mod.rs:59-193, one row per filter.
 * params per row: {t0, t1, tapset0, tapset1}; gains per row: {g0, g1}. */
int opn_op_comb_filter_inplace(int device, float *y, size_t row_stride, size_t y_offset, size_t n,
                               uint32_t n_rows, const int32_t *params4, const float *gains2,
                               size_t overlap);
int opn_op_comb_filter(int device, float *y, const float *x, size_t row_stride, size_t offset,
                       size_t n, uint32_t n_rows, const int32_t *params4, const float *gains2,
                       size_t overlap);
/* smooth_fade_into_in1 / smooth_fade_into_in2, src/decoder.rs:833-865 (the cross-fade decode_frame applies at a mode
 * transition, decoder.rs:731-788): out = w^2 * in2 + (1 - w^2) * in1 over the first `overlap` samples per channel of
 * n_rows interleaved rows, w = WINDOW[i * 48000 / fs_hz].  `out` may be in1 or in2 (the crate's two in-place forms);
 * samples past the overlap are copied from in1. */
int opn_op_smooth_fade(int device, const float *in1, const float *in2, float *out, size_t row_stride,
                       size_t overlap, int channels, int32_t fs_hz, uint32_t n_rows);
/* pcm_soft_clip, src/lib.rs:526-632: n_rows independent interleaved buffers. */
int opn_op_pcm_soft_clip(int device, float *pcm, size_t row_stride, size_t row_len, int channels,
                         uint32_t n_rows, float *softclip_mem /* [n_rows][channels] */);

/* bitexact_cos (src/math.rs:51-55) on x[0..n_cos) and bitexact_log2tan (math.rs:59-69) on (isin, icos)[0..n_log2tan):
 * the Q15 integer trigonometry CELT's stereo/theta split uses.  Either half may be empty. */
int opn_op_bitexact_trig(int device, const int16_t *x, int16_t *cos_out, uint32_t n_cos, const int32_t *isin,
                         const int32_t *icos, int32_t *log2tan_out, uint32_t n_log2tan);

/* ---- SYNTH-CELT/1 frames (DESIGN.md): side information the symbol kernel reports ------ */
typedef struct {
    int32_t silence, postfilter, octave, period, gain_idx, tapset, transient, intra;
    int32_t coarse[2][21];
    int32_t fine[2][21];
    uint32_t final_rng, tell_frac, n_pulses;
} opn_synth_side;
/* Symbol decode only (kernel 0): payloads (bytes after the TOC) -> side info, pulses, coefficients.
 * y_out / coef_out: [n_packets][channels][120<<lm]; either may be NULL. */
int opn_op_synth_symbols(int device, const uint8_t *arena, const uint32_t *offsets,
                         const uint32_t *lens, uint32_t n_packets, int lm, int channels,
                         opn_synth_side *side_out, int32_t *y_out, float *coef_out);

/* ---- SYNTH-CELT/2 frames: everything the frame decode derives besides the coefficients ---------------------------- */
typedef struct {
    int32_t silence, postfilter, octave, period, gain_idx, tapset, transient, intra;
    int32_t spread, alloc_trim, coded_bands, intensity, dual_stereo, anti_collapse, balance;
    int32_t offsets[21], pulses[21], ebits[21], fine_priority[21]; /* band boosts; compute_allocation's outputs */
    int32_t coarse[2][21], fine[2][21], fine_final[2][21];
    int32_t energy_q9[2][21]; /* band energy = log2 of the band's gain, in 1/512: coarse + fine + final refinement */
    uint32_t n_parts, n_pulses, n_splits, theta_sum;
    uint32_t final_rng, tell_frac;
} opn_celt2_side;
/* Symbol decode + expansion only: payloads (bytes after the TOC) -> side record, pulses, coefficients.
 * y_out / coef_out: [n_packets][channels][120<<lm]; any output may be NULL. */
int opn_op_celt2_symbols(int device, const uint8_t *arena, const uint32_t *offsets, const uint32_t *lens, uint32_t n_packets,
                         int lm, int channels, opn_celt2_side *side_out, int32_t *y_out, float *coef_out);
/* Generator (host): one packet of exactly pkt_bytes (TOC + SYNTH-CELT/2 payload) / a [frame][stream][pkt_bytes] block. */
int opn_celt2_packet(uint64_t stream_id, uint64_t frame_idx, int lm, int channels, uint32_t pkt_bytes,
                     uint32_t transient_permille, uint8_t *out, opn_celt2_side *truth);
int opn_celt2_fill(uint64_t first_stream, uint32_t n_streams, uint64_t first_frame, uint32_t n_frames, int lm, int channels,
                   uint32_t pkt_bytes, uint32_t transient_permille, int n_threads, uint8_t *out);

/* ---- SYNTH-SILK/1 frames (DESIGN.md section 3c) -------------------------------------------------------------------- */
typedef struct {
    int32_t type, gidx[4], rc_idx[16], lag[4], ltp_idx[4], seed;
    int32_t pulses[20];
    uint32_t index[20];
} opn_silk_chan_side;
typedef struct {
    opn_silk_chan_side ch[2];
    uint32_t final_rng, tell_frac;
    int32_t lbrr; /* the packet carries a redundant copy of the previous frame (in-band FEC) */
} opn_silk_side;
/* One SILK-only packet (TOC included) per row, each decoded by a fresh decoder of `channels` output channels; every packet
 * must hold one frame of frame_size samples (480 or 960) and `stream_channels` coded channels.  side_out [n_packets], exc_out
 * [n_packets][2][320] (excitation after long-term prediction, Q14, per coded channel), out16 [n_packets][2][320] (internal-rate
 * samples per output channel), pcm_out [n_packets][frame_size*channels], result [n_packets]; any output may be NULL.  decode_fec:
 * decode each packet's redundant copy of the previous frame instead of its own (a packet without one conceals: silence from rest). */
int opn_op_silk_frames(int device, const uint8_t *arena, const uint32_t *offsets, const uint32_t *lens, uint32_t n_packets,
                       int stream_channels, int channels, size_t frame_size, int decode_fec, opn_silk_side *side_out, int32_t *exc_out,
                       int16_t *out16, float *pcm_out, int32_t *result);
/* Generator (host): one packet of exactly pkt_bytes (TOC + SYNTH-SILK/1 payload) / a [frame][stream][pkt_bytes] block.
 * bandwidth 0 NB (8 kHz), 1 MB (12 kHz), 2 WB (16 kHz); frame_ms 10 or 20. */
int opn_silk_packet(uint64_t stream_id, uint64_t frame_idx, int bandwidth, int frame_ms, int channels, uint32_t pkt_bytes,
                    uint32_t lbrr_permille /* chance in 1/1000 that the packet carries an LBRR copy of the previous frame */, uint8_t *out);
int opn_silk_fill(uint64_t first_stream, uint32_t n_streams, uint64_t first_frame, uint32_t n_frames, int bandwidth, int frame_ms,
                  int channels, uint32_t pkt_bytes, uint32_t lbrr_permille, int n_threads, uint8_t *out);

/* ---- synthetic stream generator (host; uses the library's own range ENCODER) --------- */
/* Writes one packet of exactly pkt_bytes (TOC + SYNTH-CELT/1 payload) for (stream_id, frame).
 * truth (optional) receives the values that were encoded.  Returns pkt_bytes or an error
 * (OPN_ERR_BUFFER_TOO_SMALL when the frame does not fit). */
int opn_synth_packet(uint64_t stream_id, uint64_t frame_idx, int lm, int channels,
                     uint32_t pkt_bytes, uint32_t transient_permille, uint8_t *out,
                     opn_synth_side *truth);
/* n_streams*n_frames packets, layout [frame][stream][pkt_bytes], generated on n_threads threads. */
int opn_synth_fill(uint64_t first_stream, uint32_t n_streams, uint64_t first_frame,
                   uint32_t n_frames, int lm, int channels, uint32_t pkt_bytes,
                   uint32_t transient_permille, int n_threads, uint8_t *out);

/* host range ENCODER, src/range_coder/encoder.rs (packet synthesis and round-trip tests) */
int opn_enc_run_script(uint8_t *buf, uint32_t len, const opn_op *ops, const uint32_t *values,
                       uint32_t n_ops, const uint8_t *icdf_pool, const int32_t *y_in,
                       uint32_t *tell_frac_out, uint32_t *range_bytes, uint32_t *final_tell_frac);

#ifdef __cplusplus
}
#endif
#endif /* OPUSB200_H */
