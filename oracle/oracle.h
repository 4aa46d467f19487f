/* oracle.h -- CPU ORACLE (TEST INFRASTRUCTURE, NOT PRODUCT CODE).
 *
 * A plain-C restatement of the algorithms of the reference crate hasenbanck/opus-native
 * (pure Rust, not buildable here: no rustc/cargo in the image) for the batched-decode hot
 * path.  Every function cites the reference file:line it follows.  Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load
 * this library; the product (opus-native_b200/) never links or calls it.
 *
 * Parity pinning: the restatement is checked against every known-answer test the reference
 * holds for this path (tests/test_oracle_kat.py; SURVEY.md section 8c).
 *
 * Build: make -C oracle   (gcc -O2 -ffp-contract=off -fno-fast-math: Rust never contracts
 * a*b+c into an FMA, so neither may the oracle).
 */
#ifndef ORACLE_H
#define ORACLE_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- range coder: src/range_coder/{mod,decoder,encoder}.rs ---- */
typedef struct {
    const uint8_t *buffer;
    uint32_t storage, end_offs, end_window, end_bits, bits_total, offs, rng, val, ext;
    uint8_t rem;
} orc_dec;

typedef struct {
    uint8_t *buffer;
    uint32_t buffer_len;
    uint32_t storage, end_offs, end_window, end_bits, bits_total, offs, rng, val, ext;
    int32_t rem; /* -1 = None */
    int error;   /* sticky: 0 ok, ORC_ERR_* otherwise (Rust returns Result per call) */
} orc_enc;

enum { ORC_OK = 0, ORC_ERR_BAD_ARG = -1, ORC_ERR_BUFFER_TOO_SMALL = -2, ORC_ERR_INTERNAL = -3,
       ORC_ERR_INVALID_PACKET = -4, ORC_ERR_FRAME_SIZE_TOO_SMALL = -5 };

uint32_t orc_ilog(uint32_t x);
uint32_t orc_tell(uint32_t bits_total, uint32_t rng);
uint32_t orc_tell_frac(uint32_t bits_total, uint32_t rng);
uint32_t orc_laplace_freq1(uint32_t fs0, uint32_t decay);
uint32_t orc_laplace_start_freq(uint32_t decay);

void orc_dec_init(orc_dec *d, const uint8_t *buf, uint32_t len);
void orc_dec_shrink_storage(orc_dec *d, uint32_t by);
uint32_t orc_dec_decode(orc_dec *d, uint32_t ft);
uint32_t orc_dec_decode_bin(orc_dec *d, uint32_t bits);
void orc_dec_update(orc_dec *d, uint32_t fl, uint32_t fh, uint32_t ft);
int orc_dec_bit_logp(orc_dec *d, uint32_t logp);
uint32_t orc_dec_icdf(orc_dec *d, const uint8_t *icdf, uint32_t ftb);
uint32_t orc_dec_uint(orc_dec *d, uint32_t ft);
uint32_t orc_dec_bits(orc_dec *d, uint32_t bits);
int32_t orc_dec_laplace(orc_dec *d, uint32_t fs, uint32_t decay);
uint32_t orc_dec_tell(const orc_dec *d);
uint32_t orc_dec_tell_frac(const orc_dec *d);

void orc_enc_init(orc_enc *e, uint8_t *buf, uint32_t len);
int orc_enc_encode(orc_enc *e, uint32_t fl, uint32_t fh, uint32_t ft);
int orc_enc_encode_bin(orc_enc *e, uint32_t fl, uint32_t fh, uint32_t bits);
int orc_enc_bit_logp(orc_enc *e, uint32_t val, uint32_t logp);
int orc_enc_icdf(orc_enc *e, uint32_t s, const uint8_t *icdf, uint32_t ftb);
int orc_enc_uint(orc_enc *e, uint32_t fl, uint32_t ft);
int orc_enc_bits(orc_enc *e, uint32_t fl, uint32_t bits);
int orc_enc_patch_initial_bits(orc_enc *e, uint32_t val, uint32_t nbits);
void orc_enc_shrink(orc_enc *e, uint32_t len);
int orc_enc_done(orc_enc *e);
int orc_enc_laplace(orc_enc *e, int32_t *value, uint32_t fs, uint32_t decay);
uint32_t orc_enc_range_bytes(const orc_enc *e);
uint32_t orc_enc_tell(const orc_enc *e);
uint32_t orc_enc_tell_frac(const orc_enc *e);

/* A flat "symbol script": one record per range-coder call, so the same sequence can be
 * replayed by the oracle and by the CUDA warp decoder and compared record by record. */
enum { ORC_OP_UINT = 0, ORC_OP_BITS = 1, ORC_OP_BIT_LOGP = 2, ORC_OP_ICDF = 3, ORC_OP_LAPLACE = 4,
       ORC_OP_BIT_VIA_DECODE = 5, ORC_OP_BIT_VIA_DECODE_BIN = 6, ORC_OP_PULSES = 7,
       ORC_OP_SHRINK = 8, ORC_OP_TELL = 9 };
typedef struct { uint32_t op, a, b; } orc_op;
typedef struct { uint32_t value, tell_frac, rng; } orc_op_out;
/* pulses (ORC_OP_PULSES) are appended to y_out; returns number of ints written. */
uint32_t orc_dec_run_script(const uint8_t *buf, uint32_t len, const orc_op *ops, uint32_t n_ops,
                            const uint8_t *icdf_pool, orc_op_out *out, int32_t *y_out);
int orc_enc_run_script(uint8_t *buf, uint32_t len, const orc_op *ops, const uint32_t *values,
                       uint32_t n_ops, const uint8_t *icdf_pool, const int32_t *y_in,
                       uint32_t *tell_frac_out, uint32_t *range_bytes, uint32_t *final_tell_frac);

/* ---- PVQ: src/celt/pvc.rs ---- */
uint32_t orc_pvq_u(uint32_t n, uint32_t k);
uint32_t orc_pvq_v(uint32_t n, uint32_t k);
uint32_t orc_icwrs(const int32_t *y, uint32_t n);
float orc_cwrsi(int32_t *y, uint32_t n, uint32_t k, uint32_t i);
float orc_decode_pulses(orc_dec *d, int32_t *y, uint32_t n, uint32_t k);
int orc_encode_pulses(orc_enc *e, const int32_t *y, uint32_t n, uint32_t k);

/* ---- FFT / MDCT: src/celt/kiss_fft.rs, src/celt/mdct.rs ---- */
/* data: nfft interleaved complex, already in bit-reversed order (kiss_fft.rs:24-53) */
void orc_fft_process(int shift, float *data);
const uint16_t *orc_fft_bitrev(int shift);
float orc_fft_scale(int shift);
void orc_mdct_backward(const float *input, float *output, const float *window, int overlap,
                       int shift, int stride);
void orc_mdct_forward(const float *input, float *output, const float *window, int overlap,
                      int shift, int stride);
const float *orc_window(void);
const float *orc_trig(void);

/* ---- comb filter: src/celt/comb_filter/{mod,fallback}.rs ---- */
void orc_comb_filter(float *y, size_t y_offset, const float *x, size_t x_offset, size_t t0,
                     size_t t1, size_t n, float g0, float g1, size_t tapset0, size_t tapset1,
                     size_t overlap);
void orc_comb_filter_inplace(float *y, size_t y_offset, size_t t0, size_t t1, size_t n, float g0,
                             float g1, size_t tapset0, size_t tapset1, size_t overlap);

/* ---- math: src/math.rs ---- */
int16_t orc_bitexact_cos(int16_t x);
int32_t orc_bitexact_log2tan(int32_t isin, int32_t icos);

/* ---- packets: src/lib.rs ---- */
int orc_packet_bandwidth(const uint8_t *p);            /* 0 NB 1 MB 2 WB 3 SWB 4 FB */
int orc_packet_channels(const uint8_t *p);
int orc_packet_frame_count(const uint8_t *p, size_t len);
int orc_packet_samples_per_frame(const uint8_t *p, int fs);
int orc_packet_sample_count(const uint8_t *p, size_t len, int fs);
int orc_packet_mode(const uint8_t *p);                 /* 0 silk 1 hybrid 2 celt */
int orc_parse_packet(const uint8_t *p, size_t len, int self_delimited, uint32_t frames[48],
                     uint32_t sizes[48], uint32_t *payload_offset, uint32_t *packet_offset);
void orc_pcm_soft_clip(float *pcm, size_t total_len, size_t channels, float *softclip_mem,
                       size_t mem_len);
void orc_smooth_fade(const float *in1, const float *in2, float *out, int overlap, int channels,
                     int fs);
int orc_sample_from_f32(int format, const float *in, void *out, size_t n); /* lib.rs:63-107 */

/* ---- SYNTH-CELT/1 frame decode (SURVEY.md 8d): the oracle side of the fused pipeline ---- */
typedef struct {
    int32_t silence, postfilter, octave, period, gain_idx, tapset, transient, intra;
    int32_t coarse[2][21];
    int32_t fine[2][21];
    uint32_t final_rng, tell_frac, n_pulses;
} orc_synth_side;

#define ORC_SYNTH_HIST 1024 /* T + 2 <= 1024 */
#define ORC_SYNTH_BUF (ORC_SYNTH_HIST + 8 * 960 + 60)
typedef struct {
    /* Rolling output buffer per channel: [.. history | frame | 60-sample un-windowed IMDCT tail].  Frames are
     * appended at `pos` (the previous frame's tail is already there, the comb history directly below it); when
     * the buffer is full the last 1024 samples + tail move to the front (once per 8 long frames). */
    float buf[2][ORC_SYNTH_BUF];
    uint32_t pos;
    int32_t pf_period, pf_tapset;  /* post-filter parameters of the previous frame  */
    float pf_gain;
} orc_synth_state;

void orc_synth_state_init(orc_synth_state *s);
/* coefficients (channel-major) -> interleaved PCM; the back half of every SYNTH-CELT frame decode */
int orc_synth_finish_frame(orc_synth_state *st, const float *coef, int lm, int channels, int apply_comb, int lost, int postfilter,
                           int period, int gain_idx, int tapset, int transient, float *pcm_out);
/* payload = frame bytes after the TOC.  y_out: >= channels*100<<LM ints; coef_out: same, floats
 * (channel-major, frequency order); pcm_out: interleaved frame_size*channels floats. */
int orc_synth_decode_frame(orc_synth_state *st, const uint8_t *payload, uint32_t len, int lm,
                           int channels, int apply_comb, orc_synth_side *side, int32_t *y_out,
                           float *coef_out, float *pcm_out);
/* A packet of stream_channels channels in a decoder of `channels` channels: mono -> stereo copies the spectrum, stereo -> mono
 * averages it (stream_channels, src/decoder.rs:332,376,395; mapping restated from libopus' celt_synthesis). */
void orc_map_channels(float *coef, int nf, int stream_channels, int channels);
int orc_synth_decode_frame_mapped(orc_synth_state *st, const uint8_t *payload, uint32_t len, int lm, int stream_channels, int channels,
                                  int apply_comb, orc_synth_side *side, float *pcm_out);
/* ---- SYNTH-CELT/2 (oracle/celt2.c): allocation-driven CELT frame decode, PARITY UNPINNED (no reference code exists) ---- */
#define ORC_CELT2_MAX_PARTS 192
typedef struct {
    int32_t silence, postfilter, octave, period, gain_idx, tapset, transient, intra;
    int32_t spread, alloc_trim, coded_bands, intensity, dual_stereo, anti_collapse, balance;
    int32_t offsets[21], pulses[21], ebits[21], fine_priority[21];
    int32_t coarse[2][21], fine[2][21], fine_final[2][21];
    int32_t energy_q9[2][21]; /* band energy (log2 of the band's gain) in 1/512 */
    uint32_t n_parts, n_pulses, n_splits, theta_sum;
    uint32_t final_rng, tell_frac;
} orc_celt2_side;
/* one PVQ leaf: normalised coefficients [pos, pos+n) of the channel-major frame = cwrsi(n, k, index) * gain / sqrt(yy);
 * base = pos | band << 11 */
typedef struct {
    uint16_t base;
    uint8_t n, k;
    uint32_t index;
    float gain;
} orc_celt2_part;
/* payload = frame bytes after the TOC.  y_out / coef_out: [channels][120<<lm] (channel-major); parts may be NULL. */
int orc_celt2_decode_symbols(const uint8_t *payload, uint32_t len, int lm, int channels, orc_celt2_side *side, orc_celt2_part *parts,
                             int32_t *y_out, float *coef_out);
int orc_celt2_decode_frame(orc_synth_state *st, const uint8_t *payload, uint32_t len, int lm, int channels, int apply_comb,
                           orc_celt2_side *side, float *pcm_out);
int orc_celt2_decode_frame_mapped(orc_synth_state *st, const uint8_t *payload, uint32_t len, int lm, int stream_channels, int channels,
                                  int apply_comb, orc_celt2_side *side, float *pcm_out);
int orc_celt2_packet(uint64_t stream_id, uint64_t frame_idx, int lm, int channels, uint32_t pkt_bytes, uint32_t transient_permille,
                     uint8_t *out, orc_celt2_side *truth);

/* ---- SYNTH-SILK/1 (oracle/silk.c): SILK-only frames, PARITY UNPINNED (src/silk/decoder.rs:71-80 is unimplemented!()) ---- */
#define ORC_SILK_MAX_FRAME 320 /* 20 ms at 16 kHz */
#define ORC_SILK_HIST 320      /* excitation history of the long-term predictor (>= 18 ms + 2 samples) */
typedef struct {
    int32_t type, gidx[4], rc_idx[16], lag[4], ltp_idx[4], seed;
    int32_t pulses[20];
    uint32_t index[20];
} orc_silk_chan_side;
typedef struct {
    orc_silk_chan_side ch[2];
    uint32_t final_rng, tell_frac;
    int32_t lbrr; /* the packet carries a redundant copy of the previous frame */
} orc_silk_side;
typedef struct {
    int32_t slpc[16];            /* sLPC_Q14 of the last 16 samples, [15] = newest */
    int32_t hist[ORC_SILK_HIST]; /* excitation after long-term prediction, [ORC_SILK_HIST-1] = newest */
    int16_t a_q12[16];
    int32_t gain_q10;
} orc_silk_chan;
typedef struct {
    orc_silk_chan ch[2];
    float rs[2][8];              /* resampler history per output channel: rs[c][j] = x[-1-j] */
    int32_t fs_khz, stream_channels;
} orc_silk_state;
void orc_silk_state_init(orc_silk_state *st);
/* payload = frame bytes after the TOC; bandwidth 0 NB / 1 MB / 2 WB; frame_ms 10 or 20.  exc_out: [2][ORC_SILK_MAX_FRAME]
 * excitation after long-term prediction (Q14) or NULL; out16: [2][ORC_SILK_MAX_FRAME] internal-rate samples per OUTPUT channel
 * or NULL; pcm_out: interleaved frame_ms*48*channels floats.  lost: 0 decode the packet's frame, 1 conceal, 2 decode the packet's
 * redundant copy of the previous frame (LostFlag::DecodeFec; conceals when the packet has none).  Returns samples per channel at 48 kHz. */
int orc_silk_decode_frame(orc_silk_state *st, const uint8_t *payload, uint32_t len, int bandwidth, int frame_ms, int stream_channels,
                          int channels, int lost, orc_silk_side *side, int32_t *exc_out, int16_t *out16, float *pcm_out);
int orc_silk_packet(uint64_t stream_id, uint64_t frame_idx, int bandwidth, int frame_ms, int channels, uint32_t pkt_bytes,
                    uint32_t lbrr_permille, uint8_t *out);
int orc_silk_fill(uint64_t first_stream, uint32_t n_streams, uint64_t first_frame, uint32_t n_frames, int bandwidth, int frame_ms,
                  int channels, uint32_t pkt_bytes, uint32_t lbrr_permille, int n_threads, uint8_t *out);
double orc_silk_bench(const uint8_t *packets, uint32_t n_streams, uint32_t n_frames, uint32_t pkt_bytes, int bandwidth, int frame_ms,
                      int channels, int n_threads, float *pcm_last, uint32_t *final_rng_xor);

/* SYNTH-CELT/1 packet generator on the oracle's own range encoder (same seeded draws as opn_synth_packet). */
int orc_synth_packet(uint64_t stream_id, uint64_t frame_idx, int lm, int channels, uint32_t pkt_bytes,
                     uint32_t transient_permille, uint8_t *out);
int orc_synth_fill(uint64_t first_stream, uint32_t n_streams, uint64_t first_frame, uint32_t n_frames, int lm, int channels,
                   uint32_t pkt_bytes, uint32_t transient_permille, int n_threads, uint8_t *out);
/* Multithreaded CPU baseline: streams statically partitioned over n_threads; each thread walks
 * its streams frame by frame.  packets: [n_frames][n_streams][pkt_bytes].  Returns seconds. */
double orc_synth_bench(const uint8_t *packets, uint32_t n_streams, uint32_t n_frames,
                       uint32_t pkt_bytes, int lm, int channels, int apply_comb, int n_threads,
                       float *pcm_last /* [n_streams][frame*channels] or NULL */,
                       uint32_t *final_rng_xor);

/* ---- one step of a batch (oracle/step.c): every stream advanced by one packet, n_threads threads over contiguous stream
 * ranges.  states: [n_streams]; packets: row s at packets + s * pkt_stride, TOC first, lens[s] bytes (0 = lost); pcm_out: row s
 * at pcm_out + s * pcm_stride floats, interleaved; final_rng: [n_streams], 0 for a lost frame.  The CELT steps take each
 * stream's frame size (lm[s]: 120 << lm[s] samples, a lost frame conceals one frame of that size) and write hist[s] (or NULL),
 * the comb history samples the GPU frame kernel counts for the frame: channels * (max(T_old, T_new, 15) + 2) when the
 * post-filter runs, else 0.  The SILK step reads bandwidth and coded channel count from each TOC.  Returns 0 or the first
 * error of a per-stream decode.  lens[s] == ORC_STEP_SKIP leaves stream s out of the step: its state stays untouched and
 * its row, final_rng and hist entries are not written. */
#define ORC_STEP_SKIP 0xFFFFFFFFu
int orc_synth_step(orc_synth_state *states, uint32_t n_streams, const uint8_t *packets, size_t pkt_stride, const uint32_t *lens,
                   const uint8_t *lm, int channels, int apply_comb, int n_threads, float *pcm_out, size_t pcm_stride,
                   uint32_t *final_rng, uint32_t *hist);
int orc_celt2_step(orc_synth_state *states, uint32_t n_streams, const uint8_t *packets, size_t pkt_stride, const uint32_t *lens,
                   const uint8_t *lm, int channels, int apply_comb, int n_threads, float *pcm_out, size_t pcm_stride,
                   uint32_t *final_rng, uint32_t *hist);
int orc_silk_step(orc_silk_state *states, uint32_t n_streams, const uint8_t *packets, size_t pkt_stride, const uint32_t *lens,
                  int frame_ms, int channels, int n_threads, float *pcm_out, size_t pcm_stride, uint32_t *final_rng);

#ifdef __cplusplus
}
#endif
#endif
