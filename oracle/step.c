/* CPU ORACLE (test infrastructure) -- one step of a batch: every stream advanced by one packet.
 *
 * The GPU decodes a step of thousands of streams at once; checking every stream of every step through one ctypes call per
 * stream and frame is slow, and orc_synth_bench / orc_silk_bench keep only the last frame.  These functions take an array
 * of per-stream decoder states and one packet (or a loss) per stream, and decode the step on n_threads threads, streams
 * statically partitioned as in orc_synth_bench.  Each stream goes through exactly the per-stream functions the tests call
 * otherwise (orc_synth_decode_frame, orc_celt2_decode_frame, orc_silk_decode_frame), so the results are the same bits.
 *
 * packets: row s at packets + s * pkt_stride, TOC first; lens[s] bytes of it, 0 = lost (so is a TOC-only packet,
 * src/decoder.rs:467), ORC_STEP_SKIP = the stream takes no part in this step: its state stays untouched, its row and
 * final_rng are not written (a host-buffer call that conceals several frames for some streams is modelled as several
 * steps, each over the streams that still have a frame to go).  pcm_out: row s at pcm_out + s * pcm_stride, the frame's interleaved samples; final_rng[s]: the range
 * coder's final state, 0 for a lost frame. */
#include "oracle.h"

#include <pthread.h>
#include <stdlib.h>

typedef struct {
    int kind; /* 0 SYNTH-CELT/1, 1 SYNTH-CELT/2, 2 SYNTH-SILK/1 */
    void *states;
    uint32_t s0, s1;
    const uint8_t *packets;
    size_t pkt_stride, pcm_stride;
    const uint32_t *lens;
    const uint8_t *lm;
    int channels, apply_comb, frame_ms;
    float *pcm_out;
    uint32_t *final_rng, *hist;
    int rc;
} step_job;

static int max3(int a, int b, int c)
{
    int m = a > b ? a : b;
    return m > c ? m : c;
}

static void celt_stream(step_job *j, uint32_t s)
{
    if (j->lens[s] == ORC_STEP_SKIP) return;
    orc_synth_state *st = (orc_synth_state *)j->states + s;
    const uint8_t *pkt = j->packets + (size_t)s * j->pkt_stride;
    const uint32_t len = j->lens[s] ? j->lens[s] - 1u : 0u; /* byte 0 is the TOC */
    const int lm = j->lm[s], nf = 120 << lm;
    const int old_period = st->pf_period;
    const float old_gain = st->pf_gain;
    float *pcm = j->pcm_out + (size_t)s * j->pcm_stride;
    int r;
    uint32_t rng;
    if (j->kind == 0) {
        orc_synth_side side;
        r = orc_synth_decode_frame(st, len ? pkt + 1 : NULL, len, lm, j->channels, j->apply_comb, &side, NULL, NULL, pcm);
        rng = side.final_rng;
    } else {
        orc_celt2_side side;
        r = orc_celt2_decode_frame(st, len ? pkt + 1 : NULL, len, lm, j->channels, j->apply_comb, &side, pcm);
        rng = side.final_rng;
    }
    if (r != nf) {
        j->rc = r < 0 ? r : ORC_ERR_INTERNAL;
        return;
    }
    j->final_rng[s] = len > 1 ? rng : 0u;
    /* The frame kernel's count of comb history samples (opus-native_b200/csrc/frame_warp.cuh): the post-filter runs when the
     * previous or this frame's gain is non-zero and reads max(T_old, T_new, 15) + 2 samples of history per channel. */
    if (j->hist)
        j->hist[s] = j->apply_comb && (old_gain != 0.0f || st->pf_gain != 0.0f)
                         ? (uint32_t)j->channels * (uint32_t)(max3(old_period, st->pf_period, 15) + 2)
                         : 0u;
}

static void silk_stream(step_job *j, uint32_t s)
{
    if (j->lens[s] == ORC_STEP_SKIP) return;
    orc_silk_state *st = (orc_silk_state *)j->states + s;
    const uint8_t *pkt = j->packets + (size_t)s * j->pkt_stride;
    const uint32_t len = j->lens[s] ? j->lens[s] - 1u : 0u;
    orc_silk_side side;
    const int lost = len <= 1;
    /* bandwidth and coded channel count come from the TOC, as on the device */
    const int bw = lost ? 0 : orc_packet_bandwidth(pkt), cs = lost ? j->channels : orc_packet_channels(pkt);
    const int r = orc_silk_decode_frame(st, lost ? NULL : pkt + 1, len, bw, j->frame_ms, cs, j->channels, lost, &side, NULL, NULL,
                                        j->pcm_out + (size_t)s * j->pcm_stride);
    if (r != j->frame_ms * 48) {
        j->rc = r < 0 ? r : ORC_ERR_INTERNAL;
        return;
    }
    j->final_rng[s] = lost ? 0u : side.final_rng;
}

static void *step_thread(void *arg)
{
    step_job *j = (step_job *)arg;
    for (uint32_t s = j->s0; s < j->s1 && j->rc == 0; s++) {
        if (j->kind == 2) silk_stream(j, s);
        else celt_stream(j, s);
    }
    return NULL;
}

static int run_step(const step_job *proto, uint32_t n_streams, int n_threads)
{
    if (n_threads < 1) n_threads = 1;
    if ((uint32_t)n_threads > n_streams) n_threads = (int)n_streams;
    if (n_threads < 1) return 0;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)n_threads);
    step_job *jobs = (step_job *)calloc((size_t)n_threads, sizeof(step_job));
    if (!th || !jobs) {
        free(th);
        free(jobs);
        return ORC_ERR_INTERNAL;
    }
    for (int t = 0; t < n_threads; t++) {
        jobs[t] = *proto;
        jobs[t].s0 = (uint32_t)((uint64_t)n_streams * (uint64_t)t / (uint64_t)n_threads);
        jobs[t].s1 = (uint32_t)((uint64_t)n_streams * (uint64_t)(t + 1) / (uint64_t)n_threads);
        pthread_create(&th[t], NULL, step_thread, &jobs[t]);
    }
    int rc = 0;
    for (int t = 0; t < n_threads; t++) {
        pthread_join(th[t], NULL);
        if (jobs[t].rc && !rc) rc = jobs[t].rc;
    }
    free(th);
    free(jobs);
    return rc;
}

static int celt_step(int kind, orc_synth_state *states, uint32_t n_streams, const uint8_t *packets, size_t pkt_stride,
                     const uint32_t *lens, const uint8_t *lm, int channels, int apply_comb, int n_threads, float *pcm_out,
                     size_t pcm_stride, uint32_t *final_rng, uint32_t *hist)
{
    if (!states || !packets || !lens || !lm || !pcm_out || !final_rng || channels < 1 || channels > 2) return ORC_ERR_BAD_ARG;
    for (uint32_t s = 0; s < n_streams; s++)
        if (lm[s] > 3 || (size_t)(120 << lm[s]) * (size_t)channels > pcm_stride || (lens[s] > pkt_stride && lens[s] != ORC_STEP_SKIP))
            return ORC_ERR_BAD_ARG;
    step_job j = {0};
    j.kind = kind;
    j.states = states;
    j.packets = packets;
    j.pkt_stride = pkt_stride;
    j.lens = lens;
    j.lm = lm;
    j.channels = channels;
    j.apply_comb = apply_comb;
    j.pcm_out = pcm_out;
    j.pcm_stride = pcm_stride;
    j.final_rng = final_rng;
    j.hist = hist;
    return run_step(&j, n_streams, n_threads);
}

int orc_synth_step(orc_synth_state *states, uint32_t n_streams, const uint8_t *packets, size_t pkt_stride, const uint32_t *lens,
                   const uint8_t *lm, int channels, int apply_comb, int n_threads, float *pcm_out, size_t pcm_stride,
                   uint32_t *final_rng, uint32_t *hist)
{
    return celt_step(0, states, n_streams, packets, pkt_stride, lens, lm, channels, apply_comb, n_threads, pcm_out, pcm_stride,
                     final_rng, hist);
}

int orc_celt2_step(orc_synth_state *states, uint32_t n_streams, const uint8_t *packets, size_t pkt_stride, const uint32_t *lens,
                   const uint8_t *lm, int channels, int apply_comb, int n_threads, float *pcm_out, size_t pcm_stride,
                   uint32_t *final_rng, uint32_t *hist)
{
    return celt_step(1, states, n_streams, packets, pkt_stride, lens, lm, channels, apply_comb, n_threads, pcm_out, pcm_stride,
                     final_rng, hist);
}

int orc_silk_step(orc_silk_state *states, uint32_t n_streams, const uint8_t *packets, size_t pkt_stride, const uint32_t *lens,
                  int frame_ms, int channels, int n_threads, float *pcm_out, size_t pcm_stride, uint32_t *final_rng)
{
    if (!states || !packets || !lens || !pcm_out || !final_rng || channels < 1 || channels > 2) return ORC_ERR_BAD_ARG;
    if ((frame_ms != 10 && frame_ms != 20) || (size_t)frame_ms * 48u * (size_t)channels > pcm_stride) return ORC_ERR_BAD_ARG;
    for (uint32_t s = 0; s < n_streams; s++)
        if (lens[s] > pkt_stride && lens[s] != ORC_STEP_SKIP) return ORC_ERR_BAD_ARG;
    step_job j = {0};
    j.kind = 2;
    j.states = states;
    j.packets = packets;
    j.pkt_stride = pkt_stride;
    j.lens = lens;
    j.channels = channels;
    j.frame_ms = frame_ms;
    j.pcm_out = pcm_out;
    j.pcm_stride = pcm_stride;
    j.final_rng = final_rng;
    return run_step(&j, n_streams, n_threads);
}
