"""Oracle side of mixed-mode device-resident steps (OPN_FLAG_MIXED_MODES): a batch of CELT + SILK decoder pairs that switch
codec as Decoder::decode does, built on oracle_lib's batched steps, and the traffic generator the tests and
tools/bench_mixed_modes.py share."""
import ctypes as C

import numpy as np

from oracle_lib import CeltBatch, SilkBatch, lib, ptr

CELT, SILK = 1, 2  # MixedModeBatch.mode: codec of a stream's last packet (0 = none yet)


class MixedModeBatch:
    """Oracle side of a batch of decoders that take, per stream and step, a single-frame CELT packet (SYNTH-CELT/1 or /2), a
    single-frame SYNTH-SILK/1 packet or a loss, and switch codec as Decoder::decode does (decoder.rs:519-557, 703-705, 765-788):
      - SILK after CELT: the SILK decoder starts from rest, the CELT decoder conceals 5 ms (decode_frame(None) of 240 samples),
        whose first 2.5 ms replace the start of the SILK frame and whose next 2.5 ms cross-fade into it (smooth_fade);
      - CELT after SILK: the CELT decoder starts from rest;
      - a loss conceals one frame of the stream's last size with the codec of its last packet; before any packet, one CELT
        frame of the step's row capacity (zeros).  A PLC/DTX packet (lens 1 or 2) sets codec and size from its TOC.
    Built on CeltBatch / SilkBatch steps with skip and on resets of single states, so it runs at tens of thousands of streams.
    Stream s decodes exactly as one SynthStream / Celt2Stream and one SilkStream composed by hand would."""

    def __init__(self, n_streams, channels, bitstream=1, cap=960, n_threads=None, apply_comb=True):
        """bitstream: the CELT layout, 1 or 2; 0 (OPN_BITSTREAM_OPUS): CELT packets are rejected (OPN_ERR_UNIMPLEMENTED).
        apply_comb: the CELT post-filter (a batch created with postfilter = false runs without it)"""
        self.n, self.channels, self.cap, self.celt_ok = n_streams, channels, cap, bitstream != 0
        self.celt = CeltBatch(n_streams, channels, bitstream or 1, apply_comb=apply_comb, n_threads=n_threads)
        self.silk = SilkBatch(n_streams, channels, n_threads=n_threads)
        self.mode = np.zeros(n_streams, np.uint8)
        self.lm = np.zeros(n_streams, np.uint8)     # the size a loss conceals once a packet was decoded (LM; SILK: 2 = 10 ms, 3 = 20 ms)
        self.final = np.zeros(n_streams, np.uint32)  # Decoder::final_range() of each stream's last decoded frame

    def classify(self, packets, lens):
        """-> (codec [n]: CELT, SILK or 0 for a stream whose packet is rejected, lm [n], err [n]: OPN_ERR_* or 0), as the
        device step checks the TOC; lost packets take the stream's last codec and size"""
        packets = np.asarray(packets)
        toc = packets[:, 0].astype(np.int64)
        got = np.asarray(lens) > 0
        codec = np.where(self.mode == SILK, SILK, CELT).astype(np.uint8)
        cap_lm = 3 if self.cap >= 960 else 2 if self.cap >= 480 else 1 if self.cap >= 240 else 0
        lm = np.where(self.mode != 0, self.lm, cap_lm).astype(np.uint8)  # before any packet: this step's row capacity
        err = np.zeros(self.n, np.int32)
        celt = (toc & 0x80) != 0
        config = toc >> 3
        bad = (toc & 3) != 0
        bad |= np.where(toc & 4, 2, 1) != self.channels
        bad |= ~celt & ((config >= 12) | ((config & 3) > 1))
        bad |= celt & (not self.celt_ok)
        p_lm = np.where(celt, (toc >> 3) & 3, np.where(config & 1, 3, 2))
        codec = np.where(got, np.where(celt, CELT, SILK), codec).astype(np.uint8)
        lm = np.where(got, p_lm, lm).astype(np.uint8)
        err[got & bad] = -6
        big = (err == 0) & ((120 << lm.astype(np.int64)) > self.cap)
        err[big] = -5
        codec[err != 0] = 0
        return codec, lm, err

    def step(self, packets, lens, cap=None):
        """packets uint8 [n, stride] (TOC first), lens [n] (0 = lost) -> (pcm float32 [n, cap * C]: the row, zeros after the
        frame; pre: the same before the transition's cross-fade (what the decoder's ring holds); result int32 [n]: samples or
        OPN_ERR_*; final_rng uint32 [n] (a rejected packet leaves the stream's previous one); hist uint32 [n]: comb history samples of the CELT frames, concealments included).
        cap: this step's row capacity in samples per channel, if not the batch's"""
        full, self.cap = self.cap, cap or self.cap
        try:
            return self._step(packets, lens)
        finally:
            self.cap = full

    def _step(self, packets, lens):
        packets = np.ascontiguousarray(packets, np.uint8)
        lens = np.asarray(lens, np.uint32)
        n, nch = self.n, self.channels
        codec, lm, err = self.classify(packets, lens)
        got = (lens > 0) & (err == 0)
        to_silk = got & (codec == SILK) & (self.mode == CELT)
        to_celt = got & (codec == CELT) & (self.mode == SILK)
        for s in np.nonzero(to_celt)[0]:                              # decoder.rs:703-705
            lib().orc_synth_state_init(C.byref(self.celt.states[int(s)]))
        trans = hist_t = None
        if to_silk.any():                                             # decoder.rs:519-543: the old decoder's 5 ms
            trans, _, hist_t = self.celt.step(packets, np.zeros(n, np.uint32), 1, cap=240, skip=~to_silk)
            for s in np.nonzero(to_silk)[0]:                          # decoder.rs:555-557
                lib().orc_silk_state_init(C.byref(self.silk.states[int(s)]))
        pcm = np.zeros((n, self.cap * nch), np.float32)
        rng = np.zeros(n, np.uint32)
        hist = np.zeros(n, np.uint32)
        is_celt = (codec == CELT) & (err == 0)
        if is_celt.any():
            p, r, h = self.celt.step(packets, lens, np.where(is_celt, lm, 0), cap=self.cap, skip=~is_celt)
            pcm[is_celt], rng[is_celt], hist[is_celt] = p[is_celt], r[is_celt], h[is_celt]
        for ms, l in ((10, 2), (20, 3)):
            sel = (codec == SILK) & (err == 0) & (lm == l)
            if sel.any():
                p, r = self.silk.step(packets, lens, ms, skip=~sel)
                pcm[sel, :p.shape[1]], rng[sel] = p[sel], r[sel]
        pre = pcm.copy()
        if trans is not None:                                         # decoder.rs:765-788
            n2 = 120 * nch
            hist[to_silk] += hist_t[to_silk]
            for s in np.nonzero(to_silk)[0]:
                faded = np.zeros(n2, np.float32)
                lib().orc_smooth_fade(ptr(trans[s, n2:2 * n2].copy()), ptr(pcm[s, n2:2 * n2].copy()), ptr(faded), 120, nch, 48000)
                pcm[s, :n2] = trans[s, :n2]
                pcm[s, n2:2 * n2] = faded
        result = np.where(err != 0, err, 120 << lm.astype(np.int32)).astype(np.int32)
        rng = np.where(err != 0, self.final, rng).astype(np.uint32)
        self.final = rng
        self.mode = np.where(got, codec, self.mode).astype(np.uint8)
        self.lm = np.where(got, lm, self.lm).astype(np.uint8)
        return pcm, pre, result, rng, hist


def mixed_mode_traffic(n, nsteps, channels, rnd, celt_fill, silk_fill, seed=0, silk_share=0.5, switch=0.1, loss=0.03, plc=0.03, first_loss=0.1,
                       transient_permille=100, celt_lm_p=(0.1, 0.1, 0.3, 0.5)):
    """Packets of streams that each stay in one codec with some stickiness: per step a stream switches codec with probability
    `switch`, loses its packet with `loss` (the first one with loss + first_loss) or sends a PLC/DTX packet (the TOC alone
    or with one byte) with `plc`.  CELT frames of 2.5-20 ms (celt_lm_p), SILK NB/MB/WB at 10 or 20 ms.
    celt_fill(first_stream, n, frame, lm, channels, nbytes, transient_permille) and silk_fill(first_stream, n, frame, bw, ms,
    channels, nbytes) -> uint8 [n, nbytes].  -> packets uint8 [nsteps, n, stride], lens uint32 [nsteps, n]"""
    celt_bytes = {0: 64, 1: 80, 2: 110, 3: 160}
    silk_bytes = 120 * channels
    stride = max(160, silk_bytes)
    packets = np.zeros((nsteps, n, stride), np.uint8)
    lens = np.zeros((nsteps, n), np.uint32)
    silk = rnd.random(n) < silk_share
    for f in range(nsteps):
        silk ^= rnd.random(n) < switch
        lm = rnd.choice(4, size=n, p=np.array(celt_lm_p) / np.sum(celt_lm_p))
        bw = rnd.integers(0, 3, n)
        ms = np.where(rnd.random(n) < 0.5, 10, 20)
        for l in range(4):
            ids = np.nonzero(~silk & (lm == l))[0]
            if len(ids):
                packets[f, ids, :celt_bytes[l]] = celt_fill(seed + 11 * l, n, f, l, channels, celt_bytes[l], transient_permille)[ids]
                lens[f, ids] = celt_bytes[l]
        for b in range(3):
            for m in (10, 20):
                ids = np.nonzero(silk & (bw == b) & (ms == m))[0]
                if len(ids):
                    packets[f, ids, :silk_bytes] = silk_fill(seed + 100 + 7 * b + m, n, f, b, m, channels, silk_bytes)[ids]
                    lens[f, ids] = silk_bytes
        ev = rnd.random(n)
        lens[f, ev < loss + (first_loss if f == 0 else 0.0)] = 0
        short = (ev >= 0.5) & (ev < 0.5 + plc)
        lens[f, short] = 1 + rnd.integers(0, 2, int(short.sum()))
    return packets, lens
