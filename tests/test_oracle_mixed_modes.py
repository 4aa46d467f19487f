"""The oracle of mixed-mode steps (mixed_modes_oracle.MixedModeBatch), pinned bit for bit to one SynthStream and one SilkStream per stream
composed by hand, as Decoder::decode composes its CELT and SILK decoders (decoder.rs:519-557, 703-705, 765-788).  CPU only."""
import numpy as np

import mixed_modes_oracle as M
import oracle_lib as O


def _celt_fill(first, n, frame, lm, channels, nbytes, transient):
    return O.synth_fill(first, n, frame, 1, lm, channels, nbytes, transient)[0]


def _silk_fill(first, n, frame, bw, ms, channels, nbytes):
    return O.silk_fill(first, n, frame, 1, bw, ms, channels, nbytes)[0]


def _per_stream(packets, lens, channels, cap=960, apply_comb=True):
    """-> per step (pcm [n, cap * C], result [n], final_rng [n]) from one decoder pair per stream"""
    nsteps, n = lens.shape
    celt = [O.SynthStream(3, channels, apply_comb) for _ in range(n)]
    silk = [O.SilkStream(channels) for _ in range(n)]
    mode = [0] * n
    last = [3] * n  # LM of the last packet; before any, the row's capacity
    n2 = 120 * channels
    out = []
    for f in range(nsteps):
        pcm = np.zeros((n, cap * channels), np.float32)
        res = np.zeros(n, np.int32)
        rng = np.zeros(n, np.uint32)
        for s in range(n):
            L = int(lens[f, s])
            pk = packets[f, s, :L]
            if L == 0:
                if mode[s] == M.SILK:
                    w = silk[s].decode(b"", 0, 10 if last[s] == 2 else 20, channels, lost=True)[3]
                else:
                    w = celt[s].conceal(last[s])
                pcm[s, :len(w)] = w
                res[s] = len(w) // channels
                continue
            toc = int(pk[0])
            if toc & 0x80:
                lm = (toc >> 3) & 3
                if mode[s] == M.SILK:
                    celt[s] = O.SynthStream(3, channels, apply_comb)        # decoder.rs:703-705
                celt[s].lm = lm
                side, _, _, w = celt[s].decode(pk[1:])
                rng[s] = side.final_rng if L > 2 else 0
                mode[s], last[s] = M.CELT, lm
            else:
                ms = 20 if (toc >> 3) & 1 else 10
                bw = (toc >> 5) & 3
                switch = mode[s] == M.CELT
                if switch:
                    silk[s] = O.SilkStream(channels)                        # decoder.rs:555-557
                    trans = celt[s].conceal(1)                              # decoder.rs:519-543
                lost = L <= 2
                side, _, _, w = silk[s].decode(b"" if lost else pk[1:], 0 if lost else bw, ms, channels, lost=lost)
                w = w.copy()
                rng[s] = 0 if lost else side.final_rng
                if switch:                                                  # decoder.rs:765-778
                    faded = np.zeros(n2, np.float32)
                    O.lib().orc_smooth_fade(O.ptr(trans[n2:2 * n2].copy()), O.ptr(w[n2:2 * n2].copy()), O.ptr(faded), 120, channels, 48000)
                    w[:n2] = trans[:n2]
                    w[n2:2 * n2] = faded
                mode[s], last[s] = M.SILK, 3 if ms == 20 else 2
            pcm[s, :len(w)] = w
            res[s] = len(w) // channels
        out.append((pcm, res, rng))
    return out


def test_mixed_mode_batch_equals_per_stream_composition():
    """60 streams, 16 steps: codec switches both ways, losses (some before any packet), TOC-only and one-byte packets of both
    codecs, CELT frames of 2.5-20 ms and SILK frames of every bandwidth at 10 and 20 ms."""
    _against_per_stream(apply_comb=True)


def _against_per_stream(apply_comb):
    rnd = np.random.default_rng(77)
    for channels in (2, 1):
        n, nsteps = 60, 16
        packets, lens = M.mixed_mode_traffic(n, nsteps, channels, rnd, _celt_fill, _silk_fill, seed=5, switch=0.2, loss=0.08, plc=0.08)
        want = _per_stream(packets, lens, channels, apply_comb=apply_comb)
        batch = M.MixedModeBatch(n, channels, n_threads=4, apply_comb=apply_comb)
        switches = 0
        for f in range(nsteps):
            before = batch.mode.copy()
            pcm, pre, res, rng, _ = batch.step(packets[f], lens[f])
            switches += int(((before != 0) & (batch.mode != before)).sum())
            assert np.array_equal(res, want[f][1]), f
            assert np.array_equal(rng, want[f][2]), f
            assert np.array_equal(pcm, want[f][0]), f
        assert switches > 20
        assert (lens == 1).any() and (lens == 2).any() and (lens[0] == 0).any()


def test_mixed_mode_batch_without_post_filter_equals_per_stream_composition():
    """apply_comb=False (a batch created with postfilter = false): the same traffic against SynthStream(apply_comb=False) and
    SilkStream pairs, and the post-filter changes the PCM of that traffic"""
    _against_per_stream(apply_comb=False)
    rnd = np.random.default_rng(78)
    packets, lens = M.mixed_mode_traffic(40, 6, 2, rnd, _celt_fill, _silk_fill, seed=6)
    on, off = M.MixedModeBatch(40, 2, n_threads=4), M.MixedModeBatch(40, 2, n_threads=4, apply_comb=False)
    differ = False
    for f in range(6):
        a, b = on.step(packets[f], lens[f])[0], off.step(packets[f], lens[f])[0]
        differ |= not np.array_equal(a, b)
    assert differ
