"""The oracle's batched steps (oracle/step.c: orc_synth_step, orc_celt2_step, orc_silk_step) against the per-stream classes the
GPU tests otherwise use, bit for bit.  The batched steps are what tests/test_gpu_workloads.py checks every stream of every step
with, at the benchmark's sizes; this pins them to SynthStream / Celt2Stream / SilkStream first: chained frames, per-stream
frame sizes that change from step to step, lost packets, and the comb history count the GPU frame kernel keeps in timed passes."""
import numpy as np
import pytest

import oracle_lib as O

NS, NSTEPS = 50, 10
CELT_BYTES = {0: 64, 1: 80, 2: 112, 3: 160}


def _hist_want(state, old_period, old_gain, channels):
    """channels * (max(T_old, T_new, 15) + 2) when the post-filter runs (either gain non-zero), else 0"""
    if old_gain == 0.0 and state.pf_gain == 0.0:
        return 0
    return channels * (max(old_period, state.pf_period, 15) + 2)


def _celt_packets(bitstream, rnd, channels):
    """[NSTEPS, NS, 160] packets of a frame size drawn per stream and step, lens (3 % lost after the first step), lm"""
    packets = np.zeros((NSTEPS, NS, 160), np.uint8)
    lm = rnd.choice(4, size=(NSTEPS, NS), p=[0.1, 0.1, 0.3, 0.5]).astype(np.uint8)
    lens = np.zeros((NSTEPS, NS), np.uint32)
    for f in range(NSTEPS):
        for s in range(NS):
            nb = CELT_BYTES[int(lm[f, s])]
            if bitstream == 1:
                packets[f, s, :nb] = O.synth_fill(300 + s, 1, f, 1, int(lm[f, s]), channels, nb, transient_permille=200)[0, 0]
            else:
                packets[f, s, :nb] = O.celt2_packet(300 + s, f, int(lm[f, s]), channels, nb, transient_permille=200)[0]
            lens[f, s] = nb
        if f > 0:
            lens[f, rnd.random(NS) < 0.05] = 0
    lens[4, 7] = 1  # a TOC alone is a lost frame too (decoder.rs:467)
    return packets, lens, lm


@pytest.mark.parametrize("bitstream,channels", [(1, 2), (1, 1), (2, 2), (2, 1)])
def test_celt_step_equals_per_stream_decoders(bitstream, channels):
    rnd = np.random.default_rng(17 * bitstream + channels)
    packets, lens, lm = _celt_packets(bitstream, rnd, channels)
    batch = O.CeltBatch(NS, channels, bitstream, n_threads=4)
    ref = [(O.SynthStream if bitstream == 1 else O.Celt2Stream)(3, channels) for _ in range(NS)]
    n_hist = 0
    for f in range(NSTEPS):
        pcm, rng, hist = batch.step(packets[f], lens[f], lm[f])
        for s in range(NS):
            r = ref[s]
            r.lm = int(lm[f, s])
            old_period, old_gain = r.state.pf_period, r.state.pf_gain
            payload = packets[f, s, 1:lens[f, s]] if lens[f, s] else b""
            if bitstream == 1:
                side, _, _, want = r.decode(payload)
            else:
                side, want = r.decode(payload)
            nf = 120 << int(lm[f, s])
            assert np.array_equal(pcm[s, :nf * channels].view(np.uint32), want.view(np.uint32)), (f, s)
            assert not pcm[s, nf * channels:].any()
            assert rng[s] == (side.final_rng if lens[f, s] > 1 else 0), (f, s)
            assert hist[s] == _hist_want(r.state, old_period, old_gain, channels), (f, s)
            n_hist += hist[s] > 0
        assert bytes(batch.states[NS - 1]) == bytes(ref[NS - 1].state)
    assert n_hist > NS  # the post-filter ran in many frames: the count was exercised


def test_celt_step_without_postfilter_counts_no_history():
    packets = O.synth_fill(5, 8, 0, 3, 3, 2, 160)
    batch = O.CeltBatch(8, 2, apply_comb=False, n_threads=2)
    ref = [O.SynthStream(3, 2, apply_comb=False) for _ in range(8)]
    for f in range(3):
        pcm, rng, hist = batch.step(packets[f], np.full(8, 160), 3)
        assert not hist.any()
        for s in range(8):
            side, _, _, want = ref[s].decode(packets[f, s, 1:])
            assert np.array_equal(pcm[s], want) and rng[s] == side.final_rng


@pytest.mark.parametrize("channels", [1, 2])
def test_silk_step_equals_per_stream_decoders(channels):
    """bandwidths mixed across the streams (read from the TOC), 10 and 20 ms steps, lost packets"""
    rnd = np.random.default_rng(40 + channels)
    nb = 96 * channels
    bws = rnd.integers(0, 3, NS)
    ms_of = [20, 20, 10, 20, 10, 10, 20, 20, 20, 10]
    batch = O.SilkBatch(NS, channels, n_threads=4)
    ref = [O.SilkStream(channels) for _ in range(NS)]
    for f, ms in enumerate(ms_of):
        packets = np.zeros((NS, nb), np.uint8)
        for s in range(NS):
            packets[s] = O.silk_fill(200 + s, 1, f, 1, int(bws[s]), ms, channels, nb)[0, 0]
        lens = np.full(NS, nb, np.uint32)
        lens[rnd.random(NS) < 0.06] = 0
        if f == 0:
            lens[3] = 0  # lost before anything was decoded: silence, state untouched
        pcm, rng = batch.step(packets, lens, ms)
        for s in range(NS):
            if lens[s]:
                side, _, _, want = ref[s].decode(packets[s, 1:], int(bws[s]), ms, channels)
            else:
                side, _, _, want = ref[s].decode(b"", int(bws[s]), ms, channels, lost=True)
            assert np.array_equal(pcm[s].view(np.uint32), want.view(np.uint32)), (f, s)
            assert rng[s] == (side.final_rng if lens[s] else 0), (f, s)
    assert np.abs(pcm).max() > 0.01


@pytest.mark.parametrize("bitstream", [1, 2, 0])
def test_skipped_streams_are_left_untouched(bitstream):
    """skip: a stream left out of a step keeps its state, as a per-stream decoder that was not called (SYNTH-CELT/1, /2 and,
    for bitstream 0, SYNTH-SILK/1); its row, final range and history count are zero.  A host-buffer call that conceals
    several frames for some streams is modelled with such steps."""
    rnd = np.random.default_rng(90 + bitstream)
    channels = 2
    if bitstream:
        packets, lens, lm = _celt_packets(bitstream, rnd, channels)
        batch = O.CeltBatch(NS, channels, bitstream, n_threads=4)
        ref = [(O.SynthStream if bitstream == 1 else O.Celt2Stream)(3, channels) for _ in range(NS)]
    else:
        bws = rnd.integers(0, 3, NS)
        packets = np.stack([O.silk_fill(200 + s, 1, 0, NSTEPS, int(bws[s]), 20, channels, 192)[:, 0] for s in range(NS)], axis=1)
        lens = np.full((NSTEPS, NS), 192, np.uint32)
        lens[1:][rnd.random((NSTEPS - 1, NS)) < 0.1] = 0
        batch = O.SilkBatch(NS, channels, n_threads=4)
        ref = [O.SilkStream(channels) for _ in range(NS)]
    n_skipped = 0
    for f in range(NSTEPS):
        skip = rnd.random(NS) < 0.3
        if bitstream:
            pcm, rng, hist = batch.step(packets[f], lens[f], lm[f], cap=960, skip=skip)
        else:
            pcm, rng = batch.step(packets[f], lens[f], 20, skip=skip)
            hist = np.zeros(NS, np.uint32)
        for s in range(NS):
            if skip[s]:
                assert not pcm[s].any() and rng[s] == 0 and hist[s] == 0, (f, s)
                n_skipped += 1
                continue
            payload = packets[f, s, 1:lens[f, s]] if lens[f, s] else b""
            if bitstream == 1:
                ref[s].lm = int(lm[f, s])
                side, _, _, want = ref[s].decode(payload)
            elif bitstream == 2:
                ref[s].lm = int(lm[f, s])
                side, want = ref[s].decode(payload)
            else:
                side, _, _, want = ref[s].decode(payload, int(bws[s]), 20, channels, lost=not lens[f, s])
            assert np.array_equal(pcm[s, :len(want)].view(np.uint32), want.view(np.uint32)), (f, s)
            assert rng[s] == (side.final_rng if lens[f, s] > 1 else 0), (f, s)
    for s in range(NS):
        assert bytes(batch.states[s]) == bytes(ref[s].state), s
    assert n_skipped > NS
