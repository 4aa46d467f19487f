"""The paths bench.py times, at the sizes and with the flags it times them, and the step pipeline's batch-size edges, against
the CPU oracle.  Every stream of every step is compared bit for bit with the oracle's batched step (oracle/step.c), which
advances one decoder state per stream exactly as SynthStream / Celt2Stream / SilkStream do (tests/test_oracle_step.py).

A. Each bench.py workload (the default, --transient-permille 1000, --bitstream 2, --mix, --silk) at its own stream count,
   built with the same packet fills.  Pass 1 runs the benchmark's flags (FLAG_NO_PCM_COPY: the PCM exists only in the
   decoder's ring) for 20 steps back to back, so each of the 8 buffer sets is reused and the ring wraps, and reads the last
   frame back the way bench.py --dump-outputs does.  Pass 2 decodes the same steps into a dense row per step.  The CELT
   workloads also run a timed pass (enable_timing), whose comb history count is the number behind bench.py's roofline.
B. Batch sizes at the launch geometry's edges (warp, CTA and bucket-padding multiples, the 2048-stream cut into three
   frame-kernel groups and the ranges of those groups), for every device-resident step kind.
C. Step kinds interleaved on one grouped batch: uniform steps cut the streams into groups on the host, mixed-frame steps
   again on the device (k_mix_key); both cuts and the state each kind keeps must agree for every stream."""
import numpy as np
import pytest

import bench
import opus_native_b200 as opn
import oracle_lib as O

pytestmark = pytest.mark.gpu
NSTEPS_A = 20  # more than twice the 8 buffer sets
NSTEPS_B = 12  # more than the 8 buffer sets
SILK = opn.BITSTREAM_SYNTH_CELT_1 | opn.BITSTREAM_SYNTH_SILK_1
RESIDENT = opn.FLAG_DEVICE_PTRS | opn.FLAG_INPUTS_READY
MIX_LOSS = 0.03


def _torch():
    return pytest.importorskip("torch")


def _same(got, want, what):
    """PCM rows equal value for value (as everywhere in the suite); names the streams that differ"""
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.nonzero(~(got == want).all(axis=1))[0]
    assert len(bad) == 0, f"{what}: {len(bad)} of {len(got)} streams differ from the oracle, first {bad[:8].tolist()}"


def _groups(n):
    return 3 if n >= 2048 else 1


class Steps:
    """Packets of one batch, resident on the device: arena [nsteps, n, stride], lens [nsteps, n]."""

    def __init__(self, packets, lens, dev):
        torch = _torch()
        self.packets, self.lens = packets, lens
        self.nsteps, self.n, self.stride = packets.shape
        self.d_arena = torch.from_numpy(packets.reshape(-1).copy()).to(dev)
        self.d_off = (torch.arange(self.n, dtype=torch.int64, device=dev) * self.stride).to(torch.int32)
        self.d_len = torch.from_numpy(lens.astype(np.int32)).to(dev)

    def run(self, dec, f, flags, frame_size, row=None, res=None):
        """one device-resident step; row: a dense PCM tensor [n, frame_size * C] or None (FLAG_NO_PCM_COPY)"""
        if row is None:
            flags |= opn.FLAG_NO_PCM_COPY
        dec.decode_float_ptrs(self.d_arena.data_ptr() + f * self.n * self.stride, self.d_off.data_ptr(), self.d_len[f].data_ptr(),
                              row.data_ptr() if row is not None else None, row.stride(0) if row is not None else 0, frame_size,
                              res.data_ptr(), flags)


def _ring_frames(dec, n, nf, channels, cap, dev):
    """The last frame of every stream, read from the decoder's PCM ring (opn_batch_ring) as bench.dump_outputs reads it, for
    frames of each stream's own size nf [n]: -> float32 [n, cap * channels], the frame at the start of the row"""
    torch = _torch()
    ring_ptr, ring_n, pos_ptr = dec.ring()
    ring = torch.as_tensor(bench._DeviceArray(ring_ptr, (n, ring_n, channels), "<f4"), device=dev)
    pos = torch.as_tensor(bench._DeviceArray(pos_ptr, (n,), "<i4"), device=dev).long()
    nf_d = torch.from_numpy(np.asarray(nf, np.int64)).to(dev)
    k = torch.arange(cap, device=dev)
    idx = (pos[:, None] - nf_d[:, None] + k[None, :]) % ring_n
    pcm = torch.gather(ring, 1, idx[:, :, None].expand(-1, -1, channels))
    pcm = torch.where((k[None, :] < nf_d[:, None])[:, :, None], pcm, torch.zeros((), device=dev))
    return pcm.reshape(n, cap * channels).cpu().numpy()


# ------------------------------------------------------------------ A. the benchmark's workloads
def _celt_workload(bitstream, transient_permille):
    fill = opn.synth_fill if bitstream == 1 else opn.celt2_fill
    n = 4096
    packets = fill(0, n, 0, NSTEPS_A, bench.LM, bench.CHANNELS, bench.PKT_BYTES, transient_permille)
    lens = np.full((NSTEPS_A, n), bench.PKT_BYTES, np.uint32)
    return dict(n=n, channels=bench.CHANNELS, bitstream=bitstream, packets=packets, lens=lens,
                lm=np.full((NSTEPS_A, n), bench.LM, np.uint8), flags=RESIDENT, frame=bench.NF)


def _mix_workload():
    """bench.run_mix's packets for rank 0 of one GPU: every step every stream draws a frame size, 10 % transient frames"""
    n, tp = 4096, 100
    rnd = np.random.default_rng(1234)
    stride = max(bench.MIX_PKT_BYTES)
    arena = np.zeros((NSTEPS_A, n, stride), np.uint8)
    lens = np.zeros((NSTEPS_A, n), np.uint32)
    lm_of = rnd.choice(4, size=(NSTEPS_A, n), p=bench.MIX_WEIGHTS)
    for f in range(NSTEPS_A):
        for lm in range(4):
            ids = np.nonzero(lm_of[f] == lm)[0]
            if len(ids):
                arena[f, ids, :bench.MIX_PKT_BYTES[lm]] = opn.synth_fill(7 * lm, len(ids), f, 1, lm, bench.CHANNELS, bench.MIX_PKT_BYTES[lm], tp)[0]
                lens[f, ids] = bench.MIX_PKT_BYTES[lm]
    return dict(n=n, channels=bench.CHANNELS, bitstream=1, packets=arena, lens=lens, lm=lm_of.astype(np.uint8),
                flags=RESIDENT | opn.FLAG_MIXED_FRAMES, frame=bench.NF)


def _silk_workload():
    n, nb = 16384, bench.SILK_PKT_BYTES
    packets = opn.silk_fill(0, n, 0, NSTEPS_A, 2, 20, 1, nb)
    return dict(n=n, channels=1, bitstream=SILK, packets=packets, lens=np.full((NSTEPS_A, n), nb, np.uint32), lm=None,
                flags=RESIDENT | opn.FLAG_SILK_FRAMES, frame=960)


WORKLOADS = {
    "default": lambda: _celt_workload(1, 0),
    "all-transient": lambda: _celt_workload(1, 1000),
    "celt2": lambda: _celt_workload(2, 0),
    "mix": _mix_workload,
    "silk": _silk_workload,
}


@pytest.mark.parametrize("name", list(WORKLOADS))
def test_benchmark_workload_at_its_own_size(name, tmp_path):
    torch = _torch()
    dev = torch.device("cuda:0")
    w = WORKLOADS[name]()
    n, channels, frame, flags = w["n"], w["channels"], w["frame"], w["flags"]
    mixed, silk = bool(flags & opn.FLAG_MIXED_FRAMES), w["lm"] is None
    steps = Steps(w["packets"], w["lens"], dev)
    row = frame * channels
    cfg = opn.DecoderConfiguration(48000, channels, 0)
    want_res = (120 << w["lm"].astype(np.int32)) if not silk else np.full((NSTEPS_A, n), frame, np.int32)

    # pass 1: the benchmark's own flags, PCM left in the ring
    dec1 = opn.BatchDecoder(n, cfg, bitstream=w["bitstream"])
    res1 = torch.zeros(n, dtype=torch.int32, device=dev)
    for f in range(NSTEPS_A):
        steps.run(dec1, f, flags, frame, None, res1)
    dec1.join()
    dec1.synchronize()
    assert np.array_equal(res1.cpu().numpy(), want_res[-1])
    if mixed:
        ring_last = _ring_frames(dec1, n, want_res[-1], channels, frame, dev)
    else:
        bench.dump_outputs(str(tmp_path), dec1, n, frame, channels, dev)
        assert np.array_equal(np.load(tmp_path / "stream.npy"), np.arange(n))  # below DUMP_BYTES every stream is written
        ring_last = np.load(tmp_path / "pcm.npy")
        dump_rng = np.load(tmp_path / "final_range.npy")

    # pass 2: the same steps, a dense row per step; a timed pass of the CELT workloads
    def dense_pass(timing):
        dec = opn.BatchDecoder(n, cfg, bitstream=w["bitstream"])
        dec.enable_timing(timing)
        pcm = torch.full((NSTEPS_A, n, row), 7.0, dtype=torch.float32, device=dev)
        if mixed:
            pcm.zero_()
        res = torch.full((NSTEPS_A, n), -99, dtype=torch.int32, device=dev)
        for f in range(NSTEPS_A):
            steps.run(dec, f, flags, frame, pcm[f], res[f])
        dec.join()
        dec.synchronize()
        return dec, pcm, res.cpu().numpy()

    dec2, pcm2, res2 = dense_pass(False)
    assert np.array_equal(res2, want_res)
    passes = [("pipelined", pcm2)]
    if not silk:
        dec3, pcm3, res3 = dense_pass(True)
        assert np.array_equal(res3, want_res)
        passes.append(("timed", pcm3))

    # the oracle, step by step
    ora = O.SilkBatch(n, channels) if silk else O.CeltBatch(n, channels, w["bitstream"])
    hist_sum = 0
    for f in range(NSTEPS_A):
        if silk:
            want, rng = ora.step(steps.packets[f], steps.lens[f], 20)
        else:
            want, rng, hist = ora.step(steps.packets[f], steps.lens[f], w["lm"][f], cap=frame)
            hist_sum += int(hist.sum(dtype=np.uint64))
        for what, pcm in passes:
            _same(pcm[f].cpu().numpy(), want, f"{name} {what} step {f}")
    _same(ring_last, want, f"{name}: last frame in the ring")
    assert np.abs(want).max() > 0.01
    for dec in [dec1, dec2] + ([dec3] if not silk else []):
        assert np.array_equal(dec.final_ranges(), rng)
    if not mixed:
        assert np.array_equal(dump_rng, rng.astype(np.float64))
    if not silk:
        # the comb history samples behind bench.py's roofline.achieved: counted by the frame kernel in timed passes only
        assert dec2.history_samples() == 0
        assert hist_sum > 0 and dec3.history_samples() == hist_sum


# ------------------------------------------------------------------ B. batch-size edges
MIX_BYTES = {0: 64, 1: 80, 2: 110, 3: 160}


def _kind_steps(kind, n, nsteps, rnd):
    """-> (packets [nsteps, n, stride], lens, lm [nsteps, n] or None, channels, bitstream, flags, frame)"""
    if kind in ("celt1-stereo", "celt1-mono", "celt2-stereo"):
        channels = 1 if kind == "celt1-mono" else 2
        bitstream = 2 if kind == "celt2-stereo" else 1
        nb = 160 if channels == 2 else 100
        fill = opn.synth_fill if bitstream == 1 else opn.celt2_fill
        packets = fill(900 + n, n, 0, nsteps, 3, channels, nb, 150)
        lens = np.full((nsteps, n), nb, np.uint32)
        lens[1:][rnd.random((nsteps - 1, n)) < MIX_LOSS] = 0
        return packets, lens, np.full((nsteps, n), 3, np.uint8), channels, bitstream, RESIDENT, 960
    if kind in ("silk-mono-wb", "silk-stereo-mixed-bw"):
        channels = 1 if kind == "silk-mono-wb" else 2
        nb = 96 * channels
        bws = np.full(n, 2) if channels == 1 else rnd.integers(0, 3, n)
        packets = np.zeros((nsteps, n, nb), np.uint8)
        for bw in range(3):
            ids = np.nonzero(bws == bw)[0]
            if len(ids):
                packets[:, ids] = opn.silk_fill(1000 * bw + n, len(ids), 0, nsteps, bw, 20, channels, nb)
        lens = np.full((nsteps, n), nb, np.uint32)
        lens[1:][rnd.random((nsteps - 1, n)) < MIX_LOSS] = 0
        return packets, lens, None, channels, SILK, RESIDENT | opn.FLAG_SILK_FRAMES, 960
    assert kind == "mixed-stereo"
    packets, lens, lm = _mixed_packets(n, nsteps, rnd, 2)
    return packets, lens, lm, 2, 1, RESIDENT | opn.FLAG_MIXED_FRAMES, 960


def _mixed_packets(n, nsteps, rnd, channels, first=0):
    """every stream draws a frame size per step (10/10/30/50 % of 2.5/5/10/20 ms), 10 % transient frames; lens 0 = lost"""
    packets = np.zeros((nsteps, n, 160), np.uint8)
    lens = np.zeros((nsteps, n), np.uint32)
    lm = rnd.choice(4, size=(nsteps, n), p=bench.MIX_WEIGHTS).astype(np.uint8)
    for f in range(nsteps):
        for l in range(4):
            ids = np.nonzero(lm[f] == l)[0]
            if len(ids):
                packets[f, ids, :MIX_BYTES[l]] = opn.synth_fill(4000 + 10 * l + n, len(ids), first + f, 1, l, channels, MIX_BYTES[l], 100)[0]
                lens[f, ids] = MIX_BYTES[l]
        if first + f > 0:
            lens[f, rnd.random(n) < MIX_LOSS] = 0
    return packets, lens, lm


class MixedOracle:
    """Frame sizes of a mixed-frame step as a decoder sees them: a lost packet conceals one frame of the stream's previous
    size, whatever kind of step decoded that (decoder.rs:427-441); any packet of lens >= 1, PLC/DTX ones included, sets
    that size from its TOC; before any packet, one frame of the row's capacity."""

    def __init__(self, n, cap_lm=3):
        self.last = np.full(n, cap_lm, np.uint8)

    def sizes(self, lens, lm):
        out = np.where(lens > 0, lm, self.last).astype(np.uint8)
        self.last = np.where(lens > 0, lm, self.last).astype(np.uint8)
        return out


SIZES_SMALL = [1, 2, 5, 6, 31, 33, 161]
SIZES_LARGE = [2047, 2048, 2049, 2050, 4097]
KINDS_ALL = ["celt1-stereo", "celt1-mono", "celt2-stereo", "silk-mono-wb", "silk-stereo-mixed-bw", "mixed-stereo"]
KINDS_LARGE = ["celt1-stereo", "celt2-stereo", "silk-mono-wb", "mixed-stereo"]
EDGE_CASES = [(k, n) for n in SIZES_SMALL for k in KINDS_ALL] + [(k, n) for n in SIZES_LARGE for k in KINDS_LARGE]


@pytest.mark.parametrize("kind,n", EDGE_CASES)
def test_batch_size_edges(kind, n):
    """NSTEPS_B device-resident steps enqueued without a host wait, a few percent of the packets lost; every stream of every
    step against the oracle, and the launches per step: one frame-kernel launch below 2048 streams, three from 2048 up."""
    torch = _torch()
    dev = torch.device("cuda:0")
    rnd = np.random.default_rng([KINDS_ALL.index(kind), n])
    packets, lens, lm, channels, bitstream, flags, frame = _kind_steps(kind, n, NSTEPS_B, rnd)
    steps = Steps(packets, lens, dev)
    dec = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, channels, 0), bitstream=bitstream)
    pcm = torch.zeros((NSTEPS_B, n, frame * channels), dtype=torch.float32, device=dev)
    res = torch.full((NSTEPS_B, n), -99, dtype=torch.int32, device=dev)
    for f in range(NSTEPS_B):
        steps.run(dec, f, flags, frame, pcm[f], res[f])
    dec.join()
    dec.synchronize()
    mixed = bool(flags & opn.FLAG_MIXED_FRAMES)
    assert dec.stats()["launches"] == [NSTEPS_B, NSTEPS_B * _groups(n), 2 * NSTEPS_B if mixed else 0]
    got_res = res.cpu().numpy()
    silk = lm is None
    ora = O.SilkBatch(n, channels) if silk else O.CeltBatch(n, channels, bitstream)
    sizes = MixedOracle(n)
    for f in range(NSTEPS_B):
        if silk:
            want, rng = ora.step(packets[f], lens[f], 20)
            want_res = np.full(n, 960)
        else:
            lm_f = sizes.sizes(lens[f], lm[f]) if mixed else lm[f]
            want, rng, _ = ora.step(packets[f], lens[f], lm_f, cap=frame)
            want_res = 120 << lm_f.astype(np.int32)
        assert np.array_equal(got_res[f], want_res), f
        _same(pcm[f].cpu().numpy(), want, f"{kind} n={n} step {f}")
    assert np.array_equal(dec.final_ranges(), rng)


# ------------------------------------------------------------------ C. step kinds interleaved on one grouped batch
@pytest.mark.parametrize("n", [2050, 4097])
def test_step_kinds_interleaved_on_a_grouped_batch(n):
    """SYNTH-CELT/1 stereo, one batch: uniform 20 ms, mixed, uniform 5 ms, mixed, uniform 20 ms with losses -- enqueued without
    a host wait -- then a host-buffer call (per-stream frame sizes, bucketed on the host), then mixed and uniform 10 ms.  Every
    stream of every step against one oracle decoder per stream that follows the stream's frame sizes."""
    torch = _torch()
    dev = torch.device("cuda:0")
    rnd = np.random.default_rng(n)
    channels, cap = 2, 960
    plan = ["u3", "mix", "u1", "mix", "u3-lost", "host", "mix", "u2"]
    nsteps = len(plan)
    packets = np.zeros((nsteps, n, 160), np.uint8)
    lens = np.zeros((nsteps, n), np.uint32)
    lm = np.zeros((nsteps, n), np.uint8)
    for f, kind in enumerate(plan):
        if kind in ("mix", "host"):
            p, l, m = _mixed_packets(n, 1, rnd, channels, first=f)
            packets[f], lens[f], lm[f] = p[0], l[0], m[0]
            if kind == "host":
                lens[f] = np.array([MIX_BYTES[int(x)] for x in lm[f]], np.uint32)  # the host call: no losses
        else:
            l = int(kind[1])
            nb = MIX_BYTES[l]
            packets[f, :, :nb] = opn.synth_fill(6000 + l, n, f, 1, l, channels, nb, 100)[0]
            lens[f], lm[f] = nb, l
            if kind == "u3-lost":
                lens[f, rnd.random(n) < 0.05] = 0
    steps = Steps(packets, lens, dev)
    dec = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, channels, 0), bitstream=1)
    pcm = torch.zeros((nsteps, n, cap * channels), dtype=torch.float32, device=dev)
    res = torch.full((nsteps, n), -99, dtype=torch.int32, device=dev)
    host_pcm = np.zeros((n, cap * channels), np.float32)
    host_res = None
    for f, kind in enumerate(plan):
        if kind == "mix":
            steps.run(dec, f, RESIDENT | opn.FLAG_MIXED_FRAMES, cap, pcm[f], res[f])
        elif kind == "host":
            host_res = dec.decode_float(packets[f].reshape(-1), (np.arange(n) * 160).astype(np.uint32), lens[f].copy(), host_pcm, cap)
        else:
            nf = 120 << int(lm[f, 0])
            steps.run(dec, f, RESIDENT, nf, pcm[f, :, :nf * channels], res[f])
    dec.join()
    dec.synchronize()
    got, got_res = pcm.cpu().numpy(), res.cpu().numpy()
    ora = O.CeltBatch(n, channels, 1)
    sizes = MixedOracle(n)
    for f, kind in enumerate(plan):
        lm_f = sizes.sizes(lens[f], lm[f])  # a lost packet of a uniform step conceals the step's frame size
        if kind.startswith("u"):
            lm_f = lm[f]
        want, rng, _ = ora.step(packets[f], lens[f], lm_f, cap=cap)
        want_res = 120 << lm_f.astype(np.int32)
        if kind == "host":
            assert np.array_equal(host_res, want_res)
            _same(host_pcm, want, f"n={n} step {f} ({kind})")
            continue
        if kind.startswith("u"):
            nf = 120 << int(lm[f, 0])
            assert np.all(got_res[f] == nf), f
            _same(np.ascontiguousarray(got[f, :, :nf * channels]), want[:, :nf * channels], f"n={n} step {f} ({kind})")
        else:
            assert np.array_equal(got_res[f], want_res), f
            _same(got[f], want, f"n={n} step {f} ({kind})")
    assert np.array_equal(dec.final_ranges(), rng)
