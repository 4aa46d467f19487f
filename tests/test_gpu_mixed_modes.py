"""Mixed-mode device-resident steps (OPN_FLAG_MIXED_MODES): CELT and SILK packets in one step, with mode switches on the
device, against the CPU oracle (mixed_modes_oracle.MixedModeBatch, pinned to per-stream decoders by tests/test_oracle_mixed_modes.py).
Dense rows, result_per_stream and final_ranges() are compared bit for bit for every stream.

A. Randomised traffic: streams keep their codec with some stickiness and switch both ways; CELT 2.5-20 ms (10 % transient),
   SILK NB/MB/WB at 10 and 20 ms, losses (also at step 0), PLC/DTX packets of both codecs.  16 steps back to back, mono and
   stereo, SYNTH-CELT/1 and /2, below and above the 2048-stream cut into frame groups.  A FLAG_NO_PCM_COPY pass reads the last
   frame from the ring: the PCM before the gain and before the transition's cross-fade.
B. Every stream switches at the same step, CELT -> SILK and back, with a decoder gain of +6 and -6 dB.
C. Against the other step kinds: an all-CELT step equals a mixed-frame step, an all-SILK one a SILK-frames step, and loss-free
   traffic the host-buffer path (ring and ring positions too).
D. Per-stream errors leave the stream's state untouched and its neighbours exact; flag validation.
E. Interleaving with uniform, mixed-frame, SILK-frames and host-buffer calls on one grouped batch.
F. A timed pass equals an untimed one; launches per step; the comb history count.
G. The per-GPU size of the mixed-mode workload: 32 768 stereo streams."""
import numpy as np
import pytest

import opus_native_b200 as opn
import mixed_modes_oracle as M
import oracle_lib as O
from test_gpu_stream_state import _gain
from test_gpu_workloads import RESIDENT, _ring_frames

pytestmark = pytest.mark.gpu
MODES = RESIDENT | opn.FLAG_MIXED_MODES
CAP = 960


def _torch():
    return pytest.importorskip("torch")


def _fills(bitstream):
    fill = opn.celt2_fill if bitstream == 2 else opn.synth_fill

    def celt(first, n, frame, lm, channels, nbytes, transient):
        return fill(first, n, frame, 1, lm, channels, nbytes, transient)[0]

    def silk(first, n, frame, bw, ms, channels, nbytes):
        return opn.silk_fill(first, n, frame, 1, bw, ms, channels, nbytes)[0]
    return celt, silk


def _traffic(n, nsteps, channels, bitstream, seed, **kw):
    celt, silk = _fills(bitstream or 1)
    return M.mixed_mode_traffic(n, nsteps, channels, np.random.default_rng(seed), celt, silk, seed=seed, **kw)


def _decoder(n, channels, bitstream=1, gain=0):
    return opn.BatchDecoder(n, opn.DecoderConfiguration(48000, channels, gain), bitstream=bitstream | opn.BITSTREAM_SYNTH_SILK_1)


class Device:
    """All steps' packets on the device, a dense row and a result row per step"""

    def __init__(self, packets, lens, channels, cap=CAP, rows=True):
        torch = _torch()
        self.dev = torch.device("cuda:0")
        self.nsteps, self.n, self.stride = packets.shape
        self.arena = torch.from_numpy(packets.reshape(-1).copy()).to(self.dev)
        self.off = (torch.arange(self.n, dtype=torch.int64, device=self.dev) * self.stride).to(torch.int32)
        self.lens = torch.from_numpy(lens.astype(np.int32)).to(self.dev)
        self.rows = torch.zeros((self.nsteps, self.n, cap * channels), dtype=torch.float32, device=self.dev) if rows else None
        self.res = torch.zeros((self.nsteps, self.n), dtype=torch.int32, device=self.dev)
        torch.cuda.synchronize()

    def run(self, dec, f, flags=MODES, frame_size=CAP, dense=True):
        row = self.rows[f] if dense else None
        if row is None:
            flags |= opn.FLAG_NO_PCM_COPY
        dec.decode_float_ptrs(self.arena.data_ptr() + f * self.n * self.stride, self.off.data_ptr(), self.lens[f].data_ptr(),
                              row.data_ptr() if row is not None else None, row.stride(0) if row is not None else 0, frame_size,
                              self.res[f].data_ptr(), flags)

    def pcm(self, f):
        return self.rows[f].cpu().numpy()

    def result(self, f):
        return self.res[f].cpu().numpy()


def _same(got, want, what):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.nonzero(~(got == want).reshape(len(got), -1).all(axis=1))[0]
    assert len(bad) == 0, f"{what}: {len(bad)} of {len(got)} streams differ, first {bad[:8].tolist()}"


def _host(dec, packets, lens, frame_size=CAP):
    n, stride = lens.shape[0], packets.shape[1]
    pcm = np.zeros((n, frame_size * dec.channels), np.float32)
    res = dec.decode_float(np.ascontiguousarray(packets).reshape(-1), (np.arange(n) * stride).astype(np.uint32),
                           lens.astype(np.uint32), pcm, frame_size)
    return pcm, res


# ------------------------------------------------------------------ A. randomised traffic
@pytest.mark.parametrize("n,channels,bitstream", [(300, 2, 1), (300, 1, 2), (2050, 2, 2), (2050, 1, 1), (4097, 2, 1), (4097, 1, 2)])
def test_random_traffic_against_the_oracle(n, channels, bitstream):
    nsteps = 16
    packets, lens = _traffic(n, nsteps, channels, bitstream, seed=n + 10 * channels + bitstream)
    d = Device(packets, lens, channels)
    dec = _decoder(n, channels, bitstream)
    for f in range(nsteps):
        d.run(dec, f)
    dec.synchronize()
    oracle = M.MixedModeBatch(n, channels, bitstream)
    switches = 0
    for f in range(nsteps):
        before = oracle.mode.copy()
        pcm, pre, res, rng, _ = oracle.step(packets[f], lens[f])
        switches += int(((before != 0) & (oracle.mode != before)).sum())
        assert np.array_equal(d.result(f), res), f
        _same(d.pcm(f), pcm, f"step {f}")
    assert np.array_equal(dec.final_ranges(), rng)
    assert switches > n // 10
    # the same steps without dense rows: the last frame of each stream, read from the ring, is the PCM before the fade
    nr = Device(packets, lens, channels, rows=False)
    dec2 = _decoder(n, channels, bitstream)
    for f in range(nsteps):
        nr.run(dec2, f, dense=False)
    dec2.synchronize()
    assert np.array_equal(nr.result(nsteps - 1), res)
    ok = (lens[-1] > 2) & (res > 0)
    ring = _ring_frames(dec2, n, np.where(ok, res, 0), channels, CAP, nr.dev)
    _same(ring[ok], pre[ok], "ring")


# ------------------------------------------------------------------ B. every stream switches at once
@pytest.mark.parametrize("gain_q8", [1536, -1536])
def test_every_stream_switches_at_the_same_step(gain_q8):
    n, channels = 300, 2
    celt, silk = _fills(1)
    plan = ["celt"] * 3 + ["silk"] * 3 + ["celt"] * 3
    packets = np.zeros((len(plan), n, 240), np.uint8)
    lens = np.zeros((len(plan), n), np.uint32)
    rnd = np.random.default_rng(gain_q8 & 0xFFFF)
    for f, kind in enumerate(plan):
        for s0 in range(0, n, 50):
            ids = np.arange(s0, s0 + 50)
            if kind == "celt":
                lm = int(rnd.integers(0, 4))
                nb = {0: 64, 1: 80, 2: 110, 3: 160}[lm]
                packets[f, ids, :nb] = celt(40 + lm, n, f, lm, channels, nb, 100)[ids]
            else:
                nb = 240
                packets[f, ids, :nb] = silk(50, n, f, int(rnd.integers(0, 3)), int(rnd.choice([10, 20])), channels, nb)[ids]
            lens[f, ids] = nb
    d = Device(packets, lens, channels)
    dec = _decoder(n, channels, 1, gain_q8)
    oracle = M.MixedModeBatch(n, channels, 1)
    g = _gain(gain_q8)
    for f in range(len(plan)):
        d.run(dec, f)
        dec.synchronize()
        pcm, _, res, rng, _ = oracle.step(packets[f], lens[f])
        assert np.array_equal(d.result(f), res), f
        assert np.array_equal(dec.final_ranges(), rng), f
        _same(d.pcm(f), pcm * g, f"step {f}")


# ------------------------------------------------------------------ C. against the other step kinds
def test_all_celt_equals_mixed_frames_and_all_silk_equals_silk_frames():
    n, channels = 2050, 2
    packets, lens = _traffic(n, 8, channels, 1, seed=3, silk_share=0.0, switch=0.0)
    a, b = Device(packets, lens, channels), Device(packets, lens, channels)
    d1, d2 = _decoder(n, channels), _decoder(n, channels)
    for f in range(8):
        a.run(d1, f)
        b.run(d2, f, RESIDENT | opn.FLAG_MIXED_FRAMES)
    d1.synchronize()
    d2.synchronize()
    for f in range(8):
        assert np.array_equal(a.result(f), b.result(f))
        _same(a.pcm(f), b.pcm(f), f"celt step {f}")
    assert np.array_equal(d1.final_ranges(), d2.final_ranges())
    # SILK at 20 ms, every bandwidth
    celt, silk = _fills(1)
    packets = np.zeros((6, n, 240), np.uint8)
    bw = np.random.default_rng(4).integers(0, 3, n)
    for f in range(6):
        for w in range(3):
            packets[f, bw == w] = silk(70 + w, n, f, w, 20, channels, 240)[bw == w]
    lens = np.full((6, n), 240, np.uint32)
    lens[2, ::17] = 0
    a, b = Device(packets, lens, channels), Device(packets, lens, channels)
    d1, d2 = _decoder(n, channels), _decoder(n, channels)
    for f in range(6):
        a.run(d1, f)
        b.run(d2, f, RESIDENT | opn.FLAG_SILK_FRAMES)
    d1.synchronize()
    d2.synchronize()
    for f in range(6):
        assert np.array_equal(a.result(f), b.result(f))
        _same(a.pcm(f), b.pcm(f), f"silk step {f}")
    assert np.array_equal(d1.final_ranges(), d2.final_ranges())


@pytest.mark.parametrize("channels", [2, 1])
def test_loss_free_traffic_equals_the_host_path(channels):
    torch = _torch()
    n, nsteps = 2050, 10
    packets, lens = _traffic(n, nsteps, channels, 1, seed=21 + channels, loss=0.0, first_loss=0.0, switch=0.15)
    d = Device(packets, lens, channels)
    dev_dec, host_dec = _decoder(n, channels), _decoder(n, channels)
    for f in range(nsteps):
        d.run(dev_dec, f)
        dev_dec.synchronize()
        pcm, res = _host(host_dec, packets[f], lens[f])
        assert np.array_equal(d.result(f), res), f
        _same(d.pcm(f), pcm, f"step {f}")
        assert np.array_equal(dev_dec.final_ranges(), host_dec.final_ranges()), f
    import bench
    rings = []
    for dec in (dev_dec, host_dec):
        ptr, ring_n, pos_ptr = dec.ring()
        r = torch.as_tensor(bench._DeviceArray(ptr, (n, ring_n * channels), "<f4"), device=d.dev).cpu().numpy()
        p = torch.as_tensor(bench._DeviceArray(pos_ptr, (n,), "<i4"), device=d.dev).cpu().numpy()
        rings.append((r, p))
    _same(rings[0][0], rings[1][0], "ring")
    assert np.array_equal(rings[0][1], rings[1][1])


# ------------------------------------------------------------------ D. errors
def test_per_stream_errors_leave_the_stream_untouched():
    n, channels = 96, 2
    packets, lens = _traffic(n, 6, channels, 1, seed=9, loss=0.0, plc=0.0)
    bad = packets[3].copy()
    blens = lens[3].copy()
    kinds = {}
    for s in range(0, n, 6):
        k = (s // 6) % 6
        toc = int(bad[s, 0])
        if k == 0:
            bad[s, 0] = (12 + (s % 4)) << 3 | 4                       # hybrid
        elif k == 1:
            bad[s, 0] = (4 * (s % 3) + 2) << 3 | 4                    # SILK 40 ms
        elif k == 2:
            bad[s, 0] = toc | 1                                       # two frames
        elif k == 3:
            bad[s, 0] = toc & ~4                                      # mono packet
        elif k == 4:
            bad[s, 0] = 0x80 | (3 << 3) | 4                           # CELT 20 ms in a 10 ms row
        kinds[s] = k
    packets[3] = bad
    oracle = M.MixedModeBatch(n, channels, 1)
    d = Device(packets, lens, channels)
    dec = _decoder(n, channels)
    for f in range(6):
        cap = 480 if f == 3 else CAP
        d.run(dec, f, frame_size=cap)
        dec.synchronize()
        pcm, _, res, rng, _ = oracle.step(packets[f], lens[f], cap=cap)
        assert np.array_equal(d.result(f), res), (f, d.result(f)[:12], res[:12])
        _same(d.pcm(f)[:, :cap * channels], pcm, f"step {f}")
        assert np.array_equal(dec.final_ranges(), rng), f
        if f == 3:
            got = d.result(f)
            assert all(got[s] == (-5 if k == 4 else -6) for s, k in kinds.items() if k < 5 and blens[s] > 0)


def test_opus_celt_layout_rejects_celt_packets_per_stream():
    n, channels = 64, 1
    packets, lens = _traffic(n, 4, channels, 1, seed=12, loss=0.0, plc=0.0)
    oracle = M.MixedModeBatch(n, channels, 0)
    d = Device(packets, lens, channels)
    dec = _decoder(n, channels, opn.BITSTREAM_OPUS)
    for f in range(4):
        d.run(dec, f)
        dec.synchronize()
        pcm, _, res, rng, _ = oracle.step(packets[f], lens[f])
        assert np.array_equal(d.result(f), res), f
        _same(d.pcm(f), pcm, f"step {f}")
    assert (res == -6).any() and (res > 0).any()


def test_flag_validation():
    torch = _torch()
    n = 8
    dev = torch.device("cuda:0")
    arena = torch.zeros(64, dtype=torch.uint8, device=dev)
    off = torch.zeros(n, dtype=torch.int32, device=dev)
    lens = torch.zeros(n, dtype=torch.int32, device=dev)
    rows = torch.zeros((n, 1920), dtype=torch.float32, device=dev)
    res = torch.zeros(n, dtype=torch.int32, device=dev)

    def call(dec, flags, host=False):
        if host:
            a, o, l, p, r = np.zeros(64, np.uint8), np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.zeros((n, 1920), np.float32), np.zeros(n, np.int32)
            return opn.lib().opn_batch_decode_float(dec._h, a.ctypes.data, o.ctypes.data, l.ctypes.data, p.ctypes.data, 1920, 960, r.ctypes.data, flags)
        return opn.lib().opn_batch_decode_float(dec._h, arena.data_ptr(), off.data_ptr(), lens.data_ptr(), rows.data_ptr(), 1920, 960,
                                                res.data_ptr(), flags)
    with_silk = _decoder(n, 2)
    celt_only = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, 2, 0), bitstream=opn.BITSTREAM_SYNTH_CELT_1)
    assert call(celt_only, MODES) == -1
    assert call(with_silk, MODES | opn.FLAG_SILK_FRAMES) == -1
    assert call(with_silk, opn.FLAG_MIXED_MODES, host=True) == -1
    assert call(with_silk, MODES) == 0
    assert call(with_silk, MODES | opn.FLAG_MIXED_FRAMES) == 0
    with_silk.synchronize()


# ------------------------------------------------------------------ E. interleaving with the other step kinds
def test_interleaved_with_other_step_kinds():
    n, channels = 2050, 2
    celt, silk = _fills(1)
    oracle = M.MixedModeBatch(n, channels, 1)
    dec = _decoder(n, channels)
    rnd = np.random.default_rng(31)

    def device_step(packets, lens, flags, frame_size=CAP):
        d = Device(packets[None], lens[None], channels)
        d.run(dec, 0, flags, frame_size)
        dec.synchronize()
        pcm, _, res, rng, _ = oracle.step(packets, lens)
        assert np.array_equal(d.result(0), res)
        _same(d.pcm(0)[:, :CAP * channels], pcm, f"flags {flags}")
        assert np.array_equal(dec.final_ranges(), rng)

    def host_step(packets, lens):
        pcm, res = _host(dec, packets, lens)
        want, _, wres, rng, _ = oracle.step(packets, lens)
        assert np.array_equal(res, wres)
        _same(pcm, want, "host call")
        assert np.array_equal(dec.final_ranges(), rng)

    def uniform(kind):
        p = np.zeros((n, 240), np.uint8)
        if kind == "celt":
            p[:, :160] = celt(90, n, int(rnd.integers(0, 99)), 3, channels, 160, 100)
            return p, np.full(n, 160, np.uint32)
        p[:, :240] = silk(91, n, int(rnd.integers(0, 99)), 2, 20, channels, 240)
        return p, np.full(n, 240, np.uint32)

    def traffic(seed, **kw):
        p, l = _traffic(n, 1, channels, 1, seed=seed, **kw)
        return np.pad(p[0], ((0, 0), (0, 240 - p.shape[2]))), l[0]

    for k in range(3):
        device_step(*traffic(100 + k), MODES)
    host_step(*traffic(110, loss=0.0, first_loss=0.0))                                   # switches on the host path
    device_step(*traffic(111), MODES)                                    # sees them
    device_step(*uniform("silk"), MODES)                                 # every stream SILK 20 ms
    device_step(*uniform("silk"), RESIDENT | opn.FLAG_SILK_FRAMES)
    p, l = traffic(112, silk_share=1.0, switch=0.0)
    l[::7] = 0
    device_step(p, l, MODES)                                             # SILK losses after a SILK-frames step
    device_step(*uniform("celt"), MODES)                                 # every stream CELT 20 ms
    device_step(*uniform("celt"), RESIDENT)
    p, l = traffic(113, silk_share=0.0, switch=0.0)
    device_step(p, l, RESIDENT | opn.FLAG_MIXED_FRAMES)
    device_step(*traffic(114), MODES)
    p, l = traffic(115, loss=0.0)
    device_step(p, l, MODES)
    # a host-buffer loss after mixed-mode steps conceals with the stream's codec: streams whose last frame was 20 ms lose theirs
    p, l = traffic(116, loss=0.0, first_loss=0.0)
    lost = (oracle.lm == 3) & (oracle.mode != 0) & (rnd.random(n) < 0.3)
    l[lost] = 0
    assert (lost & (oracle.mode == M.SILK)).any() and (lost & (oracle.mode == M.CELT)).any()
    host_step(p, l)
    device_step(*traffic(117), MODES)


# ------------------------------------------------------------------ F. timing, launches, history
@pytest.mark.parametrize("n", [300, 2050])
def test_timed_pass_equals_untimed_and_counts_launches(n):
    channels, nsteps = 2, 6
    packets, lens = _traffic(n, nsteps, channels, 1, seed=50 + n)
    a, b = Device(packets, lens, channels), Device(packets, lens, channels)
    plain, timed = _decoder(n, channels), _decoder(n, channels)
    timed.enable_timing(True)
    timed.stats(reset=True)
    timed.history_samples(reset=True)
    for f in range(nsteps):
        a.run(plain, f)
        b.run(timed, f)
    plain.synchronize()
    timed.synchronize()
    launches = timed.stats(reset=True)["launches"]
    G = 3 if n >= 2048 else 1
    assert list(launches) == [2 * nsteps, 2 * G * nsteps, (2 + 2 * G) * nsteps], launches
    oracle = M.MixedModeBatch(n, channels, 1)
    hist = 0
    for f in range(nsteps):
        _, _, _, _, h = oracle.step(packets[f], lens[f])
        hist += int(h.sum())
        assert np.array_equal(a.result(f), b.result(f))
        _same(a.pcm(f), b.pcm(f), f"step {f}")
    assert np.array_equal(plain.final_ranges(), timed.final_ranges())
    assert timed.history_samples() == hist


# ------------------------------------------------------------------ G. the workload's per-GPU size
def test_per_gpu_size_of_the_mixed_mode_workload():
    n, channels, nsteps = 32768, 2, 8
    packets, lens = _traffic(n, nsteps, channels, 1, seed=8, switch=0.02, loss=0.02, plc=0.01)
    d = Device(packets, lens, channels)
    dec = _decoder(n, channels)
    for f in range(nsteps):
        d.run(dec, f)
    dec.synchronize()
    oracle = M.MixedModeBatch(n, channels, 1)
    for f in range(nsteps):
        pcm, _, res, rng, _ = oracle.step(packets[f], lens[f])
        assert np.array_equal(d.result(f), res), f
        _same(d.pcm(f), pcm, f"step {f}")
    assert np.array_equal(dec.final_ranges(), rng)
