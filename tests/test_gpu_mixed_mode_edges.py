"""Mixed-mode device-resident steps (OPN_FLAG_MIXED_MODES) at the edges random traffic does not reach, against the CPU oracle
(mixed_modes_oracle.MixedModeBatch).  Dense rows, result_per_stream and final_ranges() are compared bit for bit for every
stream of every step; test_gpu_mixed_modes.py covers random traffic at full rows.

1. Batch sizes at the cut into frame groups (1 to 2049 streams), 12 steps in flight, so the 8 buffer sets are reused; the
   launches per step.
2. Constructed bucket counts: per group, SILK buckets of 0-33 items around the SILK frame CTA (16 stereo / 32 mono items) and
   SILK_PAD, CELT buckets of 0-33 items around FRAME_WARPS and MIX_PAD; CELT bucket (g, 1) holding 5 ms packets and CELT->SILK
   concealment items whose sum straddles 32; groups without CELT or without SILK items; a group in which every stream
   switches next to one in which none does; a step in which every packet is rejected.
3. Rows of 480, 240 and 120 samples, and a capacity that changes every step: frames and concealments that do not fit.
4. opn_batch_reset with mixed-mode steps in flight, then a loss-only step and every step kind a SILK batch takes.
5. Inputs ordered by the caller (no FLAG_INPUTS_READY): one arena and one lens buffer, rewritten on opn_batch_cuda_stream
   after every call, without a host wait.
6. The decoder gain on random traffic: dense rows are the oracle's (faded) PCM times the gain, the ring the PCM before both.
7. A batch without the post-filter.
8. Silence frames in mixed-mode traffic (also right after a SILK -> CELT switch); a timed pass without dense rows."""
import numpy as np
import pytest

import opus_native_b200 as opn
import mixed_modes_oracle as M
from test_gpu_mixed_modes import CAP, MODES, Device, _decoder, _fills, _same, _torch, _traffic
from test_gpu_stream_state import _gain, silence_payload
from test_gpu_workloads import RESIDENT, _ring_frames

pytestmark = pytest.mark.gpu
CELT_BYTES = {0: 64, 1: 80, 2: 110, 3: 160}
STRIDE = 240


def _groups(n):
    return 3 if n >= 2048 else 1


def _enqueue_and_compare(d, dec, oracle, packets, lens, what, caps=None, flags=MODES):
    """every step enqueued without a host wait, then each against the oracle -> the oracle's outputs per step"""
    nsteps, n = lens.shape
    caps = caps if caps is not None else [CAP] * nsteps
    for f in range(nsteps):
        d.run(dec, f, flags, frame_size=caps[f])
    dec.synchronize()
    out = []
    for f in range(nsteps):
        pcm, pre, res, rng, hist = oracle.step(packets[f], lens[f], cap=caps[f])
        assert np.array_equal(d.result(f), res), (what, f)
        _same(d.pcm(f)[:, :caps[f] * oracle.channels], pcm, f"{what} step {f}")
        out.append((pcm, pre, res, rng, hist))
    assert np.array_equal(dec.final_ranges(), out[-1][3]), what
    return out


# ------------------------------------------------------------------ 1. batch sizes at the group cut
SIZES = [(1, 2, 1), (1, 1, 2), (2, 2, 1), (2, 1, 2), (31, 2, 1), (31, 1, 2), (32, 2, 1), (32, 1, 2), (33, 2, 1), (33, 1, 2),
         (2047, 2, 1), (2048, 1, 2), (2049, 2, 1)]


@pytest.mark.parametrize("n,channels,bitstream", SIZES)
def test_batch_sizes_at_the_group_cut(n, channels, bitstream):
    nsteps = 12
    packets, lens = _traffic(n, nsteps, channels, bitstream, seed=7 * n + channels, switch=0.3)
    d = Device(packets, lens, channels)
    dec = _decoder(n, channels, bitstream)
    dec.stats(reset=True)
    _enqueue_and_compare(d, dec, M.MixedModeBatch(n, channels, bitstream), packets, lens, f"n={n}")
    G = _groups(n)
    assert list(dec.stats()["launches"]) == [2 * nsteps, 2 * G * nsteps, (2 + 2 * G) * nsteps]


# ------------------------------------------------------------------ 2. constructed bucket counts
SILK_COUNTS = [0, 1, 15, 16, 17, 31, 32, 33]
CELT_COUNTS = [0, 1, 4, 5, 6, 31, 32, 33]
# (5 ms packets, CELT -> SILK switches) in CELT bucket (g, 1)
STRADDLE = [(20, 11), (20, 12), (20, 13), (31, 1), (1, 31), (0, 33), (16, 16), (17, 16)]
ALL = -1


class Built:
    """Packets built step by step against the oracle, so that every group of every step gets exact item counts.  A step
    is a dict per group {(kind, size): count}: kind "celt" (a CELT stream keeps CELT, size = LM), "silk" (a SILK stream
    keeps SILK, size = ms), "to_silk" (CELT -> SILK, size = ms), "to_celt" (SILK -> CELT, size = LM); count ALL = every
    stream of the pool left.  Every other stream of the group sends a hybrid packet, a per-stream error that makes no item."""

    def __init__(self, n, channels, bitstream, seed):
        self.n, self.channels, self.G = n, channels, _groups(n)
        self.bounds = [n * g // self.G for g in range(self.G + 1)]
        self.celt, self.silk = _fills(bitstream)
        self.oracle = M.MixedModeBatch(n, channels, bitstream)
        self.rnd = np.random.default_rng(seed)
        self.packets, self.lens = [], []

    def step(self, groups):
        n, ch, f, rnd = self.n, self.channels, len(self.packets), self.rnd
        p = np.zeros((n, STRIDE), np.uint8)
        p[:, 0] = ((12 + rnd.integers(0, 4, n)) << 3) | (4 if ch == 2 else 0)
        l = np.full(n, 40, np.uint32)
        mode = self.oracle.mode
        fills = {}

        def fill(kind, size, bw=0):  # one fill of every stream per kind of packet and step
            if (kind, size, bw) not in fills:
                if kind == "celt":
                    fills[kind, size, bw] = self.celt(300 + 11 * size, n, f, size, ch, CELT_BYTES[size], 100)
                else:
                    fills[kind, size, bw] = self.silk(400 + 7 * bw + size, n, f, bw, size, ch, 120 * ch)
            return fills[kind, size, bw]
        want_celt = np.zeros((self.G, 4), np.int64)  # CELT items per (group, LM), the switches' concealments included
        want_silk = np.zeros((self.G, 2), np.int64)
        want_sw = np.zeros((self.G, 2), np.int64)
        for g, counts in enumerate(groups):
            ids = np.arange(self.bounds[g], self.bounds[g + 1])
            if not mode[ids].any():  # every stream's first packet
                shared = list(rnd.permutation(ids))
                pools = {M.CELT: shared, M.SILK: shared}
            else:
                pools = {m: list(rnd.permutation(ids[mode[ids] == m])) for m in (M.CELT, M.SILK)}
            for (kind, size), k in counts.items():
                pool = pools[M.SILK if kind in ("silk", "to_celt") else M.CELT]
                k = len(pool) if k == ALL else k
                assert len(pool) >= k, (kind, size, k, len(pool))
                take = np.array(pool[:k], np.int64)
                del pool[:k]
                if kind in ("celt", "to_celt"):
                    nb = CELT_BYTES[size]
                    p[take, :nb] = fill("celt", size)[take]
                    want_celt[g, size] += k
                else:
                    nb = 120 * ch
                    bw = rnd.integers(0, 3, k)
                    for b in range(3):
                        sel = take[bw == b]
                        if len(sel):
                            p[sel, :nb] = fill("silk", size, b)[sel]
                    want_silk[g, size // 20] += k
                    if kind == "to_silk":
                        want_celt[g, 1] += k
                l[take] = nb
                if kind.startswith("to_"):
                    want_sw[g, int(kind == "to_celt")] += k
        # the counts the step is meant to have, from the oracle's view of its packets
        codec, lm, err = self.oracle.classify(p, l)
        group = np.searchsorted(self.bounds, np.arange(n), side="right") - 1
        for g in range(self.G):
            in_g = (group == g) & (err == 0)
            switch = in_g & (mode != 0) & (codec != mode)
            to_silk = switch & (codec == M.SILK)
            for lmv in range(4):
                assert ((in_g & (codec == M.CELT) & (lm == lmv)).sum() + (to_silk.sum() if lmv == 1 else 0)) == want_celt[g, lmv]
            for k, lmv in enumerate((2, 3)):
                assert (in_g & (codec == M.SILK) & (lm == lmv)).sum() == want_silk[g, k]
            assert to_silk.sum() == want_sw[g, 0] and (switch & (codec == M.CELT)).sum() == want_sw[g, 1]
        self.oracle.step(p, l)
        self.packets.append(p)
        self.lens.append(l)

    def arrays(self):
        return np.stack(self.packets), np.stack(self.lens)


def _count_plan(b):
    G = b.G
    # step 0: every stream's first packet, CELT 20 ms or SILK 20 ms
    b.step([{("celt", 3): (b.bounds[g + 1] - b.bounds[g]) // 2, ("silk", 20): ALL} for g in range(G)])
    # every bucket count, a different one per group and bucket
    for f in range(8):
        b.step([{**{("celt", lm): CELT_COUNTS[(f + 3 * g + 2 * lm) % 8] for lm in range(4)},
                 **{("silk", ms): SILK_COUNTS[(f + 3 * g + 5 * k) % 8] for k, ms in enumerate((10, 20))}} for g in range(G)])
    # 5 ms packets and CELT -> SILK concealments in bucket (g, 1); as many SILK -> CELT switches keep the pools' sizes
    for f in range(8):
        steps = []
        for g in range(G):
            a, s = STRADDLE[(f + 3 * g) % 8]
            steps.append({("celt", 1): a, ("to_silk", 10): s // 2, ("to_silk", 20): s - s // 2, ("to_celt", (0, 2, 3)[f % 3]): s,
                          ("celt", 3): 5, ("silk", 20): 16})
        b.step(steps)
    # a group in which every stream switches, one with SILK items only, one with CELT items only (in turn, on one group)
    roles = [{("to_silk", 20): ALL, ("to_celt", 2): ALL}, {("silk", 10): ALL}, {("celt", 0): 7, ("celt", 3): ALL}]
    for r in range(3):
        b.step([roles[(g + r) % 3] for g in range(G)])
    b.step([{} for _ in range(G)])  # every packet rejected: no item at all
    b.step([{("celt", 2): 33, ("celt", 1): 32, ("silk", 20): 17, ("silk", 10): 16} for _ in range(G)])


@pytest.mark.parametrize("n,channels,bitstream", [(300, 2, 1), (300, 1, 2), (2050, 2, 2), (2050, 1, 1)])
def test_constructed_bucket_counts(n, channels, bitstream):
    b = Built(n, channels, bitstream, seed=n + channels)
    _count_plan(b)
    packets, lens = b.arrays()
    d = Device(packets, lens, channels)
    dec = _decoder(n, channels, bitstream)
    out = _enqueue_and_compare(d, dec, M.MixedModeBatch(n, channels, bitstream), packets, lens, f"n={n} C={channels}")
    rejected = out[-2][2]
    assert np.all(rejected == -6)


# ------------------------------------------------------------------ 3. row capacity
@pytest.mark.parametrize("cap", [480, 240, 120, "changing"])
@pytest.mark.parametrize("n,channels,bitstream", [(300, 2, 1), (2050, 1, 2)])
def test_row_capacity(n, channels, bitstream, cap):
    nsteps = 14
    rnd = np.random.default_rng([n, channels, 0 if cap == "changing" else cap])
    packets, lens = _traffic(n, nsteps, channels, bitstream, seed=n + channels + 3, switch=0.2, loss=0.08)
    if cap == "changing":
        caps = [int(c) for c in rnd.choice([960, 480, 240, 120], nsteps)]
        caps[:3] = [960, 960, 480]  # frames of 20 ms, then a row they do not fit
        oracle = M.MixedModeBatch(n, channels, bitstream)
    else:
        caps = [cap] * nsteps
        oracle = M.MixedModeBatch(n, channels, bitstream, cap=cap)
    d = Device(packets, lens, channels, cap=max(caps))
    dec = _decoder(n, channels, bitstream)
    for f in range(nsteps):
        d.run(dec, f, frame_size=caps[f])
    dec.synchronize()
    seen = dict(silk_too_big=0, switch_too_big=0, loss_too_big=0, switch_10ms_in_480=0)
    for f in range(nsteps):
        mode = oracle.mode.copy()
        pcm, _, res, rng, _ = oracle.step(packets[f], lens[f], cap=caps[f])
        assert np.array_equal(d.result(f), res), (cap, f)
        _same(d.pcm(f)[:, :caps[f] * channels], pcm, f"cap {cap} step {f}")
        toc = packets[f, :, 0]
        silk = (lens[f] > 0) & ((toc & 0x80) == 0)
        seen["silk_too_big"] += int((silk & (res == -5)).sum())
        seen["switch_too_big"] += int((silk & (mode == M.CELT) & (res == -5)).sum())
        seen["loss_too_big"] += int(((lens[f] == 0) & (res == -5)).sum())
        if caps[f] == 480:
            seen["switch_10ms_in_480"] += int((silk & (mode == M.CELT) & (res == 480)).sum())
    assert np.array_equal(dec.final_ranges(), rng)
    assert seen["silk_too_big"] > 0 and seen["switch_too_big"] > 0, seen
    if cap == 480:
        assert seen["switch_10ms_in_480"] > 0, seen
    if cap == "changing":
        assert seen["loss_too_big"] > 0, seen


# ------------------------------------------------------------------ 4. reset with mixed-mode steps in flight
@pytest.mark.parametrize("n,channels,bitstream", [(300, 2, 1), (2050, 1, 2)])
def test_reset_with_mixed_mode_steps_in_flight(n, channels, bitstream):
    _, silk = _fills(bitstream)
    before, blens = _traffic(n, 5, channels, bitstream, seed=40 + n)
    pre = Device(before, blens, channels)
    dec = _decoder(n, channels, bitstream)
    for f in range(5):
        pre.run(dec, f)
    dec.reset()  # no synchronize: the steps above are still in flight
    old = M.MixedModeBatch(n, channels, bitstream)
    for f in range(5):
        pcm, _, res, _, _ = old.step(before[f], blens[f])
        assert np.array_equal(pre.result(f), res), f
        _same(pre.pcm(f), pcm, f"before the reset, step {f}")

    steps = []  # (packets [n, STRIDE], lens [n], flags, frame_size)

    def traffic(seed, **kw):
        p, l = _traffic(n, 1, channels, bitstream, seed=seed, **kw)
        return np.pad(p[0], ((0, 0), (0, STRIDE - p.shape[2]))), l[0]

    def all_silk(f):
        p = np.zeros((n, STRIDE), np.uint8)
        p[:, :120 * channels] = silk(60, n, f, 2, 20, channels, 120 * channels)
        return p, np.full(n, 120 * channels, np.uint32)

    steps.append((np.zeros((n, STRIDE), np.uint8), np.zeros(n, np.uint32), MODES, 480))  # conceals 10 ms of CELT (zeros)
    p, l = traffic(41, silk_share=0.0, switch=0.0)
    steps.append((p, l, RESIDENT | opn.FLAG_MIXED_FRAMES, CAP))                           # CELT packets only
    for k in range(3):
        steps.append((*traffic(42 + k, switch=0.3), MODES, CAP))
    steps.append((*all_silk(5), MODES, CAP))                                              # every stream SILK 20 ms
    steps.append((*all_silk(6), RESIDENT | opn.FLAG_SILK_FRAMES, CAP))
    p, l = traffic(46)
    l[::5] = 0
    steps.append((p, l, MODES, CAP))
    packets = np.stack([s[0] for s in steps])
    lens = np.stack([s[1] for s in steps])
    d = Device(packets, lens, channels)
    for f, (_, _, flags, fs) in enumerate(steps):
        d.run(dec, f, flags, frame_size=fs)
    dec.synchronize()
    oracle = M.MixedModeBatch(n, channels, bitstream)  # a fresh decoder per stream
    for f, (_, _, flags, fs) in enumerate(steps):
        pcm, _, res, rng, _ = oracle.step(packets[f], lens[f], cap=fs)
        assert np.array_equal(d.result(f), res), f
        _same(d.pcm(f)[:, :fs * channels], pcm, f"after the reset, step {f}")
        if f == 0:
            assert np.all(res == 480) and not pcm.any()
    assert np.array_equal(dec.final_ranges(), rng)


# ------------------------------------------------------------------ 5. inputs ordered by the caller
@pytest.mark.parametrize("n,channels,bitstream", [(300, 2, 1), (2050, 1, 2)])
def test_inputs_ordered_by_the_caller(n, channels, bitstream):
    """FLAG_DEVICE_PTRS without FLAG_INPUTS_READY: the step is ordered after what opn_batch_cuda_stream holds, and the
    caller may rewrite the packets on that stream right after the call"""
    torch = _torch()
    dev = torch.device("cuda:0")
    nsteps = 12
    packets, lens = _traffic(n, nsteps, channels, bitstream, seed=60 + n, switch=0.2)
    stride = packets.shape[2]
    src_packets = torch.from_numpy(packets.reshape(nsteps, -1).copy()).to(dev)
    src_lens = torch.from_numpy(lens.astype(np.int32)).to(dev)
    arena = torch.zeros(n * stride, dtype=torch.uint8, device=dev)
    d_lens = torch.zeros(n, dtype=torch.int32, device=dev)
    off = (torch.arange(n, dtype=torch.int64, device=dev) * stride).to(torch.int32)
    rows = torch.zeros((nsteps, n, CAP * channels), dtype=torch.float32, device=dev)
    res = torch.zeros((nsteps, n), dtype=torch.int32, device=dev)
    dec = _decoder(n, channels, bitstream)
    ext = torch.cuda.ExternalStream(dec.cuda_stream, device=dev)
    arena.copy_(src_packets[0])
    d_lens.copy_(src_lens[0])
    torch.cuda.synchronize()
    for f in range(nsteps):
        dec.decode_float_ptrs(arena.data_ptr(), off.data_ptr(), d_lens.data_ptr(), rows[f].data_ptr(), rows.stride(1), CAP,
                              res[f].data_ptr(), opn.FLAG_DEVICE_PTRS | opn.FLAG_MIXED_MODES)
        if f + 1 < nsteps:
            with torch.cuda.stream(ext):
                arena.copy_(src_packets[f + 1])
                d_lens.copy_(src_lens[f + 1])
    dec.synchronize()
    torch.cuda.synchronize()
    got, got_res = rows.cpu().numpy(), res.cpu().numpy()
    oracle = M.MixedModeBatch(n, channels, bitstream)
    for f in range(nsteps):
        pcm, _, want_res, rng, _ = oracle.step(packets[f], lens[f])
        assert np.array_equal(got_res[f], want_res), f
        _same(got[f], pcm, f"step {f}")
    assert np.array_equal(dec.final_ranges(), rng)


# ------------------------------------------------------------------ 6. decoder gain on random traffic
@pytest.mark.parametrize("gain_q8", [1, 1536, -1536])
@pytest.mark.parametrize("channels,bitstream", [(2, 1), (1, 2)])
def test_decoder_gain_on_random_traffic(channels, bitstream, gain_q8):
    n, nsteps = 2050, 8
    packets, lens = _traffic(n, nsteps, channels, bitstream, seed=80 + channels + (gain_q8 & 0xFFFF), switch=0.2)
    g = _gain(gain_q8)
    assert g != np.float32(1.0)
    d = Device(packets, lens, channels)
    dec = _decoder(n, channels, bitstream, gain_q8)
    for f in range(nsteps):
        d.run(dec, f)
    dec.synchronize()
    oracle = M.MixedModeBatch(n, channels, bitstream)
    switched = 0
    for f in range(nsteps):
        mode = oracle.mode.copy()
        pcm, pre, res, rng, _ = oracle.step(packets[f], lens[f])
        switched += int(((mode == M.CELT) & (oracle.mode == M.SILK) & (res > 0)).sum())
        assert np.array_equal(d.result(f), res), f
        _same(d.pcm(f), pcm * g, f"gain_q8={gain_q8} step {f}")
    assert np.array_equal(dec.final_ranges(), rng)
    assert switched > 0
    # without dense rows the ring holds the last frame before the fade and before the gain
    nr = Device(packets, lens, channels, rows=False)
    dec2 = _decoder(n, channels, bitstream, gain_q8)
    for f in range(nsteps):
        nr.run(dec2, f, dense=False)
    dec2.synchronize()
    assert np.array_equal(nr.result(nsteps - 1), res)
    ok = (lens[-1] > 2) & (res > 0)
    ring = _ring_frames(dec2, n, np.where(ok, res, 0), channels, CAP, nr.dev)
    _same(ring[ok], pre[ok], "ring")


# ------------------------------------------------------------------ 7. post-filter off
@pytest.mark.parametrize("n,channels,bitstream", [(300, 2, 1), (2050, 1, 2), (2050, 2, 1)])
def test_without_the_post_filter(n, channels, bitstream):
    """mixed-frame steps on CELT streams, mixed-mode steps with switches, a mixed-mode step that brings every stream back to
    CELT, and mixed-frame steps again, on a batch created with postfilter = false"""
    plan = [("mf", dict(silk_share=0.0, switch=0.0))] * 2 + [("mm", dict(switch=0.2))] * 6 + \
           [("mm", dict(silk_share=0.0, switch=0.0, loss=0.0, first_loss=0.0)), ("mf", dict(silk_share=0.0, switch=0.0))]
    steps = [_traffic(n, 1, channels, bitstream, seed=90 + f, **kw) for f, (_, kw) in enumerate(plan)]
    packets = np.stack([np.pad(p[0], ((0, 0), (0, STRIDE - p.shape[2]))) for p, _ in steps])
    lens = np.stack([l[0] for _, l in steps])
    d = Device(packets, lens, channels)
    dec = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, channels, 0), postfilter=False,
                           bitstream=bitstream | opn.BITSTREAM_SYNTH_SILK_1)
    for f, (kind, _) in enumerate(plan):
        d.run(dec, f, MODES if kind == "mm" else RESIDENT | opn.FLAG_MIXED_FRAMES)
    dec.synchronize()
    oracle = M.MixedModeBatch(n, channels, bitstream, apply_comb=False)
    with_comb = M.MixedModeBatch(n, channels, bitstream)
    differ = False
    for f in range(len(plan)):
        pcm, _, res, rng, _ = oracle.step(packets[f], lens[f])
        differ |= not np.array_equal(with_comb.step(packets[f], lens[f])[0], pcm)
        assert np.array_equal(d.result(f), res), f
        _same(d.pcm(f), pcm, f"step {f} ({plan[f][0]})")
        if f == len(plan) - 2:
            assert np.all(oracle.mode == M.CELT)
    assert np.array_equal(dec.final_ranges(), rng)
    assert differ


# ------------------------------------------------------------------ 8. silence frames; timing without dense rows
@pytest.mark.parametrize("n,channels,bitstream", [(300, 2, 1), (2050, 1, 2)])
def test_silence_frames_and_timing_without_dense_rows(n, channels, bitstream):
    nsteps = 10
    rnd = np.random.default_rng([n, channels, 8])
    packets, lens = _traffic(n, nsteps, channels, bitstream, seed=110 + n, switch=0.25)
    last = np.zeros(n, np.uint8)  # codec of each stream's last packet
    silence = {nb: silence_payload(nb - 1) for nb in CELT_BYTES.values()}
    after_switch = 0
    for f in range(nsteps):
        got = lens[f] > 0
        celt = got & ((packets[f, :, 0] & 0x80) != 0)
        full = celt & (lens[f] > 2)
        sw = full & (last == M.SILK)
        silent = full & ((rnd.random(n) < 0.15) | (sw & (rnd.random(n) < 0.6)))
        after_switch += int((silent & sw).sum())
        for s in np.nonzero(silent)[0]:
            nb = int(lens[f, s])
            packets[f, s, 1:nb] = silence[nb]
        last = np.where(got, np.where(celt, M.CELT, M.SILK), last).astype(np.uint8)
    assert after_switch > 0
    d = Device(packets, lens, channels)
    dec = _decoder(n, channels, bitstream)
    out = _enqueue_and_compare(d, dec, M.MixedModeBatch(n, channels, bitstream), packets, lens, "silence")
    hist = sum(int(h.sum(dtype=np.uint64)) for *_, h in out)
    # a timed pass without dense rows: no fade is launched; the comb history count and the ring as the oracle's
    nr = Device(packets, lens, channels, rows=False)
    timed = _decoder(n, channels, bitstream)
    timed.enable_timing(True)
    timed.stats(reset=True)
    timed.history_samples(reset=True)
    for f in range(nsteps):
        nr.run(timed, f, dense=False)
    timed.synchronize()
    G = _groups(n)
    assert list(timed.stats(reset=True)["launches"]) == [2 * nsteps, 2 * G * nsteps, (2 + G) * nsteps]
    for f in range(nsteps):
        assert np.array_equal(nr.result(f), out[f][2]), f
    assert hist > 0 and timed.history_samples() == hist
    assert np.array_equal(timed.final_ranges(), out[-1][3])
    _, pre, res = out[-1][:3]
    ok = (lens[-1] > 2) & (res > 0)
    ring = _ring_frames(timed, n, np.where(ok, res, 0), channels, CAP, nr.dev)
    _same(ring[ok], pre[ok], "ring")
