"""Per-stream state across packets the generators never write and call orders the other files never make, against the CPU
oracle, bit for bit (PCM, result_per_stream, final_ranges()) for every stream of every step.

A. Short packets and silence frames on every device-resident step kind.  Per stream and step: a full packet, a loss, a
   TOC-only packet (lens 1), a one-byte payload (lens 2) -- both PLC/DTX (decoder.rs:467) -- or a SYNTH-CELT silence frame.
   A short packet still sets the frame size the stream conceals its next loss with (libopus takes st->frame_size from the
   TOC before it decodes the frames): in mixed-frame steps its TOC size differs from the stream's previous size and a loss
   follows it.  Then a timed pass (comb history count) and a host-buffer call over the same kinds of packets.
B. Host-buffer calls between device-resident steps, with losses, short packets and a frame_size larger than the stream's
   last frame: the host call conceals from the state the device steps left (several frames of the last size), and a
   device step after it conceals with the size the host call left.
C. The decoder gain on device-resident steps: dense rows carry one f32 multiply by the gain, the PCM ring holds the PCM
   before it (it is the post-filter's history).
D. Silence frames through the range-decode kernels at operator level: the whole side record.

Device-resident steps do not switch a stream between CELT and SILK, so every test keeps each stream in one mode."""
import ctypes
import ctypes.util

import numpy as np
import pytest

import opus_native_b200 as opn
import oracle_lib as O
from test_gpu_workloads import MIX_BYTES, RESIDENT, SILK, Steps, _ring_frames, _same

pytestmark = pytest.mark.gpu
NSTEPS = 12
FULL, LOSS, TOC_ONLY, ONE_BYTE, SILENCE = range(5)
EVENT_P = [0.55, 0.1, 0.1, 0.1, 0.15]
KINDS = ["celt1-stereo", "celt1-mono", "celt2-stereo", "mixed-stereo", "silk-mono-wb", "silk-stereo-mixed-bw"]


def _torch():
    return pytest.importorskip("torch")


def _gain(gain_q8):
    """the decoder's linear gain: exp(6.48814081e-4 * gain_q8 * ln 2) in f32 (decoder.rs:790-791, math.rs:17-19), with the C
    library's expf as f32::exp uses it.  numpy's float32 exp is one ulp off it for some gains (-1536 among them)."""
    libm = ctypes.CDLL(ctypes.util.find_library("m"))
    libm.expf.restype, libm.expf.argtypes = ctypes.c_float, [ctypes.c_float]
    x = np.float32(np.float32(6.48814081e-4) * np.float32(gain_q8)) * np.float32(0.6931471805599453)
    return np.float32(libm.expf(float(x)))


def silence_payload(nbytes):
    """a SYNTH-CELT/1 or /2 frame whose first symbol, the silence flag (bit_logp 15), is 1; nbytes of range-coder output"""
    ops = np.zeros(1, O.OP_DTYPE)
    ops[0] = (O.OP_BIT_LOGP, 15, 0)
    buf, _, _, _, err = O.enc_run_script(nbytes, ops, [1])
    assert err == 0
    return buf


def plc_frames(frame_size, last_nf):
    """decode_native(None, frame_size) conceals in frames of the stream's last size (decoder.rs:427-441)"""
    out, done = [], 0
    while done < frame_size:
        a = min(frame_size - done, last_nf)
        if a > 960:
            a = 960
        elif a < 960:
            if a > 480:
                a = 480
            elif 240 < a < 480:
                a = 240
        out.append(a)
        done += a
    return out


class Sizes:
    """The frame size each stream conceals a loss with: a packet of lens >= 1 (a short one too) sets it from its TOC, a loss
    keeps it; before any packet, one frame of the row's capacity.  seen: the stream has had a packet, so a host-buffer call
    conceals a loss from its state instead of writing zeros (decoder.rs:478-487)."""

    def __init__(self, n, cap_lm=3):
        self.last = np.full(n, cap_lm, np.uint8)
        self.seen = np.zeros(n, bool)

    def step(self, lens, lm_toc):
        """-> the LM every stream decodes or conceals in a mixed-frame step"""
        got = lens > 0
        out = np.where(got, lm_toc, self.last).astype(np.uint8)
        self.last = out
        self.seen |= got
        return out

    def uniform(self, lens, lm):
        """a uniform step of LM lm: a loss conceals lm, the stream's size does not change"""
        self.step(lens, np.full(len(lens), lm, np.uint8))
        return np.full(len(lens), lm, np.uint8)


# ------------------------------------------------------------------ packets
def _events(rnd, shape, silence=True):
    p = np.array(EVENT_P)
    if not silence:
        p[FULL] += p[SILENCE]
        p[SILENCE] = 0
    return rnd.choice(5, size=shape, p=p)


def _apply(ev, packets, lens, nb):
    """one step: events [n] onto full packets [n, stride] of nb bytes (nb per stream) -> lens"""
    nb = np.broadcast_to(nb, ev.shape)
    lens[:] = nb
    lens[ev == LOSS] = 0
    lens[ev == TOC_ONLY] = 1
    lens[ev == ONE_BYTE] = 2
    for s in np.nonzero(ev == SILENCE)[0]:
        packets[s, 1:nb[s]] = silence_payload(int(nb[s]) - 1)


def _uniform_celt(kind, n, nsteps, rnd, lm=3, first=0, seed=0):
    """SYNTH-CELT/1 or /2 packets of LM lm for every stream -> packets [nsteps, n, 160], lens"""
    channels = 1 if kind == "celt1-mono" else 2
    nb = MIX_BYTES[lm] if lm < 3 or channels == 2 else 100
    fill = opn.celt2_fill if kind == "celt2-stereo" else opn.synth_fill
    packets = np.zeros((nsteps, n, 160), np.uint8)
    packets[:, :, :nb] = fill(seed + 700 + n, n, first, nsteps, lm, channels, nb, 150)
    lens = np.zeros((nsteps, n), np.uint32)
    ev = _events(rnd, (nsteps, n))
    for f in range(nsteps):
        _apply(ev[f], packets[f], lens[f], nb)
    return packets, lens, np.full((nsteps, n), lm, np.uint8)


def _mixed_celt(n, nsteps, rnd, sizes_last, channels=2, first=0, max_lm=3, seed=0):
    """SYNTH-CELT/1 packets of a frame size drawn per stream and step.  A short packet's TOC size differs from the stream's
    previous size (sizes_last, updated), and a loss follows it in the next step."""
    packets = np.zeros((nsteps, n, 160), np.uint8)
    lens = np.zeros((nsteps, n), np.uint32)
    lm = np.zeros((nsteps, n), np.uint8)
    w = np.array([0.10, 0.10, 0.30, 0.50])[:max_lm + 1]
    last = sizes_last.copy()
    force_loss = np.zeros(n, bool)
    for f in range(nsteps):
        ev = _events(rnd, n)
        ev[force_loss] = LOSS
        lm[f] = rnd.choice(max_lm + 1, size=n, p=w / w.sum())
        short = (ev == TOC_ONLY) | (ev == ONE_BYTE)
        for s in np.nonzero(short & (lm[f] == last))[0]:
            lm[f, s] = (int(last[s]) + 1 + rnd.integers(0, max_lm)) % (max_lm + 1)
        assert not (short & (lm[f] == last)).any()
        for l in range(max_lm + 1):
            ids = np.nonzero(lm[f] == l)[0]
            if len(ids):
                packets[f, ids, :MIX_BYTES[l]] = opn.synth_fill(seed + 4100 + 10 * l + n, n, first + f, 1, l, channels, MIX_BYTES[l], 100)[0][ids]
        _apply(ev, packets[f], lens[f], np.array([MIX_BYTES[int(l)] for l in lm[f]]))
        last = np.where(lens[f] > 0, lm[f], last)
        force_loss = short
    sizes_last[:] = last
    return packets, lens, lm


def _silk(kind, n, nsteps, rnd, first=0, bws=None):
    """SYNTH-SILK/1 20 ms packets; a short packet carries a TOC of another bandwidth than the stream's packets"""
    channels = 1 if kind == "silk-mono-wb" else 2
    nb = 96 * channels
    if bws is None:
        bws = np.full(n, 2) if channels == 1 else rnd.integers(0, 3, n)
    packets = np.zeros((nsteps, n, nb), np.uint8)
    for bw in range(3):
        ids = np.nonzero(bws == bw)[0]
        if len(ids):
            packets[:, ids] = opn.silk_fill(1000 * bw + n, len(ids), first, nsteps, bw, 20, channels, nb)
    lens = np.zeros((nsteps, n), np.uint32)
    ev = _events(rnd, (nsteps, n), silence=False)
    for f in range(nsteps):
        _apply(ev[f], packets[f], lens[f], nb)
        short = np.nonzero((ev[f] == TOC_ONLY) | (ev[f] == ONE_BYTE))[0]
        other = (bws[short] + 1 + rnd.integers(0, 2, len(short))) % 3
        toc = packets[f, short, 0]
        packets[f, short, 0] = (toc & 0x07) | (((4 * other) + ((toc >> 3) & 3)) << 3)
    return packets, lens, bws


def _kind(kind):
    """-> channels, bitstream, device-step flags"""
    channels = 1 if kind in ("celt1-mono", "silk-mono-wb") else 2
    if kind.startswith("silk"):
        return channels, SILK, RESIDENT | opn.FLAG_SILK_FRAMES
    if kind == "mixed-stereo":
        return channels, 1, RESIDENT | opn.FLAG_MIXED_FRAMES
    return channels, 2 if kind == "celt2-stereo" else 1, RESIDENT


# ------------------------------------------------------------------ the oracle of a host-buffer call
def _host_oracle(ora, sizes, packets, lens, lm_toc, frame_size, channels):
    """A host-buffer call of frame_size samples per row on CELT streams: a packet decodes its frame at the start of the row,
    a loss of a stream that has had a packet conceals frame_size samples in frames of its last size, a loss of a stream that
    has not writes zeros and leaves the state alone -> (pcm [n, frame_size * C], final_rng, result_per_stream)"""
    n = len(lens)
    got = lens > 0
    pcm = np.zeros((n, frame_size * channels), np.float32)
    rng = np.zeros(n, np.uint32)
    res = np.where(got, 120 << lm_toc.astype(np.int32), frame_size).astype(np.int32)
    w, r, _ = ora.step(packets, lens, np.where(got, lm_toc, 0), cap=frame_size, skip=~got)
    pcm[got], rng[got] = w[got], r[got]
    conceal = ~got & sizes.seen
    chunks = {s: plc_frames(frame_size, 120 << int(sizes.last[s])) for s in np.nonzero(conceal)[0]}
    at = np.zeros(n, np.int64)
    zero = np.zeros(n, np.uint32)
    for k in range(max((len(c) for c in chunks.values()), default=0)):
        active = np.zeros(n, bool)
        lm_k = np.zeros(n, np.uint8)
        for s, c in chunks.items():
            if k < len(c):
                active[s], lm_k[s] = True, c[k].bit_length() - 7  # 120 << lm
        w, _, _ = ora.step(packets, zero, lm_k, cap=960, skip=~active)
        for s in np.nonzero(active)[0]:
            nf = 120 << int(lm_k[s])
            pcm[s, at[s] * channels:(at[s] + nf) * channels] = w[s, :nf * channels]
            at[s] += nf
    sizes.step(lens, lm_toc)
    return pcm, rng, res


def _host_call(dec, packets, lens, frame_size, channels):
    n, stride = packets.shape
    pcm = np.full((n, frame_size * channels), 7.0, np.float32)
    res = dec.decode_float(np.ascontiguousarray(packets).reshape(-1), (np.arange(n) * stride).astype(np.uint32), lens.astype(np.uint32), pcm,
                           frame_size)
    return pcm, res


# ------------------------------------------------------------------ A. short packets and silence on every step kind
@pytest.mark.parametrize("n", [300, 2050])
@pytest.mark.parametrize("kind", KINDS)
def test_short_packets_and_silence(kind, n):
    torch = _torch()
    dev = torch.device("cuda:0")
    rnd = np.random.default_rng([KINDS.index(kind), n, 1])
    channels, bitstream, flags = _kind(kind)
    silk, mixed = kind.startswith("silk"), kind == "mixed-stereo"
    frame = 960
    sizes = Sizes(n)
    if silk:
        packets, lens, bws = _silk(kind, n, NSTEPS + 1, rnd)
        lm = None
    elif mixed:
        last = np.full(n, 3, np.uint8)
        packets, lens, lm = _mixed_celt(n, NSTEPS + 1, rnd, last, channels)
    else:
        packets, lens, lm = _uniform_celt(kind, n, NSTEPS + 1, rnd)
    steps = Steps(packets[:NSTEPS], lens[:NSTEPS], dev)
    assert (lens == 1).any() and (lens == 2).any() and (lens == 0).any()

    def device_pass(timing):
        dec = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, channels, 0), bitstream=bitstream)
        dec.enable_timing(timing)
        pcm = torch.zeros((NSTEPS, n, frame * channels), dtype=torch.float32, device=dev)
        res = torch.full((NSTEPS, n), -99, dtype=torch.int32, device=dev)
        for f in range(NSTEPS):
            steps.run(dec, f, flags, frame, pcm[f], res[f])
        dec.join()
        dec.synchronize()
        return dec, pcm.cpu().numpy(), res.cpu().numpy()

    dec, got, got_res = device_pass(False)
    passes = [("pipelined", got, got_res)]
    if not silk:
        dec_t, got_t, res_t = device_pass(True)
        passes.append(("timed", got_t, res_t))
    ora = O.SilkBatch(n, channels) if silk else O.CeltBatch(n, channels, bitstream)
    hist_sum = 0
    for f in range(NSTEPS):
        if silk:
            want, rng = ora.step(packets[f], lens[f], 20)
            want_res = np.full(n, 960)
        else:
            lm_f = sizes.step(lens[f], lm[f]) if mixed else sizes.uniform(lens[f], 3)
            want, rng, hist = ora.step(packets[f], lens[f], lm_f, cap=frame)
            hist_sum += int(hist.sum(dtype=np.uint64))
            want_res = 120 << lm_f.astype(np.int32)
        for what, g, r in passes:
            assert np.array_equal(r[f], want_res), (what, f)
            _same(g[f], want, f"{kind} n={n} {what} step {f}")
    assert np.abs(want).max() > 0.01
    assert np.array_equal(dec.final_ranges(), rng)
    if not silk:
        assert np.array_equal(dec_t.final_ranges(), rng)
        assert hist_sum > 0 and dec_t.history_samples() == hist_sum

    # a host-buffer call over the same kinds of packets, after the device-resident steps
    f = NSTEPS
    host_pcm, host_res = _host_call(dec, packets[f], lens[f], frame, channels)
    if silk:
        want, rng = ora.step(packets[f], lens[f], 20)
        want_res = np.full(n, 960)
    else:
        want, rng, want_res = _host_oracle(ora, sizes, packets[f], lens[f], lm[f], frame, channels)
    assert np.array_equal(host_res, want_res)
    _same(host_pcm, want, f"{kind} n={n} host-buffer call after device steps")
    assert np.array_equal(dec.final_ranges(), rng)


# ------------------------------------------------------------------ B. host-buffer calls between device-resident steps
CELT_PLANS = {
    "device-host-device": ["u3", "mix", "host960", "mix", "u1", "host480", "u3"],
    "host-first": ["host960", "u3", "mix", "u2", "mix"],
}


@pytest.mark.parametrize("n", [300, 2050])
@pytest.mark.parametrize("plan", list(CELT_PLANS))
def test_host_calls_between_device_steps(plan, n):
    """SYNTH-CELT/1 stereo: uniform (u<LM>) and mixed-frame device-resident steps with host-buffer calls (host<frame_size>)
    between them; every kind of step gets losses and short packets.  A host call conceals frame_size samples in frames of
    the stream's last size, whatever kind of step decoded it; the mixed-frame step after it conceals with the size the
    host call left (its packets' TOC sizes, short packets included)."""
    torch = _torch()
    dev = torch.device("cuda:0")
    rnd = np.random.default_rng([list(CELT_PLANS).index(plan), n, 2])
    channels, cap = 2, 960
    kinds = CELT_PLANS[plan]
    last = np.full(n, 3, np.uint8)
    dec = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, channels, 0), bitstream=1)
    ora = O.CeltBatch(n, channels, 1)
    sizes = Sizes(n)
    n_multi = 0
    for f, kind in enumerate(kinds):
        what = f"{plan} n={n} step {f} ({kind})"
        if kind.startswith("u"):
            l = int(kind[1])
            packets, lens, lm = _uniform_celt("celt1-stereo", n, 1, rnd, lm=l, first=f, seed=f)
            last = np.where(lens[0] > 0, l, last).astype(np.uint8)
        else:
            fs = int(kind[4:]) if kind.startswith("host") else cap
            packets, lens, lm = _mixed_celt(n, 1, rnd, last, channels, first=f, max_lm=fs.bit_length() - 7, seed=f)
        packets, lens, lm = packets[0], lens[0], lm[0]
        if kind.startswith("host"):
            fs = int(kind[4:])
            chunks = [len(plc_frames(fs, 120 << int(sizes.last[s]))) for s in np.nonzero((lens == 0) & sizes.seen)[0]]
            n_multi += sum(c > 1 for c in chunks)
            want, rng, want_res = _host_oracle(ora, sizes, packets, lens, lm, fs, channels)
            got, got_res = _host_call(dec, packets, lens, fs, channels)
            assert np.array_equal(got_res, want_res), what
            _same(got, want, what)
            continue
        steps = Steps(packets[None], lens[None], dev)
        res = torch.full((n,), -99, dtype=torch.int32, device=dev)
        if kind == "mix":
            lm_f = sizes.step(lens, lm)
            pcm = torch.zeros((n, cap * channels), dtype=torch.float32, device=dev)
            steps.run(dec, 0, RESIDENT | opn.FLAG_MIXED_FRAMES, cap, pcm, res)
        else:
            lm_f = sizes.uniform(lens, int(kind[1]))
            nf = 120 << int(kind[1])
            pcm = torch.zeros((n, nf * channels), dtype=torch.float32, device=dev)
            steps.run(dec, 0, RESIDENT, nf, pcm, res)
        want, rng, _ = ora.step(packets, lens, lm_f, cap=cap)
        dec.join()
        dec.synchronize()
        got = pcm.cpu().numpy()
        assert np.array_equal(res.cpu().numpy(), 120 << lm_f.astype(np.int32)), what
        _same(got, want[:, :got.shape[1]], what)
    assert np.array_equal(dec.final_ranges(), rng)
    if plan == "device-host-device":
        assert n_multi > 0  # a host call concealed several frames for some stream


def test_silk_host_call_between_device_steps():
    """SILK mono wideband, 300 streams: 20 ms device-resident steps, a lossy host-buffer call, another device step.  The
    host call conceals from the SILK state the device steps left."""
    torch = _torch()
    dev = torch.device("cuda:0")
    n, channels, kind = 300, 1, "silk-mono-wb"
    rnd = np.random.default_rng(3)
    packets, lens, _ = _silk(kind, n, 4, rnd)
    lens[2, rnd.random(n) < 0.2] = 0  # the host call: more losses
    dec = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, channels, 0), bitstream=SILK)
    steps = Steps(packets, lens, dev)
    ora = O.SilkBatch(n, channels)
    for f, kind_f in enumerate(["device", "device", "host", "device"]):
        want, rng = ora.step(packets[f], lens[f], 20)
        if kind_f == "host":
            got, got_res = _host_call(dec, packets[f], lens[f], 960, channels)
        else:
            pcm = torch.zeros((n, 960 * channels), dtype=torch.float32, device=dev)
            res = torch.full((n,), -99, dtype=torch.int32, device=dev)
            steps.run(dec, f, RESIDENT | opn.FLAG_SILK_FRAMES, 960, pcm, res)
            dec.join()
            dec.synchronize()
            got, got_res = pcm.cpu().numpy(), res.cpu().numpy()
        assert np.all(got_res == 960), f
        _same(got, want, f"SILK step {f} ({kind_f})")
    assert np.array_equal(dec.final_ranges(), rng)


# ------------------------------------------------------------------ C. decoder gain on device-resident steps
@pytest.mark.parametrize("gain_q8", [1536, -1536, 1])
@pytest.mark.parametrize("kind", KINDS)
def test_decoder_gain_on_device_steps(kind, gain_q8):
    """dense rows = np.float32(oracle) * g, the one f32 multiply the kernels do; the ring holds the PCM before the gain"""
    torch = _torch()
    dev = torch.device("cuda:0")
    n = 300
    rnd = np.random.default_rng([KINDS.index(kind), gain_q8 & 0xFFFF])
    channels, bitstream, flags = _kind(kind)
    silk, mixed = kind.startswith("silk"), kind == "mixed-stereo"
    if silk:
        packets, lens, _ = _silk(kind, n, NSTEPS, rnd)
        lm = None
    elif mixed:
        packets, lens, lm = _mixed_celt(n, NSTEPS, rnd, np.full(n, 3, np.uint8), channels)
    else:
        packets, lens, lm = _uniform_celt(kind, n, NSTEPS, rnd)
    g = _gain(gain_q8)
    assert g != np.float32(1.0)
    steps = Steps(packets, lens, dev)
    dec = opn.BatchDecoder(n, opn.DecoderConfiguration(48000, channels, gain_q8), bitstream=bitstream)
    pcm = torch.zeros((NSTEPS, n, 960 * channels), dtype=torch.float32, device=dev)
    res = torch.full((NSTEPS, n), -99, dtype=torch.int32, device=dev)
    for f in range(NSTEPS):
        steps.run(dec, f, flags, 960, pcm[f], res[f])
    dec.join()
    dec.synchronize()
    got, got_res = pcm.cpu().numpy(), res.cpu().numpy()
    ora = O.SilkBatch(n, channels) if silk else O.CeltBatch(n, channels, bitstream)
    sizes = Sizes(n)
    for f in range(NSTEPS):
        if silk:
            want, rng = ora.step(packets[f], lens[f], 20)
            lm_f = np.full(n, 3, np.uint8)
        else:
            lm_f = sizes.step(lens[f], lm[f]) if mixed else sizes.uniform(lens[f], 3)
            want, rng, _ = ora.step(packets[f], lens[f], lm_f, cap=960)
        assert np.array_equal(got_res[f], 120 << lm_f.astype(np.int32)), f
        _same(got[f], want * g, f"{kind} gain_q8={gain_q8} step {f}")
    assert np.abs(want).max() > 0.01
    ring = _ring_frames(dec, n, 120 << lm_f.astype(np.int64), channels, 960, dev)
    _same(ring, want, f"{kind} gain_q8={gain_q8}: last frame in the ring")
    assert np.array_equal(dec.final_ranges(), rng)


# ------------------------------------------------------------------ D. silence at operator level
@pytest.mark.parametrize("bitstream", [1, 2])
@pytest.mark.parametrize("channels", [1, 2])
@pytest.mark.parametrize("lm", [0, 1, 2, 3])
def test_silence_frame_symbols(bitstream, channels, lm):
    """opn_op_synth_symbols / opn_op_celt2_symbols on silence frames of 2..159 bytes: silence = 1, the final range and
    tell_frac of the oracle, every other field of the side record zero, no pulses, no coefficients"""
    lens = np.array([2, 3, 5, 8, 20, 64, 159], np.uint32)
    offsets = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint32)
    arena = np.concatenate([silence_payload(int(l)) for l in lens])
    op = opn.op_synth_symbols if bitstream == 1 else opn.op_celt2_symbols
    side, y, coef = op(arena, offsets, lens, lm, channels)
    assert not y.any() and not coef.any()
    for s, l in enumerate(lens):
        payload = arena[offsets[s]:offsets[s] + l]
        if bitstream == 1:
            w = O.SynthStream(lm, channels).decode(payload)[0]
        else:
            w = O.celt2_decode_symbols(payload, lm, channels)[0]
        assert w.silence == 1
        for f in side.dtype.names:
            v = getattr(w, f)
            v = np.ctypeslib.as_array(v) if hasattr(v, "__len__") else v
            assert np.array_equal(side[s][f], v), (s, f)
            if f not in ("silence", "final_rng", "tell_frac"):
                assert not np.any(side[s][f]), (s, f)
        assert side[s]["final_rng"] != 0 and side[s]["tell_frac"] > 0
