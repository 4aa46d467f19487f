"""ctypes binding of the CPU oracle (oracle/liboracle.so).  Test infrastructure only."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SO = os.path.join(ROOT, "oracle", "liboracle.so")


def build():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])


class Dec(C.Structure):
    _fields_ = [("buffer", C.c_void_p)] + [(n, C.c_uint32) for n in
                ("storage", "end_offs", "end_window", "end_bits", "bits_total", "offs", "rng", "val", "ext")] + [("rem", C.c_uint8)]


class Enc(C.Structure):
    _fields_ = [("buffer", C.c_void_p), ("buffer_len", C.c_uint32)] + [(n, C.c_uint32) for n in
                ("storage", "end_offs", "end_window", "end_bits", "bits_total", "offs", "rng", "val", "ext")] + [("rem", C.c_int32), ("error", C.c_int)]


class Op(C.Structure):
    _fields_ = [("op", C.c_uint32), ("a", C.c_uint32), ("b", C.c_uint32)]


class OpOut(C.Structure):
    _fields_ = [("value", C.c_uint32), ("tell_frac", C.c_uint32), ("rng", C.c_uint32)]


class SynthSide(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("silence", "postfilter", "octave", "period", "gain_idx", "tapset", "transient", "intra")] + [
        ("coarse", (C.c_int32 * 21) * 2), ("fine", (C.c_int32 * 21) * 2),
        ("final_rng", C.c_uint32), ("tell_frac", C.c_uint32), ("n_pulses", C.c_uint32)]


class Celt2Side(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("silence", "postfilter", "octave", "period", "gain_idx", "tapset", "transient", "intra",
                                          "spread", "alloc_trim", "coded_bands", "intensity", "dual_stereo", "anti_collapse", "balance")] + [
        (n, C.c_int32 * 21) for n in ("offsets", "pulses", "ebits", "fine_priority")] + [
        (n, (C.c_int32 * 21) * 2) for n in ("coarse", "fine", "fine_final", "energy_q9")] + [
        (n, C.c_uint32) for n in ("n_parts", "n_pulses", "n_splits", "theta_sum", "final_rng", "tell_frac")]


class Celt2Part(C.Structure):
    _fields_ = [("base", C.c_uint16), ("n", C.c_uint8), ("k", C.c_uint8), ("index", C.c_uint32), ("gain", C.c_float)]


CELT2_MAX_PARTS = 192


class SynthState(C.Structure):
    _fields_ = [("buf", (C.c_float * (1024 + 8 * 960 + 60)) * 2), ("pos", C.c_uint32),
                ("pf_period", C.c_int32), ("pf_tapset", C.c_int32), ("pf_gain", C.c_float)]


class SilkChanSide(C.Structure):
    _fields_ = [("type", C.c_int32), ("gidx", C.c_int32 * 4), ("rc_idx", C.c_int32 * 16), ("lag", C.c_int32 * 4), ("ltp_idx", C.c_int32 * 4),
                ("seed", C.c_int32), ("pulses", C.c_int32 * 20), ("index", C.c_uint32 * 20)]


class SilkSide(C.Structure):
    _fields_ = [("ch", SilkChanSide * 2), ("final_rng", C.c_uint32), ("tell_frac", C.c_uint32), ("lbrr", C.c_int32)]


SILK_MAX_FRAME = 320


class SilkChan(C.Structure):
    _fields_ = [("slpc", C.c_int32 * 16), ("hist", C.c_int32 * 320), ("a_q12", C.c_int16 * 16), ("gain_q10", C.c_int32)]


class SilkState(C.Structure):
    _fields_ = [("ch", SilkChan * 2), ("rs", (C.c_float * 8) * 2), ("fs_khz", C.c_int32), ("stream_channels", C.c_int32)]


OP_UINT, OP_BITS, OP_BIT_LOGP, OP_ICDF, OP_LAPLACE, OP_BIT_VIA_DECODE, OP_BIT_VIA_DECODE_BIN, OP_PULSES, OP_SHRINK, OP_TELL = range(10)
OP_DTYPE = np.dtype([("op", "<u4"), ("a", "<u4"), ("b", "<u4")])
OUT_DTYPE = np.dtype([("value", "<u4"), ("tell_frac", "<u4"), ("rng", "<u4")])

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        build()
    L = C.CDLL(_SO)
    u32, i32, vp, f32, sz = C.c_uint32, C.c_int32, C.c_void_p, C.c_float, C.c_size_t

    def sig(name, res, *args):
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = list(args)

    sig("orc_ilog", u32, u32)
    sig("orc_tell", u32, u32, u32)
    sig("orc_tell_frac", u32, u32, u32)
    sig("orc_laplace_start_freq", u32, u32)
    sig("orc_dec_init", None, C.POINTER(Dec), vp, u32)
    sig("orc_dec_shrink_storage", None, C.POINTER(Dec), u32)
    sig("orc_dec_decode", u32, C.POINTER(Dec), u32)
    sig("orc_dec_decode_bin", u32, C.POINTER(Dec), u32)
    sig("orc_dec_update", None, C.POINTER(Dec), u32, u32, u32)
    sig("orc_dec_bit_logp", C.c_int, C.POINTER(Dec), u32)
    sig("orc_dec_icdf", u32, C.POINTER(Dec), vp, u32)
    sig("orc_dec_uint", u32, C.POINTER(Dec), u32)
    sig("orc_dec_bits", u32, C.POINTER(Dec), u32)
    sig("orc_dec_laplace", i32, C.POINTER(Dec), u32, u32)
    sig("orc_dec_tell", u32, C.POINTER(Dec))
    sig("orc_dec_tell_frac", u32, C.POINTER(Dec))
    sig("orc_enc_init", None, C.POINTER(Enc), vp, u32)
    sig("orc_enc_encode", C.c_int, C.POINTER(Enc), u32, u32, u32)
    sig("orc_enc_encode_bin", C.c_int, C.POINTER(Enc), u32, u32, u32)
    sig("orc_enc_bit_logp", C.c_int, C.POINTER(Enc), u32, u32)
    sig("orc_enc_icdf", C.c_int, C.POINTER(Enc), u32, vp, u32)
    sig("orc_enc_uint", C.c_int, C.POINTER(Enc), u32, u32)
    sig("orc_enc_bits", C.c_int, C.POINTER(Enc), u32, u32)
    sig("orc_enc_patch_initial_bits", C.c_int, C.POINTER(Enc), u32, u32)
    sig("orc_enc_shrink", None, C.POINTER(Enc), u32)
    sig("orc_enc_done", C.c_int, C.POINTER(Enc))
    sig("orc_enc_laplace", C.c_int, C.POINTER(Enc), C.POINTER(i32), u32, u32)
    sig("orc_enc_range_bytes", u32, C.POINTER(Enc))
    sig("orc_enc_tell", u32, C.POINTER(Enc))
    sig("orc_enc_tell_frac", u32, C.POINTER(Enc))
    sig("orc_dec_run_script", u32, vp, u32, vp, u32, vp, vp, vp)
    sig("orc_enc_run_script", C.c_int, vp, u32, vp, vp, u32, vp, vp, vp, C.POINTER(u32), C.POINTER(u32))
    sig("orc_pvq_u", u32, u32, u32)
    sig("orc_pvq_v", u32, u32, u32)
    sig("orc_icwrs", u32, vp, u32)
    sig("orc_cwrsi", f32, vp, u32, u32, u32)
    sig("orc_fft_process", None, C.c_int, vp)
    sig("orc_fft_bitrev", C.POINTER(C.c_uint16), C.c_int)
    sig("orc_fft_scale", f32, C.c_int)
    sig("orc_mdct_backward", None, vp, vp, vp, C.c_int, C.c_int, C.c_int)
    sig("orc_mdct_forward", None, vp, vp, vp, C.c_int, C.c_int, C.c_int)
    sig("orc_window", C.POINTER(f32))
    sig("orc_trig", C.POINTER(f32))
    sig("orc_comb_filter", None, vp, sz, vp, sz, sz, sz, sz, f32, f32, sz, sz, sz)
    sig("orc_comb_filter_inplace", None, vp, sz, sz, sz, sz, f32, f32, sz, sz, sz)
    sig("orc_bitexact_cos", C.c_int16, C.c_int16)
    sig("orc_bitexact_log2tan", i32, i32, i32)
    sig("orc_packet_bandwidth", C.c_int, vp)
    sig("orc_packet_channels", C.c_int, vp)
    sig("orc_packet_frame_count", C.c_int, vp, sz)
    sig("orc_packet_samples_per_frame", C.c_int, vp, C.c_int)
    sig("orc_packet_sample_count", C.c_int, vp, sz, C.c_int)
    sig("orc_packet_mode", C.c_int, vp)
    sig("orc_parse_packet", C.c_int, vp, sz, C.c_int, vp, vp, C.POINTER(u32), C.POINTER(u32))
    sig("orc_pcm_soft_clip", None, vp, sz, sz, vp, sz)
    sig("orc_smooth_fade", None, vp, vp, vp, C.c_int, C.c_int, C.c_int)
    sig("orc_sample_from_f32", C.c_int, C.c_int, vp, vp, sz)
    sig("orc_synth_state_init", None, C.POINTER(SynthState))
    sig("orc_synth_decode_frame", C.c_int, C.POINTER(SynthState), vp, u32, C.c_int, C.c_int, C.c_int,
        C.POINTER(SynthSide), vp, vp, vp)
    sig("orc_celt2_decode_symbols", C.c_int, vp, u32, C.c_int, C.c_int, C.POINTER(Celt2Side), vp, vp, vp)
    sig("orc_celt2_decode_frame", C.c_int, C.POINTER(SynthState), vp, u32, C.c_int, C.c_int, C.c_int, C.POINTER(Celt2Side), vp)
    sig("orc_celt2_decode_frame_mapped", C.c_int, C.POINTER(SynthState), vp, u32, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(Celt2Side), vp)
    sig("orc_synth_decode_frame_mapped", C.c_int, C.POINTER(SynthState), vp, u32, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(SynthSide), vp)
    sig("orc_celt2_packet", C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, u32, u32, vp, C.POINTER(Celt2Side))
    sig("orc_synth_packet", C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, u32, u32, vp)
    sig("orc_synth_fill", C.c_int, C.c_uint64, u32, C.c_uint64, u32, C.c_int, C.c_int, u32, u32, C.c_int, vp)
    sig("orc_synth_bench", C.c_double, vp, u32, u32, u32, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.POINTER(u32))
    sig("orc_silk_state_init", None, C.POINTER(SilkState))
    sig("orc_silk_decode_frame", C.c_int, C.POINTER(SilkState), vp, u32, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(SilkSide),
        vp, vp, vp)
    sig("orc_silk_packet", C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int, u32, u32, vp)
    sig("orc_silk_fill", C.c_int, C.c_uint64, u32, C.c_uint64, u32, C.c_int, C.c_int, C.c_int, u32, u32, C.c_int, vp)
    sig("orc_silk_bench", C.c_double, vp, u32, u32, u32, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.POINTER(u32))
    for name in ("orc_synth_step", "orc_celt2_step"):
        sig(name, C.c_int, vp, u32, vp, sz, vp, vp, C.c_int, C.c_int, C.c_int, vp, sz, vp, vp)
    sig("orc_silk_step", C.c_int, vp, u32, vp, sz, vp, C.c_int, C.c_int, C.c_int, vp, sz, vp)
    _lib = L
    return L


def ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def window():
    return np.ctypeslib.as_array(lib().orc_window(), shape=(120,)).copy()


def dec_run_script(buf, ops, icdf_pool=None, y_cap=0):
    """buf: bytes/uint8 array; ops: structured array OP_DTYPE -> (out OUT_DTYPE array, y int32 array)"""
    b = np.frombuffer(bytes(buf), dtype=np.uint8).copy() if not isinstance(buf, np.ndarray) else np.ascontiguousarray(buf)
    ops = np.ascontiguousarray(ops, dtype=OP_DTYPE)
    out = np.zeros(len(ops), dtype=OUT_DTYPE)
    y = np.zeros(max(y_cap, 1), dtype=np.int32)
    pool = np.ascontiguousarray(icdf_pool, dtype=np.uint8) if icdf_pool is not None else np.zeros(1, np.uint8)
    ny = lib().orc_dec_run_script(ptr(b), len(b), ptr(ops), len(ops), ptr(pool), ptr(out), ptr(y))
    return out, y[:ny]


def enc_run_script(nbytes, ops, values, icdf_pool=None, y_in=None):
    """-> (buffer uint8[nbytes], per-op tell_frac, range_bytes, final_tell_frac, err)"""
    ops = np.ascontiguousarray(ops, dtype=OP_DTYPE)
    values = np.ascontiguousarray(values, dtype=np.uint32)
    buf = np.zeros(nbytes, dtype=np.uint8)
    tf = np.zeros(len(ops), dtype=np.uint32)
    pool = np.ascontiguousarray(icdf_pool, dtype=np.uint8) if icdf_pool is not None else np.zeros(1, np.uint8)
    yin = np.ascontiguousarray(y_in, dtype=np.int32) if y_in is not None else np.zeros(1, np.int32)
    rb, ftf = C.c_uint32(0), C.c_uint32(0)
    err = lib().orc_enc_run_script(ptr(buf), nbytes, ptr(ops), ptr(values), len(ops), ptr(pool), ptr(yin), ptr(tf), C.byref(rb), C.byref(ftf))
    return buf, tf, rb.value, ftf.value, err


def mdct_backward(coefs, out, shift, stride=1, overlap=120, window_arr=None):
    w = window() if window_arr is None else np.ascontiguousarray(window_arr, dtype=np.float32)
    coefs = np.ascontiguousarray(coefs, dtype=np.float32)
    assert out.dtype == np.float32 and out.flags.c_contiguous
    lib().orc_mdct_backward(ptr(coefs), ptr(out), ptr(w), overlap, shift, stride)
    return out


def comb_filter_inplace(y, y_offset, t0, t1, n, g0, g1, tap0, tap1, overlap):
    assert y.dtype == np.float32 and y.flags.c_contiguous
    lib().orc_comb_filter_inplace(ptr(y), y_offset, t0, t1, n, g0, g1, tap0, tap1, overlap)
    return y


def comb_filter(y, y_offset, x, x_offset, t0, t1, n, g0, g1, tap0, tap1, overlap):
    x = np.ascontiguousarray(x, dtype=np.float32)
    lib().orc_comb_filter(ptr(y), y_offset, ptr(x), x_offset, t0, t1, n, g0, g1, tap0, tap1, overlap)
    return y


def synth_fill(first_stream, n_streams, first_frame, n_frames, lm, channels, pkt_bytes, transient_permille=0, n_threads=1):
    """-> uint8 [n_frames, n_streams, pkt_bytes], generated with the oracle's range encoder"""
    out = np.zeros((n_frames, n_streams, pkt_bytes), np.uint8)
    rc = lib().orc_synth_fill(first_stream, n_streams, first_frame, n_frames, lm, channels, pkt_bytes, transient_permille, n_threads, ptr(out))
    assert rc == 0, rc
    return out


def celt2_packet(stream_id, frame_idx, lm, channels, pkt_bytes, transient_permille=0):
    """-> (packet uint8[pkt_bytes] incl. TOC, Celt2Side truth) from the oracle's SYNTH-CELT/2 generator"""
    out = np.zeros(pkt_bytes, np.uint8)
    truth = Celt2Side()
    rc = lib().orc_celt2_packet(stream_id, frame_idx, lm, channels, pkt_bytes, transient_permille, ptr(out), C.byref(truth))
    assert rc == pkt_bytes, rc
    return out, truth


def celt2_decode_symbols(payload, lm, channels):
    """-> (Celt2Side, parts array, y int32 [C*nf], coef float32 [C*nf])"""
    payload = np.ascontiguousarray(payload, np.uint8)
    nf = 120 << lm
    side = Celt2Side()
    parts = (Celt2Part * CELT2_MAX_PARTS)()
    y = np.zeros(channels * nf, np.int32)
    coef = np.zeros(channels * nf, np.float32)
    rc = lib().orc_celt2_decode_symbols(ptr(payload), len(payload), lm, channels, C.byref(side), parts, ptr(y), ptr(coef))
    assert rc == 0, rc
    return side, parts, y, coef


class Celt2Stream:
    """One stream's oracle-side SYNTH-CELT/2 decoder state."""

    def __init__(self, lm, channels, apply_comb=True):
        self.lm, self.channels, self.apply_comb = lm, channels, apply_comb
        self.state = SynthState()
        lib().orc_synth_state_init(C.byref(self.state))

    def decode(self, payload):
        """-> (Celt2Side, pcm) or (error code, None) for a rejected frame"""
        nf = 120 << self.lm
        payload = np.frombuffer(bytes(payload), dtype=np.uint8).copy()
        side = Celt2Side()
        pcm = np.zeros(self.channels * nf, np.float32)
        r = lib().orc_celt2_decode_frame(C.byref(self.state), ptr(payload) if len(payload) else None, len(payload), self.lm, self.channels,
                                        int(self.apply_comb), C.byref(side), ptr(pcm))
        return (side, pcm) if r == nf else (r, None)


class MappedStream:
    """One decoder of `channels` channels fed packets of either channel count (stream_channels, decoder.rs:332): oracle side,
    SYNTH-CELT/1 (bitstream 1) or /2."""

    def __init__(self, channels, bitstream=1, apply_comb=True):
        self.channels, self.bitstream, self.apply_comb = channels, bitstream, apply_comb
        self.state = SynthState()
        lib().orc_synth_state_init(C.byref(self.state))

    def decode(self, payload, lm, stream_channels):
        """-> (final_rng, pcm [nf*channels])"""
        nf = 120 << lm
        payload = np.frombuffer(bytes(payload), dtype=np.uint8).copy()
        pcm = np.zeros(self.channels * nf, np.float32)
        side = SynthSide() if self.bitstream == 1 else Celt2Side()
        fn = lib().orc_synth_decode_frame_mapped if self.bitstream == 1 else lib().orc_celt2_decode_frame_mapped
        r = fn(C.byref(self.state), ptr(payload) if len(payload) else None, len(payload), lm, stream_channels, self.channels,
               int(self.apply_comb), C.byref(side), ptr(pcm))
        assert r == nf, r
        return side.final_rng, pcm


class SynthStream:
    """One stream's oracle-side SYNTH-CELT/1 decoder state."""

    def __init__(self, lm, channels, apply_comb=True):
        self.lm, self.channels, self.apply_comb = lm, channels, apply_comb
        self.state = SynthState()
        lib().orc_synth_state_init(C.byref(self.state))

    def decode(self, payload):
        nf = 120 << self.lm
        payload = np.frombuffer(bytes(payload), dtype=np.uint8).copy()
        side = SynthSide()
        y = np.zeros(self.channels * nf, np.int32)
        coef = np.zeros(self.channels * nf, np.float32)
        pcm = np.zeros(self.channels * nf, np.float32)
        r = lib().orc_synth_decode_frame(C.byref(self.state), ptr(payload) if len(payload) else None, len(payload), self.lm,
                                        self.channels, int(self.apply_comb), C.byref(side), ptr(y), ptr(coef), ptr(pcm))
        assert r == nf
        return side, y, coef, pcm

    def conceal(self, lm):
        """One lost frame of 120 << lm samples (decode_frame(None)): -> pcm [nf * channels]"""
        nf = 120 << lm
        side = SynthSide()
        pcm = np.zeros(self.channels * nf, np.float32)
        r = lib().orc_synth_decode_frame(C.byref(self.state), None, 0, lm, self.channels, int(self.apply_comb), C.byref(side), None, None, ptr(pcm))
        assert r == nf
        return pcm


STEP_SKIP = 0xFFFFFFFF  # ORC_STEP_SKIP


def _with_skip(lens, skip):
    lens = np.array(lens, np.uint32)
    if skip is not None:
        lens[np.asarray(skip, bool)] = STEP_SKIP
    return lens


def _threads():
    return min(len(os.sched_getaffinity(0)), 64)


class CeltBatch:
    """Oracle side of a batch of SYNTH-CELT/1 (bitstream 1) or /2 decoders, every stream advanced by one packet per step
    (orc_synth_step / orc_celt2_step, multithreaded).  Stream s decodes exactly as a SynthStream / Celt2Stream would."""

    def __init__(self, n_streams, channels, bitstream=1, apply_comb=True, n_threads=None):
        self.n, self.channels, self.apply_comb = n_streams, channels, apply_comb
        self.n_threads = n_threads or _threads()
        self.fn = lib().orc_synth_step if bitstream == 1 else lib().orc_celt2_step
        self.states = (SynthState * n_streams)()
        for s in range(n_streams):
            lib().orc_synth_state_init(C.byref(self.states[s]))

    def step(self, packets, lens, lm, cap=None, skip=None):
        """packets uint8 [n, stride] (TOC first); lens [n] (0 = lost); lm: int or [n]; skip: bool [n] or None, streams left out
        of the step (state untouched, row, final_rng and hist zero) -> (pcm float32 [n, cap * C] (cap: samples per channel,
        default 120 << max lm), the frame at the start of each row, zeros after it; final_rng uint32 [n], 0 for a lost frame;
        hist uint32 [n], the comb history samples the frame kernel counts for each frame)"""
        packets = np.ascontiguousarray(packets, np.uint8)
        lens = _with_skip(lens, skip)
        lm = np.ascontiguousarray(np.broadcast_to(lm, (self.n,)), np.uint8)
        assert packets.shape[0] == self.n and lens.shape == (self.n,)
        pcm = np.zeros((self.n, (cap or 120 << int(lm.max())) * self.channels), np.float32)
        rng = np.zeros(self.n, np.uint32)
        hist = np.zeros(self.n, np.uint32)
        rc = self.fn(self.states, self.n, ptr(packets), packets.shape[1], ptr(lens), ptr(lm), self.channels, int(self.apply_comb),
                     self.n_threads, ptr(pcm), pcm.shape[1], ptr(rng), ptr(hist))
        assert rc == 0, rc
        return pcm, rng, hist


class SilkBatch:
    """Oracle side of a batch of SYNTH-SILK/1 decoders of `channels` channels, every stream advanced by one packet per step
    (orc_silk_step, multithreaded; bandwidth and coded channel count from each packet's TOC)."""

    def __init__(self, n_streams, channels, n_threads=None):
        self.n, self.channels = n_streams, channels
        self.n_threads = n_threads or _threads()
        self.states = (SilkState * n_streams)()
        for s in range(n_streams):
            lib().orc_silk_state_init(C.byref(self.states[s]))

    def step(self, packets, lens, frame_ms, skip=None):
        """skip as for CeltBatch.step -> (pcm float32 [n, frame_ms * 48 * C], final_rng uint32 [n], 0 for a lost frame)"""
        packets = np.ascontiguousarray(packets, np.uint8)
        lens = _with_skip(lens, skip)
        assert packets.shape[0] == self.n and lens.shape == (self.n,)
        pcm = np.zeros((self.n, frame_ms * 48 * self.channels), np.float32)
        rng = np.zeros(self.n, np.uint32)
        rc = lib().orc_silk_step(self.states, self.n, ptr(packets), packets.shape[1], ptr(lens), frame_ms, self.channels, self.n_threads,
                                 ptr(pcm), pcm.shape[1], ptr(rng))
        assert rc == 0, rc
        return pcm, rng


def silk_fill(first_stream, n_streams, first_frame, n_frames, bandwidth, frame_ms, channels, pkt_bytes, n_threads=1, lbrr_permille=0):
    """-> uint8 [n_frames, n_streams, pkt_bytes]: SYNTH-SILK/1 packets (TOC included) from the oracle's generator"""
    out = np.zeros((n_frames, n_streams, pkt_bytes), np.uint8)
    rc = lib().orc_silk_fill(first_stream, n_streams, first_frame, n_frames, bandwidth, frame_ms, channels, pkt_bytes, lbrr_permille, n_threads, ptr(out))
    assert rc == 0, rc
    return out


class SilkStream:
    """One decoder's oracle-side SYNTH-SILK/1 state (decoder of `channels` output channels)."""

    def __init__(self, channels):
        self.channels = channels
        self.state = SilkState()
        lib().orc_silk_state_init(C.byref(self.state))

    def decode(self, payload, bandwidth, frame_ms, stream_channels, lost=False, fec=False):
        """-> (SilkSide, exc int32 [2, 320], out16 int16 [2, 320], pcm float32 [frame_ms*48*channels]); fec: the packet's redundant
        copy of the previous frame (LostFlag::DecodeFec)"""
        payload = np.frombuffer(bytes(payload), dtype=np.uint8).copy()
        side = SilkSide()
        exc = np.zeros((2, SILK_MAX_FRAME), np.int32)
        out16 = np.zeros((2, SILK_MAX_FRAME), np.int16)
        pcm = np.zeros(frame_ms * 48 * self.channels, np.float32)
        r = lib().orc_silk_decode_frame(C.byref(self.state), ptr(payload) if len(payload) else None, len(payload), bandwidth, frame_ms,
                                       stream_channels, self.channels, 2 if fec else int(lost), C.byref(side), ptr(exc), ptr(out16), ptr(pcm))
        assert r == frame_ms * 48, r
        return side, exc, out16, pcm
