"""ctypes binding of libopusb200.so (include/opusb200.h)."""
import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libopusb200.so")

OP_UINT, OP_BITS, OP_BIT_LOGP, OP_ICDF, OP_LAPLACE, OP_BIT_VIA_DECODE, OP_BIT_VIA_DECODE_BIN, OP_PULSES, OP_SHRINK, OP_TELL, OP_PULSES_EVENTS = range(11)
FLAG_DEVICE_PTRS, FLAG_NO_PCM_COPY, FLAG_INPUTS_READY, FLAG_SUBMIT_ONLY, FLAG_MIXED_FRAMES, FLAG_SILK_FRAMES, FLAG_DECODE_FEC = 1, 2, 4, 8, 16, 32, 64
FLAG_MIXED_MODES = 128
# OPN_BITSTREAM_*: CELT frames are Unimplemented (as in the crate, whose CeltDecoder::decode is todo!()) unless the caller
# opts in to the synthetic SYNTH-CELT/1 frame layout (DESIGN.md section 3; not Opus-interoperable)
BITSTREAM_OPUS, BITSTREAM_SYNTH_CELT_1, BITSTREAM_SYNTH_CELT_2 = 0, 1, 2
# OR-ed onto one of the above: SILK-only frames decode with the synthetic SYNTH-SILK/1 layout (DESIGN.md section 3c) instead of Unimplemented
BITSTREAM_SYNTH_SILK_1 = 0x100
SILK_MAX_FRAME = 320
# OPN_SAMPLE_*: the types the crate implements `Sample` for (lib.rs:63-107)
SAMPLE_F32, SAMPLE_I16, SAMPLE_I32, SAMPLE_U16, SAMPLE_U32, SAMPLE_F64 = 0, 1, 2, 3, 4, 5
SAMPLE_FORMAT_OF = {np.dtype(np.float32): SAMPLE_F32, np.dtype(np.int16): SAMPLE_I16, np.dtype(np.int32): SAMPLE_I32,
                    np.dtype(np.uint16): SAMPLE_U16, np.dtype(np.uint32): SAMPLE_U32, np.dtype(np.float64): SAMPLE_F64}
OP_DTYPE = np.dtype([("op", "<u4"), ("a", "<u4"), ("b", "<u4")])
OUT_DTYPE = np.dtype([("value", "<u4"), ("tell_frac", "<u4"), ("rng", "<u4")])
SIDE_DTYPE = np.dtype([(n, "<i4") for n in ("silence", "postfilter", "octave", "period", "gain_idx", "tapset", "transient", "intra")]
                      + [("coarse", "<i4", (2, 21)), ("fine", "<i4", (2, 21)), ("final_rng", "<u4"), ("tell_frac", "<u4"), ("n_pulses", "<u4")])

CELT2_SIDE_DTYPE = np.dtype([(n, "<i4") for n in ("silence", "postfilter", "octave", "period", "gain_idx", "tapset", "transient", "intra",
                                                  "spread", "alloc_trim", "coded_bands", "intensity", "dual_stereo", "anti_collapse", "balance")]
                            + [(n, "<i4", (21,)) for n in ("offsets", "pulses", "ebits", "fine_priority")]
                            + [(n, "<i4", (2, 21)) for n in ("coarse", "fine", "fine_final", "energy_q9")]
                            + [(n, "<u4") for n in ("n_parts", "n_pulses", "n_splits", "theta_sum", "final_rng", "tell_frac")])

_SILK_CH = [("type", "<i4"), ("gidx", "<i4", (4,)), ("rc_idx", "<i4", (16,)), ("lag", "<i4", (4,)), ("ltp_idx", "<i4", (4,)), ("seed", "<i4"),
            ("pulses", "<i4", (20,)), ("index", "<u4", (20,))]
SILK_SIDE_DTYPE = np.dtype([("ch", np.dtype(_SILK_CH), (2,)), ("final_rng", "<u4"), ("tell_frac", "<u4"), ("lbrr", "<i4")])

_ERR_NAMES = {-1: "BadArguments", -2: "BufferToSmall", -3: "InternalError", -4: "InvalidPacket",
              -5: "FrameSizeTooSmall", -6: "Unimplemented", -7: "Cuda"}


class OpusError(Exception):
    """Mirror of `OpusError` (src/error.rs:5-16); `.code` is the C-ABI error code."""

    def __init__(self, code, detail=""):
        self.code = code
        self.kind = _ERR_NAMES.get(code, "Unknown")
        msg = lib().opn_strerror(code).decode()
        if code == -7:
            detail = detail or lib().opn_last_cuda_error().decode()
        super().__init__(f"{self.kind}: {msg}" + (f" ({detail})" if detail else ""))


def library_path():
    return _SO


def build_library(force=False):
    """Compile libopusb200.so in-tree (nvcc -gencode arch=compute_100a,code=sm_100a)."""
    args = ["make", "-s", "-C", os.path.join(_HERE, "csrc")]
    if force:
        subprocess.check_call(args + ["clean"])
    subprocess.check_call(args)


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise ImportError(f"{_SO} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
    L = C.CDLL(_SO)
    u8p, u32, i32, vp, sz, f32 = C.c_void_p, C.c_uint32, C.c_int32, C.c_void_p, C.c_size_t, C.c_float

    def sig(name, res, *args):
        if not hasattr(L, name) and os.environ.get("OPN_ALLOW_OLD_LIBRARY") == "1":
            return  # A/B runs of an older build (tools/experiments/variants.sh): entry points added since are simply absent
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = list(args)

    sig("opn_strerror", C.c_char_p, C.c_int)
    sig("opn_last_cuda_error", C.c_char_p)
    sig("opn_device_count", C.c_int)
    sig("opn_packet_bandwidth", C.c_int, u8p)
    sig("opn_packet_channels", C.c_int, u8p)
    sig("opn_packet_frame_count", C.c_int, u8p, sz)
    sig("opn_packet_samples_per_frame", C.c_int, u8p, i32)
    sig("opn_packet_sample_count", C.c_int, u8p, sz, i32)
    sig("opn_packet_mode", C.c_int, u8p)
    sig("opn_parse_packet", C.c_int, u8p, sz, C.c_int, vp, vp, C.POINTER(u32), C.POINTER(u32))
    sig("opn_decoder_create", C.c_int, C.c_int, i32, i32, C.c_int16, i32, C.POINTER(vp))
    sig("opn_decoder_destroy", None, vp)
    sig("opn_decoder_reset", C.c_int, vp)
    sig("opn_decode_float", C.c_int, vp, u8p, sz, vp, sz, C.c_int)
    sig("opn_decode_i16", C.c_int, vp, u8p, sz, vp, sz, sz, C.c_int)
    sig("opn_decode_pcm", C.c_int, vp, u8p, sz, vp, sz, C.c_int, sz, C.c_int)
    sig("opn_sample_size", sz, C.c_int)
    for g in ("sampling_rate", "channels", "gain", "bandwidth", "pitch", "last_packet_duration"):
        sig("opn_decoder_" + g, i32, vp)
    sig("opn_decoder_final_range", u32, vp)
    sig("opn_host_alloc", vp, sz)
    sig("opn_host_free", None, vp)
    sig("opn_host_register", C.c_int, vp, sz)
    sig("opn_host_unregister", C.c_int, vp)
    sig("opn_batch_create", C.c_int, C.c_int, u32, vp, C.POINTER(vp))
    sig("opn_batch_destroy", None, vp)
    sig("opn_batch_reset", C.c_int, vp)
    sig("opn_batch_decode_float", C.c_int, vp, vp, vp, vp, vp, sz, sz, vp, u32)
    sig("opn_batch_synchronize", C.c_int, vp)
    sig("opn_batch_final_ranges", C.c_int, vp, vp)
    sig("opn_batch_ring", C.c_int, vp, C.POINTER(vp), C.POINTER(u32), C.POINTER(vp))
    sig("opn_batch_enable_timing", C.c_int, vp, C.c_int)
    sig("opn_batch_stats", C.c_int, vp, vp, vp, C.c_int)
    sig("opn_batch_wait", C.c_int, vp, C.c_int)
    sig("opn_batch_decode_i16", C.c_int, vp, vp, vp, vp, vp, C.c_size_t, C.c_size_t, vp, C.c_uint32)
    sig("opn_batch_decode_pcm", C.c_int, vp, vp, vp, vp, vp, C.c_size_t, C.c_int, C.c_size_t, vp, C.c_uint32)
    sig("opn_batch_join", C.c_int, vp)
    sig("opn_batch_history_samples", C.c_int, vp, C.POINTER(C.c_uint64), C.c_int)
    sig("opn_op_bitexact_trig", C.c_int, C.c_int, vp, vp, C.c_uint32, vp, vp, vp, C.c_uint32)
    sig("opn_batch_cuda_stream", vp, vp)
    sig("opn_op_rangedec_script", C.c_int, C.c_int, vp, vp, vp, u32, vp, u32, vp, u32, vp, vp, u32)
    sig("opn_op_imdct_tdac", C.c_int, C.c_int, vp, sz, vp, sz, u32, C.c_int, C.c_int, C.c_int)
    sig("opn_op_comb_filter_inplace", C.c_int, C.c_int, vp, sz, sz, sz, u32, vp, vp, sz)
    sig("opn_op_comb_filter", C.c_int, C.c_int, vp, vp, sz, sz, sz, u32, vp, vp, sz)
    sig("opn_op_pcm_soft_clip", C.c_int, C.c_int, vp, sz, sz, C.c_int, u32, vp)
    sig("opn_op_smooth_fade", C.c_int, C.c_int, vp, vp, vp, sz, sz, C.c_int, C.c_int32, u32)
    sig("opn_op_synth_symbols", C.c_int, C.c_int, vp, vp, vp, u32, C.c_int, C.c_int, vp, vp, vp)
    sig("opn_op_celt2_symbols", C.c_int, C.c_int, vp, vp, vp, u32, C.c_int, C.c_int, vp, vp, vp)
    sig("opn_celt2_packet", C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, u32, u32, vp, vp)
    sig("opn_celt2_fill", C.c_int, C.c_uint64, u32, C.c_uint64, u32, C.c_int, C.c_int, u32, u32, C.c_int, vp)
    sig("opn_synth_packet", C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, u32, u32, vp, vp)
    sig("opn_synth_fill", C.c_int, C.c_uint64, u32, C.c_uint64, u32, C.c_int, C.c_int, u32, u32, C.c_int, vp)
    sig("opn_op_silk_frames", C.c_int, C.c_int, vp, vp, vp, u32, C.c_int, C.c_int, sz, C.c_int, vp, vp, vp, vp, vp)
    sig("opn_silk_packet", C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int, u32, u32, vp)
    sig("opn_silk_fill", C.c_int, C.c_uint64, u32, C.c_uint64, u32, C.c_int, C.c_int, C.c_int, u32, u32, C.c_int, vp)
    sig("opn_enc_run_script", C.c_int, vp, u32, vp, vp, u32, vp, vp, vp, C.POINTER(u32), C.POINTER(u32))
    _lib = L
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _chk(rc):
    if rc < 0:
        raise OpusError(rc)
    return rc


def _bytes(packet):
    a = np.frombuffer(bytes(packet), dtype=np.uint8) if not isinstance(packet, np.ndarray) else packet
    return np.ascontiguousarray(a, dtype=np.uint8)


# ---------------------------------------------------------------- packet inspection (src/lib.rs:219-498)
_BW = ("Narrowband", "Mediumband", "Wideband", "Superwideband", "Fullband")
_MODE = ("SilkOnly", "Hybrid", "CeltOnly")


def query_packet_bandwidth(packet):
    return _BW[lib().opn_packet_bandwidth(_p(_bytes(packet)))]


def query_packet_channel_count(packet):
    return lib().opn_packet_channels(_p(_bytes(packet)))


def query_packet_frame_count(packet):
    b = _bytes(packet)
    return _chk(lib().opn_packet_frame_count(_p(b), len(b)))


def query_packet_samples_per_frame(packet, sampling_rate=48000):
    return lib().opn_packet_samples_per_frame(_p(_bytes(packet)), sampling_rate)


def query_packet_sample_count(packet, sampling_rate=48000):
    b = _bytes(packet)
    return _chk(lib().opn_packet_sample_count(_p(b), len(b), sampling_rate))


def query_packet_codec_mode(packet):
    return _MODE[lib().opn_packet_mode(_p(_bytes(packet)))]


def parse_packet(packet, self_delimited=False):
    """-> (count, frame_offsets, sizes, payload_offset, packet_offset)   (lib.rs:345-498)"""
    b = _bytes(packet)
    fr, sz = np.zeros(48, np.uint32), np.zeros(48, np.uint32)
    po, ko = C.c_uint32(0), C.c_uint32(0)
    n = _chk(lib().opn_parse_packet(_p(b), len(b), int(self_delimited), _p(fr), _p(sz), C.byref(po), C.byref(ko)))
    return n, fr[:n].tolist(), sz[:n].tolist(), po.value, ko.value


# ---------------------------------------------------------------- Decoder (src/decoder.rs:27-232)
@dataclass
class DecoderConfiguration:
    sampling_rate: int = 48000
    channels: int = 2
    gain: int = 0


class Decoder:
    """`Decoder` of the reference crate: one stream, packets in order, `None` = lost packet."""

    def __init__(self, configuration: DecoderConfiguration = None, device: int = 0, bitstream: int = BITSTREAM_OPUS):
        cfg = configuration or DecoderConfiguration()
        h = C.c_void_p()
        _chk(lib().opn_decoder_create(device, cfg.sampling_rate, cfg.channels, cfg.gain, bitstream, C.byref(h)))
        self._h, self._cfg = h, cfg

    def __del__(self):
        if getattr(self, "_h", None):
            lib().opn_decoder_destroy(self._h)
            self._h = None

    def reset(self):
        _chk(lib().opn_decoder_reset(self._h))

    def decode_float(self, packet, samples: np.ndarray, frame_size: int, decode_fec: bool = False) -> int:
        assert samples.dtype == np.float32 and samples.flags.c_contiguous
        if samples.size < frame_size * self._cfg.channels:
            raise OpusError(-2)
        if packet is None:
            return _chk(lib().opn_decode_float(self._h, None, 0, _p(samples), frame_size, int(decode_fec)))
        b = _bytes(packet)
        if len(b) == 0:
            raise OpusError(-1, "packet is empty")
        return _chk(lib().opn_decode_float(self._h, _p(b), len(b), _p(samples), frame_size, int(decode_fec)))

    def decode(self, packet, samples: np.ndarray, frame_size: int, decode_fec: bool = False) -> int:
        """Generic `decode<S>` (soft clip + Sample::from_f32); S is the dtype of `samples`: int16, int32, uint16,
        uint32, float32 or float64."""
        assert samples.flags.c_contiguous
        fmt = SAMPLE_FORMAT_OF[samples.dtype]
        if packet is None:
            return _chk(lib().opn_decode_pcm(self._h, None, 0, _p(samples), samples.size, fmt, frame_size, int(decode_fec)))
        b = _bytes(packet)
        return _chk(lib().opn_decode_pcm(self._h, _p(b), len(b), _p(samples), samples.size, fmt, frame_size, int(decode_fec)))

    sampling_rate = property(lambda s: lib().opn_decoder_sampling_rate(s._h))
    channels = property(lambda s: lib().opn_decoder_channels(s._h))
    gain = property(lambda s: lib().opn_decoder_gain(s._h))
    final_range = property(lambda s: lib().opn_decoder_final_range(s._h))

    @property
    def bandwidth(self):
        v = lib().opn_decoder_bandwidth(self._h)
        return None if v < 0 else _BW[v]

    @property
    def pitch(self):
        v = lib().opn_decoder_pitch(self._h)
        return None if v < 0 else v

    @property
    def last_packet_duration(self):
        v = lib().opn_decoder_last_packet_duration(self._h)
        return None if v < 0 else v


class _Config(C.Structure):
    _fields_ = [("fs_hz", C.c_int32), ("channels", C.c_int32), ("gain_q8", C.c_int16), ("postfilter", C.c_int16), ("bitstream", C.c_int32)]


class BatchDecoder:
    """Batch-of-streams entry point: n independent `Decoder`s advanced by one call per step."""

    def __init__(self, n_streams: int, configuration: DecoderConfiguration = None, device: int = 0, postfilter: bool = True,
                 bitstream: int = BITSTREAM_OPUS):
        cfg = configuration or DecoderConfiguration()
        c = _Config(cfg.sampling_rate, cfg.channels, cfg.gain, int(postfilter), bitstream)
        h = C.c_void_p()
        _chk(lib().opn_batch_create(device, n_streams, C.byref(c), C.byref(h)))
        self._h, self.n_streams, self.channels, self.device = h, n_streams, cfg.channels, device

    def __del__(self):
        if getattr(self, "_h", None):
            lib().opn_batch_destroy(self._h)
            self._h = None

    def reset(self):
        _chk(lib().opn_batch_reset(self._h))

    def decode_float(self, arena: np.ndarray, offsets: np.ndarray, lens: np.ndarray, pcm: np.ndarray, frame_size: int,
                     flags: int = 0):
        """Host buffers.  pcm: float32 [n_streams, >= frame_size*channels].  -> int32 results per stream."""
        assert arena.dtype == np.uint8 and offsets.dtype == np.uint32 and lens.dtype == np.uint32
        res = np.zeros(self.n_streams, np.int32)
        stride = 0
        if pcm is not None:
            assert pcm.dtype == np.float32 and pcm.ndim == 2 and pcm.shape[0] == self.n_streams and pcm.strides[1] == 4
            stride = pcm.strides[0] // 4
        _chk(lib().opn_batch_decode_float(self._h, _p(arena), _p(offsets), _p(lens), _p(pcm), stride, frame_size, _p(res), flags))
        return res

    def decode_float_ptrs(self, arena_ptr, offsets_ptr, lens_ptr, pcm_ptr, pcm_stride_floats, frame_size, result_ptr, flags):
        """Raw pointers (host or device according to `flags`); used with pinned / device tensors."""
        return _chk(lib().opn_batch_decode_float(self._h, arena_ptr, offsets_ptr, lens_ptr, pcm_ptr, pcm_stride_floats,
                                                 frame_size, result_ptr, flags))

    def decode_i16(self, arena, offsets, lens, pcm, frame_size, flags=0):
        """`Decoder::decode::<i16>` for every stream: soft clip + Sample::from_f32 on the device; pcm is int16
        [n_streams, >= frame_size*channels].  Returns (result_per_stream, ticket-or-0)."""
        arena = np.ascontiguousarray(arena, np.uint8)
        offsets = np.ascontiguousarray(offsets, np.uint32)
        lens = np.ascontiguousarray(lens, np.uint32)
        assert pcm.dtype == np.int16 and pcm.ndim == 2 and pcm.shape[0] == self.n_streams and pcm.flags.c_contiguous
        res = np.zeros(self.n_streams, np.int32)
        t = _chk(lib().opn_batch_decode_i16(self._h, _p(arena), _p(offsets), _p(lens), _p(pcm), pcm.shape[1], frame_size, _p(res), flags))
        return res, t

    def decode_pcm(self, arena, offsets, lens, pcm, frame_size, flags=0):
        """`Decoder::decode::<S>` for every stream, S = pcm.dtype (int16, int32, uint16, uint32, float32, float64);
        pcm is [n_streams, >= frame_size*channels].  Returns (result_per_stream, ticket-or-0)."""
        arena = np.ascontiguousarray(arena, np.uint8)
        offsets = np.ascontiguousarray(offsets, np.uint32)
        lens = np.ascontiguousarray(lens, np.uint32)
        assert pcm.ndim == 2 and pcm.shape[0] == self.n_streams and pcm.flags.c_contiguous
        res = np.zeros(self.n_streams, np.int32)
        t = _chk(lib().opn_batch_decode_pcm(self._h, _p(arena), _p(offsets), _p(lens), _p(pcm), pcm.shape[1], SAMPLE_FORMAT_OF[pcm.dtype],
                                            frame_size, _p(res), flags))
        return res, t

    def decode_i16_ptrs(self, arena_ptr, offsets_ptr, lens_ptr, pcm_ptr, pcm_stride_samples, frame_size, result_ptr, flags):
        return _chk(lib().opn_batch_decode_i16(self._h, arena_ptr, offsets_ptr, lens_ptr, pcm_ptr, pcm_stride_samples, frame_size,
                                               result_ptr, flags))

    def wait(self, ticket):
        """Completion of a host-buffer call submitted with FLAG_SUBMIT_ONLY (its return value is the ticket)."""
        _chk(lib().opn_batch_wait(self._h, int(ticket)))

    def join(self):
        """Order everything enqueued so far before whatever comes next on `cuda_stream` (no host wait)."""
        _chk(lib().opn_batch_join(self._h))

    def synchronize(self):
        _chk(lib().opn_batch_synchronize(self._h))

    def final_ranges(self):
        out = np.zeros(self.n_streams, np.uint32)
        _chk(lib().opn_batch_final_ranges(self._h, _p(out)))
        return out

    def ring(self):
        ring, pos, n = C.c_void_p(), C.c_void_p(), C.c_uint32(0)
        _chk(lib().opn_batch_ring(self._h, C.byref(ring), C.byref(n), C.byref(pos)))
        return ring.value, n.value, pos.value

    def enable_timing(self, on=True):
        _chk(lib().opn_batch_enable_timing(self._h, int(on)))

    def stats(self, reset=False):
        launches = (C.c_uint64 * 3)()
        ms = (C.c_double * 3)()
        _chk(lib().opn_batch_stats(self._h, launches, ms, int(reset)))
        return {"launches": list(launches), "ms": list(ms)}

    def history_samples(self, reset=False):
        """Comb history samples (summed over channel-frames) the frame kernel read in timed passes."""
        v = C.c_uint64(0)
        _chk(lib().opn_batch_history_samples(self._h, C.byref(v), int(reset)))
        return v.value

    @property
    def cuda_stream(self):
        return lib().opn_batch_cuda_stream(self._h)


# ---------------------------------------------------------------- host memory
class HostBuffer:
    """Page-locked host memory from opn_host_alloc, viewed as a numpy array (freed with the object)."""

    def __init__(self, shape, dtype):
        self.dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * self.dtype.itemsize
        self._p = lib().opn_host_alloc(n)
        if not self._p:
            raise MemoryError("opn_host_alloc failed")
        self.array = np.ctypeslib.as_array((C.c_uint8 * n).from_address(self._p)).view(self.dtype).reshape(shape)

    def __del__(self):
        if getattr(self, "_p", None):
            self.array = None
            lib().opn_host_free(self._p)
            self._p = None


def host_register(a: np.ndarray):
    _chk(lib().opn_host_register(_p(a), a.nbytes))


def host_unregister(a: np.ndarray):
    _chk(lib().opn_host_unregister(_p(a)))


# ---------------------------------------------------------------- operator level
def op_rangedec_script(arena, offsets, lens, ops, icdf_pool=None, y_stride=0, device=0):
    arena = np.ascontiguousarray(arena, np.uint8)
    offsets = np.ascontiguousarray(offsets, np.uint32)
    lens = np.ascontiguousarray(lens, np.uint32)
    ops = np.ascontiguousarray(ops, OP_DTYPE)
    pool = np.ascontiguousarray(icdf_pool if icdf_pool is not None else [0], np.uint8)
    n = len(offsets)
    out = np.zeros((n, len(ops)), OUT_DTYPE)
    y = np.zeros((n, max(y_stride, 1)), np.int32)
    _chk(lib().opn_op_rangedec_script(device, _p(arena), _p(offsets), _p(lens), n, _p(ops), len(ops), _p(pool), len(pool),
                                      _p(out), _p(y) if y_stride else None, y_stride))
    return out, y


def op_imdct_tdac(coefs, out, shift, blocks=1, device=0):
    """coefs [rows, >= n2*blocks]; out [rows, >= n2*blocks+60] (first 60 = previous tail), in place."""
    assert coefs.dtype == np.float32 and out.dtype == np.float32 and coefs.flags.c_contiguous and out.flags.c_contiguous
    _chk(lib().opn_op_imdct_tdac(device, _p(coefs), coefs.shape[1], _p(out), out.shape[1], coefs.shape[0], shift, blocks, blocks))
    return out


def op_comb_filter_inplace(y, y_offset, n, params4, gains2, overlap, device=0):
    assert y.dtype == np.float32 and y.ndim == 2 and y.flags.c_contiguous
    p = np.ascontiguousarray(params4, np.int32)
    g = np.ascontiguousarray(gains2, np.float32)
    _chk(lib().opn_op_comb_filter_inplace(device, _p(y), y.shape[1], y_offset, n, y.shape[0], _p(p), _p(g), overlap))
    return y


def op_comb_filter(y, x, offset, n, params4, gains2, overlap, device=0):
    assert y.dtype == np.float32 and x.dtype == np.float32 and y.shape == x.shape and y.flags.c_contiguous and x.flags.c_contiguous
    p = np.ascontiguousarray(params4, np.int32)
    g = np.ascontiguousarray(gains2, np.float32)
    _chk(lib().opn_op_comb_filter(device, _p(y), _p(x), y.shape[1], offset, n, y.shape[0], _p(p), _p(g), overlap))
    return y


def op_pcm_soft_clip(pcm, row_len, channels, mem, device=0):
    assert pcm.dtype == np.float32 and pcm.ndim == 2 and mem.dtype == np.float32 and mem.shape == (pcm.shape[0], channels)
    _chk(lib().opn_op_pcm_soft_clip(device, _p(pcm), pcm.shape[1], row_len, channels, pcm.shape[0], _p(mem)))
    return pcm


def op_smooth_fade(in1, in2, overlap, channels, fs=48000, device=0):
    """smooth_fade_into_in1 (src/decoder.rs:833-848) on rows of interleaved samples; returns the faded copy of in1."""
    in1 = np.ascontiguousarray(in1, np.float32)
    in2 = np.ascontiguousarray(in2, np.float32)
    assert in1.ndim == 2 and in1.shape == in2.shape
    out = np.empty_like(in1)
    _chk(lib().opn_op_smooth_fade(device, _p(in1), _p(in2), _p(out), in1.shape[1], overlap, channels, fs, in1.shape[0]))
    return out


def op_bitexact_trig(x=None, isin=None, icos=None, device=0):
    """bitexact_cos(x) and/or bitexact_log2tan(isin, icos) on the device (src/math.rs:51-69)."""
    x = np.zeros(0, np.int16) if x is None else np.ascontiguousarray(x, np.int16)
    isin = np.zeros(0, np.int32) if isin is None else np.ascontiguousarray(isin, np.int32)
    icos = np.zeros(0, np.int32) if icos is None else np.ascontiguousarray(icos, np.int32)
    assert len(isin) == len(icos)
    c, l = np.zeros(len(x), np.int16), np.zeros(len(isin), np.int32)
    _chk(lib().opn_op_bitexact_trig(device, _p(x), _p(c), len(x), _p(isin), _p(icos), _p(l), len(isin)))
    return c, l


def op_synth_symbols(arena, offsets, lens, lm, channels, device=0):
    arena = np.ascontiguousarray(arena, np.uint8)
    offsets = np.ascontiguousarray(offsets, np.uint32)
    lens = np.ascontiguousarray(lens, np.uint32)
    n, nf = len(offsets), 120 << lm
    side = np.zeros(n, SIDE_DTYPE)
    y = np.zeros((n, channels, nf), np.int32)
    coef = np.zeros((n, channels, nf), np.float32)
    _chk(lib().opn_op_synth_symbols(device, _p(arena), _p(offsets), _p(lens), n, lm, channels, _p(side), _p(y), _p(coef)))
    return side, y, coef


# ---------------------------------------------------------------- synthetic streams (host)
def synth_packet(stream_id, frame_idx, lm, channels, pkt_bytes, transient_permille=0):
    out = np.zeros(pkt_bytes, np.uint8)
    truth = np.zeros(1, SIDE_DTYPE)
    _chk(lib().opn_synth_packet(stream_id, frame_idx, lm, channels, pkt_bytes, transient_permille, _p(out), _p(truth)))
    return out, truth[0]


def synth_fill(first_stream, n_streams, first_frame, n_frames, lm, channels, pkt_bytes, transient_permille=0, n_threads=None,
               out=None):
    """-> uint8 [n_frames, n_streams, pkt_bytes]"""
    if out is None:
        out = np.zeros((n_frames, n_streams, pkt_bytes), np.uint8)
    assert out.dtype == np.uint8 and out.flags.c_contiguous and out.size == n_frames * n_streams * pkt_bytes
    nt = n_threads or min(os.cpu_count() or 1, 32)
    _chk(lib().opn_synth_fill(first_stream, n_streams, first_frame, n_frames, lm, channels, pkt_bytes, transient_permille, nt, _p(out)))
    return out


def silk_fill(first_stream, n_streams, first_frame, n_frames, bandwidth, frame_ms, channels, pkt_bytes, n_threads=None, out=None, lbrr_permille=0):
    """SYNTH-SILK/1 packets (TOC + payload) -> uint8 [n_frames, n_streams, pkt_bytes]; bandwidth 0 NB, 1 MB, 2 WB; frame_ms 10 or 20"""
    if out is None:
        out = np.zeros((n_frames, n_streams, pkt_bytes), np.uint8)
    assert out.dtype == np.uint8 and out.flags.c_contiguous and out.size == n_frames * n_streams * pkt_bytes
    nt = n_threads or min(os.cpu_count() or 1, 32)
    _chk(lib().opn_silk_fill(first_stream, n_streams, first_frame, n_frames, bandwidth, frame_ms, channels, pkt_bytes, lbrr_permille, nt, _p(out)))
    return out


def op_silk_frames(arena, offsets, lens, stream_channels, channels, frame_size, device=0, decode_fec=False):
    """One SILK-only packet per row, each through a fresh decoder -> (side, exc [n, 2, 320], out16 [n, 2, 320], pcm, results)"""
    arena = np.ascontiguousarray(arena, np.uint8)
    offsets = np.ascontiguousarray(offsets, np.uint32)
    lens = np.ascontiguousarray(lens, np.uint32)
    n = len(offsets)
    side = np.zeros(n, SILK_SIDE_DTYPE)
    exc = np.zeros((n, 2, SILK_MAX_FRAME), np.int32)
    out16 = np.zeros((n, 2, SILK_MAX_FRAME), np.int16)
    pcm = np.zeros((n, frame_size * channels), np.float32)
    res = np.zeros(n, np.int32)
    _chk(lib().opn_op_silk_frames(device, _p(arena), _p(offsets), _p(lens), n, stream_channels, channels, frame_size, int(decode_fec), _p(side), _p(exc),
                                  _p(out16), _p(pcm), _p(res)))
    return side, exc, out16, pcm, res


def celt2_packet(stream_id, frame_idx, lm, channels, pkt_bytes, transient_permille=0):
    """One SYNTH-CELT/2 packet (TOC + payload) and the side record the generator's own frame logic produced."""
    out = np.zeros(pkt_bytes, np.uint8)
    truth = np.zeros(1, CELT2_SIDE_DTYPE)
    _chk(lib().opn_celt2_packet(stream_id, frame_idx, lm, channels, pkt_bytes, transient_permille, _p(out), _p(truth)))
    return out, truth[0]


def celt2_fill(first_stream, n_streams, first_frame, n_frames, lm, channels, pkt_bytes, transient_permille=0, n_threads=None):
    """-> uint8 [n_frames, n_streams, pkt_bytes]"""
    out = np.zeros((n_frames, n_streams, pkt_bytes), np.uint8)
    nt = n_threads or min(os.cpu_count() or 1, 32)
    _chk(lib().opn_celt2_fill(first_stream, n_streams, first_frame, n_frames, lm, channels, pkt_bytes, transient_permille, nt, _p(out)))
    return out


def op_celt2_symbols(arena, offsets, lens, lm, channels, device=0):
    arena = np.ascontiguousarray(arena, np.uint8)
    offsets = np.ascontiguousarray(offsets, np.uint32)
    lens = np.ascontiguousarray(lens, np.uint32)
    n, nf = len(offsets), 120 << lm
    side = np.zeros(n, CELT2_SIDE_DTYPE)
    y = np.zeros((n, channels, nf), np.int32)
    coef = np.zeros((n, channels, nf), np.float32)
    _chk(lib().opn_op_celt2_symbols(device, _p(arena), _p(offsets), _p(lens), n, lm, channels, _p(side), _p(y), _p(coef)))
    return side, y, coef


def enc_run_script(nbytes, ops, values, icdf_pool=None, y_in=None):
    ops = np.ascontiguousarray(ops, OP_DTYPE)
    values = np.ascontiguousarray(values, np.uint32)
    buf = np.zeros(nbytes, np.uint8)
    tf = np.zeros(len(ops), np.uint32)
    pool = np.ascontiguousarray(icdf_pool if icdf_pool is not None else [0], np.uint8)
    yin = np.ascontiguousarray(y_in if y_in is not None else [0], np.int32)
    rb, ftf = C.c_uint32(0), C.c_uint32(0)
    err = lib().opn_enc_run_script(_p(buf), nbytes, _p(ops), _p(values), len(ops), _p(pool), _p(yin), _p(tf), C.byref(rb), C.byref(ftf))
    return buf, tf, rb.value, ftf.value, err
