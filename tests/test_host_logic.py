"""CPU-only tests of the product's host side: C-ABI export surface, packet inspection, the host
range encoder and the SYNTH-CELT/1 generator -- each cross-checked against the oracle."""
import ctypes as C
import json
import os
import re
import subprocess

import numpy as np
import pytest

import opus_native_b200 as opn
import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KATS = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_kats.json")))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "opusb200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(opn_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 40
    out = subprocess.check_output(["nm", "-D", "--defined-only", opn.library_path()], text=True)
    exported = set(re.findall(r" T (opn_[a-z0-9_]+)", out))
    assert declared <= exported, sorted(declared - exported)
    L = opn.lib()
    for name in declared:
        assert getattr(L, name) is not None


def test_no_fma_in_the_fused_float_kernels():
    """The float kernels must round exactly like the reference (no contraction of a*b+c): the TU is built with -fmad=false
    and only SUMS are packed (FADD2); ptxas would contract a packed multiply feeding a packed add into FFMA2 regardless
    of --fmad=false, so there must be none.  The only FMAs allowed are the division / square-root expansions of the PVQ
    gain (2^-5 / sqrt(yy)) in the kernels that expand pulses, and of the soft clip."""
    import collections
    sass = subprocess.run(["cuobjdump", "-sass", opn.library_path()], capture_output=True, text=True, check=True).stdout
    counts, cur = collections.defaultdict(collections.Counter), None
    for ln in sass.split("\n"):
        m = re.search(r"Function : (\S+)", ln)
        if m:
            cur = m.group(1)
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+([A-Z0-9]+)", ln)
        if m and cur:
            counts[cur][m.group(1)] += 1
    frame = [k for k in counts if "k_frame_w" in k]
    # 4 frame sizes x mono/stereo x {SYNTH-CELT/1, SYNTH-CELT/2}, plus the mono<->stereo mapping variants
    # (4 frame sizes x 2 directions x the two SYNTH layouts)
    assert len(frame) == 16 + 16
    for k, c in counts.items():
        assert c["FFMA2"] == 0 and c["FMUL2"] == 0, (k, dict(c))
        if "k_frame_w" in k:
            assert c["FADD2"] > 100, k                      # the packed sums are there
            assert c["FFMA"] <= 24, (k, c["FFMA"])
        if "k_op_imdct_w" in k or "k_op_comb" in k:
            assert c["FFMA"] == 0, (k, c["FFMA"])


def test_no_gpu_means_loud_failure():
    if opn.lib().opn_device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(opn.OpusError) as e:
        opn.BatchDecoder(4)
    assert e.value.kind == "Cuda"
    with pytest.raises(opn.OpusError):
        opn.Decoder()


# ---- src/lib.rs:653-860 through the product's own host functions
def test_query_packet_tables():
    assert [opn.query_packet_bandwidth([c << 3]) for c in range(32)] == (
        ["Narrowband"] * 4 + ["Mediumband"] * 4 + ["Wideband"] * 4 + ["Superwideband"] * 2 + ["Fullband"] * 2
        + ["Narrowband"] * 4 + ["Wideband"] * 4 + ["Superwideband"] * 4 + ["Fullband"] * 4)
    assert [opn.query_packet_samples_per_frame([c << 3]) for c in range(32)] == (
        [480, 960, 1920, 2880] * 3 + [480, 960, 480, 960] + [120, 240, 480, 960] * 4)
    assert opn.query_packet_channel_count([0]) == 1 and opn.query_packet_channel_count([4]) == 2
    assert [opn.query_packet_frame_count([c]) for c in (0, 1, 2)] == [1, 2, 2]
    with pytest.raises(opn.OpusError):
        opn.query_packet_frame_count([3])
    assert opn.query_packet_frame_count([3, 5]) == 5
    assert opn.query_packet_sample_count([70]) == 960
    with pytest.raises(opn.OpusError):
        opn.query_packet_sample_count([3])
    assert opn.query_packet_sample_count([255, 5]) == 4800
    assert [opn.query_packet_codec_mode([t]) for t in (0x00, 0x60, 0x80, 0xFC)] == ["SilkOnly", "Hybrid", "CeltOnly", "CeltOnly"]


def test_parse_packet_kats():
    assert opn.parse_packet(KATS["packet_single"]) == (1, [1], [11], 1, 12)
    assert opn.parse_packet(KATS["packet_cbr"]) == (2, [1, 6], [5, 5], 1, 11)
    assert opn.parse_packet(KATS["packet_vbr"]) == (2, [2, 6], [4, 6], 2, 12)
    with pytest.raises(opn.OpusError) as e:
        opn.parse_packet(KATS["packet_invalid"])
    assert e.value.kind == "InvalidPacket"


def test_parse_packet_matches_oracle_on_random_packets():
    rnd = np.random.default_rng(7)
    L = O.lib()
    n_ok = 0
    for trial in range(4000):
        ln = int(rnd.integers(1, 64))
        pkt = rnd.integers(0, 256, ln).astype(np.uint8)
        if trial % 3 == 0:  # bias towards code 3 with plausible headers
            pkt[0] = (pkt[0] & 0xFC) | 3
            if ln > 1:
                pkt[1] = (pkt[1] & 0xC0) | int(rnd.integers(0, 8))
        for sd in (0, 1):
            fr, sz = np.zeros(48, np.uint32), np.zeros(48, np.uint32)
            po, ko = C.c_uint32(0), C.c_uint32(0)
            want = L.orc_parse_packet(O.ptr(pkt), ln, sd, O.ptr(fr), O.ptr(sz), C.byref(po), C.byref(ko))
            try:
                got = opn.parse_packet(pkt, bool(sd))
            except opn.OpusError as e:
                assert want < 0 and e.code == want
                continue
            assert want == got[0]
            assert got[1] == fr[:want].tolist() and got[2] == sz[:want].tolist()
            assert (got[3], got[4]) == (po.value, ko.value)
            n_ok += 1
    assert n_ok > 500


# ---- host range encoder == oracle encoder, byte for byte
def test_host_encoder_matches_oracle_encoder():
    rnd = np.random.default_rng(3)
    pool = np.array([2, 1, 0, 1, 0], np.uint8)
    for _ in range(200):
        ops, vals, ys = [], [], []
        for _ in range(int(rnd.integers(20, 200))):
            kind = int(rnd.integers(0, 8))
            if kind == 0:
                ft = int(rnd.integers(2, 2 ** int(rnd.integers(2, 32))))
                ops.append((opn.OP_UINT, ft, 0)); vals.append(int(rnd.integers(0, ft)))
            elif kind == 1:
                nb = int(rnd.integers(1, 26))
                ops.append((opn.OP_BITS, nb, 0)); vals.append(int(rnd.integers(0, 1 << nb)))
            elif kind == 2:
                ops.append((opn.OP_BIT_LOGP, int(rnd.integers(1, 16)), 0)); vals.append(int(rnd.integers(0, 2)))
            elif kind == 3:
                ops.append((opn.OP_ICDF, 0, 2)); vals.append(int(rnd.integers(0, 3)))
            elif kind == 4:
                decay = int(rnd.integers(5000, 16000))
                ops.append((opn.OP_LAPLACE, O.lib().orc_laplace_start_freq(decay), decay))
                vals.append(int(rnd.integers(-20, 21)) & 0xFFFFFFFF)
            elif kind == 5:
                ops.append((opn.OP_BIT_VIA_DECODE, int(rnd.integers(1, 16)), 0)); vals.append(int(rnd.integers(0, 2)))
            elif kind == 6:
                ops.append((opn.OP_BIT_VIA_DECODE_BIN, int(rnd.integers(1, 16)), 0)); vals.append(int(rnd.integers(0, 2)))
            else:
                i = int(rnd.integers(0, 22))
                n, kmax = KATS["pvc_pn"][i], KATS["pvc_pk_max"][i]
                k = int(rnd.integers(1, kmax + 1))
                y = np.zeros(n, np.int32)
                O.lib().orc_cwrsi(O.ptr(y), n, k, int(rnd.integers(0, O.lib().orc_pvq_v(n, k))))
                ops.append((opn.OP_PULSES, n, k)); vals.append(0); ys.extend(y.tolist())
        ops = np.array(ops, opn.OP_DTYPE)
        a = opn.enc_run_script(2048, ops, vals, pool, ys or None)
        b = O.enc_run_script(2048, ops, vals, pool, ys or None)
        assert a[4] == b[4] == 0
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2:4] == b[2:4]
        out, y = O.dec_run_script(a[0], ops, pool, y_cap=len(ys))
        ok = ops["op"] != opn.OP_LAPLACE  # the Laplace encoder may clamp its input
        assert np.array_equal(out["value"][ok & (ops["op"] != opn.OP_PULSES)],
                              np.array(vals, np.uint32)[ok & (ops["op"] != opn.OP_PULSES)])
        assert y.tolist() == ys


# ---- SYNTH-CELT/1: generator truth == oracle decode, for every frame size and channel count
@pytest.mark.parametrize("lm,channels,pkt_bytes", [(3, 2, 160), (3, 1, 100), (2, 2, 130), (1, 2, 100), (0, 2, 80), (0, 1, 48)])
def test_synth_packets_decode_to_truth(lm, channels, pkt_bytes):
    for stream in range(24):
        dec = O.SynthStream(lm, channels)
        for frame in range(3):
            pkt, truth = opn.synth_packet(stream, frame, lm, channels, pkt_bytes, transient_permille=300)
            assert opn.query_packet_codec_mode(pkt) == "CeltOnly"
            assert opn.query_packet_samples_per_frame(pkt) == 120 << lm
            assert opn.query_packet_channel_count(pkt) == channels
            assert opn.parse_packet(pkt) == (1, [1], [pkt_bytes - 1], 1, pkt_bytes)
            side, y, coef, pcm = dec.decode(pkt[1:])
            for f in ("silence", "postfilter", "octave", "period", "gain_idx", "tapset", "transient", "intra", "n_pulses", "tell_frac"):
                assert getattr(side, f) == truth[f], f
            assert np.array_equal(np.ctypeslib.as_array(side.coarse)[:channels], truth["coarse"][:channels])
            assert np.array_equal(np.ctypeslib.as_array(side.fine)[:channels], truth["fine"][:channels])
            nf = 120 << lm
            y = y.reshape(channels, nf)
            assert np.all(y[:, 100 << lm:] == 0)
            # every band part has unit norm * 2^-5
            e = (coef.reshape(channels, nf).astype(np.float64) ** 2).sum(axis=1)
            assert np.all(e > 0) and np.all(np.isfinite(pcm))


def test_synth_packet_budget_errors():
    with pytest.raises(opn.OpusError) as e:
        opn.synth_packet(0, 0, 3, 2, 60)
    assert e.value.kind == "BufferToSmall"
    with pytest.raises(opn.OpusError):
        opn.synth_packet(0, 0, 4, 2, 160)


def test_synth_fill_is_deterministic_and_threaded():
    a = opn.synth_fill(5, 16, 2, 3, 3, 2, 160, n_threads=1)
    b = opn.synth_fill(5, 16, 2, 3, 3, 2, 160, n_threads=4)
    assert np.array_equal(a, b)
    pkt, _ = opn.synth_packet(5 + 7, 2 + 1, 3, 2, 160)
    assert np.array_equal(a[1, 7], pkt)


def test_digit_reversal_closed_form():
    """imdct_warp.cuh resolves the kiss-fft digit reversal at compile time: the aligned group g (of
    GS = 32 >> shift positions) holds exactly the inputs i = r + 15 q, r = g // 3 + 5 (g % 3), and the
    in-group position p maps to q by w_qmap.  Check that closed form against the generated tables."""
    src = open(os.path.join(ROOT, "opus-native_b200", "csrc", "opn_tables.h")).read()

    def table(name):
        body = re.search(r"%s\[\d+\] = \{(.*?)\};" % name, src, re.S).group(1)
        return [int(v) for v in body.replace("\n", " ").split(",") if v.strip()]

    def qmap(shift, p):
        if shift == 0:
            return (p >> 3) + 4 * ((p >> 2) & 1) + 8 * (p & 3)
        if shift == 1:
            return (p >> 2) + 4 * (p & 3)
        if shift == 2:
            return (p >> 2) + 2 * (p & 3)
        return p

    for shift, nfft in [(0, 480), (1, 240), (2, 120), (3, 60)]:
        bitrev = table("OPN_BITREV_%d" % nfft)
        gs = 32 >> shift
        seen = set()
        for g in range(15):
            j1, j2 = divmod(g, 3)
            r = j1 + 5 * j2
            for p in range(gs):
                i = r + 15 * qmap(shift, p)
                assert bitrev[i] == gs * g + p
                seen.add(i)
        assert len(seen) == nfft


def test_cpp_mirror_compiles_and_fails_loudly_without_gpu():
    """include/opusb200.hpp (the C++ mirror of Decoder / DecoderConfiguration / OpusError) builds against the
    library; without a CUDA device the example exits with the library's Cuda error, never with PCM."""
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "examples")], stdout=subprocess.DEVNULL)
    exe = os.path.join(ROOT, "examples", "decode_batch")
    assert os.path.exists(exe)
    if opn.lib().opn_device_count() > 0:
        pytest.skip("a CUDA device is present (the GPU suite runs the example)")
    r = subprocess.run([exe, "4", "1"], capture_output=True, text=True)
    assert r.returncode == 2 and "OpusError(-7)" in r.stderr and r.stdout == ""
