#!/usr/bin/env python3
"""Generate the constant tables of the CELT 48 kHz / 960 standard mode.

Nothing here is copied from the reference: every table is recomputed from its
defining formula and the result is checked (tests/test_tables_vs_reference.py)
against the literals in the reference crate, kept in tests/golden/reference_tables.json:

  TRIG[1800]      /root/reference/src/celt/mdct.rs:265-626
                  f32(cos(2*PI_F*(i+1/8)/N)) for N = 1920, 960, 480, 240 (i < N/2), where
                  PI_F is the *single precision* constant 3.141592653f the upstream C
                  generator used, then rounded through an 8-significant-digit decimal
                  (the precision the literals were printed with).  Reproduces 1800/1800.
  WINDOW[120]     src/celt/mode.rs:43-68
                  sin(pi/2 * sin^2(pi/2 * (i+1/2)/120)) in double, printed with 8 significant
                  digits, parsed as f32.  Reproduces 120/120.
  TWIDDLES[480]   src/celt/kiss_fft.rs:341-582
                  (cos, sin)(-2*pi*k/480) in double, 8 significant digits, parsed as f32.
                  Reproduces 957/960 scalars; the three that differ are the "zero"
                  crossings, where the upstream table holds x87 `fcos/fsin` argument
                  reduction residue instead of the IEEE double result.  They are listed
                  in X87_RESIDUE below (value ~1e-16, no effect on PCM at the 1e-5 bar,
                  but kept so that the table is bit-identical).
  BITREV_*        src/celt/kiss_fft.rs:281-336  (kiss-fft recursive digit reversal of the
                  factor lists at kiss_fft.rs:251,259,267,275)
  PVQ_U           src/celt/pvc.rs:301-429  U(n,k)=U(n-1,k)+U(n,k-1)+U(n-1,k-1) (pvc.rs:293)

Outputs two headers with the same numbers and different symbol prefixes, so that the
oracle and the product never include each other's files:
    oracle/oracle_tables.h                 (prefix ORC_)
    opus-native_b200/csrc/opn_tables.h     (prefix OPN_)
"""
import math
import os
import struct

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def f32(x: float) -> float:
    return struct.unpack("<f", struct.pack("<f", x))[0]


def via_text8(x: float) -> float:
    """8 significant decimal digits -> nearest f32 (how the literals were produced)."""
    return f32(float("%.8g" % x))


PI_F = f32(3.141592653)

# (index, component) -> value ; see module docstring.
X87_RESIDUE = {(120, "r"): 6.1230318e-17, (360, "r"): -1.8369095e-16, (240, "i"): -1.2246064e-16}

FACTORS = {
    480: [5, 96, 3, 32, 4, 8, 2, 4, 4, 1],
    240: [5, 48, 3, 16, 4, 4, 4, 1],
    120: [5, 24, 3, 8, 2, 4, 4, 1],
    60: [5, 12, 3, 4, 4, 1],
}

# last column stored for row r = min(n,k)  (pvc.rs:316-427)
PVQ_ROW_LAST = [176, 176, 176, 176, 176, 176, 96, 54, 37, 28, 24, 19, 18, 16, 14]

E_BANDS = [0, 1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 14, 16, 20, 24, 28, 34, 40, 48, 60, 78, 100]
LOG_N = [0, 0, 0, 0, 0, 0, 0, 0, 8, 8, 8, 8, 16, 16, 16, 21, 21, 24, 29, 34, 36]
# Q15 tap gains / 32768 (comb_filter/mod.rs:45-55)
COMB_GAINS_Q15 = [10048, 7112, 4248, 15200, 8784, 0, 26208, 3280, 0]


# ---- static allocation data of the standard 48 kHz / 960 mode.  These are DATA of the codec (RFC 6716 section 4.3.3:
# the static allocation table in 1/32 bit per sample; libopus ships the pulse cache of its compute_pulse_cache() as
# literals in static_modes_float.h), not formulas; tests/test_tables_vs_reference.py checks them against
# src/celt/mode.rs:13-28 and :70-111.
NB_ALLOC_VECTORS = 11
ALLOC_VECTORS = [
    0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
    90, 80, 75, 69, 63, 56, 49, 40, 34, 29, 20, 18, 10, 0, 0, 0, 0, 0, 0, 0, 0,
    110, 100, 90, 84, 78, 71, 65, 58, 51, 45, 39, 32, 26, 20, 12, 0, 0, 0, 0, 0, 0,
    118, 110, 103, 93, 86, 80, 75, 70, 65, 59, 53, 47, 40, 31, 23, 15, 4, 0, 0, 0, 0,
    126, 119, 112, 104, 95, 89, 83, 78, 72, 66, 60, 54, 47, 39, 32, 25, 17, 12, 1, 0, 0,
    134, 127, 120, 114, 103, 97, 91, 85, 78, 72, 66, 60, 54, 47, 41, 35, 29, 23, 16, 10, 1,
    144, 137, 130, 124, 113, 107, 101, 95, 88, 82, 76, 70, 64, 57, 51, 45, 39, 33, 26, 15, 1,
    152, 145, 138, 132, 123, 117, 111, 105, 98, 92, 86, 80, 74, 67, 61, 55, 49, 43, 36, 20, 1,
    162, 155, 148, 142, 133, 127, 121, 115, 108, 102, 96, 90, 84, 77, 71, 65, 59, 53, 46, 30, 1,
    172, 165, 158, 152, 143, 137, 131, 125, 118, 112, 106, 100, 94, 87, 81, 75, 69, 63, 56, 45, 20,
    200, 200, 200, 200, 200, 200, 200, 200, 198, 193, 188, 183, 178, 173, 168, 163, 158, 153, 148, 129, 104,
]
CACHE_INDEX = [
    -1, -1, -1, -1, -1, -1, -1, -1, 0, 0, 0, 0, 41, 41, 41, 82, 82, 123, 164, 200, 222,
    0, 0, 0, 0, 0, 0, 0, 0, 41, 41, 41, 41, 123, 123, 123, 164, 164, 240, 266, 283, 295,
    41, 41, 41, 41, 41, 41, 41, 41, 123, 123, 123, 123, 240, 240, 240, 266, 266, 305, 318, 328, 336,
    123, 123, 123, 123, 123, 123, 123, 123, 240, 240, 240, 240, 305, 305, 305, 318, 318, 343, 351, 358, 364,
    240, 240, 240, 240, 240, 240, 240, 240, 305, 305, 305, 305, 343, 343, 343, 351, 351, 370, 376, 382, 387,
]
CACHE_BITS = [
    40, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7,
    7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 7, 40, 15, 23, 28, 31, 34, 36,
    38, 39, 41, 42, 43, 44, 45, 46, 47, 47, 49, 50, 51, 52, 53, 54, 55, 55, 57, 58, 59, 60, 61, 62,
    63, 63, 65, 66, 67, 68, 69, 70, 71, 71, 40, 20, 33, 41, 48, 53, 57, 61, 64, 66, 69, 71, 73, 75,
    76, 78, 80, 82, 85, 87, 89, 91, 92, 94, 96, 98, 101, 103, 105, 107, 108, 110, 112, 114, 117, 119, 121, 123,
    124, 126, 128, 40, 23, 39, 51, 60, 67, 73, 79, 83, 87, 91, 94, 97, 100, 102, 105, 107, 111, 115, 118, 121,
    124, 126, 129, 131, 135, 139, 142, 145, 148, 150, 153, 155, 159, 163, 166, 169, 172, 174, 177, 179, 35, 28, 49, 65,
    78, 89, 99, 107, 114, 120, 126, 132, 136, 141, 145, 149, 153, 159, 165, 171, 176, 180, 185, 189, 192, 199, 205, 211,
    216, 220, 225, 229, 232, 239, 245, 251, 21, 33, 58, 79, 97, 112, 125, 137, 148, 157, 166, 174, 182, 189, 195, 201,
    207, 217, 227, 235, 243, 251, 17, 35, 63, 86, 106, 123, 139, 152, 165, 177, 187, 197, 206, 214, 222, 230, 237, 250,
    25, 31, 55, 75, 91, 105, 117, 128, 138, 146, 154, 161, 168, 174, 180, 185, 190, 200, 208, 215, 222, 229, 235, 240,
    245, 255, 16, 36, 65, 89, 110, 128, 144, 159, 173, 185, 196, 207, 217, 226, 234, 242, 250, 11, 41, 74, 103, 128,
    151, 172, 191, 209, 225, 241, 255, 9, 43, 79, 110, 138, 163, 186, 207, 227, 246, 12, 39, 71, 99, 123, 144, 164,
    182, 198, 214, 228, 241, 253, 9, 44, 81, 113, 142, 168, 192, 214, 235, 255, 7, 49, 90, 127, 160, 191, 220, 247,
    6, 51, 95, 134, 170, 203, 234, 7, 47, 87, 123, 155, 184, 212, 237, 6, 52, 97, 137, 174, 208, 240, 5, 57,
    106, 151, 192, 231, 5, 59, 111, 158, 202, 243, 5, 55, 103, 147, 187, 224, 5, 60, 113, 161, 206, 248, 4, 65,
    122, 175, 224, 4, 67, 127, 182, 234,
]
CACHE_CAPS = [
    224, 224, 224, 224, 224, 224, 224, 224, 160, 160, 160, 160, 185, 185, 185, 178, 178, 168, 134, 61, 37,
    224, 224, 224, 224, 224, 224, 224, 224, 240, 240, 240, 240, 207, 207, 207, 198, 198, 183, 144, 66, 40,
    160, 160, 160, 160, 160, 160, 160, 160, 185, 185, 185, 185, 193, 193, 193, 183, 183, 172, 138, 64, 38,
    240, 240, 240, 240, 240, 240, 240, 240, 207, 207, 207, 207, 204, 204, 204, 193, 193, 180, 143, 66, 40,
    185, 185, 185, 185, 185, 185, 185, 185, 193, 193, 193, 193, 193, 193, 193, 183, 183, 172, 138, 65, 39,
    207, 207, 207, 207, 207, 207, 207, 207, 204, 204, 204, 204, 201, 201, 201, 188, 188, 176, 141, 66, 40,
    193, 193, 193, 193, 193, 193, 193, 193, 193, 193, 193, 193, 194, 194, 194, 184, 184, 173, 139, 65, 39,
    204, 204, 204, 204, 204, 204, 204, 204, 201, 201, 201, 201, 198, 198, 198, 187, 187, 175, 140, 66, 40,
]
# log2(n) in 1/8 bit, n = 0..23: the cost of the intensity-stereo parameter (libopus rate.c LOG2_FRAC_TABLE)
LOG2_FRAC_TABLE = [0, 8, 13, 16, 19, 21, 23, 24, 26, 27, 28, 29, 30, 31, 32, 32, 33, 34, 34, 35, 36, 36, 37, 37]


def trig_table():
    out = []
    for shift in range(4):
        n = 1920 >> shift
        for i in range(n // 2):
            out.append(via_text8(f32(math.cos(2 * PI_F * (i + 0.125) / n))))
    return out


def window_table():
    out = []
    for i in range(120):
        s = math.sin(0.5 * math.pi * (i + 0.5) / 120)
        out.append(via_text8(math.sin(0.5 * math.pi * s * s)))
    return out


def twiddle_table():
    out = []
    for k in range(480):
        ph = (-2 * math.pi / 480) * k
        r = via_text8(math.cos(ph))
        i = via_text8(math.sin(ph))
        if (k, "r") in X87_RESIDUE:
            r = f32(X87_RESIDUE[(k, "r")])
        if (k, "i") in X87_RESIDUE:
            i = f32(X87_RESIDUE[(k, "i")])
        out.append((r, i))
    return out


def bitrev_table(nfft):
    """kiss-fft compute_bitrev_table: recursive digit reversal."""
    fac = FACTORS[nfft]
    table = [0] * nfft

    def rec(fout, f_base, fstride, in_stride, fi):
        p, m = fac[fi], fac[fi + 1]
        if m == 1:
            for j in range(p):
                table[f_base + j] = fout
                fout += fstride * in_stride
        else:
            for j in range(p):
                rec(fout, f_base, fstride * p, in_stride, fi + 2)
                f_base += m
                fout += fstride * in_stride

    # Table maps natural index -> position; the reference stores bitrev[i] = position of
    # input i, which is the inverse of the kiss-fft "f" walk below.
    order = [0] * nfft
    pos = [0]

    def walk(fout, fstride, fi):
        p, m = fac[fi], fac[fi + 1]
        if m == 1:
            for j in range(p):
                order[pos[0]] = fout + j * fstride
                pos[0] += 1
        else:
            for j in range(p):
                walk(fout + j * fstride, fstride * p, fi + 2)

    walk(0, 1, 0)
    # order[q] = natural input index stored at position q  ->  bitrev[input] = q
    inv = [0] * nfft
    for q, i in enumerate(order):
        inv[i] = q
    return inv


def pvq_tables():
    nmax = 177
    # U(0,0)=1, U(0,k>0)=0, U(n>0,0)=0; only cells with min(n,k) <= 15 are needed.
    full = [[0] * (nmax + 1) for _ in range(nmax + 1)]
    full[0][0] = 1
    for n in range(1, nmax + 1):
        for k in range(1, nmax + 1):
            if min(n, k) > 15:
                continue
            full[n][k] = full[n - 1][k] + full[n][k - 1] + full[n - 1][k - 1]
    data, rows = [], []
    for r, last in enumerate(PVQ_ROW_LAST):
        rows.append(len(data) - r)
        for c in range(r, last + 1):
            v = full[r][c]
            assert v < 2 ** 32, (r, c, v)
            data.append(v)
    return rows, data


# pvc.rs:463-469 (test_pvc): band sizes reachable by splitting and the largest K whose V(N,K)
# fits in 32 bits.
PVQ_N = [2, 3, 4, 6, 8, 9, 11, 12, 16, 18, 22, 24, 32, 36, 44, 48, 64, 72, 88, 96, 144, 176]
PVQ_KMAX = [128, 128, 128, 88, 36, 26, 18, 16, 12, 11, 9, 9, 7, 7, 6, 6, 5, 5, 5, 5, 4, 4]
SYNTH_RATE = 0.65  # bits per coefficient (SURVEY.md 8d, SYNTH-CELT/1)


def synth_schedule():
    """SYNTH-CELT/1 PVQ schedule (SURVEY.md 8d): for every (LM, band) the part size n, the
    number of parts and the pulse count K.  n == 1 means "one raw sign bit"."""
    nmax = 177
    full = [[0] * (nmax + 2) for _ in range(nmax + 2)]
    full[0][0] = 1
    for n in range(1, nmax + 1):
        for k in range(1, nmax + 1):
            if min(n, k) <= 15:
                full[n][k] = full[n - 1][k] + full[n][k - 1] + full[n - 1][k - 1]

    def V(n, k):
        return full[n][k] + full[n][k + 1]

    kmax = dict(zip(PVQ_N, PVQ_KMAX))
    sched = []
    for lm in range(4):
        row = []
        for b in range(21):
            nb = (E_BANDS[b + 1] - E_BANDS[b]) << lm
            if nb == 1:
                row.append((1, 1, 0))
                continue
            n, parts = nb, 1
            budget = SYNTH_RATE * nb
            while True:
                if n not in kmax:
                    n //= 2
                    parts *= 2
                    continue
                if parts * math.log2(V(n, kmax[n])) < budget and (n // 2) in kmax and n % 2 == 0:
                    n //= 2
                    parts *= 2
                    continue
                break
            k = 1
            for kk in range(1, kmax[n] + 1):
                if parts * math.log2(V(n, kk)) <= budget:
                    k = kk
            assert V(n, k) < 2 ** 32
            row.append((n, parts, k))
        sched.append(row)
    return sched


def silk_up_filter(L, taps=8, beta=8.0):
    """Polyphase interpolator by L: phase p, tap j weighs input x[i - j] for output L*i + p."""
    n = L * taps
    centre = (n - 1) / 2.0
    def i0(x):  # modified Bessel function of the first kind, order 0
        t, term, k = 1.0, 1.0, 1
        while term > 1e-18 * t:
            term *= (x / (2.0 * k)) ** 2
            t += term
            k += 1
        return t
    proto = []
    for m in range(n):
        x = (m - centre) / L                      # in input samples
        s = 1.0 if x == 0 else math.sin(math.pi * 0.9 * x) / (math.pi * 0.9 * x)
        r = 2.0 * m / (n - 1) - 1.0
        proto.append(0.9 * s * i0(beta * math.sqrt(max(0.0, 1.0 - r * r))) / i0(beta))
    phases = []
    for p in range(L):
        ph = [proto[p + L * j] for j in range(taps)]
        g = sum(ph)
        phases.append([v / g for v in ph])
    return phases


def silk_ltp_filters():
    """SYNTH-SILK/1 long-term predictor codebook: 8 symmetric 5-tap filters in Q14, total gain 0.20 .. 0.76."""
    out = []
    for f in range(8):
        g = 0.2 + 0.08 * f
        w0 = 0.5 + 0.05 * f
        w1 = (1.0 - w0) / 2.0 * 0.8
        w2 = (1.0 - w0) / 2.0 * 0.2
        out += [int(round(16384.0 * g * w)) for w in (w2, w1, w0, w1, w2)]
    return out


SILK_TYPE_ICDF = [230, 154, 0]                                # frame type: 0 inactive, 1 unvoiced, 2 voiced
SILK_DELTA_GAIN_ICDF = [250, 240, 220, 180, 76, 36, 16, 6, 0]  # gain index step - 4, subframes 1..3
SILK_CONTOUR_ICDF = [200, 60, 20, 0]                          # pitch lag of a subframe - frame lag + 1
SILK_LTP_ICDF = [224, 192, 160, 128, 96, 64, 32, 0]           # LTP filter of a subframe
SILK_PULSES_ICDF = [120, 60, 30, 14, 6, 3, 2, 1, 0,           # pulses K of a 16-sample shell block, inactive frames
                    200, 130, 80, 45, 25, 12, 5, 2, 0]        # ... active frames


def fhex(x: float) -> str:
    if x == 0.0:
        return "-0.0f" if math.copysign(1, x) < 0 else "0.0f"
    m, e = float.hex(x).split("p")
    m = m.rstrip("0")
    if m.endswith("."):
        m += "0"
    return f"{m}p{e}f"


def emit(path, prefix, guard):
    trig, win, tw = trig_table(), window_table(), twiddle_table()
    rows, data = pvq_tables()
    L = []
    w = L.append
    w("/* GENERATED by tools/gen_tables.py -- do not edit. CELT 48 kHz/960 standard mode constants,")
    w(" * recomputed from their defining formulas (see the generator's docstring for the formulas")
    w(" * and for the reference file:line each table is checked against). */")
    w(f"#ifndef {guard}\n#define {guard}\n#include <stdint.h>\n")
    w(f"#define {prefix}OVERLAP 120\n#define {prefix}NB_EBANDS 21\n#define {prefix}MAX_LM 3")
    w(f"#define {prefix}MDCT_N 1920\n#define {prefix}COMB_MINPERIOD 15\n#define {prefix}COMB_MAXPERIOD 1024\n")
    w("/* C++ translation units get constexpr tables: kernels that index them with compile-time")
    w(" * constants receive the values as instruction immediates. */")
    w(f"#ifdef __cplusplus\n#define {prefix}TABLE static constexpr\n#else\n#define {prefix}TABLE static const\n#endif\n")

    def arr(ctype, name, vals, fmt, per=8):
        w(f"{prefix}TABLE {ctype} {prefix}{name}[{len(vals)}] = {{")
        for i in range(0, len(vals), per):
            w("  " + ", ".join(fmt(v) for v in vals[i:i + per]) + ",")
        w("};\n")

    arr("float", "TRIG", trig, fhex, 6)
    arr("float", "WINDOW", win, fhex, 6)
    flat = [c for p in tw for c in p]
    w("/* interleaved (re, im) */")
    arr("float", "TWIDDLES", flat, fhex, 6)
    for n in (480, 240, 120, 60):
        arr("uint16_t", f"BITREV_{n}", bitrev_table(n), str, 16)
        arr("uint8_t", f"FFT_FACTORS_{n}", FACTORS[n] + [0] * (16 - len(FACTORS[n])), str, 16)
    arr("uint16_t", "PVQ_U_ROW", rows, str, 15)
    arr("uint32_t", "PVQ_U_DATA", data, lambda v: f"{v}u", 8)
    arr("uint8_t", "E_BANDS", E_BANDS, str, 22)
    arr("uint8_t", "LOG_N", LOG_N, str, 21)
    w(f"#define {prefix}NB_ALLOC_VECTORS {NB_ALLOC_VECTORS}")
    arr("uint8_t", "ALLOC_VECTORS", ALLOC_VECTORS, str, 21)
    arr("int16_t", "CACHE_INDEX", CACHE_INDEX, str, 21)
    arr("uint8_t", "CACHE_BITS", CACHE_BITS, str, 24)
    arr("uint8_t", "CACHE_CAPS", CACHE_CAPS, str, 21)
    arr("uint8_t", "LOG2_FRAC_TABLE", LOG2_FRAC_TABLE, str, 24)
    sched = synth_schedule()
    w("/* SYNTH-CELT/1 PVQ schedule [LM][band] = {part size n, parts, pulses K}; n==1: one sign bit */")
    w(f"static const uint8_t {prefix}SYNTH_SCHED[4][21][3] = {{")
    for row in sched:
        w("  {" + ", ".join("{%d,%d,%d}" % t for t in row) + "},")
    w("};\n")
    arr("float", "COMB_GAINS", [f32(g / 32768.0) for g in COMB_GAINS_Q15], fhex, 3)
    # SILK output resampler (RFC 6716 4.2.9: not normative, "any resampler"): polyphase windowed-sinc interpolators from the
    # internal rates 8/12/16/24 kHz to 48 kHz.  Factor L, 8 taps per phase, prototype = sinc at 0.45 fs_in x Kaiser(beta 8),
    # each phase normalised to unity DC gain.  Stored [L][8]: out[L i + p] = sum_j h[p][j] x[i - j].
    for up in (2, 3, 4, 6):
        w(f"/* {48 // up} kHz -> 48 kHz: {up} phases x 8 taps */")
        arr("float", f"SILK_UP{up}", [f32(v) for ph in silk_up_filter(up) for v in ph], fhex, 8)
    w("/* SYNTH-SILK/1 (DESIGN.md 3c): subframe gain 2^(1 + i*11/63) in Q10; LTP codebook [8][5] in Q14; symbol models */")
    arr("int32_t", "SILK_GAIN_Q10", [int(round(1024.0 * 2.0 ** (1.0 + i * 11.0 / 63.0))) for i in range(64)], str, 8)
    arr("int16_t", "SILK_LTP_Q14", silk_ltp_filters(), str, 5)
    arr("uint8_t", "SILK_TYPE_ICDF", SILK_TYPE_ICDF, str, 16)
    arr("uint8_t", "SILK_DELTA_GAIN_ICDF", SILK_DELTA_GAIN_ICDF, str, 16)
    arr("uint8_t", "SILK_CONTOUR_ICDF", SILK_CONTOUR_ICDF, str, 16)
    arr("uint8_t", "SILK_LTP_ICDF", SILK_LTP_ICDF, str, 16)
    arr("uint8_t", "SILK_PULSES_ICDF", SILK_PULSES_ICDF, str, 9)
    w("/* 2^(j/512), j = 0..511, rounded to f32: the fractional part of a band energy (SYNTH-CELT/2 denormalisation); */")
    w("/* the crate's fast_exp2 (src/math.rs:17-19) goes through libm's exp, which no two platforms round alike */")
    arr("float", "EXP2_Q9", [f32(2.0 ** (j / 512.0)) for j in range(512)], fhex, 6)
    w(f"#endif /* {guard} */")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        f.write("\n".join(L) + "\n")


if __name__ == "__main__":
    emit(os.path.join(ROOT, "oracle", "oracle_tables.h"), "ORC_", "ORACLE_TABLES_H")
    emit(os.path.join(ROOT, "opus-native_b200", "csrc", "opn_tables.h"), "OPN_", "OPN_TABLES_H")
    print("tables written")
