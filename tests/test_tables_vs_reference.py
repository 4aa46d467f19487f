"""The tables tools/gen_tables.py recomputes from formulas are bit-identical to the literals in the reference
crate, stored in tests/golden/reference_tables.json (f32 bit patterns; tests/golden/make_golden.py extracts them
from the crate's source).  The stored values are those the generator produced while this test still read the
crate's source directly and found every table bit-identical."""
import importlib.util
import json
import os
import struct

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_tables.json")))


def _gen():
    spec = importlib.util.spec_from_file_location("gen_tables", os.path.join(ROOT, "tools", "gen_tables.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _bits(x):
    return struct.unpack("<I", struct.pack("<f", x))[0]


def _is_zero(bits):
    return bits & 0x7FFFFFFF == 0


def test_trig_bit_identical():
    g = _gen()
    ref = REF["TRIG"]
    mine = g.trig_table()
    assert len(ref) == len(mine) == 1800
    assert ref == [_bits(b) for b in mine]


def test_window_bit_identical():
    g = _gen()
    ref = REF["WINDOW"]
    mine = g.window_table()
    assert len(ref) == len(mine) == 120
    assert ref == [_bits(b) for b in mine]


def test_twiddles_bit_identical():
    g = _gen()
    pairs = REF["TWIDDLES"]
    mine = g.twiddle_table()
    assert len(pairs) == len(mine) == 480
    for (r, i), (mr, mi) in zip(pairs, mine):
        assert r == _bits(mr) or (_is_zero(r) and mr == 0.0)
        assert i == _bits(mi) or (_is_zero(i) and mi == 0.0)


@pytest.mark.parametrize("n", [480, 240, 120, 60])
def test_bitrev_identical(n):
    g = _gen()
    assert REF[f"BITREV_{n}"] == g.bitrev_table(n)


def test_fft_factors_identical():
    g = _gen()
    found = REF["FFT_FACTORS"]
    assert len(found) == 4
    for nfft, fac in found.items():
        mine = g.FACTORS[int(nfft)]
        assert fac[: len(mine)] == mine and not any(fac[len(mine):])


def test_pvq_u_identical():
    g = _gen()
    rows, data = g.pvq_tables()
    assert rows == REF["CELT_PVQ_U_ROW"]
    assert data == REF["CELT_PVQ_U_DATA"] and len(data) == 1272


def test_allocation_tables_identical():
    g = _gen()
    for name, mine in (("ALLOC_VECTORS", g.ALLOC_VECTORS), ("CACHE_INDEX", g.CACHE_INDEX), ("CACHE_BITS", g.CACHE_BITS), ("CACHE_CAPS", g.CACHE_CAPS)):
        assert REF[name] == mine, name
    assert len(g.ALLOC_VECTORS) == 231 and len(g.CACHE_INDEX) == 105 and len(g.CACHE_BITS) == 392 and len(g.CACHE_CAPS) == 168


def test_mode_constants_identical():
    g = _gen()
    assert REF["E_BANDS"] == g.E_BANDS and REF["LOG_N"] == g.LOG_N
    assert REF["GAINS"] == [_bits(g.f32(q / 32768.0)) for q in g.COMB_GAINS_Q15]
