#!/usr/bin/env python3
"""Extract golden data from the reference crate's source tree (hasenbanck/opus-native):

  tests/golden/reference_kats.json    the known-answer vectors of the crate's own unit tests
  tests/golden/reference_tables.json  the crate's literal constant tables (float tables as f32 bit patterns)

Usage: python tests/golden/make_golden.py <reference crate>/src
The JSON files are committed, so the tests that read them need no copy of the reference.

Sources (relative to the crate's src/):
  range_coder/mod.rs:155-188   test_tell / test_tell_frac / test_tell_frac_limits literals
  celt/pvc.rs:439-451          test_pvq_v literals
  celt/comb_filter/mod.rs:207-224  TEST_VECTOR1 / TEST_VECTOR2 (+ the test's parameters :197-204)
  lib.rs:641-651               TEST_PACKET_* byte strings
  celt/mdct.rs, celt/mode.rs, celt/kiss_fft.rs, celt/pvc.rs, celt/comb_filter/mod.rs: the tables
                               tests/test_tables_vs_reference.py compares tools/gen_tables.py with
"""
import json
import os
import re
import struct
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "reference_kats.json")
OUT_TABLES = os.path.join(HERE, "reference_tables.json")
NUM = r"-?\d+\.\d+(?:e-?\d+)?"
TABLES_NOTE = ("Literal tables of the reference crate (hasenbanck/opus-native: celt/mdct.rs TRIG, celt/mode.rs WINDOW, E_BANDS, "
               "LOG_N and the allocation data, celt/kiss_fft.rs TWIDDLES_480000_960, BITREV_* and the factor lists, celt/pvc.rs "
               "CELT_PVQ_U_*, celt/comb_filter/mod.rs GAINS). Float tables hold f32 bit patterns.")


def f32_bits(x):
    return struct.unpack("<I", struct.pack("<f", x))[0]


def write_tables(tables, path=OUT_TABLES):
    """One line per table, so that a change to one table is one line of diff."""
    body = ",\n".join(f" {json.dumps(k)}: {json.dumps(v)}" for k, v in [("_note", TABLES_NOTE)] + list(tables.items()))
    with open(path, "w") as f:
        f.write("{\n" + body + "\n}\n")


def extract_tables(ref):
    def read(p):
        return open(os.path.join(ref, p)).read()

    def block(path, start_pat):
        """The lines after the first line matching start_pat, up to the closing `];`, comments dropped."""
        out, on = [], False
        for line in read(path).split("\n"):
            if re.search(start_pat, line):
                on = True
                continue
            if on:
                if re.match(r"^\s*\];", line):
                    break
                out.append(line.split("//")[0])
        return "\n".join(out)

    t = {}
    t["TRIG"] = [f32_bits(float(s)) for s in re.findall(NUM, block("celt/mdct.rs", r"const TRIG"))]
    t["WINDOW"] = [f32_bits(float(s)) for s in re.findall(NUM, block("celt/mode.rs", r"const WINDOW"))]
    pairs = re.findall(r"r:\s*(" + NUM + r"),\s*i:\s*(" + NUM + ")", block("celt/kiss_fft.rs", r"const TWIDDLES_480000_960"))
    t["TWIDDLES"] = [[f32_bits(float(r)), f32_bits(float(i))] for r, i in pairs]
    for n in (480, 240, 120, 60):
        t[f"BITREV_{n}"] = [int(s) for s in re.findall(r"\d+", block("celt/kiss_fft.rs", rf"const BITREV_{n}:"))]
    found = re.findall(r"nfft: (\d+),.*?factors: \[([^\]]*)\]", read("celt/kiss_fft.rs"), flags=re.S)
    t["FFT_FACTORS"] = {nfft: [int(x) for x in fac.split(",") if x.strip()] for nfft, fac in found}
    t["CELT_PVQ_U_ROW"] = [int(s) for s in re.findall(r"\d+", block("celt/pvc.rs", r"const CELT_PVQ_U_ROW"))]
    t["CELT_PVQ_U_DATA"] = [int(s) for s in re.findall(r"\d+", block("celt/pvc.rs", r"const CELT_PVQ_U_DATA"))]
    for name in ("ALLOC_VECTORS", "CACHE_INDEX", "CACHE_BITS", "CACHE_CAPS"):
        t[name] = [int(x) for x in re.findall(r"-?\d+", block("celt/mode.rs", rf"const {name}:"))]
    t["E_BANDS"] = [int(s) for s in re.findall(r"\d+", block("celt/mode.rs", r"const E_BANDS"))]
    t["LOG_N"] = [int(s) for s in re.findall(r"\d+", block("celt/mode.rs", r"const LOG_N"))]
    t["GAINS"] = [f32_bits(float(s)) for s in re.findall(NUM, block("celt/comb_filter/mod.rs", r"const GAINS"))]
    return t


def main(ref):
    def read(p):
        return open(os.path.join(ref, p)).read()

    kats = {}
    rc = read("range_coder/mod.rs")
    tell = re.findall(r"TellImpl \{ bits_total: (\w+|u32::MAX), range: (\w+|u32::MAX) \}\.(tell|tell_frac)\(\), (\w+)\)", rc)

    def num(s):
        return 0xFFFFFFFF if s == "u32::MAX" else int(s, 0)

    kats["tell"] = [[num(a), num(b), num(d)] for a, b, f, d in tell if f == "tell"]
    kats["tell_frac"] = [[num(a), num(b), num(d)] for a, b, f, d in tell if f == "tell_frac"]
    m = re.search(r"entropy - ([\d.]+)\)", rc)
    kats["simple_uint_bits"] = {
        "entropy": float(m.group(1)),
        "tell_frac_over_8": float(re.search(r"-3\.0\) - ([\d.]+)\)", rc).group(1)),
        "range_bytes": int(re.search(r"range_bytes\(\), (\d+)\);\n\n        drop", rc).group(1)),
    }
    pvc = read("celt/pvc.rs")
    kats["pvq_v"] = [[int(a), int(b), int(c)] for a, b, c in re.findall(r"assert_eq!\(pvq_v\((\d+), (\d+)\), (\d+)\)", pvc)]
    pn = re.search(r"let pn: \[u32; 22\] = \[([^\]]*)\]", pvc).group(1)
    pk = re.search(r"let pk_max: \[u32; 22\] = \[([^\]]*)\]", pvc).group(1)
    kats["pvc_pn"] = [int(x) for x in pn.replace("\n", " ").split(",") if x.strip()]
    kats["pvc_pk_max"] = [int(x) for x in pk.replace("\n", " ").split(",") if x.strip()]
    comb = read("celt/comb_filter/mod.rs")
    for name in ("TEST_VECTOR1", "TEST_VECTOR2"):
        blk = re.search(name + r": &\[f32; N\] = &\[([^\]]*)\]", comb).group(1)
        kats["comb_" + name.lower()] = [float(x) for x in blk.replace("\n", " ").split(",") if x.strip()]
    consts = dict(re.findall(r"const (T0|T1|SIZE|N|OVERLAP): usize = (\d+);", comb))
    kats["comb_params"] = {k: int(v) for k, v in consts.items()}
    kats["comb_params"]["G0"] = float(re.search(r"const G0: f32 = ([\d.]+);", comb).group(1))
    kats["comb_params"]["G1"] = float(re.search(r"const G1: f32 = ([\d.]+);", comb).group(1))
    lib = read("lib.rs")
    for name in ("SINGLE", "CBR", "VBR", "INVALID"):
        blk = re.search(r"TEST_PACKET_" + name + r": &\[u8\] = &\[([^\]]*)\]", lib).group(1)
        kats["packet_" + name.lower()] = [int(x, 0) for x in blk.replace("\n", " ").split(",") if x.strip()]
    with open(OUT, "w") as f:
        json.dump(kats, f, indent=1)
    print("wrote", OUT, {k: (len(v) if hasattr(v, "__len__") else v) for k, v in kats.items()})
    tables = extract_tables(ref)
    write_tables(tables)
    print("wrote", OUT_TABLES, {k: len(v) for k, v in tables.items()})


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit("usage: make_golden.py <reference crate>/src")
    main(sys.argv[1])
