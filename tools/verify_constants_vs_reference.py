#!/usr/bin/env python
"""Dev-time check (needs /root/reference; never runs on the GPU box): every constant the oracle
derives from a closed form equals, bit for bit, the f32 the reference's decimal literal parses to.

Rust parses a float literal to the nearest f32 (correctly rounded); numpy.float32(float(str)) is
double rounding but cannot differ unless the decimal sits within 2^-53 relative of an f32 tie,
which a 16-19 digit literal of an irrational never does.
"""
import ctypes
import os
import re
import sys

import numpy as np

REF = "/root/reference"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def literals(path, name):
    src = open(os.path.join(REF, path)).read()
    m = re.search(r"const " + name + r": \[f32; \d+\] = \[(.*?)\];", src, re.S)
    body = re.sub(r"//.*", "", m.group(1))
    out = []
    for tok in body.replace("\n", " ").split(","):
        tok = tok.strip().replace("_", "")
        if not tok:
            continue
        if tok == "std::f32::consts::SQRT2" or tok.endswith("SQRT2"):
            out.append(np.float32(np.sqrt(np.float64(2.0))))
        else:
            out.append(np.float32(float(tok)))
    return np.array(out, dtype=np.float32)


def main():
    lib = ctypes.CDLL(os.path.join(ROOT, "oracle/_build/liboracle.so"))
    lib.oracle_mp3_tables.restype = ctypes.c_size_t
    n = lib.oracle_mp3_tables(None, 0)
    buf = np.zeros(n, dtype=np.float32)
    lib.oracle_mp3_tables(buf.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(n))
    off = {}
    pos = 0
    for name, k in [("synth_d", 512), ("imdct_win", 144), ("half_cos12", 36), ("cs", 8), ("ca", 8),
                    ("is1", 14), ("is2", 128), ("dct_iv_scale", 18), ("sdct18_scale", 9),
                    ("sdct9_d", 7), ("lee16", 16), ("lee8", 8), ("lee4", 4), ("lee2", 2), ("lee1", 1)]:
        off[name] = buf[pos:pos + k]
        pos += k
    assert pos == n
    bad = 0

    def check(label, mine, ref):
        nonlocal bad
        same = mine.view(np.uint32) == ref.view(np.uint32)
        print(f"{label:28s} {int(same.sum())}/{len(ref)} bit-identical")
        if not same.all():
            bad += 1
            for i in np.nonzero(~same)[0]:
                print("   idx", i, repr(mine[i]), repr(ref[i]))

    syn = "symphonia-bundle-mp3/src/synthesis.rs"
    hyb = "symphonia-bundle-mp3/src/layer3/hybrid_synthesis.rs"
    src = open(os.path.join(REF, syn)).read()
    m = re.search(r"static SYNTHESIS_D: \[f32; 512\] = \[(.*?)\];", src, re.S)
    d = np.array([np.float32(float(v)) for v in m.group(1).replace("\n", " ").split(",") if v.strip()],
                 dtype=np.float32)
    check("SYNTHESIS_D", off["synth_d"], d)
    check("COS_16", off["lee16"], literals(syn, "COS_16"))
    check("COS_8", off["lee8"], literals(syn, "COS_8"))
    check("COS_4", off["lee4"], literals(syn, "COS_4"))
    check("COS_2", off["lee2"], literals(syn, "COS_2"))
    m = re.search(r"const COS_1: f32 = ([0-9._]+);", src)
    check("COS_1", off["lee1"], np.array([np.float32(float(m.group(1).replace("_", "")))], dtype=np.float32))
    hsrc = open(os.path.join(REF, hyb)).read()
    scales = re.findall(r"const SCALE: \[f32; (\d+)\] = \[(.*?)\];", hsrc, re.S)
    for cnt, body in scales:
        body = re.sub(r"//.*", "", body)
        vals = []
        for tok in body.replace("\n", " ").split(","):
            tok = tok.strip().replace("_", "")
            if not tok:
                continue
            vals.append(np.float32(np.sqrt(2.0)) if "SQRT2" in tok else np.float32(float(tok)))
        vals = np.array(vals, dtype=np.float32)
        check(f"SCALE[{cnt}]", off["dct_iv_scale"] if cnt == "18" else off["sdct18_scale"], vals)
    check("sdct9 D", off["sdct9_d"], literals(hyb, "D"))

    # band tables
    csrc = open(os.path.join(REF, "symphonia-bundle-mp3/src/layer3/common.rs")).read()
    hdr = open(os.path.join(ROOT, "oracle/mp3_iso_data.h")).read()

    def ref_tab(name):
        m = re.search(name + r".*?= \[(.*?)\n\];", csrc, re.S)
        body = re.sub(r"//.*", "", m.group(1))
        return [[int(x) for x in g.replace("\n", " ").split(",") if x.strip()]
                for g in re.findall(r"\[(.*?)\]", body, re.S)]

    def my_tab(name):
        m = re.search(name + r"\[9\]\[\d+\] = \{(.*?)\n\};", hdr, re.S)
        body = re.sub(r"//.*", "", m.group(1))
        return [[int(x) for x in g.split(",") if x.strip()] for g in re.findall(r"\{(.*?)\}", body, re.S)]

    for rname, mname in [("SFB_LONG_BANDS", "kLongEdges"), ("SFB_SHORT_BANDS", "kShortEdges"),
                         ("SFB_MIXED_BANDS", "kMixedEdges")]:
        r, mm = ref_tab(rname), my_tab(mname)
        ok = all(a == b[:len(a)] and not any(b[len(a):]) for a, b in zip(r, mm)) and len(r) == len(mm)
        print(f"{rname:28s} {'OK' if ok else 'MISMATCH'}")
        bad += 0 if ok else 1
    # the mixed-block switch points and band counts (tests/_mp3_f64_model.py reads them from the header too)
    ref_switch = [int(x) for x in re.search(r"SFB_MIXED_SWITCH_POINT: \[usize; 9\] = \[(.*?)\];", csrc).group(1).split(",")]
    my_count, my_switch = ([int(x) for x in re.search(name + r"\[9\] = \{(.*?)\};", hdr).group(1).split(",")]
                           for name in ("kMixedCount", "kMixedSwitch"))
    ok = my_switch == ref_switch and my_count == [len(r) for r in ref_tab("SFB_MIXED_BANDS")]
    print(f"{'SFB_MIXED_SWITCH_POINT':28s} {'OK' if ok else 'MISMATCH'}")
    bad += 0 if ok else 1
    print("FAILED" if bad else "ALL CONSTANTS MATCH THE REFERENCE")
    return 1 if bad else 0




def verify_fft_literals():
    """The level-16 / level-32 twiddles the oracle and the product compute as (cos, -sin) in f64 equal the
    reference's 20-digit literals (symphonia-core/src/dsp/fft/no_simd.rs:309-323, :376-382) bit for bit,
    and the Vorbis inverse-dB table equals the reference's 8-digit literals."""
    lib = ctypes.CDLL(os.path.join(ROOT, "oracle/_build/liboracle.so"))
    src = open(os.path.join(REF, "symphonia-core/src/dsp/fft/no_simd.rs")).read()
    bad = 0
    for fn, size in (("fft32", 32), ("fft16", 16)):
        body = src[src.index(f"fn {fn}("):]
        body = body[:body.index("\n}\n")]
        lits = re.findall(r"complex!\((-?[0-9.]+), (-?[0-9.]+)\) \* x1\[(\d+)\]", body)
        assert lits, fn
        for re_s, im_s, k in lits:
            out = (ctypes.c_float * 2)()
            lib.oracle_fft_twiddle(size, int(k), out)
            ok = np.float32(out[0]) == np.float32(float(re_s)) and np.float32(out[1]) == np.float32(float(im_s))
            bad += 0 if ok else 1
            if not ok:
                print("  mismatch", fn, k, out[0], out[1], re_s, im_s)
        print(f"{fn} literal twiddles          {len(lits)} checked")
    vsrc = open(os.path.join(REF, "symphonia-codec-vorbis/src/floor.rs")).read()
    m = re.search(r"static FLOOR1_INVERSE_DB_TABLE: \[f32; 256\] = \[(.*?)\];", vsrc, re.S)
    vals = [np.float32(float(v.strip().replace("_", ""))) for v in re.sub(r"//.*", "", m.group(1)).replace("\n", " ").split(",") if v.strip()]
    lib.oracle_vorbis_inverse_db.restype = ctypes.c_float
    same = sum(np.float32(lib.oracle_vorbis_inverse_db(i)) == vals[i] for i in range(256))
    print(f"FLOOR1_INVERSE_DB_TABLE       {same}/256 bit-identical")
    bad += 0 if same == 256 else 1
    return bad


if __name__ == "__main__":
    rc = main()
    rc |= 1 if verify_fft_literals() else 0
    sys.exit(rc)
