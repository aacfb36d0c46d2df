"""Regenerates / cross-checks tests/golden/survey_8c.json, vectors.npz and reference_outputs.json against the reference
compiled in oracle/_ref.

Needs the reference sources when oracle/_ref is built (oracle/Makefile, REF=<path>).  Usage: python tests/golden/make_goldens.py [--write]
Without --write it only verifies that the committed files match what the reference computes here.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import oracle_lib as ol  # noqa: E402


def main():
    o, r = ol.load_oracle(), ol.load_ref()
    assert r is not None, "oracle/_ref/libfastecc_ref.so missing (needs /root/reference)"
    g = json.load(open(os.path.join(HERE, "survey_8c.json")))
    bad = 0

    def chk(name, got, want):
        nonlocal bad
        if got != want:
            bad += 1
            print("MISMATCH", name, got, want)

    for k, v in g["gf_root"].items():
        chk("root" + k, r.ref_gf_root(1 << int(k)), v)
    for k, v in g["gf_inv_pow2"].items():
        chk("inv" + k, r.ref_gf_inv(1 << int(k)), v)
    for L, (h0, h1) in g["ntt_fillA_4096B"].items():
        L = int(L)
        if L > 16 and "--big" not in sys.argv:
            continue
        a = ol.fill_A(o, 1 << L, 1024)
        chk("ntt h0 %d" % L, ol.ohash(o, a), h0)
        r.ref_mfa_ntt_flat(a.ctypes.data, 1 << L, 1024, 0)
        chk("ntt h1 %d" % L, ol.ohash(o, a), h1)
    for fill, key in ((ol.fill_A, "encode_fillA"), (ol.fill_B, "encode_fillB")):
        for L, S, h0, h1 in g[key]:
            if L > 16 and "--big" not in sys.argv:
                continue
            a = fill(o, 1 << L, S)
            chk("enc h0 %d %d" % (L, S), ol.ohash(o, a), h0)
            r.ref_rs_encode_flat(a.ctypes.data, 1 << L, S)
            chk("enc h1 %d %d" % (L, S), ol.ohash(o, a), h1)
    # full-buffer vectors (not just hashes) produced by the reference itself, committed as a small fixture
    vec = {}
    for L, S in ((1, 4), (2, 1), (2, 8), (3, 8), (4, 8), (6, 8), (8, 8), (10, 4), (11, 4), (5, 13)):
        N = 1 << L
        x = ol.fill_B(o, N, S)
        vec["in_%d_%d" % (L, S)] = x.copy()
        for inv in (0, 1):
            y = x.copy(); r.ref_mfa_ntt_flat(y.ctypes.data, N, S, inv); vec["ntt%d_%d_%d" % (inv, L, S)] = y
        y = x.copy(); r.ref_rs_encode_flat(y.ctypes.data, N, S); vec["enc_%d_%d" % (L, S)] = y
    path = os.path.join(HERE, "vectors.npz")
    if "--write" in sys.argv:
        np.savez_compressed(path, **vec)
        print("wrote", path)
    else:
        old = np.load(path)
        for k, v in vec.items():
            if not np.array_equal(old[k], v):
                bad += 1
                print("MISMATCH vector", k)
    # field operations on random pairs, and digests of outputs too large to store, for tests/test_oracle.py
    rng = np.random.default_rng(3)
    out = {"gf_pairs": [], "transforms": []}
    for _ in range(200):
        x, y = int(rng.integers(0, ol.P)), int(rng.integers(0, ol.P))
        out["gf_pairs"].append([x, y, r.ref_gf_mul(x, y), r.ref_gf_add(x, y), r.ref_gf_sub(x, y)])
    for L, S in ((2, 3), (6, 17), (9, 1024), (10, 16), (11, 64), (13, 33)):     # flat / 2-D / cube paths of MFA_NTT
        a = ol.fill_B(o, 1 << L, S)
        t = {"L": L, "S": S, "input": ol.sha256(a)}
        for inv in (0, 1):
            b = a.copy(); r.ref_mfa_ntt_flat(b.ctypes.data, 1 << L, S, inv); t["ntt%d" % inv] = ol.sha256(b)
        b = a.copy(); r.ref_rs_encode_flat(b.ctypes.data, 1 << L, S); t["encode"] = ol.sha256(b)
        out["transforms"].append(t)
    path = os.path.join(HERE, "reference_outputs.json")
    if "--write" in sys.argv:
        with open(path, "w") as f:             # one entry per line
            f.write("{\n" + ",\n".join('"%s": [\n%s]' % (k, ",\n".join(json.dumps(e) for e in v)) for k, v in out.items()) + "}\n")
        print("wrote", path)
    elif json.load(open(path)) != out:
        bad += 1
        print("MISMATCH", path)
    print("goldens", "MISMATCH" if bad else "verified against the compiled reference")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
