"""CPU-only: pins the oracle (oracle/gfp_oracle.c) to the reference's golden values and to stored outputs of the
unmodified reference templates.  Citations: SURVEY.md section 8c."""
import json
import os

import numpy as np
import pytest

import oracle_lib as ol

G = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "survey_8c.json")))
V = np.load(os.path.join(os.path.dirname(__file__), "golden", "vectors.npz"))
R = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_outputs.json")))
P = 0xFFF00001


def test_field_constants(oracle):
    for k, v in G["gf_root"].items():
        assert oracle.oracle_gf_root(1 << int(k)) == v
    for k, v in G["gf_inv_pow2"].items():
        assert oracle.oracle_gf_inv(1 << int(k)) == v
    assert oracle.oracle_gf_root(2) == P - 1                      # main.cpp:314
    for a, b, c in G["gf_mul"]:
        assert oracle.oracle_gf_mul(a, b) == c and oracle.oracle_gf_mul32(a, b) == c
    for a, b, c in G["gf_add"]:
        assert oracle.oracle_gf_add(a, b) == c
    for a, b, c in G["gf_sub"]:
        assert oracle.oracle_gf_sub(a, b) == c


def test_gf_mul_known_answers(oracle):
    """Test_GF_Mul (main.cpp:95-115): GF_Mul(i,j) == (uint64(i)*j) % P, descending from P-1, plus random pairs."""
    rng = np.random.default_rng(1)
    xs = list(range(P - 1, P - 40, -1)) + [0, 1, 2, 0x100000, 0xFFFFF] + rng.integers(0, P, 200).tolist()
    for i in xs[:60]:
        for j in xs[:60]:
            want = (i * j) % P
            assert oracle.oracle_gf_mul(i, j) == want
            assert oracle.oracle_gf_mul32(i, j) == want


def test_gf_inv_sample(oracle):
    """Test_GF_Inv (main.cpp:25-38) on a sample: x * x^-1 == 1."""
    rng = np.random.default_rng(2)
    for x in [1, 2, 3, P - 1, P - 2] + rng.integers(1, P, 300).tolist():
        assert oracle.oracle_gf_mul(x, oracle.oracle_gf_inv(x)) == 1


def test_tiny_transforms(oracle):
    a = np.array([[1], [2], [3], [4]], dtype=np.uint32)
    assert ol.o_ntt(oracle, a, False).ravel().tolist() == G["ntt4_fwd"]
    assert ol.o_ntt(oracle, a, True).ravel().tolist() == G["ntt4_inv"]
    a = np.arange(1, 9, dtype=np.uint32).reshape(8, 1)
    assert ol.o_ntt(oracle, a, False).ravel().tolist() == G["ntt8_fwd"]


@pytest.mark.parametrize("L", [7, 10, 11, 12])
def test_ntt_hash_goldens(oracle, L):
    h0, h1 = G["ntt_fillA_4096B"][str(L)]
    a = ol.fill_A(oracle, 1 << L, 1024)
    assert ol.ohash(oracle, a) == h0
    assert ol.ohash(oracle, ol.o_ntt(oracle, a, False)) == h1


def test_ntt_small_block_goldens_and_slow_ntt(oracle):
    for L, S, h in G["ntt_small_blocks"]:
        a = ol.fill_A(oracle, 1 << L, S)
        assert ol.ohash(oracle, ol.o_ntt(oracle, a, False)) == h
    # Slow_NTT (the definition, ntt.cpp:451-483) agrees with the fast oracle
    a = ol.fill_B(oracle, 64, 5)
    b = a.copy(); oracle.oracle_slow_ntt(b.ctypes.data, 64, 5, 0)
    assert np.array_equal(b, ol.o_ntt(oracle, a, False))
    b = a.copy(); oracle.oracle_slow_ntt(b.ctypes.data, 64, 5, 1)
    assert np.array_equal(b, ol.o_ntt(oracle, a, True))


def test_published_hash_pair(oracle):
    """Benchmarks.md:491-507: N=2^20, SIZE=32 bytes: original 2679569933 -> after NTT 1187104119."""
    a = ol.fill_A(oracle, 1 << 20, 8)
    assert ol.ohash(oracle, a) == G["published_ntt_2p20_32B"][0]
    assert ol.ohash(oracle, ol.o_ntt(oracle, a, False)) == G["published_ntt_2p20_32B"][1]


def test_encode_hash_goldens(oracle):
    for fill, key in ((ol.fill_A, "encode_fillA"), (ol.fill_B, "encode_fillB")):
        for L, S, h0, h1 in G[key]:
            if L > 16:
                continue                      # the 2^19 goldens are checked on the GPU (tests/test_gpu_parity.py)
            a = fill(oracle, 1 << L, S)
            assert ol.ohash(oracle, a) == h0
            assert ol.ohash(oracle, ol.o_encode(oracle, a)) == h1


def test_encode_matches_definition(oracle):
    """SURVEY 8a13: parity[j] = f(root_2N^(2j+1)), f interpolating data[i] at root_2N^(2i)."""
    for L in (1, 3, 5):
        a = ol.fill_B(oracle, 1 << L, 3)
        want = np.empty_like(a)
        oracle.oracle_rs_encode_by_definition(a.ctypes.data, want.ctypes.data, 1 << L, 3)
        assert np.array_equal(ol.o_encode(oracle, a), want)


def test_reference_vectors(oracle):
    """Full output buffers written by the unmodified reference (tests/golden/make_goldens.py)."""
    for key in V.files:
        if not key.startswith("in_"):
            continue
        L, S = map(int, key.split("_")[1:])
        x = V[key]
        assert np.array_equal(ol.o_ntt(oracle, x, False), V["ntt0_%d_%d" % (L, S)])
        assert np.array_equal(ol.o_ntt(oracle, x, True), V["ntt1_%d_%d" % (L, S)])
        assert np.array_equal(ol.o_encode(oracle, x), V["enc_%d_%d" % (L, S)])


def test_roundtrip_and_linearity(oracle):
    a = ol.fill_B(oracle, 256, 7)
    back = ol.o_ntt(oracle, ol.o_ntt(oracle, a, False), True).astype(np.uint64)
    inv = oracle.oracle_gf_inv(256)
    assert np.array_equal((back * inv) % P, a)
    b = ol.fill_A(oracle, 256, 7)
    s = ((a.astype(np.uint64) + b) % P).astype(np.uint32)
    es = ol.o_encode(oracle, s).astype(np.uint64)
    assert np.array_equal(es, (ol.o_encode(oracle, a).astype(np.uint64) + ol.o_encode(oracle, b)) % P)


def test_against_compiled_reference(oracle):
    """Outputs of the unmodified reference templates, stored by tests/golden/make_goldens.py: field operations on random
    pairs, and SHA-256 digests of MFA_NTT (both directions) and the encode on fill B at orders that take the flat, 2-D and
    cube paths of MFA_NTT."""
    for x, y, mul, add, sub in R["gf_pairs"]:
        assert (oracle.oracle_gf_mul(x, y), oracle.oracle_gf_add(x, y), oracle.oracle_gf_sub(x, y)) == (mul, add, sub)
    for t in R["transforms"]:
        a = ol.fill_B(oracle, 1 << t["L"], t["S"])
        assert ol.sha256(a) == t["input"]
        for inv in (0, 1):
            assert ol.sha256(ol.o_ntt(oracle, a, bool(inv))) == t["ntt%d" % inv], (t["L"], t["S"], inv)
        assert ol.sha256(ol.o_encode(oracle, a)) == t["encode"], (t["L"], t["S"])
