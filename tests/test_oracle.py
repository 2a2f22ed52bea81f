"""Pins the oracle (oracle/rsx_oracle.c) before anything trusts it.

1. the reference's own known answers (tests/golden/reference_vectors.json: its tests, tutorial
   listings and README outputs -- SURVEY.md Appendix A);
2. outputs of the UNMODIFIED reference headers on seeded inputs (tests/golden/ref_outputs.json,
   made by tests/golden/make_golden.py) and, where oracle/_ref exists, the live reference;
3. an independent merge sort (no radix code) and numpy's stable sort.
CPU only.
"""
import json
import os

import numpy as np
import pytest

import pyoracle
from cases import GOLDEN_CASES, case_id, digest, make_input
from pyoracle import OrcLayout, TYPES

GOLD = os.path.join(os.path.dirname(__file__), "golden")
VEC = json.load(open(os.path.join(GOLD, "reference_vectors.json")))
REF_OUT = json.load(open(os.path.join(GOLD, "ref_outputs.json")))


def records_from_keys(layout, keys):
    """Records of layout[0] bytes: key bytes at key_offset, original position in the last 4 bytes
    (or nothing for bare keys)."""
    rb, ko, kb = layout[0], layout[1], layout[2]
    n = len(keys)
    raw = np.zeros((n, rb), dtype=np.uint8)
    for i, k in enumerate(keys):
        raw[i, ko:ko + kb] = np.frombuffer(int(k).to_bytes(kb, "little"), dtype=np.uint8)
        if rb >= kb + 4:
            raw[i, rb - 4:rb] = np.frombuffer(int(i).to_bytes(4, "little"), dtype=np.uint8)
    return raw


# ---- 1. the reference's known answers ---------------------------------------------------------

@pytest.mark.parametrize("v", VEC["value_sorts"], ids=lambda v: v["name"][:40])
def test_reference_value_vectors(oracle, v):
    L = OrcLayout(*v["layout"])
    raw = records_from_keys(v["layout"], v["keys"])
    out, rep, _ = oracle.radix_sort(raw, L)
    got_order = [int.from_bytes(out[i, -4:].tobytes(), "little") for i in range(len(v["keys"]))]
    assert got_order == v["order"]
    assert rep.result_in_aux == v["result_in_aux"]


def test_reference_float_vector(oracle):
    v = VEC["float_sort"]
    data = np.array([int(x, 16) for x in v["input_bits"]], dtype=np.uint32)
    out, rep, _ = oracle.radix_sort(data, TYPES["f32"].layout())
    assert [f"{x:08x}" for x in out] == v["output_bits"]
    assert rep.result_in_aux == v["result_in_aux"]


@pytest.mark.parametrize("v", VEC["rank_sorts"], ids=lambda v: v["name"][:40])
def test_reference_rank_vectors(oracle, v):
    L = OrcLayout(*v["layout"])
    raw = records_from_keys(v["layout"], v["keys"])
    idt = np.dtype(f"u{v['idx_bytes']}")
    ranks, rep, _ = oracle.radix_sort_rank(raw, L, idt, as_shipped=False)
    assert ranks.tolist() == v["ranks"]
    assert rep.result_in_aux == v["result_in_aux"]
    shipped, rep2, _ = oracle.radix_sort_rank(raw, L, idt, as_shipped=True)
    if v["shipped_header_agrees"]:
        assert shipped.tolist() == v["ranks"]
    else:  # the witness of radix_sort_rank.hpp:82 (SURVEY.md Appendix A4)
        assert shipped.tolist() == v["shipped_header_output"]
        assert sorted(shipped.tolist()) == list(range(len(v["keys"])))


@pytest.mark.parametrize("v", VEC["kdf"], ids=lambda v: v["ref"][:30])
def test_kdf_identities(oracle, v):
    L = OrcLayout(*v["layout"])
    raw = np.frombuffer(int(v["raw"], 16).to_bytes(L.record_bytes, "little"), dtype=np.uint8)
    assert oracle.kdf(raw, L) == int(v["derived"], 16)


# ---- 2. the unmodified reference on seeded inputs -----------------------------------------------

@pytest.mark.parametrize("c", GOLDEN_CASES, ids=case_id)
def test_oracle_matches_reference_golden(oracle, c):
    t = TYPES[c[0]]
    data = make_input(c[0], c[1], 1234, c[2], c[3], c[4])
    out, rep, _ = oracle.radix_sort(data, t.layout())
    g = REF_OUT["sort"][case_id(c)]
    assert digest(out) == g["sha256"]
    assert rep.result_in_aux == g["result_in_aux"]
    if case_id(c) in REF_OUT["sort_desc"]:
        out, rep, _ = oracle.radix_sort(data, t.layout(descending=True))
        g = REF_OUT["sort_desc"][case_id(c)]
        assert digest(out) == g["sha256"] and rep.result_in_aux == g["result_in_aux"]
    if case_id(c) in REF_OUT["rank_as_shipped"]:
        g = REF_OUT["rank_as_shipped"][case_id(c)]
        shipped, rep, _ = oracle.radix_sort_rank(data, t.layout(), np.uint32, as_shipped=True)
        assert digest(shipped) == g["sha256"] and rep.result_in_aux == g["result_in_aux"]
        fixed, rep2, _ = oracle.radix_sort_rank(data, t.layout(), np.uint32, as_shipped=False)
        assert rep2.result_in_aux == g["result_in_aux"]
        if rep2.ncols <= 1:  # the shipped header is correct exactly here
            assert digest(fixed) == g["sha256"]


@pytest.mark.parametrize("tname", ["u32", "u64", "i32", "f32", "f64", "rec8_u32", "rec16_u8"])
def test_oracle_matches_live_reference(oracle, ref, tname):
    t = TYPES[tname]
    for n, seed in [(0, 1), (1, 2), (2, 3), (1023, 4), (100000, 5)]:
        data = make_input(tname, n, seed)
        want, in_aux = ref.radix_sort(t, data)
        got, rep, _ = oracle.radix_sort(data, t.layout())
        assert got.tobytes() == want.tobytes()
        assert rep.result_in_aux == in_aux
        want, in_aux = ref.radix_sort(t, data, descending=True)
        got, rep, _ = oracle.radix_sort(data, t.layout(descending=True))
        assert got.tobytes() == want.tobytes() and rep.result_in_aux == in_aux


def test_shipped_rank_header_is_not_sorted_for_two_columns(oracle):
    """Documents the upstream bug (radix_sort_rank.hpp:82): valid permutation, not sorted.  The
    shipped header's output is pinned by its stored digest (tests/golden/ref_outputs.json)."""
    c = ("u32", 257, "uniform", (1 << 64) - 1, 0)
    t = TYPES["u32"]
    data = make_input("u32", 257, 1234)
    g = REF_OUT["rank_as_shipped"][case_id(c)]
    shipped, rep, _ = oracle.radix_sort_rank(data, t.layout(), np.uint32, as_shipped=True)
    assert digest(shipped) == g["sha256"] and rep.result_in_aux == g["result_in_aux"]  # == the reference's bytes
    assert sorted(shipped.tolist()) == list(range(257))
    assert not np.all(np.diff(data[shipped].astype(np.int64)) >= 0)
    fixed, _, _ = oracle.radix_sort_rank(data, t.layout(), np.uint32)
    assert np.all(np.diff(data[fixed].astype(np.int64)) >= 0)


# ---- 3. independent cross-checks ---------------------------------------------------------------------

@pytest.mark.parametrize("tname", list(TYPES))
@pytest.mark.parametrize("desc", [False, True])
def test_oracle_equals_stable_sort(oracle, tname, desc):
    t = TYPES[tname]
    for n, mask in [(5000, (1 << 64) - 1), (5000, 0x0F0F), (777, 0xFF00FF)]:
        data = make_input(tname, n, 77, "uniform", mask)
        L = t.layout(descending=desc)
        out, rep, _ = oracle.radix_sort(data, L)
        assert out.tobytes() == oracle.stable_sort(data, L).tobytes()
        ranks, rep2, _ = oracle.radix_sort_rank(data, L, np.uint32)
        assert ranks.astype(np.uint64).tolist() == oracle.stable_argsort(data, L).tolist()
        assert rep.result_in_aux == rep2.result_in_aux == (rep.ncols & 1)


def test_oracle_equals_numpy_stable(oracle):
    data = make_input("u32", 100000, 5, "uniform", 0xFFFFF)
    out, _, _ = oracle.radix_sort(data, TYPES["u32"].layout())
    assert np.array_equal(out, np.sort(data, kind="stable"))
    ranks, _, _ = oracle.radix_sort_rank(data, TYPES["u32"].layout(), np.uint32)
    assert np.array_equal(ranks, np.argsort(data, kind="stable").astype(np.uint32))
    f = make_input("f32", 50000, 6, "uniform", 0xBFFFFFFF)  # no NaN/Inf exponent: numpy order is total
    out, _, _ = oracle.radix_sort(f, TYPES["f32"].layout())
    assert np.array_equal(out.view(np.uint32), np.sort(f, kind="stable").view(np.uint32)) or \
        np.array_equal(out, np.sort(f, kind="stable"))


def test_oracle_edge_cases(oracle):
    L = TYPES["u32"].layout()
    for n in (0, 1):
        data = make_input("u32", n, 3)
        out, rep, _ = oracle.radix_sort(data, L)
        assert rep.early_exit == 1 and rep.result_in_aux == 0 and out.tobytes() == data.tobytes()
        ranks, rep, ib = oracle.radix_sort_rank(data, L, np.uint32)
        assert rep.result_in_aux == 0 and ranks.tolist() == list(range(n))
    # presorted and constant inputs: early exit, identity ranks in the FIRST half (radix_sort_rank.hpp:55-57)
    for dist in ("sorted", "constant"):
        data = make_input("u32", 1000, 3, dist)
        out, rep, hist = oracle.radix_sort(data, L, want_hist=True)
        assert rep.early_exit == 1 and rep.result_in_aux == 0 and out.tobytes() == data.tobytes()
        assert int(hist.sum()) == 4 * 1000
        ranks, rep, _ = oracle.radix_sort_rank(data, L, np.uint32)
        assert rep.early_exit == 1 and ranks.tolist() == list(range(1000))
    # histogram is column-major, one 256-bin block per byte of the derived key (radix_sort.hpp:40-58)
    data = make_input("i32", 4096, 8)
    _, rep, hist = oracle.radix_sort(data, TYPES["i32"].layout(), want_hist=True)
    derived = data.view(np.uint32) ^ np.uint32(0x80000000)
    for c in range(4):
        assert np.array_equal(hist[c], np.bincount((derived >> (8 * c)) & 0xFF, minlength=256).astype(np.uint64))
