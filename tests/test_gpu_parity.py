"""GPU parity tests: the CUDA path (through the C ABI in librsx.so) against the oracle and the
committed golden digests of the unmodified reference.  Bit-exact: this is integer/byte work.

Run on the B200 box: python -m pytest tests -m gpu
"""
import contextlib
import json
import os

import numpy as np
import pytest

from cases import GOLDEN_CASES, case_id, digest, make_input
from pyoracle import TYPES

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")
REF_OUT = json.load(open(os.path.join(GOLD, "ref_outputs.json")))
VEC = json.load(open(os.path.join(GOLD, "reference_vectors.json")))


@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the product has no CPU path (run with -m gpu on the GPU box)")
    return torch


def to_dev(torch, a: np.ndarray):
    """numpy (any dtype, incl. structured) -> uint8 CUDA tensor with the same bytes."""
    raw = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
    return torch.from_numpy(raw.copy()).cuda()


def kf_for(rsx, tname, descending=False):
    """KeyFunc of TYPES[tname], or of `tname` itself when it is a pyoracle.ElemType."""
    t = TYPES[tname] if isinstance(tname, str) else tname
    return rsx.KeyFunc(t.kdf_kind, descending, t.record_bytes, t.key_offset, t.key_bytes)


def gpu_sort(rsx, torch, tname, data, descending=False):
    src = to_dev(torch, data)
    aux = torch.full_like(src, 0xCD)
    rep = rsx.RsxReport()
    res = rsx.radix_sort(src, aux, None, kf_for(rsx, tname, descending), report=rep)
    torch.cuda.synchronize()
    return res.cpu().numpy(), rep, (res.data_ptr() == aux.data_ptr() and data.shape[0] > 0)


def gpu_rank(rsx, torch, tname, data, idx_dtype=np.uint32, descending=False):
    src = to_dev(torch, data)
    before = src.clone()
    n = data.shape[0]
    ib_np = np.full(2 * n, 0xEE, dtype=idx_dtype)
    ib = torch.from_numpy(ib_np.view(np.uint8).copy()).cuda().view(
        {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[np.dtype(idx_dtype).itemsize])
    rep = rsx.RsxReport()
    res = rsx.radix_sort_rank(src, ib, n, kf_for(rsx, tname, descending), report=rep)
    torch.cuda.synchronize()
    assert torch.equal(src, before), "rank sort must not modify src (const T*, radix_sort_rank.hpp:97)"
    ranks = res.cpu().numpy().view(idx_dtype)
    return ranks, rep, ib.cpu().numpy().view(idx_dtype)


@pytest.fixture(params=["single-cta", "multi-kernel"])
def both_paths(request, rsx):
    """Inputs that fit one CTA take the single-launch kernel (rsx_small.cu); run the same case
    through the multi-kernel path too, so that both stay pinned on the small goldens."""
    rsx.lib().rsx_set_option(b"small_path", 1 if request.param == "single-cta" else 0)
    yield request.param
    rsx.lib().rsx_set_option(b"small_path", 1)


# ---- golden digests of the unmodified reference --------------------------------------------------

@pytest.mark.parametrize("c", GOLDEN_CASES, ids=case_id)
def test_sort_matches_reference_golden(rsx, torch, oracle, both_paths, c):
    t = TYPES[c[0]]
    data = make_input(c[0], c[1], 1234, c[2], c[3], c[4])
    out, rep, in_aux = gpu_sort(rsx, torch, c[0], data)
    g = REF_OUT["sort"][case_id(c)]
    want, orep, hist = oracle.radix_sort(data, t.layout(), want_hist=True)
    assert out.tobytes() == want.tobytes()
    assert digest(out) == g["sha256"]
    assert int(in_aux) == g["result_in_aux"] == rep.result_in_aux
    assert rep.early_exit == orep.early_exit and rep.ncols == orep.ncols
    assert rep.live_mask == sum(1 << orep.cols[i] for i in range(orep.ncols))
    if case_id(c) in REF_OUT["sort_desc"]:
        out, rep, in_aux = gpu_sort(rsx, torch, c[0], data, descending=True)
        g = REF_OUT["sort_desc"][case_id(c)]
        assert digest(out) == g["sha256"] and int(in_aux) == g["result_in_aux"]


@pytest.mark.parametrize("c", [c for c in GOLDEN_CASES if c[1] in (2, 257, 1000, 5000, 70001)], ids=case_id)
def test_rank_matches_oracle(rsx, torch, oracle, both_paths, c):
    t = TYPES[c[0]]
    data = make_input(c[0], c[1], 1234, c[2], c[3], c[4])
    for idt in (np.uint32, np.uint64):
        ranks, rep, ib = gpu_rank(rsx, torch, c[0], data, idt)
        want, orep, oib = oracle.radix_sort_rank(data, t.layout(), idt)
        assert np.array_equal(ranks, want)
        assert rep.result_in_aux == orep.result_in_aux and rep.ncols == orep.ncols
        if orep.early_exit:  # identity in the FIRST half (radix_sort_rank.hpp:52-57)
            assert np.array_equal(ib[:c[1]], np.arange(c[1], dtype=idt))
    # where the shipped header is right (<= 1 live column / early exit) we match it bit for bit
    cid = case_id(c)
    if cid in REF_OUT["rank_as_shipped"] and orep.ncols <= 1:
        ranks, rep, _ = gpu_rank(rsx, torch, c[0], data, np.uint32)
        assert digest(ranks) == REF_OUT["rank_as_shipped"][cid]["sha256"]


# ---- the reference's own test vectors ----------------------------------------------------------------

def _records(layout, keys):
    rb, ko, kb = layout[0], layout[1], layout[2]
    raw = np.zeros((len(keys), rb), dtype=np.uint8)
    for i, k in enumerate(keys):
        raw[i, ko:ko + kb] = np.frombuffer(int(k).to_bytes(kb, "little"), dtype=np.uint8)
        if rb >= kb + 4:
            raw[i, rb - 4:rb] = np.frombuffer(int(i).to_bytes(4, "little"), dtype=np.uint8)
    return raw


@pytest.mark.parametrize("v", VEC["value_sorts"], ids=lambda v: v["name"][:40])
def test_reference_value_vectors(rsx, torch, both_paths, v):
    rb, ko, kb, kind, flags = v["layout"]
    raw = _records(v["layout"], v["keys"])
    src = torch.from_numpy(raw.reshape(-1).copy()).cuda()
    aux = torch.zeros_like(src)
    rep = rsx.RsxReport()
    res = rsx.radix_sort(src, aux, None, rsx.KeyFunc(kind, bool(flags & 1), rb, ko, kb), report=rep)
    out = res.cpu().numpy().reshape(-1, rb)
    order = [int.from_bytes(out[i, -4:].tobytes(), "little") for i in range(len(v["keys"]))]
    assert order == v["order"]
    assert rep.result_in_aux == v["result_in_aux"]
    assert (res.data_ptr() == aux.data_ptr()) == bool(v["result_in_aux"])


def test_reference_float_vector(rsx, torch, both_paths):
    v = VEC["float_sort"]
    data = np.array([int(x, 16) for x in v["input_bits"]], dtype=np.uint32).view(np.float32)
    src = torch.from_numpy(data.copy()).cuda()
    aux = torch.zeros_like(src)
    res = rsx.radix_sort(src, aux)  # default KDF picked from the dtype, like radix_tests.cpp:163
    assert [f"{x:08x}" for x in res.cpu().numpy().view(np.uint32)] == v["output_bits"]
    assert res.data_ptr() == src.data_ptr()


@pytest.mark.parametrize("v", VEC["rank_sorts"], ids=lambda v: v["name"][:40])
def test_reference_rank_vectors(rsx, torch, both_paths, v):
    rb, ko, kb, kind, flags = v["layout"]
    raw = _records(v["layout"], v["keys"])
    n = len(v["keys"])
    src = torch.from_numpy(raw.reshape(-1).copy()).cuda()
    tdt = {1: torch.uint8, 4: torch.int32}[v["idx_bytes"]]
    ib = torch.zeros(2 * n, dtype=tdt, device="cuda")
    rep = rsx.RsxReport()
    res = rsx.radix_sort_rank(src, ib, n, rsx.KeyFunc(kind, bool(flags & 1), rb, ko, kb), report=rep)
    assert res.cpu().numpy().astype(np.int64).tolist() == v["ranks"]
    assert rep.result_in_aux == v["result_in_aux"]


def test_int_then_reverse_resort(rsx, torch, oracle):
    """radix_tests.cpp:179-207: sort 50 000 ints, then re-sort the RESULT descending with
    kdf_int_reverse, passing the other buffer as aux."""
    rng = np.random.default_rng(0)
    vals = np.clip(rng.normal(-2147483648.0, 2147483647.0, 50000), -2147483648.0, 2147483647.0).astype(np.int32)
    src = torch.from_numpy(vals.copy()).cuda()
    aux = torch.zeros_like(src)
    res = rsx.radix_sort(src, aux)
    assert np.array_equal(res.cpu().numpy(), np.sort(vals, kind="stable"))
    other = aux if res.data_ptr() == src.data_ptr() else src
    res2 = rsx.radix_sort(res, other, None, rsx.default_kdf(torch.int32, descending=True))
    assert np.array_equal(res2.cpu().numpy(), np.sort(vals, kind="stable")[::-1])


# ---- halves of the path --------------------------------------------------------------------------------

@pytest.mark.parametrize("tname", ["u8", "u16", "u32", "u64", "i32", "i64", "f32", "f64", "rec8_u32", "rec16_u8", "rec16_u64"])
@pytest.mark.parametrize("n,dist,mask", [(2, "uniform", -1), (1000, "uniform", -1), (300001, "uniform", -1),
                                          (300001, "uniform", 0x00FF00FF00FF00FF), (50000, "sorted", -1),
                                          (50000, "constant", -1), (262144, "and3", -1)])
def test_histogram_kernel(rsx, torch, oracle, tname, n, dist, mask):
    t = TYPES[tname]
    data = make_input(tname, n, 99, dist, mask & ((1 << 64) - 1))
    hist, descents, rep = rsx.histogram(to_dev(torch, data), kf_for(rsx, tname))
    _, orep, ohist = oracle.radix_sort(data, t.layout(), want_hist=True)
    assert np.array_equal(hist, ohist)
    assert descents + 1 == orep.n_unsorted  # n_unsorted = n - #ordered pairs = 1 + descents
    assert rep.early_exit == orep.early_exit
    if not orep.early_exit:
        assert rep.live_mask == sum(1 << orep.cols[i] for i in range(orep.ncols))


@pytest.mark.parametrize("tname", ["u16", "u32", "u64", "i32", "i64", "f32", "f64", "rec8_u32", "rec16_u64", "rec16_f64"])
def test_histogram_column_kernel(rsx, torch, oracle, tname):
    """rsx_histogram_column: one column of the derived key's digit histogram (the multi-GPU routing
    histogram) == that column of the oracle's full histogram; descending layouts too."""
    import ctypes as C
    t = TYPES[tname]
    data = make_input(tname, 300001, 55, "and2")
    src = to_dev(torch, data)
    for desc in (False, True):
        _, _, ohist = oracle.radix_sort(data, t.layout(descending=desc), want_hist=True)
        L = rsx.RsxLayout(t.record_bytes, t.key_offset, t.key_bytes, t.kdf_kind, 1 if desc else 0)
        cols = [t.key_bytes - 1] if t.kdf_kind == 2 else range(t.key_bytes)
        for col in cols:
            out = np.zeros(256, dtype=np.uint64)
            st = rsx.lib().rsx_histogram_column(src.data_ptr(), 300001, C.byref(L), col,
                                                out.ctypes.data_as(C.POINTER(C.c_uint64)), None)
            assert st == 0
            assert np.array_equal(out, ohist[col]), (tname, desc, col)
    if t.kdf_kind == 2:  # a lower column of a float key needs the sign bit: rejected
        out = np.zeros(256, dtype=np.uint64)
        assert rsx.lib().rsx_histogram_column(src.data_ptr(), 300001, C.byref(L), 0,
                                              out.ctypes.data_as(C.POINTER(C.c_uint64)), None) == rsx.RSX_ERR_INVALID


@pytest.mark.parametrize("off", [1, 2, 3, 5])
def test_unaligned_pointers(rsx, torch, oracle, off):
    """Buffers that are element-aligned but not 16-byte aligned (head/tail path of K1)."""
    n = 100003
    data = make_input("u32", n, 7)
    base = torch.zeros(n + 8, dtype=torch.int32, device="cuda")
    base2 = torch.zeros(n + 8, dtype=torch.int32, device="cuda")
    src = base[off:off + n]
    src.copy_(torch.from_numpy(data.view(np.int32).copy()).cuda())
    aux = base2[off:off + n]
    res = rsx.radix_sort(src, aux, None, rsx.KeyFunc(rsx.KDF_UNSIGNED))
    want, _, _ = oracle.radix_sort(data, TYPES["u32"].layout())
    assert np.array_equal(res.cpu().numpy().view(np.uint32), want)


@pytest.mark.parametrize("tname,col", [("u32", 0), ("u32", 3), ("u64", 5), ("i32", 3), ("f32", 3), ("f32", 1), ("f64", 7), ("rec8_u32", 2)])
def test_single_scatter_pass_is_stable(rsx, torch, oracle, tname, col):
    """One K3 pass == one stable counting-sort pass on that column (radix_sort.hpp:83-88)."""
    t = TYPES[tname]
    n = 200001
    data = make_input(tname, n, 11, "and2")
    src = to_dev(torch, data)
    dst = torch.zeros_like(src)
    pl_src = torch.arange(n, dtype=torch.int32, device="cuda")
    pl_dst = torch.zeros_like(pl_src)
    rsx.scatter_pass(src, dst, col, kf_for(rsx, tname), pl_src, pl_dst)
    torch.cuda.synchronize()
    # vectorised derived digits
    keys = data["key"] if data.dtype.names else data
    u = keys.view(f"<u{t.key_bytes}").astype(np.uint64)
    top = np.uint64(1 << (8 * t.key_bytes - 1))
    m = np.uint64((1 << (8 * t.key_bytes)) - 1)
    if t.kdf_kind == 1:
        u = u ^ top
    elif t.kdf_kind == 2:
        u = np.where(u & top, u ^ m, u ^ top)
    digits = ((u >> np.uint64(8 * col)) & np.uint64(0xFF)).astype(np.int64)
    perm = np.argsort(digits, kind="stable")
    assert np.array_equal(pl_dst.cpu().numpy(), perm.astype(np.int32))
    assert dst.cpu().numpy().tobytes() == data[perm].tobytes()


# ---- edges --------------------------------------------------------------------------------------------------

def test_trivial_sizes(rsx, torch):
    for n in (0, 1):
        src = torch.arange(n, dtype=torch.int32, device="cuda")
        aux = torch.zeros_like(src)
        rep = rsx.RsxReport()
        res = rsx.radix_sort(src, aux, report=rep)
        assert res.data_ptr() == src.data_ptr() and rep.early_exit == 1
        ib = torch.full((2 * n + 2,), 7, dtype=torch.int32, device="cuda")
        r = rsx.radix_sort_rank(src, ib, n)
        assert r.cpu().tolist() == list(range(n))  # radix_sort_rank.hpp:28-32


def test_presorted_leaves_buffers_untouched(rsx, torch):
    n = 1 << 20
    src = torch.arange(n, dtype=torch.int32, device="cuda")
    aux = torch.full_like(src, -1)
    rep = rsx.RsxReport()
    res = rsx.radix_sort(src, aux, report=rep)
    assert rep.early_exit == 1 and res.data_ptr() == src.data_ptr()
    assert torch.equal(src, torch.arange(n, dtype=torch.int32, device="cuda"))
    assert bool((aux == -1).all())  # radix_sort.hpp:60-62: nothing written


def test_host_buffers_are_staged(rsx, torch, oracle):
    """The reference sorts host memory; host pointers go H2D -> sort -> D2H into the buffer
    the reference would have returned."""
    for mask, tname in [((1 << 64) - 1, "u32"), (0x00FFFFFF, "u32"), ((1 << 64) - 1, "u64")]:
        data = make_input(tname, 300000, 5, "uniform", mask)
        src = torch.from_numpy(data.view(np.int32 if tname == "u32" else np.int64).copy())
        aux = torch.zeros_like(src)
        rep = rsx.RsxReport()
        res = rsx.radix_sort(src, aux, None, rsx.KeyFunc(rsx.KDF_UNSIGNED), report=rep)
        want, orep, _ = oracle.radix_sort(data, TYPES[tname].layout())
        assert rep.staged == 1 and rep.result_in_aux == orep.result_in_aux
        assert res.numpy().tobytes() == want.tobytes()
        ib = torch.zeros(2 * 300000, dtype=torch.int32)
        r = rsx.radix_sort_rank(torch.from_numpy(data.view(np.int32 if tname == "u32" else np.int64).copy()), ib,
                                300000, rsx.KeyFunc(rsx.KDF_UNSIGNED))
        wr, _, _ = oracle.radix_sort_rank(data, TYPES[tname].layout(), np.uint32)
        assert np.array_equal(r.numpy().view(np.uint32), wr)


def test_error_paths(rsx, torch):
    src = torch.zeros(16, dtype=torch.int32, device="cuda")
    with pytest.raises(rsx.RsxError) as e:  # float KDF needs a 4/8-byte key
        rsx.radix_sort(src.view(torch.uint8), torch.zeros(64, dtype=torch.uint8, device="cuda"), None,
                       rsx.KeyFunc(rsx.KDF_FLOAT, False, 2, 0, 2))
    assert e.value.status == rsx.RSX_ERR_INVALID
    import ctypes as C
    res = C.c_void_p()
    L = rsx.RsxLayout(4, 0, 4, 0, 0)
    host = torch.zeros(16, dtype=torch.int32)  # host src, device aux
    st = rsx.lib().rsx_sort(host.data_ptr(), src.data_ptr(), 16, C.byref(L), C.byref(res), None, None)
    assert st == rsx.RSX_ERR_MIXED_MEMORY
    with pytest.raises(rsx.RsxError) as e:  # 300 records cannot be ranked with uint8 indices
        rsx.radix_sort_rank(torch.zeros(300, dtype=torch.int32, device="cuda"),
                            torch.zeros(600, dtype=torch.uint8, device="cuda"))
    assert e.value.status == rsx.RSX_ERR_IDX_RANGE


# ---- large sizes: size-independent properties (no CPU oracle needed) ---------------------------------------

@pytest.mark.parametrize("tname,n", [("u32", 1 << 26), ("u64", 1 << 25), ("f32", 40_000_000)])
def test_large_sort_properties(rsx, torch, tname, n):
    """sortedness (0 descents of the derived key) + multiset checksum before == after, and
    idempotence: sorting the result again is an early exit."""
    tdt = {"u32": torch.int32, "u64": torch.int64, "f32": torch.float32}[tname]
    src = torch.empty(n, dtype=tdt, device="cuda")
    aux = torch.empty_like(src)
    rsx.fill_keys(src, seed=42)
    kf = kf_for(rsx, tname)
    d0, s0, x0 = rsx.verify(src, kf)
    assert d0 > 0
    rep = rsx.RsxReport()
    res = rsx.radix_sort(src, aux, None, kf, report=rep)
    d1, s1, x1 = rsx.verify(res, kf)
    assert d1 == 0 and (s1, x1) == (s0, x0)
    assert rep.ncols == TYPES[tname].key_bytes
    other = aux if res.data_ptr() == src.data_ptr() else src
    rep2 = rsx.RsxReport()
    res2 = rsx.radix_sort(res, other, None, kf, report=rep2)
    assert rep2.early_exit == 1 and res2.data_ptr() == res.data_ptr()


def test_device_keygen_matches_host(rsx, torch, keygen):
    for dist in keygen.DISTS:
        for kb, tdt in [(4, torch.int32), (8, torch.int64)]:
            dst = torch.empty(10007, dtype=tdt, device="cuda")
            rsx.fill_keys(dst, seed=17, start=123456789, dist=dist, mask=0x00FFFFFFFFFFFF0F, orv=0x3)
            want = keygen.fill(17, 123456789, 10007, kb, dist, 0x00FFFFFFFFFFFF0F, 0x3)
            assert np.array_equal(dst.cpu().numpy().view(f"<u{kb}"), want), (dist, kb)


# ---- the n >= 2^30 code path (64-bit look-back words and offsets) -----------------------------------------

@pytest.mark.parametrize("tname", ["u32", "u64", "f32", "rec8_u32", "rec16_u64"])
def test_wide_offset_kernels_at_small_n(rsx, torch, oracle, tname):
    """radix_sort.hpp:111-113 switches to 64-bit counters at n >= 2^32; our look-back words and
    offsets go 64-bit at n >= 2^30.  force_wide runs those kernels on oracle-sized inputs."""
    t = TYPES[tname]
    data = make_input(tname, 250007, 31, "and2")
    try:
        assert rsx.lib().rsx_set_option(b"force_wide", 1) == 0
        out, rep, _ = gpu_sort(rsx, torch, tname, data)
        ranks, _, _ = gpu_rank(rsx, torch, tname, data, np.uint64)
    finally:
        rsx.lib().rsx_set_option(b"force_wide", 0)
    want, orep, _ = oracle.radix_sort(data, t.layout())
    assert out.tobytes() == want.tobytes() and rep.result_in_aux == orep.result_in_aux
    wr, _, _ = oracle.radix_sort_rank(data, t.layout(), np.uint64)
    assert np.array_equal(ranks, wr)


def test_more_than_2_pow_30_keys(rsx, torch):
    """1.2 G u32 keys (> 2^30): sortedness + multiset checksum; masked to 3 live columns so the
    result must land in aux."""
    n = 1_200_000_000
    src = torch.empty(n, dtype=torch.int32, device="cuda")
    aux = torch.empty_like(src)
    rsx.fill_keys(src, seed=9, mask=0x00FFFFFF)
    kf = rsx.KeyFunc(rsx.KDF_UNSIGNED)
    _, s0, x0 = rsx.verify(src, kf)
    rep = rsx.RsxReport()
    res = rsx.radix_sort(src, aux, None, kf, report=rep)
    d1, s1, x1 = rsx.verify(res, kf)
    assert d1 == 0 and (s1, x1) == (s0, x0)
    assert rep.ncols == 3 and res.data_ptr() == aux.data_ptr()


# ---- fused partition + exchange pass (multi-GPU building block), on one device ----------------------------

@pytest.mark.parametrize("tname,col", [("u32", 3), ("u64", 7), ("rec8_u32", 3), ("f32", 3), ("rec16_u64", 7),
                                       ("rec16_u8", 0), ("u16", 1), ("u8", 0)])
def test_scatter_pass_to_destinations(rsx, torch, oracle, tname, col):
    """rsx_scatter_pass_to with three local 'destinations': each receives exactly the records whose
    routing bucket it owns, in an order that a stable local sort turns into the oracle's order."""
    t = TYPES[tname]
    n = 300007
    data = make_input(tname, n, 21, "and2" if tname != "f32" else "uniform")
    src = to_dev(torch, data)
    L = t.layout()
    u = (data["key"] if data.dtype.names else data).view(f"<u{t.key_bytes}").astype(np.uint64)
    top = np.uint64(1 << (8 * t.key_bytes - 1))
    m = np.uint64((1 << (8 * t.key_bytes)) - 1)
    if t.kdf_kind == 2:
        u = np.where(u & top, u ^ m, u ^ top)
    digits = ((u >> np.uint64(8 * col)) & np.uint64(0xFF)).astype(np.int64)
    owner = np.zeros(256, dtype=np.int64)
    owner[40:200] = 1
    owner[200:] = 2
    counts = [int((owner[digits] == d).sum()) for d in range(3)]
    bufs = [torch.full((max(c, 1) * t.record_bytes,), 0xAB, dtype=torch.uint8, device="cuda") for c in counts]
    rsx.scatter_pass_to(src, col, owner, [b.data_ptr() for b in bufs], kf_for(rsx, tname))
    torch.cuda.synchronize()
    for d in range(3):
        sub = data[owner[digits] == d]
        got = bufs[d][: counts[d] * t.record_bytes]
        aux = torch.zeros_like(got)
        res = rsx.radix_sort(got, aux, None, kf_for(rsx, tname))
        want, _, _ = oracle.radix_sort(sub, L)
        assert res.cpu().numpy().tobytes() == want.tobytes(), f"destination {d}"


@pytest.mark.parametrize("tname,col", [("u32", 3), ("u64", 7), ("f32", 3), ("i64", -1), ("u32", -1)])
def test_scatter_pass_append(rsx, torch, tname, col):
    """rsx_scatter_pass_append (keys-only multi-GPU exchange without a routing histogram) with three
    local 'destinations': every destination's append cursor ends at the number of keys it owns and
    its buffer holds exactly those keys (as a multiset: the landing order of runs is arbitrary);
    a destination that is too small raises the overflow flag and is not written beyond its capacity."""
    import ctypes as C
    import importlib
    dsort = importlib.import_module("radix-sorting_b200.dist")
    t = TYPES[tname]
    n = 1_500_007
    data = make_input(tname, n, 91, "uniform" if col >= 0 else "zipf")
    L = rsx.RsxLayout(t.record_bytes, 0, t.key_bytes, t.kdf_kind, 0)
    derived = dsort.derive_np(np.ascontiguousarray(data).view(np.uint8).reshape(n, t.record_bytes), L)
    owner = np.zeros(256, dtype=np.uint8)
    owner[40:200] = 1
    owner[200:] = 2
    if col >= 0:
        dest = owner[((derived >> np.uint64(8 * col)) & np.uint64(0xFF)).astype(np.int64)].astype(np.int64)
        splitters = []
    else:
        splitters = dsort.choose_splitters(derived[::53], 3)
        dest = np.searchsorted(np.array(splitters, dtype=np.uint64), derived, side="right")
    counts = [int((dest == d).sum()) for d in range(3)]
    src = to_dev(torch, data)
    u = f"<u{t.record_bytes}"
    for shrink in (False, True):
        caps = [c + 1000 for c in counts]
        if shrink:
            caps[1] = counts[1] // 2  # destination 1 cannot take its share
        bufs = [torch.full((max(c, 1) * t.record_bytes + 64,), 0xAB, dtype=torch.uint8, device="cuda") for c in caps]
        cursors = torch.zeros(3, dtype=torch.int64, device="cuda")
        base = (C.c_uint64 * 3)(*[b.data_ptr() for b in bufs])
        cur = (C.c_uint64 * 3)(*[cursors.data_ptr() + 8 * d for d in range(3)])
        cap = (C.c_uint64 * 3)(*caps)
        own = (C.c_uint8 * 256)(*owner.tolist())
        sp = (C.c_uint64 * max(len(splitters), 1))(*splitters) if splitters else None
        ovf = C.c_uint32(7)
        st = rsx.lib().rsx_scatter_pass_append(src.data_ptr(), n, C.byref(L), col, own, sp, len(splitters), base, cur, cap, 3,
                                               C.byref(ovf), None)
        assert st == 0, st
        torch.cuda.synchronize()
        got_counts = cursors.cpu().tolist()
        if not shrink:
            assert ovf.value == 0 and got_counts == counts
            for d in range(3):
                got = bufs[d][: counts[d] * t.record_bytes].cpu().numpy().view(u)
                assert np.array_equal(np.sort(got), np.sort(data[dest == d].view(u))), f"destination {d}"
                assert bool((bufs[d][counts[d] * t.record_bytes:] == 0xAB).all())
        else:
            assert ovf.value == 1
            assert bool((bufs[1][caps[1] * t.record_bytes:] == 0xAB).all()), "written beyond the stated capacity"


def test_sampled_histogram_and_key_sample(rsx, torch):
    import ctypes as C
    n, stride = 1_000_003, 37
    data = make_input("u32", n, 5, "and2")
    src = to_dev(torch, data)
    L = rsx.RsxLayout(4, 0, 4, 0, 0)
    out = np.zeros(256, dtype=np.uint64)
    assert rsx.lib().rsx_histogram_column_sampled(src.data_ptr(), n, C.byref(L), 2, stride,
                                                  out.ctypes.data_as(C.POINTER(C.c_uint64)), None) == 0
    assert np.array_equal(out, np.bincount((data[::stride] >> 16) & 0xFF, minlength=256).astype(np.uint64))
    keys = np.zeros(2048, dtype=np.uint64)
    assert rsx.lib().rsx_sample_keys(src.data_ptr(), n, C.byref(L), 2048, keys.ctypes.data_as(C.POINTER(C.c_uint64)), None) == 0
    assert np.array_equal(keys, data[np.arange(2048) * (n // 2048)].astype(np.uint64))


def test_more_than_2_pow_32_records(rsx, torch):
    """n >= 2^32 -- the reference's 64-bit counter tier (radix_sort.hpp:111-113): 4.3 G one-byte
    keys, one live column, result in aux; checked by descents + multiset checksum."""
    n = (1 << 32) + 12345
    src = torch.empty(n, dtype=torch.uint8, device="cuda")
    aux = torch.empty_like(src)
    rsx.fill_keys(src, seed=3)
    kf = rsx.KeyFunc(rsx.KDF_UNSIGNED)
    _, s0, x0 = rsx.verify(src, kf)
    rep = rsx.RsxReport()
    res = rsx.radix_sort(src, aux, None, kf, report=rep)
    d1, s1, x1 = rsx.verify(res, kf)
    assert d1 == 0 and (s1, x1) == (s0, x0)
    assert rep.ncols == 1 and res.data_ptr() == aux.data_ptr()
    hist, descents, _ = rsx.histogram(res, kf)
    assert int(hist.sum()) == n and descents == 0


@pytest.mark.parametrize("tname", ["u32", "u64", "i64", "f32", "rec8_u32", "rec16_u64", "rec16_u8", "rec16_f64"])
def test_key_range_routing(rsx, torch, oracle, tname):
    """rsx_split_counts / rsx_split_pass_to: destination = number of splitters <= derived key."""
    import importlib
    dsort = importlib.import_module("radix-sorting_b200.dist")
    t = TYPES[tname]
    n = 200003
    data = make_input(tname, n, 77, "zipf" if tname in ("u32", "u64", "rec8_u32", "rec16_u64") else "uniform")
    L = t.layout()
    derived = dsort.derive_np(np.ascontiguousarray(data).view(np.uint8).reshape(n, t.record_bytes), L)
    splitters = dsort.choose_splitters(derived[::37], 5)
    dest = np.searchsorted(np.array(splitters, dtype=np.uint64), derived, side="right")
    src = to_dev(torch, data)
    kf = kf_for(rsx, tname)
    counts = rsx.split_counts(src, splitters, kf)
    assert counts == [int((dest == j).sum()) for j in range(5)]
    bufs = [torch.full((max(c, 1) * t.record_bytes,), 0xAB, dtype=torch.uint8, device="cuda") for c in counts]
    rsx.split_pass_to(src, splitters, [b.data_ptr() for b in bufs], kf)
    torch.cuda.synchronize()
    for j in range(5):
        got = bufs[j][: counts[j] * t.record_bytes].cpu().numpy()
        if t.record_bytes == t.key_bytes:
            # keys-only: equal records are indistinguishable, the pass may permute a tile's run (its
            # body leaves as one TMA bulk store) -- the multiset per range is what is defined
            u = f"<u{t.record_bytes}"
            assert np.array_equal(np.sort(got.view(u)), np.sort(data[dest == j].view(u))), f"range {j}"
        else:
            assert got.tobytes() == data[dest == j].tobytes(), f"range {j}: not the stable sub-sequence"
    if t.record_bytes == t.key_bytes:  # with bulk stores off the pass is order-preserving for every type
        try:
            rsx.lib().rsx_set_option(b"fused_bulk", 0)
            rsx.split_pass_to(src, splitters, [b.data_ptr() for b in bufs], kf)
            torch.cuda.synchronize()
        finally:
            rsx.lib().rsx_set_option(b"fused_bulk", 1)
        for j in range(5):
            got = bufs[j][: counts[j] * t.record_bytes].cpu().numpy()
            assert got.tobytes() == data[dest == j].tobytes(), f"range {j}: not the stable sub-sequence"


@pytest.mark.parametrize("tname", ["rec16_f64", "rec16_f32"])
@pytest.mark.parametrize("n", [3001, 70001, 300007])
def test_float_key_inside_16_byte_record(rsx, torch, oracle, tname, n):
    """basic_kdfs::by_member<&Rec::float_member> on a 16-byte record: the float KDF
    (radix_sort_basic_kdf.hpp:32-46) applied to a member, through the single-CTA kernel (n = 3001) and
    the multi-kernel path alike (the latter used to reject this layout with RSX_ERR_CUDA)."""
    t = TYPES[tname]
    data = make_input(tname, n, 13, "uniform")
    for desc in (False, True):
        out, rep, _ = gpu_sort(rsx, torch, tname, data, descending=desc)
        want, orep, _ = oracle.radix_sort(data, t.layout(descending=desc))
        assert out.tobytes() == want.tobytes() and rep.result_in_aux == orep.result_in_aux
    ranks, rrep, _ = gpu_rank(rsx, torch, tname, data, np.uint32)
    wr, worep, _ = oracle.radix_sort_rank(data, t.layout(), np.uint32)
    assert np.array_equal(ranks, wr) and rrep.result_in_aux == worep.result_in_aux


@pytest.mark.parametrize("tname", ["rec12_u32", "rec24_f64", "rec7_i16"])
@pytest.mark.parametrize("n,dist,mask", [(2, "uniform", -1), (1000, "uniform", -1), (300007, "uniform", 0xFFFFF), (300007, "and3", -1),
                                          (50000, "sorted", -1), (2_000_003, "uniform", -1)])
def test_records_of_any_size(rsx, torch, oracle, tname, n, dist, mask):
    """Record sizes the tile kernels do not move (12-byte {u32 key, 64-bit payload} like
    radix_sort_u32.c:7-10 on ILP32, a double key straddling two 8-byte words, a 7-byte record):
    keys are ranked, records gathered once; result and returned buffer as the reference's
    radix_sort<T> would give (device and host buffers, value and rank sort)."""
    t = TYPES[tname]
    data = make_input(tname, n, 17, dist, mask & ((1 << 64) - 1))
    for desc in (False, True):
        out, rep, in_aux = gpu_sort(rsx, torch, tname, data, descending=desc)
        want, orep, _ = oracle.radix_sort(data, t.layout(descending=desc))
        assert out.tobytes() == want.tobytes(), (tname, n, desc)
        assert rep.result_in_aux == orep.result_in_aux == int(in_aux) and rep.early_exit == orep.early_exit
    ranks, rrep, _ = gpu_rank(rsx, torch, tname, data, np.uint32)
    wr, worep, _ = oracle.radix_sort_rank(data, t.layout(), np.uint32)
    assert np.array_equal(ranks, wr) and rrep.result_in_aux == worep.result_in_aux
    if n <= 300007:  # host buffers: staged
        raw = np.ascontiguousarray(data).view(np.uint8).reshape(-1)
        src = torch.from_numpy(raw.copy())
        aux = torch.zeros_like(src)
        res = rsx.radix_sort(src, aux, None, kf_for(rsx, tname))
        want, _, _ = oracle.radix_sort(data, t.layout())
        assert res.numpy().tobytes() == want.tobytes()
        ib = torch.full((2 * n,), -1, dtype=torch.int32)
        hranks = rsx.radix_sort_rank(torch.from_numpy(raw.copy()), ib, None, kf_for(rsx, tname))
        assert np.array_equal(hranks.numpy().view(np.uint32), wr)


@pytest.mark.parametrize("tname,mask,orv,ncols,cpasses", [
    ("u32", 0x03010103, 0, 4, 1),                        # 6 varying bits in 4 byte columns -> 1 pass, result expanded back into src
    ("u32", 0x03010103, 0xA0500000, 4, 1),                # constant ONE bits between the runs
    ("u32", 0x0F0F0F0F, 0, 4, 0),                         # 4-byte keys: two saved passes do not pay for the extra histogram
    ("u64", 0x0F0F0F0F0F0F0F0F, 0, 8, 4),
    ("u64", 0x000F0F0F0F0F0F0F, 0, 7, 4),                 # odd column count: the reference returns aux
    ("u64", 0x1F1F1F1F1F1F1F1F, 0, 8, 5),                 # 40 bits -> 5 passes, data ends where the reference wants it
    ("i32", 0x01030103, 0, 4, 1), ("i64", 0x0303030303030303, 0x8000000000000000, 8, 2),
    ("f32", 0x01030103, 0, 4, 1), ("f64", 0x0F0F0F0F0F0F0F0F, 0x8000000000000000, 8, 4),  # positive and negative floats
    ("f32", 0x3F0F0F0F, 0, 4, 0),                         # 18 varying bits: 3 passes would save only one
    ("u32", 0x00FF0F0F, 0, 3, 0),                         # would save one pass only: not compacted
    ("u64", 0x0303030303033333, 0, 8, 3),                 # 10 runs of 2 bits: the two closest pairs are merged (<= 8 runs, 24 bits)
    ("u32", 0x55555555, 0, 4, 0),                         # 16 single-bit runs: merged runs span 24 bits, only one pass saved
])
@pytest.mark.parametrize("desc", [False, True], ids=["asc", "desc"])
def test_key_compaction(rsx, torch, oracle, tname, mask, orv, ncols, cpasses, desc):
    """N4 (README.md:716-758): key bits that are constant over the input cannot influence the order;
    the varying bits are gathered into a narrower key and sorted in fewer passes.  Output, live
    column count and returned buffer stay exactly the reference's."""
    t = TYPES[tname]
    n = 600_007
    data = make_input(tname, n, 23, "uniform", mask, orv)
    try:
        assert rsx.lib().rsx_set_option(b"compact_min_n", 1000) == 0
        out, rep, in_aux = gpu_sort(rsx, torch, tname, data, descending=desc)
    finally:
        rsx.lib().rsx_set_option(b"compact_min_n", 1 << 26)
    want, orep, _ = oracle.radix_sort(data, t.layout(descending=desc))
    assert rep.compacted_passes == cpasses, (rep.compacted_passes, cpasses)
    assert rep.ncols == orep.ncols == ncols and rep.result_in_aux == orep.result_in_aux == int(in_aux)
    assert out.tobytes() == want.tobytes()


def test_key_compaction_leaves_full_entropy_keys_alone(rsx, torch):
    """and3 keys are low-entropy but no bit is constant: nothing to compact; 70 M masked keys with 6
    varying bits cross the default threshold and are."""
    n = 70_000_003
    for dist, mask, expect in (("and3", (1 << 64) - 1, 0), ("uniform", 0x03010103, 1)):
        src = torch.empty(n, dtype=torch.int32, device="cuda")
        aux = torch.empty_like(src)
        rsx.fill_keys(src, seed=5, dist=dist, mask=mask)
        kf = rsx.KeyFunc(rsx.KDF_UNSIGNED)
        _, s0, x0 = rsx.verify(src, kf)
        rep = rsx.RsxReport()
        res = rsx.radix_sort(src, aux, None, kf, report=rep)
        d1, s1, x1 = rsx.verify(res, kf)
        assert d1 == 0 and (s1, x1) == (s0, x0)
        assert rep.compacted_passes == expect and rep.ncols == 4 and res.data_ptr() == src.data_ptr()


def test_multipass_composite_key_like_listing5(rsx, torch, oracle):
    """radix_sort_u64_multipass.c:117-118 sorts a 64-bit key with two stable 32-bit sorts (low half,
    then high half).  The same composition through key_offset/key_bytes windows must equal one
    64-bit sort -- this is what makes keys wider than 64 bits sortable."""
    n = 300001
    data = make_input("rec16_u64", n, 41, "and2")
    src = to_dev(torch, data)
    aux = torch.zeros_like(src)
    lo = rsx.radix_sort(src, aux, None, rsx.KeyFunc(rsx.KDF_UNSIGNED, False, 16, 0, 4))
    other = aux if lo.data_ptr() == src.data_ptr() else src
    hi = rsx.radix_sort(lo, other, None, rsx.KeyFunc(rsx.KDF_UNSIGNED, False, 16, 4, 4))
    want, _, _ = oracle.radix_sort(data, TYPES["rec16_u64"].layout())
    assert hi.cpu().numpy().tobytes() == want.tobytes()


@pytest.mark.parametrize("tname", ["u8", "u32", "i64", "f64", "rec16_u8", "rec16_u64"])
def test_single_cta_capacity_boundary(rsx, torch, oracle, tname):
    """n at, just below and just above the single-CTA kernel's capacity (value and rank sorts)."""
    t = TYPES[tname]
    for cap in {min((65536 - 16) // t.record_bytes, 16384), min((65536 - 16) // (t.record_bytes + 4), 16384)}:
        for n in (cap - 1, cap, cap + 1):
            data = make_input(tname, n, 5, "and2")
            out, rep, _ = gpu_sort(rsx, torch, tname, data)
            want, orep, _ = oracle.radix_sort(data, t.layout())
            assert out.tobytes() == want.tobytes() and rep.result_in_aux == orep.result_in_aux, (tname, n)
            ranks, rrep, _ = gpu_rank(rsx, torch, tname, data, np.uint32)
            wr, worep, _ = oracle.radix_sort_rank(data, t.layout(), np.uint32)
            assert np.array_equal(ranks, wr) and rrep.result_in_aux == worep.result_in_aux, (tname, n)


# ---- boundary behaviour: threads, managed memory, overlapping buffers ------------------------------------

def host_sort(rsx, torch, tname, data):
    """Value sort of CPU tensors: staged through device memory."""
    raw = np.ascontiguousarray(data).view(np.uint8).reshape(-1)
    src = torch.from_numpy(raw.copy())
    aux = torch.zeros_like(src)
    rep = rsx.RsxReport()
    res = rsx.radix_sort(src, aux, None, kf_for(rsx, tname), report=rep)
    assert rep.staged == 1
    return res.numpy()


def sort_from_threads(oracle, sort, context):
    """Four host threads sorting at once, five times each inside context(); sort(tname, data) -> sorted
    records."""
    import threading
    results, errors = {}, []

    def work(k):
        try:
            t = TYPES["u32" if k % 2 == 0 else "u64"]
            data = make_input(t.name, 400000 + 1000 * k, 100 + k)
            with context():
                for _ in range(5):
                    out = sort(t.name, data)
            want, _, _ = oracle.radix_sort(data, t.layout())
            results[k] = out.tobytes() == want.tobytes()
        except Exception as e:  # noqa: BLE001
            errors.append(repr(e))

    threads = [threading.Thread(target=work, args=(k,)) for k in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors
    assert all(results.get(k) for k in range(4)), results


def test_concurrent_host_threads(rsx, torch, oracle):
    """SURVEY §8b: safe to call from several host threads (per-call workspace, no global mutable state)."""
    sort_from_threads(oracle, lambda tname, data: gpu_sort(rsx, torch, tname, data)[0],
                      lambda: torch.cuda.stream(torch.cuda.Stream()))


def test_concurrent_host_threads_on_host_buffers(rsx, torch, oracle):
    """Four threads staging CPU tensors at once: one holds the cached staging buffer, the others
    stage through buffers of their own."""
    sort_from_threads(oracle, lambda tname, data: host_sort(rsx, torch, tname, data), contextlib.nullcontext)


def test_release_while_idle(rsx, torch, oracle):
    """rsx_release frees the idle cached workspace and staging buffer; the next device sort and
    host-staged sort allocate them again."""
    t = TYPES["u64"]
    data = make_input("u64", 300007, 29)
    want, _, _ = oracle.radix_sort(data, t.layout())
    assert host_sort(rsx, torch, "u64", data).tobytes() == want.tobytes()  # the staging buffer is cached now
    rsx.reserve(64 << 20)
    rsx.lib().rsx_release()
    assert gpu_sort(rsx, torch, "u64", data)[0].tobytes() == want.tobytes()
    assert host_sort(rsx, torch, "u64", data).tobytes() == want.tobytes()


def test_managed_memory_is_sorted_in_place(rsx, torch, oracle):
    """cudaMallocManaged buffers are treated like device memory (no staging)."""
    import ctypes as C
    cudart = C.CDLL("libcudart.so.12")
    n = 123457
    data = make_input("i32", n, 8)
    src, aux = C.c_void_p(), C.c_void_p()
    assert cudart.cudaMallocManaged(C.byref(src), C.c_size_t(4 * n), C.c_uint(1)) == 0
    assert cudart.cudaMallocManaged(C.byref(aux), C.c_size_t(4 * n), C.c_uint(1)) == 0
    try:
        C.memmove(src, data.ctypes.data, 4 * n)
        L = rsx.RsxLayout(4, 0, 4, rsx.KDF_SIGNED, 0)
        res, rep = C.c_void_p(), rsx.RsxReport()
        assert rsx.lib().rsx_sort(src, aux, n, C.byref(L), C.byref(res), C.byref(rep), None) == 0
        assert rep.staged == 0
        torch.cuda.synchronize()
        out = np.empty(n, dtype=np.int32)
        C.memmove(out.ctypes.data, res, 4 * n)
        assert np.array_equal(out, np.sort(data, kind="stable"))
    finally:
        cudart.cudaFree(src)
        cudart.cudaFree(aux)


def test_overlapping_buffers_are_rejected(rsx, torch):
    import ctypes as C
    buf = torch.zeros(1000, dtype=torch.int32, device="cuda")
    L = rsx.RsxLayout(4, 0, 4, 0, 0)
    res = C.c_void_p()
    st = rsx.lib().rsx_sort(buf.data_ptr(), buf.data_ptr() + 400, 600, C.byref(L), C.byref(res), None, None)
    assert st == rsx.RSX_ERR_INVALID
