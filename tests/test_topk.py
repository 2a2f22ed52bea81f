"""Top-k selection (rsx_topk / rsx_topk_rank): the first k records or indices of the stable sort.

The CPU tests check the argument validation that needs no device.  The GPU tests compare every output
byte for byte with the oracle's radix_sort(...)[:k] and radix_sort_rank(...)[:k]: every layout with a
1/2/4/8/16-byte record, both directions and both ranking modes, inputs aimed at the threshold search
(early stop, a bucket that survives to the last column, ties across chunk boundaries) and one input
above 2^32 records checked by its known answer."""
import ctypes as C

import numpy as np
import pytest

from cases import make_input
from pyoracle import TYPES

gpu = pytest.mark.gpu

IDX_TORCH = {1: "uint8", 2: "int16", 4: "int32", 8: "int64"}
IDX_NP = {1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}
VALUE_TYPES = [t for t in TYPES if TYPES[t].record_bytes in (1, 2, 4, 8, 16)]


def small_capacity(record_bytes: int, rank: bool) -> int:
    """Records the single-CTA sort holds (rsx_small.cu small_sort_capacity)."""
    return min((65536 - 16) // (record_bytes + (4 if rank else 0)), 1024 * 16)


def launch_bound(key_bytes: int) -> int:
    """DESIGN.md "Top-k": key_bytes search launches, one select, the sort of k records."""
    return 2 * key_bytes + 6


# ---- CPU: validation before any device work ----------------------------------------------------------

def _topk(rsx, n, k, layout=(4, 0, 4, 0, 0), idx_bytes=0, out=None, src=None, rep=None):
    L = rsx.lib()
    src = src if src is not None else (C.c_uint8 * 4096)()
    out = out if out is not None else (C.c_uint8 * 4096)()
    lay = rsx.RsxLayout(*layout)
    rp = C.byref(rep) if rep is not None else None
    if idx_bytes:
        return L.rsx_topk_rank(src, n, k, C.byref(lay), idx_bytes, out, rp, None)
    return L.rsx_topk(src, n, k, C.byref(lay), out, rp, None)


def test_topk_validation_needs_no_device(rsx):
    INV = rsx.RSX_ERR_INVALID
    for idx in (0, 4):
        assert _topk(rsx, 8, 9, idx_bytes=idx) == INV                              # k > n
        assert _topk(rsx, 8, 2, layout=(4, 0, 3, 0, 0), idx_bytes=idx) == INV      # bad layout
        assert _topk(rsx, 8, 2, layout=(4, 0, 4, 3, 0), idx_bytes=idx) == INV      # bad KDF
        assert _topk(rsx, 8, 2, layout=(12, 0, 4, 0, 0), idx_bytes=idx) == INV     # record size 12
        assert _topk(rsx, 8, 2, layout=(7, 5, 2, 1, 0), idx_bytes=idx) == INV      # record size 7
    assert _topk(rsx, 8, 2, idx_bytes=3) == INV                                     # index type
    L = rsx.lib()
    buf = (C.c_uint8 * 4096)()
    lay = rsx.RsxLayout(4, 0, 4, 0, 0)
    assert L.rsx_topk(buf, 8, 2, C.byref(lay), None, None, None) == INV               # NULL out
    assert L.rsx_topk(None, 8, 2, C.byref(lay), buf, None, None) == INV               # NULL src
    assert L.rsx_topk_rank(buf, 8, 2, C.byref(lay), 4, None, None, None) == INV       # NULL index_out
    assert L.rsx_topk_rank(buf, 8, 2, C.byref(lay), 0, buf, None, None) == INV        # idx_bytes 0
    # out overlapping src (src is never written)
    base = C.addressof(buf)
    assert L.rsx_topk(buf, 8, 2, C.byref(lay), C.c_void_p(base + 24), None, None) == INV
    assert L.rsx_topk(C.c_void_p(base + 24), 8, 8, C.byref(lay), buf, None, None) == INV
    assert L.rsx_topk_rank(buf, 8, 2, C.byref(lay), 4, C.c_void_p(base + 28), None, None) == INV
    # n - 1 must fit the index type
    assert _topk(rsx, 257, 1, layout=(1, 0, 1, 0, 0), idx_bytes=1) == rsx.RSX_ERR_IDX_RANGE
    assert _topk(rsx, 256, 1, layout=(1, 0, 1, 0, 0), idx_bytes=1) != rsx.RSX_ERR_IDX_RANGE
    assert _topk(rsx, 65537, 1, layout=(1, 0, 1, 0, 0), idx_bytes=2,
                 src=(C.c_uint8 * 65537)()) == rsx.RSX_ERR_IDX_RANGE
    assert _topk(rsx, 65536, 1, layout=(1, 0, 1, 0, 0), idx_bytes=2,
                 src=(C.c_uint8 * 65536)()) != rsx.RSX_ERR_IDX_RANGE


def test_topk_k_zero_needs_no_device(rsx):
    for idx in (0, 1, 8):
        rep = rsx.RsxReport(1, 2, 3, 4, 5, 6, 7)
        out = (C.c_uint8 * 4096)(*([0xAB] * 4096))
        assert _topk(rsx, 8, 0, idx_bytes=idx, out=out, rep=rep) == rsx.RSX_OK
        assert list(out) == [0xAB] * 4096
        assert (rep.early_exit, rep.ncols, rep.live_mask, rep.result_in_aux, rep.kernel_launches,
                rep.staged, rep.compacted_passes) == (0,) * 7
    assert _topk(rsx, 0, 0) == rsx.RSX_OK
    lay = rsx.RsxLayout(4, 0, 4, 0, 0)
    assert rsx.lib().rsx_topk(None, 0, 0, C.byref(lay), None, None, None) == rsx.RSX_OK


def test_topk_no_cpu_fallback(rsx):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present; the failure path is exercised without one")
    L = rsx.lib()
    src = (C.c_uint32 * 8)(5, 4, 3, 2, 1, 0, 9, 8)
    out = (C.c_uint32 * 8)(*([77] * 8))
    lay = rsx.RsxLayout(4, 0, 4, 0, 0)
    assert L.rsx_topk(src, 8, 3, C.byref(lay), out, None, None) in (rsx.RSX_ERR_NO_DEVICE, rsx.RSX_ERR_CUDA)
    assert L.rsx_topk_rank(src, 8, 3, C.byref(lay), 4, out, None, None) in (rsx.RSX_ERR_NO_DEVICE, rsx.RSX_ERR_CUDA)
    assert list(src) == [5, 4, 3, 2, 1, 0, 9, 8] and list(out) == [77] * 8


def test_topk_is_declared_and_bound(rsx):
    assert "rsx_topk" in rsx.EXPORTS and "rsx_topk_rank" in rsx.EXPORTS
    assert callable(rsx.radix_topk) and callable(rsx.radix_topk_rank)


# ---- GPU ---------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the product has no CPU path (run with -m gpu on the GPU box)")
    # the once-per-device ranking probe (9 kernels) runs here, not inside a call whose launches are counted
    import importlib
    assert importlib.import_module("radix-sorting_b200").lib().rsx_set_option(b"query_rank_mode", 0) in (0, 1)
    return torch


@pytest.fixture(params=[0, 1], ids=["ticket", "ballot"])
def rank_mode(request, rsx):
    assert rsx.lib().rsx_set_option(b"rank_mode", request.param) == 0
    yield request.param
    rsx.lib().rsx_set_option(b"rank_mode", -1)


def to_dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


def kf_for(rsx, tname, descending=False):
    t = TYPES[tname]
    return rsx.KeyFunc(t.kdf_kind, descending, t.record_bytes, t.key_offset, t.key_bytes)


def gpu_topk(rsx, torch, tname, src, k, descending=False):
    """src: device uint8 tensor of records.  Returns (first k records as numpy, report)."""
    rb = TYPES[tname].record_bytes
    before = src.clone()
    out = torch.full((max(k, 1) * rb + 64,), 0xCD, dtype=torch.uint8, device="cuda")
    rep = rsx.RsxReport()
    res = rsx.radix_topk(src, k, out, kf_for(rsx, tname, descending), report=rep)
    torch.cuda.synchronize()
    assert torch.equal(src, before), "top-k must not modify src"
    assert res.data_ptr() == out.data_ptr() and res.numel() == k * rb
    assert (out[k * rb:].cpu().numpy() == 0xCD).all(), "top-k wrote past k records"
    return res.cpu().numpy().view(TYPES[tname].dtype), rep


def gpu_topk_rank(rsx, torch, tname, src, k, idx_bytes=4, descending=False):
    out = torch.full((k + 8,), 0x5A, dtype=getattr(torch, IDX_TORCH[idx_bytes]), device="cuda")
    rep = rsx.RsxReport()
    res = rsx.radix_topk_rank(src, k, out, kf_for(rsx, tname, descending), report=rep)
    torch.cuda.synchronize()
    assert res.data_ptr() == out.data_ptr() and res.numel() == k
    assert (out[k:].cpu() == 0x5A).all(), "top-k wrote past k indices"
    return res.cpu().numpy().view(IDX_NP[idx_bytes]), rep


def check_against_oracle(rsx, torch, oracle, tname, data, ks, descending=False, idx_bytes=4, rank=True):
    """Every k of `ks`: value and rank top-k equal the oracle's sort, sliced."""
    t = TYPES[tname]
    lay = t.layout(descending)
    want, _, _ = oracle.radix_sort(data, lay)
    want_r = oracle.radix_sort_rank(data, lay, IDX_NP[idx_bytes])[0] if rank else None
    src = to_dev(torch, data)
    reps = []
    for k in ks:
        got, rep = gpu_topk(rsx, torch, tname, src, k, descending)
        assert got.tobytes() == want[:k].tobytes(), (tname, len(data), k, "value")
        assert 1 <= rep.ncols <= t.key_bytes and rep.kernel_launches <= launch_bound(t.key_bytes), (rep.ncols, rep.kernel_launches)
        assert (rep.early_exit, rep.live_mask, rep.result_in_aux, rep.staged, rep.compacted_passes) == (0,) * 5
        reps.append(rep.ncols)
        if rank:
            got_r, rep = gpu_topk_rank(rsx, torch, tname, src, k, idx_bytes, descending)
            assert np.array_equal(got_r, want_r[:k]), (tname, len(data), k, "rank")
            assert rep.kernel_launches <= launch_bound(t.key_bytes)
    return reps


def ks_for(n):
    return sorted({k for k in (1, 2, 1000, n // 3, n - 1, n) if 1 <= k <= n})


@gpu
@pytest.mark.parametrize("descending", [False, True], ids=["asc", "desc"])
@pytest.mark.parametrize("tname", VALUE_TYPES)
def test_topk_matches_oracle_around_single_cta(rsx, torch, oracle, rank_mode, tname, descending):
    rb = TYPES[tname].record_bytes
    for n in (small_capacity(rb, False) - 1, small_capacity(rb, False) + 1, small_capacity(rb, True) + 1):
        data = make_input(tname, n, 100 + n + rb)
        check_against_oracle(rsx, torch, oracle, tname, data, ks_for(n), descending)


@gpu
@pytest.mark.parametrize("descending", [False, True], ids=["asc", "desc"])
@pytest.mark.parametrize("tname", VALUE_TYPES)
def test_topk_matches_oracle_multi_tile(rsx, torch, oracle, tname, descending):
    """n = 12 M: every CTA of the search and the select works through many steps of its chunk."""
    n = 12_000_007
    data = make_input(tname, n, 7 + TYPES[tname].record_bytes)
    check_against_oracle(rsx, torch, oracle, tname, data, ks_for(n), descending,
                         idx_bytes=8 if TYPES[tname].key_bytes == 8 else 4)


@gpu
def test_all_keys_equal_takes_the_first_k_records(rsx, torch, oracle, rank_mode):
    n = 12_000_007
    data = make_input("rec8_u32", n, 3, dist="constant")
    assert (data["key"] == data["key"][0]).all()
    src = to_dev(torch, data)
    for k in (1, 1000, n // 3, n):
        got, rep = gpu_topk(rsx, torch, "rec8_u32", src, k)
        assert got.tobytes() == data[:k].tobytes(), k
        ranks, _ = gpu_topk_rank(rsx, torch, "rec8_u32", src, k)
        assert np.array_equal(ranks, np.arange(k, dtype=np.uint32)), k


@gpu
def test_two_keys_threshold_run_crosses_chunks(rsx, torch, oracle, rank_mode):
    """Two distinct keys; the threshold key's run covers many chunk and CTA boundaries, and the quota
    of equal records ends inside one of them."""
    n = 12_000_007
    rng = np.random.default_rng(9)
    data = make_input("rec8_u32", n, 5)
    data["key"] = rng.integers(0, 2, size=n, dtype=np.uint32) * 0x01000000 + 5
    zeros = int((data["key"] == 5).sum())
    check_against_oracle(rsx, torch, oracle, "rec8_u32", data, [zeros - 1, zeros, zeros + 1, zeros + n // 5 + 12345, n - 3])
    # the smaller key only in the second half: the equal run of the larger key spans the first half
    data["key"] = np.where(np.arange(n) < n // 2, 9, 4).astype(np.uint32)
    check_against_oracle(rsx, torch, oracle, "rec8_u32", data, [n // 2 + n // 7, n - n // 2 + 1, 17])


@gpu
def test_search_stops_at_the_top_column(rsx, torch, oracle):
    """1 000 keys with top byte 0x00 and k = 1 000: the first bucket holds exactly the need."""
    n = 1_000_003
    data = make_input("rec8_u32", n, 21)
    rng = np.random.default_rng(2)
    keys = (rng.integers(1, 256, size=n, dtype=np.uint32) << 24) | (data["key"] & 0x00FFFFFF)
    low = rng.choice(n, size=1000, replace=False)
    keys[low] &= 0x00FFFFFF
    data["key"] = keys
    assert check_against_oracle(rsx, torch, oracle, "rec8_u32", data, [1000]) == [1]
    data64 = make_input("u64", n, 22) | np.uint64(1 << 56)
    data64[low] &= np.uint64((1 << 56) - 1)
    assert check_against_oracle(rsx, torch, oracle, "u64", data64, [1000], idx_bytes=8) == [1]


@gpu
def test_threshold_bucket_survives_to_the_last_column(rsx, torch, oracle, rank_mode):
    """Heavily repeated full keys: the last column's bucket is larger than the quota q."""
    n = 2_000_003
    data = make_input("rec8_u32", n, 31)
    rng = np.random.default_rng(4)
    data["key"] = rng.integers(0, 100, size=n, dtype=np.uint32) * np.uint32(0x01010101)
    ncols = check_against_oracle(rsx, torch, oracle, "rec8_u32", data, [5000, 123457, n // 2 + 1], rank=True)
    assert ncols == [4, 4, 4]
    for tname in ("rec16_u64", "i16"):
        d = make_input(tname, n, 32)
        key = rng.integers(-3, 4, size=n).astype(TYPES[tname].dtype["key"] if d.dtype.names else d.dtype)
        if d.dtype.names:
            d["key"] = key
        else:
            d = key
        for desc in (False, True):
            assert set(check_against_oracle(rsx, torch, oracle, tname, d, [1, 70001, n // 3], desc,
                                            idx_bytes=8)) == {TYPES[tname].key_bytes}


@gpu
@pytest.mark.parametrize("dist", ["sorted", "reverse", "zipf", "and3"])
def test_presorted_reversed_and_skewed(rsx, torch, oracle, dist):
    n = 3_000_017
    for tname in ("u32", "rec16_u64", "i64"):
        data = make_input(tname, n, 41, dist=dist)
        for desc in (False, True):
            check_against_oracle(rsx, torch, oracle, tname, data, [1, 1000, n // 3, n], desc,
                                 idx_bytes=8 if TYPES[tname].key_bytes == 8 else 4)


def float_specials(dt, n, seed):
    """Random bit patterns, a third of them replaced by +-0, +-inf, quiet, signalling and negative NaNs,
    denormals and the extremes.  Built on the integer view, so no NaN is quietened on the way."""
    rng = np.random.default_rng(seed)
    f = np.finfo(dt)
    ut = np.uint32 if dt == np.float32 else np.uint64
    special = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, f.tiny, -f.tiny, f.tiny / 4, -f.tiny / 4, f.max, -f.max,
                        1.0, -1.0], dtype=dt).view(ut)
    nans = [0x7FA00000, 0xFFC00001] if dt == np.float32 else [0x7FF4000000000000, 0xFFF8000000000001]
    special = np.concatenate([special, np.array(nans, dtype=ut)])
    out = rng.integers(0, np.iinfo(ut).max, size=n, dtype=ut, endpoint=True)
    pos = rng.integers(0, n, size=n // 3)
    out[pos] = special[rng.integers(0, len(special), size=pos.size)]
    return out.view(dt)


@gpu
def test_float_specials(rsx, torch, oracle, rank_mode):
    n = 1_500_001
    for tname, dt in (("f32", np.float32), ("f64", np.float64)):
        data = float_specials(dt, n, 8)
        for desc in (False, True):
            check_against_oracle(rsx, torch, oracle, tname, data, [1, 2, 1000, n // 3, n - 1], desc,
                                 idx_bytes=8 if dt == np.float64 else 4)
    rec = make_input("rec16_f32", n, 6)
    rec["key"] = float_specials(np.float32, n, 9)
    check_against_oracle(rsx, torch, oracle, "rec16_f32", rec, [1000, n // 2], True)


@gpu
@pytest.mark.parametrize("idx_bytes", [1, 2, 4, 8])
def test_rank_index_widths(rsx, torch, oracle, idx_bytes):
    n = {1: 256, 2: 65536, 4: 3_000_001, 8: 3_000_001}[idx_bytes]
    for tname in ("u8", "i32", "f64", "rec16_u8"):
        data = make_input(tname, n, 50 + idx_bytes)
        for desc in (False, True):
            lay = TYPES[tname].layout(desc)
            want = oracle.radix_sort_rank(data, lay, IDX_NP[idx_bytes])[0]
            src = to_dev(torch, data)
            for k in ks_for(n):
                got, _ = gpu_topk_rank(rsx, torch, tname, src, k, idx_bytes, desc)
                assert np.array_equal(got, want[:k]), (tname, idx_bytes, k)
    big = to_dev(torch, make_input("u8", 257, 1))
    out = torch.zeros(4, dtype=torch.uint8, device="cuda")
    with pytest.raises(rsx.RsxError) as e:
        rsx.radix_topk_rank(big, 1, out)
    assert e.value.status == rsx.RSX_ERR_IDX_RANGE


@gpu
def test_host_memory_is_refused(rsx, torch):
    src = torch.arange(100, dtype=torch.int32)
    out = torch.zeros(10, dtype=torch.int32)
    with pytest.raises(rsx.RsxError) as e:
        rsx.radix_topk(src, 5, out)
    assert e.value.status == rsx.RSX_ERR_MIXED_MEMORY
    dsrc = src.cuda()
    lay = rsx.RsxLayout(4, 0, 4, rsx.KDF_SIGNED, 0)
    assert rsx.lib().rsx_topk(dsrc.data_ptr(), 100, 5, C.byref(lay), out.data_ptr(), None, None) == rsx.RSX_ERR_MIXED_MEMORY
    assert rsx.lib().rsx_topk_rank(dsrc.data_ptr(), 100, 5, C.byref(lay), 4, out.data_ptr(), None, None) == rsx.RSX_ERR_MIXED_MEMORY
    assert (out == 0).all()


@gpu
def test_runs_on_the_current_stream(rsx, torch):
    x = torch.randint(-2**31, 2**31 - 1, (5_000_000,), dtype=torch.int32, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        src = x.clone()
        out = torch.empty(4096, dtype=torch.int32, device="cuda")
        got = rsx.radix_topk(src, 4096, out, rsx.KeyFunc(rsx.KDF_SIGNED, True)).clone()
        idx = torch.empty(4096, dtype=torch.int64, device="cuda")
        got_i = rsx.radix_topk_rank(src, 4096, idx).clone()
    torch.cuda.synchronize()
    want = torch.sort(x, descending=True, stable=True)
    assert torch.equal(got, want.values[:4096])
    assert torch.equal(got_i, torch.sort(x, stable=True).indices[:4096])


@gpu
def test_launch_bound_holds_for_very_different_n_and_k(rsx, torch):
    for tname in ("u8", "u32", "u64", "rec16_u64"):
        kb = TYPES[tname].key_bytes
        for n in (2, 5000, 3_000_000):
            data = make_input(tname, n, n)
            src = to_dev(torch, data)
            for k in sorted({1, 2, min(n, 70000), n}):
                _, rep = gpu_topk(rsx, torch, tname, src, k)
                assert kb + 2 <= rep.kernel_launches + (k < 2) <= launch_bound(kb), (tname, n, k, rep.kernel_launches)
                _, rep = gpu_topk_rank(rsx, torch, tname, src, k, 8)
                assert kb + 2 <= rep.kernel_launches <= launch_bound(kb), (tname, n, k, rep.kernel_launches)


@gpu
def test_beyond_32_bit_positions(rsx, torch):
    """More than 2^32 u8 keys of 255 with smaller keys planted at known positions, most of them beyond
    2^32: value and u64-rank top-k, with and without a quota of 255s."""
    n = 2**32 + 2**21 + 3
    src = torch.full((n,), 255, dtype=torch.uint8, device="cuda")
    plant = {2**32 + 5: 7, 2**32 + 2**20: 3, 2**32 + 2**21 + 1: 3, 2**31: 9, n - 1: 0, 2**32 - 1: 254}
    for p, v in plant.items():
        src[p] = v
    order = sorted(plant, key=lambda p: (plant[p], p))
    kf = rsx.KeyFunc(rsx.KDF_UNSIGNED)
    for k in (len(plant), len(plant) + 3):
        out = torch.empty(k, dtype=torch.uint8, device="cuda")
        got = rsx.radix_topk(src, k, out, kf).cpu().numpy()
        want = [plant[p] for p in order] + [255] * (k - len(plant))
        assert got.tolist() == want, k
        idx = torch.empty(k, dtype=torch.int64, device="cuda")
        got_i = rsx.radix_topk_rank(src, k, idx, kf).cpu().numpy().tolist()
        assert got_i == order + [0, 1, 2][:k - len(plant)], k
    # descending: the quota of 255s ends beyond 2^32 when the first records are the small ones
    src[:2**32 + 4] = 1
    idx = torch.empty(3, dtype=torch.int64, device="cuda")
    got_i = rsx.radix_topk_rank(src, 3, idx, rsx.KeyFunc(rsx.KDF_UNSIGNED, True)).cpu().numpy().tolist()
    assert got_i == [2**32 + 4, 2**32 + 6, 2**32 + 7]
    del src
    torch.cuda.empty_cache()
