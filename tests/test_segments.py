"""Segmented sort and rank (rsx_sort_segments / rsx_sort_rank_segments): many independent arrays in
one call.  The CPU tests check the argument validation that needs no device; the GPU tests compare
every segment bit for bit with the oracle's radix_sort / radix_sort_rank of that segment alone, and
the batch's result pointer and report with the reference's rule applied to the whole batch."""
import ctypes as C

import numpy as np
import pytest

from cases import make_input
from pyoracle import TYPES

gpu = pytest.mark.gpu

IDX_TORCH = {1: "uint8", 2: "int16", 4: "int32", 8: "int64"}


def group_capacity(record_bytes: int, rank: bool) -> int:
    """Records one CTA of the group kernel holds (rsx_segments.cu group_capacity)."""
    return min((65536 - 16) // (record_bytes + (4 if rank else 1)), 1024 * 16)


def offsets_of(lengths):
    return np.concatenate([[0], np.cumsum(np.asarray(lengths, dtype=np.uint64))]).astype(np.uint64)


# ---- CPU: validation before any device work ----------------------------------------------------------

def _call(rsx, n, offs, layout=(4, 0, 4, 0, 0), idx_bytes=0):
    L = rsx.lib()
    res = C.c_void_p()
    buf = (C.c_uint8 * 4096)()
    aux = (C.c_uint8 * 4096)()
    off = (C.c_uint64 * len(offs))(*offs)
    lay = rsx.RsxLayout(*layout)
    if idx_bytes:
        return L.rsx_sort_rank_segments(buf, aux, n, off, len(offs) - 1, C.byref(lay), idx_bytes, C.byref(res), None, None), res, buf
    return L.rsx_sort_segments(buf, aux, n, off, len(offs) - 1, C.byref(lay), C.byref(res), None, None), res, buf


def test_segment_validation_needs_no_device(rsx):
    bad_offsets = [
        [0, 5, 3, 8],   # not monotone
        [1, 4, 8],      # offsets[0] != 0
        [0, 4, 7],      # offsets[nseg] != n
        [0],            # nseg == 0 with n > 0
    ]
    for offs in bad_offsets:
        assert _call(rsx, 8, offs)[0] == rsx.RSX_ERR_INVALID, offs
        assert _call(rsx, 8, offs, idx_bytes=4)[0] == rsx.RSX_ERR_INVALID, offs
    assert _call(rsx, 8, [0, 8], layout=(4, 0, 3, 0, 0))[0] == rsx.RSX_ERR_INVALID       # bad layout
    assert _call(rsx, 8, [0, 8], layout=(12, 0, 4, 0, 0))[0] == rsx.RSX_ERR_INVALID      # generic record size
    assert _call(rsx, 8, [0, 8], idx_bytes=3)[0] == rsx.RSX_ERR_INVALID                  # index type
    assert _call(rsx, 400, [0, 300, 400], layout=(1, 0, 1, 0, 0), idx_bytes=1)[0] == rsx.RSX_ERR_IDX_RANGE
    assert _call(rsx, 400, [0, 256, 400], layout=(1, 0, 1, 0, 0), idx_bytes=1)[0] != rsx.RSX_ERR_IDX_RANGE


def test_segments_below_two_records_return_src(rsx):
    for n, offs in [(0, [0]), (0, [0, 0, 0]), (1, [0, 1]), (1, [0, 0, 1, 1])]:
        st, res, buf = _call(rsx, n, offs)
        assert st == 0 and res.value == C.addressof(buf)


def test_segments_no_cpu_fallback(rsx):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present; the failure path is exercised without one")
    L = rsx.lib()
    res = C.c_void_p()
    src = (C.c_uint32 * 8)(5, 4, 3, 2, 1, 0, 9, 8)
    aux = (C.c_uint32 * 8)()
    ib = (C.c_uint32 * 16)()
    off = (C.c_uint64 * 3)(0, 4, 8)
    lay = rsx.RsxLayout(4, 0, 4, 0, 0)
    st = L.rsx_sort_segments(src, aux, 8, off, 2, C.byref(lay), C.byref(res), None, None)
    assert st in (rsx.RSX_ERR_NO_DEVICE, rsx.RSX_ERR_CUDA)
    st = L.rsx_sort_rank_segments(src, ib, 8, off, 2, C.byref(lay), 4, C.byref(res), None, None)
    assert st in (rsx.RSX_ERR_NO_DEVICE, rsx.RSX_ERR_CUDA)
    assert list(src) == [5, 4, 3, 2, 1, 0, 9, 8] and list(aux) == [0] * 8 and list(ib) == [0] * 16


# ---- GPU ---------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the product has no CPU path (run with -m gpu on the GPU box)")
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


def ragged_lengths(cap, seed):
    """0, 1, 2, a run of more than 256 tiny segments, cap - 1, cap, cap + 1, 70 001, shuffled with
    random short segments (empty ones included)."""
    rng = np.random.default_rng(seed)
    special = [0, 1, 2, cap - 1, cap, cap + 1, 70001, 0, 0]
    short = list(rng.integers(0, 40, size=60))
    parts = special + short
    rng.shuffle(parts)
    k = len(parts) // 2
    tiny = list(rng.integers(1, 4, size=300))
    return parts[:k] + tiny + parts[k:]


def batch_rule(oracle, data, layout):
    """(ncols, live_mask) of the whole batch, from the oracle's histogram of the concatenation."""
    _, _, hist = oracle.radix_sort(data, layout, want_hist=True)
    n = data.shape[0]
    mask = sum(1 << c for c in range(hist.shape[0]) if hist[c].max() != n)
    return bin(mask).count("1"), mask


def gpu_sort_segments(rsx, torch, tname, data, offs, descending=False, device_offsets=False):
    src = to_dev(torch, data)
    aux = torch.full_like(src, 0xCD)
    rep = rsx.RsxReport()
    o = torch.from_numpy(offs.view(np.int64).copy())
    if device_offsets:
        o = o.cuda()
    res = rsx.radix_sort_segments(src, aux, o, kf_for(rsx, tname, descending), report=rep)
    torch.cuda.synchronize()
    return res.cpu().numpy().view(TYPES[tname].dtype), rep, res.data_ptr() == aux.data_ptr(), aux.cpu().numpy()


def gpu_rank_segments(rsx, torch, tname, data, offs, idx_dtype, descending=False):
    src = to_dev(torch, data)
    before = src.clone()
    n = data.shape[0]
    ib = torch.full((2 * n,), 0x5A, dtype=getattr(torch, IDX_TORCH[np.dtype(idx_dtype).itemsize]), device="cuda")
    rep = rsx.RsxReport()
    res = rsx.radix_sort_rank_segments(src, ib, torch.from_numpy(offs.view(np.int64).copy()), kf_for(rsx, tname, descending),
                                       report=rep)
    torch.cuda.synchronize()
    assert torch.equal(src, before), "a rank sort must not modify src"
    in_aux = res.data_ptr() != ib.data_ptr()
    return res.cpu().numpy().view(idx_dtype), rep, in_aux, ib.cpu().numpy().view(idx_dtype)


VALUE_TYPES = [t for t in TYPES if TYPES[t].record_bytes in (1, 2, 4, 8, 16)]


@gpu
@pytest.mark.parametrize("descending", [False, True], ids=["asc", "desc"])
@pytest.mark.parametrize("tname", VALUE_TYPES)
def test_segments_match_oracle(rsx, torch, oracle, rank_mode, tname, descending):
    t = TYPES[tname]
    lengths = ragged_lengths(group_capacity(t.record_bytes, False), 7 + t.record_bytes)
    offs = offsets_of(lengths)
    data = make_input(tname, int(offs[-1]), 4321)
    out, rep, in_aux, _ = gpu_sort_segments(rsx, torch, tname, data, offs, descending)
    lay = t.layout(descending)
    for s in range(len(lengths)):
        a, b = int(offs[s]), int(offs[s + 1])
        want, _, _ = oracle.radix_sort(data[a:b], lay)
        assert out[a:b].tobytes() == want.tobytes(), f"segment {s} [{a}, {b})"
    ncols, mask = batch_rule(oracle, data, lay)
    assert rep.early_exit == 0 and rep.ncols == ncols and rep.live_mask == mask
    assert in_aux == bool(ncols & 1) == bool(rep.result_in_aux)
    assert rep.kernel_launches >= 2


@gpu
@pytest.mark.parametrize("tname", ["u8", "i16", "u32", "f32", "i64", "f64", "rec16_u8", "rec8_u32", "rec16_u64"])
def test_rank_segments_match_oracle(rsx, torch, oracle, rank_mode, tname):
    t = TYPES[tname]
    long_lengths = ragged_lengths(group_capacity(t.record_bytes, True), 11 + t.record_bytes)
    rng = np.random.default_rng(5)
    short_lengths = list(rng.integers(0, 257, size=400))  # fits u8 indices: at most 256 records
    for idt, lengths in [(np.uint8, short_lengths), (np.uint16, short_lengths + [65536]),
                         (np.uint32, long_lengths), (np.uint64, long_lengths)]:
        offs = offsets_of(lengths)
        data = make_input(tname, int(offs[-1]), 99)
        for desc in (False, True):
            ranks, rep, in_aux, _ = gpu_rank_segments(rsx, torch, tname, data, offs, idt, desc)
            lay = t.layout(desc)
            for s in range(len(lengths)):
                a, b = int(offs[s]), int(offs[s + 1])
                want, _, _ = oracle.radix_sort_rank(data[a:b], lay, idt)
                assert np.array_equal(ranks[a:b], want), f"{np.dtype(idt)} segment {s} [{a}, {b})"
            ncols, mask = batch_rule(oracle, data, lay)
            assert rep.ncols == ncols and rep.live_mask == mask and in_aux == bool(ncols & 1)


@gpu
def test_every_segment_ordered_exits_early(rsx, torch, oracle, rank_mode):
    rng = np.random.default_rng(3)
    lengths = [int(x) for x in rng.integers(0, 3000, size=50)] + [20000, 1]
    offs = offsets_of(lengths)
    data = make_input("u32", int(offs[-1]), 17)
    for s in range(len(lengths)):
        data[int(offs[s]):int(offs[s + 1])].sort()
    assert (data[1:] < data[:-1]).any(), "the concatenation itself must not be ordered"
    out, rep, in_aux, aux = gpu_sort_segments(rsx, torch, "u32", data, offs)
    assert rep.early_exit == 1 and rep.ncols == 0 and not in_aux and rep.result_in_aux == 0
    assert out.tobytes() == data.tobytes()
    assert (aux == 0xCD).all(), "aux must keep its fill on early exit"
    ranks, rep, in_aux, ib = gpu_rank_segments(rsx, torch, "u32", data, offs, np.uint32)
    assert rep.early_exit == 1 and not in_aux
    want = np.concatenate([np.arange(b - a, dtype=np.uint32) for a, b in zip(offs[:-1], offs[1:])])
    assert np.array_equal(ranks, want) and np.array_equal(ib[:len(want)], want)


@gpu
def test_odd_parity_writes_every_segment_to_aux(rsx, torch, oracle, rank_mode):
    """Three live columns: the batch's result is aux, so one-record and already-ordered segments,
    and a segment longer than one group, must land there too."""
    lengths = [1, 5, 1, 300, 2, 1, 0, 7, group_capacity(4, False) + 10, 1, 40]
    offs = offsets_of(lengths)
    data = make_input("u32", int(offs[-1]), 23, mask=0x00FFFFFF)
    data[int(offs[3]):int(offs[4])].sort()  # already ordered
    data[int(offs[8]):int(offs[9])].sort()  # long and ordered
    out, rep, in_aux, _ = gpu_sort_segments(rsx, torch, "u32", data, offs)
    assert rep.ncols == 3 and in_aux and rep.result_in_aux == 1
    for s in range(len(lengths)):
        a, b = int(offs[s]), int(offs[s + 1])
        assert out[a:b].tobytes() == np.sort(data[a:b], kind="stable").tobytes(), s
    ranks, rep, in_aux, _ = gpu_rank_segments(rsx, torch, "u32", data, offs, np.uint32)
    assert in_aux
    for s in range(len(lengths)):
        a, b = int(offs[s]), int(offs[s + 1])
        assert np.array_equal(ranks[a:b], np.argsort(data[a:b], kind="stable").astype(np.uint32)), s


@gpu
def test_single_segment_equals_rsx_sort(rsx, torch, rank_mode):
    for tname in ("u32", "u64", "rec16_u8"):
        rb = TYPES[tname].record_bytes
        for n in (group_capacity(rb, False), group_capacity(rb, False) + 1, group_capacity(rb, True) + 1, 70001):
            data = make_input(tname, n, n)
            kf = kf_for(rsx, tname)
            src, aux = to_dev(torch, data), torch.full((n * rb,), 0xCD, dtype=torch.uint8, device="cuda")
            r1 = rsx.radix_sort(src, aux, None, kf)
            one = (r1.data_ptr() == aux.data_ptr(), r1.cpu().numpy().tobytes())
            out, _, in_aux, _ = gpu_sort_segments(rsx, torch, tname, data, offsets_of([n]))
            assert (in_aux, out.tobytes()) == one, (tname, n)
            ib = torch.zeros(2 * n, dtype=torch.int32, device="cuda")
            want = rsx.radix_sort_rank(to_dev(torch, data), ib, None, kf)
            want_aux = want.data_ptr() != ib.data_ptr()
            ranks, _, in_aux, _ = gpu_rank_segments(rsx, torch, tname, data, offsets_of([n]), np.uint32)
            assert in_aux == want_aux and np.array_equal(ranks, want.cpu().numpy().view(np.uint32)), (tname, n)


@gpu
def test_host_and_device_offsets_agree(rsx, torch):
    lengths = ragged_lengths(group_capacity(8, False), 31)
    offs = offsets_of(lengths)
    data = make_input("i64", int(offs[-1]), 8)
    a = gpu_sort_segments(rsx, torch, "i64", data, offs, device_offsets=False)
    b = gpu_sort_segments(rsx, torch, "i64", data, offs, device_offsets=True)
    assert a[0].tobytes() == b[0].tobytes() and a[2] == b[2] and a[1].ncols == b[1].ncols


@gpu
def test_launch_count_does_not_grow_with_segments(rsx, torch):
    counts = []
    for nseg in (1000, 100000):
        offs = offsets_of([8] * nseg)
        data = make_input("u32", int(offs[-1]), nseg)
        _, rep, _, _ = gpu_sort_segments(rsx, torch, "u32", data, offs)
        counts.append(rep.kernel_launches)
    assert counts[0] == counts[1] == 2, counts


@gpu
def test_runs_on_the_current_stream(rsx, torch):
    x = torch.randint(-2**31, 2**31 - 1, (300, 500), dtype=torch.int32, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        src = x.clone().view(-1)
        aux = torch.empty_like(src)
        res = rsx.radix_sort_segments(src, aux, torch.arange(0, 300 * 500 + 1, 500, device="cuda"))
        got = res.view(300, 500).clone()
    torch.cuda.synchronize()
    assert torch.equal(got, torch.sort(x, dim=1, stable=True).values)


@gpu
def test_rows_match_torch_sort(rsx, torch):
    B, Lr = 65536, 1024
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randint(-2**31, 2**31 - 1, (B, Lr), dtype=torch.int32, device="cuda", generator=g)
    offs = torch.arange(0, B * Lr + 1, Lr, dtype=torch.int64, device="cuda")
    want = torch.sort(x, dim=1, stable=True)
    src, aux = x.clone().view(-1), torch.empty(B * Lr, dtype=torch.int32, device="cuda")
    res = rsx.radix_sort_segments(src, aux, offs)
    assert torch.equal(res.view(B, Lr), want.values)
    ib = torch.empty(2 * B * Lr, dtype=torch.int32, device="cuda")
    ranks = rsx.radix_sort_rank_segments(x.view(-1), ib, offs)
    assert torch.equal(ranks.view(B, Lr).long(), want.indices)


@gpu
def test_offsets_beyond_32_bits(rsx, torch):
    """More than 2^32 u32 records in segments whose key ranges are disjoint and increasing: after the
    sort the whole array is ordered, which pins 64-bit offsets from the host plan to the kernels."""
    seg, width = 1024, 1000                 # keys of segment s lie in [s * width, (s + 1) * width)
    nseg = (2**32 + 2**20) // seg
    n = nseg * seg
    assert n > 2**32 and nseg * width < 2**32
    keys = torch.empty(n, dtype=torch.int32, device="cuda")
    chunk = 1 << 28
    for c0 in range(0, n, chunk):
        i = torch.arange(c0, min(n, c0 + chunk), dtype=torch.int64, device="cuda")
        h = (i * 1103515245 + 12345) % 2**31  # below 2^63 for every i here
        k = (i // seg) * width + (h % width)
        keys[c0:c0 + i.numel()] = (k - (k >= 2**31).long() * 2**32).to(torch.int32)
        del i, h, k
    kf = rsx.KeyFunc(rsx.KDF_UNSIGNED)
    before = rsx.verify(keys, kf)
    assert before[0] > 0
    aux = torch.empty_like(keys)
    offs = torch.arange(0, n + 1, seg, dtype=torch.int64, device="cuda")
    res = rsx.radix_sort_segments(keys, aux, offs, kf)
    d, s, x = rsx.verify(res, kf)
    assert d == 0 and (s, x) == before[1:]
    del keys, aux, res
    torch.cuda.empty_cache()
