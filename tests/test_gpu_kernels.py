"""Every single-GPU scatter kernel (K3) against the CPU oracle at sizes where each persistent CTA works
through several tiles.

The dispatch (csrc/rsx_scatter_dispatch.cuh) instantiates one kernel per footprint: record bytes
ES in {1, 2, 4, 8, 16} x payload lane PL in {0 value sort, 4 rank sort with <= 4-byte indices, 8 rank
sort with u64 indices} x digit mode (PLAIN, or FLOAT for ES >= 4) -- 24 footprints, each with 32- and
64-bit offsets and ticket or ballot ranking.  FOOTPRINTS below names, for every footprint, the
layouts that run it; a CPU test keeps that table in step with the dispatch.

The inputs aim at the code the small goldens never reach: tiles that share one digit which changes
from tile to tile (the hot-digit guess of the previous tile is wrong and 32 lanes hit one counter),
a partial last tile whose real records carry the padding's derived key, tile-multiple sizes, float
specials, descending order (the complement folded into digit extraction and into the padding),
unaligned buffers (plain loads instead of TMA), narrow index lanes at the top of their range, and
8-byte keys above 2^30 records.  Records carry their original position, so a misplaced tie shows.
"""
import os
import re
import zlib

import numpy as np
import pytest

from pyoracle import KDF_FLOAT, KDF_SIGNED, KDF_UNSIGNED, TYPES, ElemType
from test_gpu_large import _check_sorted_by_key_then_position
from test_gpu_parity import gpu_rank, gpu_sort, kf_for, to_dev

gpu = pytest.mark.gpu

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "radix-sorting_b200", "csrc")
N = 12_000_007  # 3.6 to 20 tiles per persistent CTA, depending on the footprint
K_TILES = 1000  # tile-multiple sizes: K_TILES * tile and K_TILES * tile + 1 records

# ---- layouts and the footprint table ------------------------------------------------------------------

LAYOUTS = {name: TYPES[name] for name in
           ["u8", "i8", "u16", "i16", "u32", "i32", "f32", "u64", "i64", "f64",
            "rec8_u32", "rec16_u64", "rec16_f64", "rec16_f32"]}
LAYOUTS.update({t.name: t for t in [
    # {u32 payload, i32 key}: a signed key in the upper half of an 8-byte word
    ElemType("rec8_i32hi", np.dtype([("payload", "<u4"), ("key", "<i4")]), 8, 4, 4, KDF_SIGNED, -1),
    # {u32 payload, f32 key}: a float key in the upper half of an 8-byte word
    ElemType("rec8_f32hi", np.dtype([("payload", "<u4"), ("key", "<f4")]), 8, 4, 4, KDF_FLOAT, -1),
    # {u64 payload, 4 pad bytes, i32 key}: a signed key in the upper half of the second 8-byte word
    ElemType("rec16_i32hi", np.dtype([("payload", "<u8"), ("pad", "V4"), ("key", "<i4")]), 16, 12, 4, KDF_SIGNED, -1),
]})

VALUE, RANK32, RANK64 = "value", "rank-u32", "rank-u64"
PL_OF = {VALUE: 0, RANK32: 4, RANK64: 8}          # make_plan: 1/2/4-byte indices travel in a 4-byte lane
IDX_OF = {RANK32: np.uint32, RANK64: np.uint64}
PLAIN, FLOAT = "plain", "float"


def footprint(t, kind):
    return (t.record_bytes, PL_OF[kind], FLOAT if t.kdf_kind == KDF_FLOAT else PLAIN)


# (ES, PL, digit mode) -> the (layout, kind) pairs that run that kernel; the first pair also runs the
# tile-multiple sizes.  Every layout of LAYOUTS appears at least once.
FOOTPRINTS = {
    (1, 0, PLAIN): [("u8", VALUE), ("i8", VALUE)],
    (1, 4, PLAIN): [("i8", RANK32)],
    (1, 8, PLAIN): [("u8", RANK64)],
    (2, 0, PLAIN): [("u16", VALUE), ("i16", VALUE)],
    (2, 4, PLAIN): [("u16", RANK32)],
    (2, 8, PLAIN): [("i16", RANK64)],
    (4, 0, PLAIN): [("u32", VALUE), ("i32", VALUE)],
    (4, 4, PLAIN): [("i32", RANK32)],
    (4, 8, PLAIN): [("u32", RANK64)],
    (4, 0, FLOAT): [("f32", VALUE)],
    (4, 4, FLOAT): [("f32", RANK32)],
    (4, 8, FLOAT): [("f32", RANK64)],
    (8, 0, PLAIN): [("rec8_u32", VALUE), ("rec8_i32hi", VALUE)],
    (8, 4, PLAIN): [("i64", RANK32)],
    (8, 8, PLAIN): [("u64", RANK64)],
    (8, 0, FLOAT): [("rec8_f32hi", VALUE), ("f64", VALUE)],
    (8, 4, FLOAT): [("f64", RANK32)],
    (8, 8, FLOAT): [("rec8_f32hi", RANK64)],
    (16, 0, PLAIN): [("rec16_u64", VALUE), ("rec16_i32hi", VALUE)],
    (16, 4, PLAIN): [("rec16_i32hi", RANK32)],
    (16, 8, PLAIN): [("rec16_u64", RANK64)],
    (16, 0, FLOAT): [("rec16_f32", VALUE), ("rec16_f64", VALUE)],
    (16, 4, FLOAT): [("rec16_f32", RANK32)],
    (16, 8, FLOAT): [("rec16_f64", RANK64)],
}

# Ticket-ranked passes of these footprints run the register-resident kernel with its own tile
# (PreferV2 / Cfg2 in rsx_scatter2.cuh); every other pass runs scatter_kernel (ScatterCfg).
TICKET_TILE = {(8, 0): 256 * 36, (4, 4): 256 * 32}


def tile_of(es, pl, ticket):
    if ticket and (es, pl) in TICKET_TILE:
        return TICKET_TILE[(es, pl)]
    return 512 * (22 if es + pl <= 4 else 192 // (es + pl))


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def test_footprint_table_covers_every_scatter_kernel():
    """FOOTPRINTS has exactly one row per footprint the dispatch can reach, and every pair in a row
    really runs that footprint (CPU only: read from the dispatch sources)."""
    api, disp = _src("rsx_api.cu"), _src("rsx_scatter_dispatch.cuh")
    es_all = {int(a) for a, b in re.findall(r"case (\d+): return launch_scatter_(\d+)\(sp", api) if a == b}
    pl_all = {int(b) for a, b in re.findall(r"case (\d+): return launch_scatter_pl<ES, (\d+)>", disp) if a == b}
    m = re.search(r"if constexpr \(((?:ES == \d+(?: \|\| )?)+)\) \{ // a float", disp)
    es_float = {int(x) for x in re.findall(r"ES == (\d+)", m.group(1))}
    assert (es_all, pl_all, es_float) == ({1, 2, 4, 8, 16}, {0, 4, 8}, {4, 8, 16})
    reachable = {(es, pl, PLAIN) for es in es_all for pl in pl_all} | \
                {(es, pl, FLOAT) for es in es_float for pl in pl_all}
    assert len(reachable) == 24
    assert set(FOOTPRINTS) == reachable, sorted(reachable ^ set(FOOTPRINTS))
    for fp, rows in FOOTPRINTS.items():
        assert rows, fp
        for lname, kind in rows:
            assert footprint(LAYOUTS[lname], kind) == fp, (lname, kind, fp)
    assert {lname for rows in FOOTPRINTS.values() for lname, _ in rows} == set(LAYOUTS)


def test_tile_table_matches_kernel_configs():
    """tile_of() mirrors ScatterCfg and the register-resident footprints (PreferV2 / Cfg2)."""
    s1, s2 = _src("rsx_scatter.cuh"), _src("rsx_scatter2.cuh")
    assert "CfgT<512, ((ES + PL <= 4) ? 22 : 192 / (ES + PL))" in s1
    v2 = re.findall(r"struct PreferV2<(\d+), (\d+)> \{\s*static constexpr bool value = true;\s*"
                    r"using Cfg = CfgT<(\d+), (\d+),", s2)
    assert {(int(a), int(b)): int(t) * int(i) for a, b, t, i in v2} == TICKET_TILE


# ---- inputs (numpy, seeded) ----------------------------------------------------------------------------

def _mask(kb):
    return np.uint64((1 << (8 * kb)) - 1)


def _rng(*key):
    return np.random.default_rng(zlib.crc32(repr(key).encode()))


def raw_from_derived(d, t, desc):
    """Key bits whose derived key (radix_sort_basic_kdf.hpp, complemented when descending) is `d`."""
    kb = t.key_bytes
    m, top = _mask(kb), np.uint64(1 << (8 * kb - 1))
    k = (~d & m) if desc else d.copy()
    if t.kdf_kind == KDF_SIGNED:
        k ^= top
    elif t.kdf_kind == KDF_FLOAT:
        k = np.where(k & top, k ^ top, k ^ m)
    return k.astype(f"<u{kb}")


def records(t, raw):
    """Scalars, or records with key = raw bits and the payload = original position."""
    if t.dtype.names is None:
        return raw.view(t.dtype).copy()
    out = np.zeros(raw.shape[0], dtype=t.dtype)
    out["key"] = raw.view(t.dtype["key"])
    payload = [f for f in t.dtype.names if f not in ("key", "pad")][0]
    out[payload] = np.arange(raw.shape[0], dtype=np.uint64).astype(t.dtype[payload])
    return out


def derived_runs(rng, n, kb, tile):
    """Runs of random length in [1, 3 tile]: each run has one random key whose lowest 0, 3 or 8 bits
    are random per record.  The upper columns are constant over a run, so in every pass whole stretches
    of a tile share one digit, and that digit changes from run to run."""
    lens = rng.integers(1, 3 * tile + 1, size=2 * n // tile + 16)
    while lens.sum() < n:
        lens = np.concatenate([lens, rng.integers(1, 3 * tile + 1, size=n // tile + 16)])
    vals = rng.integers(0, 1 << 64, size=lens.size, dtype=np.uint64, endpoint=False) & _mask(kb)
    low = (np.uint64(1) << rng.choice(np.array([0, 3, 8], dtype=np.uint64), size=lens.size)) - np.uint64(1)
    key = np.repeat(vals, lens)[:n]
    lm = np.repeat(low, lens)[:n]
    return (key & ~lm) | (rng.integers(0, 1 << 64, size=n, dtype=np.uint64, endpoint=False) & lm)


def derived_tied(rng, n, kb):
    """Random derived keys drawn from a pool of n / 16 values (ties for the stability check)."""
    pool = rng.integers(0, 1 << 64, size=max(n // 16, 1), dtype=np.uint64, endpoint=False) & _mask(kb)
    return pool[rng.integers(0, pool.size, size=n)]


def float_specials(rng, n, kb):
    """Raw float bits: random finite values, and at 1 % each +-0, +-inf, quiet and signalling NaNs of
    both signs with random mantissas, denormals of both signs."""
    if kb == 4:
        vals = (rng.standard_normal(n) * 10.0 ** rng.uniform(-30, 30, n)).astype(np.float32).view(np.uint32)
        bits, mant = 32, 23
    else:
        vals = (rng.standard_normal(n) * 10.0 ** rng.uniform(-300, 300, n)).view(np.uint64)
        bits, mant = 64, 52
    u = np.uint32 if kb == 4 else np.uint64
    sign, expo, quiet = u(1 << (bits - 1)), u(((1 << (bits - mant - 1)) - 1) << mant), u(1 << (mant - 1))
    pos = rng.permutation(n)[: 10 * (n // 100)].reshape(10, -1)
    m = pos.shape[1]
    specials = [
        np.full(m, 0, dtype=u), np.full(m, sign, dtype=u), np.full(m, expo, dtype=u), np.full(m, sign | expo, dtype=u),
        expo | quiet | rng.integers(0, int(quiet), m, dtype=u), sign | expo | quiet | rng.integers(0, int(quiet), m, dtype=u),
        expo | rng.integers(1, int(quiet), m, dtype=u), sign | expo | rng.integers(1, int(quiet), m, dtype=u),
        rng.integers(1, 1 << mant, m, dtype=u), sign | rng.integers(1, 1 << mant, m, dtype=u),
    ]
    for p, s in zip(pos, specials):
        vals[p] = s
    return vals


def tail_len(t, kind):
    """The last ceil(tile / 2) + 7 records carry the padding's derived key (the larger tile of the
    two rank modes, so that the partial last tile holds such records in every mode)."""
    es, pl = t.record_bytes, PL_OF[kind]
    return -(-max(tile_of(es, pl, True), tile_of(es, pl, False)) // 2) + 7


def make_data(t, kind, dist, n, desc):
    kb = t.key_bytes
    rng = _rng(t.name, kind, dist, n, desc)
    tile = tile_of(t.record_bytes, PL_OF[kind], False)
    if dist == "specials":
        return records(t, float_specials(rng, n, kb))
    if dist in ("runs", "runs-top"):
        d = derived_runs(rng, n, kb, tile)
        if dist == "runs-top":  # one live column: the top one
            d &= np.uint64(0xFF << (8 * (kb - 1)))
    elif dist == "tailmax":
        d = rng.integers(0, 1 << 64, size=n, dtype=np.uint64, endpoint=False) & _mask(kb)
        d[n - min(n, tail_len(t, kind)):] = _mask(kb)  # == pad_record()'s derived key
    elif dist == "reverse":
        d = np.sort(derived_tied(rng, n, kb))[::-1].copy()
    elif dist == "nearly":  # sorted, then 0.1 % random transpositions
        d = np.sort(derived_tied(rng, n, kb))
        i, j = rng.integers(0, n, size=(2, n // 1000))
        d[i], d[j] = d[j], d[i]
    else:
        raise ValueError(dist)
    return records(t, raw_from_derived(d, t, desc))


def test_inputs_carry_the_derived_keys_they_claim(oracle):
    """The builders are right by the oracle's own KDF (CPU only): raw_from_derived inverts it for every
    layout and direction, the tail of "tailmax" is the padding's derived key, "runs-top" leaves one
    live column."""
    rng = np.random.default_rng(5)
    for t in LAYOUTS.values():
        m = _mask(t.key_bytes)
        for desc in (False, True):
            L = t.layout(descending=desc)
            d = rng.integers(0, 1 << 64, 200, dtype=np.uint64, endpoint=False) & m
            data = records(t, raw_from_derived(d, t, desc))
            assert [oracle.kdf(data[i:i + 1], L) for i in range(200)] == [int(x) for x in d], (t.name, desc)
            kind = RANK32
            data = make_data(t, kind, "tailmax", 20011, desc)
            assert all(oracle.kdf(data[i:i + 1], L) == int(m) for i in range(20011 - tail_len(t, kind), 20011, 101))
            if t.key_bytes > 1:
                _, orep, _ = oracle.radix_sort_rank(make_data(t, kind, "runs-top", 200_003, desc), L)
                assert orep.ncols == 1, (t.name, desc)


_cache = {}


def _case(oracle, lname, kind, dist, n, desc):
    """Input + oracle answer, computed once and shared by the four modes (the oracle is the slow side)."""
    key = (lname, kind, dist, n, desc)
    if key not in _cache:
        t = LAYOUTS[lname]
        data = make_data(t, kind, dist, n, desc)
        if kind == VALUE:
            want, orep, _ = oracle.radix_sort(data, t.layout(descending=desc))
        else:
            want, orep, _ = oracle.radix_sort_rank(data, t.layout(descending=desc), IDX_OF[kind])
        while len(_cache) >= 3:  # a few cases resident: 12 M x 16 B x (input + answer) each
            _cache.pop(next(iter(_cache)))
        _cache[key] = (data, want, orep)
    return _cache[key]


def _first_diff(got, want, width):
    bad = np.flatnonzero((got.reshape(-1, width) != want.reshape(-1, width)).any(axis=1))
    return f"{bad.size} of {got.size // width} records differ, first at {bad[:4].tolist()}"


def compare_with_oracle(rsx, torch, oracle, lname, kind, dist, n, desc):
    data, want, orep = _case(oracle, lname, kind, dist, n, desc)
    t = LAYOUTS[lname]
    what = f"{lname} {kind} {dist} n={n} {'desc' if desc else 'asc'}"
    if kind == VALUE:
        out, rep, in_aux = gpu_sort(rsx, torch, t, data, desc)
        wb = want.view(np.uint8).reshape(-1)
        assert np.array_equal(out, wb), f"{what}: {_first_diff(out, wb, t.record_bytes)}"
        assert int(in_aux) == orep.result_in_aux, what
    else:
        ranks, rep, ib = gpu_rank(rsx, torch, t, data, IDX_OF[kind], desc)
        assert np.array_equal(ranks, want), f"{what}: {_first_diff(ranks, want, 1)}"
        assert np.array_equal(ib[n:] if orep.result_in_aux else ib[:n], want), f"{what}: not in the designated half"
    assert (rep.ncols, rep.result_in_aux, rep.early_exit) == (orep.ncols, orep.result_in_aux, orep.early_exit), what


# ---- GPU side --------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the product has no CPU path (run with -m gpu on the GPU box)")
    return torch


@pytest.fixture
def modes(request, rsx):
    """Rank mode x offset width, restored afterwards.  Parametrized indirectly by the LAST decorator,
    so the four modes of one case run back to back and share its oracle answer."""
    rank_mode, wide = request.param
    try:
        assert rsx.lib().rsx_set_option(b"rank_mode", rank_mode) == 0
        assert rsx.lib().rsx_set_option(b"force_wide", wide) == 0
        yield request.param
    finally:
        rsx.lib().rsx_set_option(b"rank_mode", -1)
        rsx.lib().rsx_set_option(b"force_wide", 0)


all_modes = pytest.mark.parametrize("modes", [(0, 0), (1, 0), (0, 1), (1, 1)], indirect=True,
                                    ids=["ticket", "ballot", "ticket-wide", "ballot-wide"])
both_dirs = pytest.mark.parametrize("desc", [False, True], ids=["asc", "desc"])

CASES = [(lname, kind, dist)
         for rows in FOOTPRINTS.values() for lname, kind in rows
         for dist in ["runs", "tailmax"]
         + (["specials"] if LAYOUTS[lname].kdf_kind == KDF_FLOAT else [])
         + (["runs-top"] if kind != VALUE and LAYOUTS[lname].key_bytes > 1 else [])]


@gpu
@all_modes
@both_dirs
@pytest.mark.parametrize("lname,kind,dist", CASES, ids=["-".join(c) for c in CASES])
def test_every_footprint_many_tiles(rsx, torch, oracle, lname, kind, dist, desc, modes):
    compare_with_oracle(rsx, torch, oracle, lname, kind, dist, N, desc)


ORDERED = [("i8", RANK32), ("i16", RANK64), ("f32", RANK32), ("rec8_i32hi", VALUE), ("rec16_f64", VALUE)]


@gpu
@all_modes
@both_dirs
@pytest.mark.parametrize("dist", ["reverse", "nearly"])
@pytest.mark.parametrize("lname,kind", ORDERED, ids=["-".join(c) for c in ORDERED])
def test_reverse_and_nearly_sorted(rsx, torch, oracle, lname, kind, dist, desc, modes):
    compare_with_oracle(rsx, torch, oracle, lname, kind, dist, N, desc)


FIRST = [(fp, rows[0][0], rows[0][1]) for fp, rows in FOOTPRINTS.items()]


@gpu
@all_modes
@pytest.mark.parametrize("extra", [0, 1], ids=["k-tiles", "k-tiles+1"])
@pytest.mark.parametrize("fp,lname,kind", FIRST, ids=["-".join(c[1:]) for c in FIRST])
def test_tile_multiple_sizes(rsx, torch, oracle, fp, lname, kind, extra, modes):
    """n = K tiles (no partial tile) and K tiles + 1 (a last tile of one real record, which carries the
    padding's derived key), descending: the tile of the kernel that runs in this mode."""
    n = K_TILES * tile_of(fp[0], fp[1], modes[0] == 0) + extra
    compare_with_oracle(rsx, torch, oracle, lname, kind, "tailmax", n, True)


UNALIGNED = [(lname, kind) for lname in ["u8", "i16", "f32", "rec8_u32"] for kind in (VALUE, RANK32)]


@gpu
@pytest.mark.parametrize("rank_mode", [0, 1], ids=["ticket", "ballot"])
@pytest.mark.parametrize("lname,kind", UNALIGNED, ids=["-".join(c) for c in UNALIGNED])
def test_unaligned_buffers_many_tiles(rsx, torch, oracle, lname, kind, rank_mode):
    """src (and aux) element-aligned but not 16-byte aligned: every tile of the passes that read them
    takes the plain-load branch instead of the TMA bulk copy."""
    t = LAYOUTS[lname]
    rb = t.record_bytes
    data, want, orep = _case(oracle, lname, kind, "runs", N, False)

    def unaligned():
        base = torch.full(((N + 2) * rb,), 0xCD, dtype=torch.uint8, device="cuda")
        v = base[rb: rb + N * rb]
        assert v.data_ptr() % 16 != 0
        return v

    src = unaligned()
    src.copy_(to_dev(torch, data))
    try:
        assert rsx.lib().rsx_set_option(b"rank_mode", rank_mode) == 0
        rep = rsx.RsxReport()
        if kind == VALUE:
            aux = unaligned()
            res = rsx.radix_sort(src, aux, None, kf_for(rsx, t), report=rep)
            torch.cuda.synchronize()
            assert (res.data_ptr() == aux.data_ptr()) == bool(orep.result_in_aux)
            got, wb = res.cpu().numpy(), want.view(np.uint8).reshape(-1)
            assert np.array_equal(got, wb), _first_diff(got, wb, rb)
        else:
            ib = torch.full((2 * N,), -1, dtype=torch.int32, device="cuda")
            ranks = rsx.radix_sort_rank(src, ib, N, kf_for(rsx, t), report=rep)
            torch.cuda.synchronize()
            assert ranks.data_ptr() == ib.data_ptr() + (4 * N if orep.result_in_aux else 0)
            got = ranks.cpu().numpy().view(np.uint32)
            assert np.array_equal(got, want), _first_diff(got, want, 1)
    finally:
        rsx.lib().rsx_set_option(b"rank_mode", -1)
    assert (rep.ncols, rep.result_in_aux) == (orep.ncols, orep.result_in_aux)


@gpu
@both_dirs
@pytest.mark.parametrize("dist", ["tied", "top-column", "sorted"])
@pytest.mark.parametrize("idt,n", [(np.uint8, 256), (np.uint16, 65536)], ids=["u8-256", "u16-65536"])
@pytest.mark.parametrize("lname", ["u16", "u32", "f64", "rec8_i32hi", "rec16_f32"])
def test_narrow_index_lanes_at_their_limit(rsx, torch, oracle, lname, idt, n, dist, desc):
    """Rank sorts with u8 indices at n = 256 and u16 indices at n = 65 536 (the largest n each can
    index): the passes carry 32-bit indices that the last step narrows.  Even column counts (all
    columns live), odd ones (only the top column), and an early exit (identity in the first half);
    through the single-CTA kernel and the multi-kernel path."""
    t = LAYOUTS[lname]
    kb = t.key_bytes
    rng = _rng(lname, n, dist, desc)
    d = derived_tied(rng, n, kb)
    if dist == "top-column":
        d &= np.uint64(0xFF << (8 * (kb - 1)))
    elif dist == "sorted":
        d = np.sort(d)
    data = records(t, raw_from_derived(d, t, desc))
    want, orep, _ = oracle.radix_sort_rank(data, t.layout(descending=desc), idt)
    assert orep.ncols == {"tied": kb, "top-column": 1, "sorted": 0}[dist]
    for small in (1, 0):
        try:
            assert rsx.lib().rsx_set_option(b"small_path", small) == 0
            ranks, rep, ib = gpu_rank(rsx, torch, t, data, idt, desc)
        finally:
            rsx.lib().rsx_set_option(b"small_path", 1)
        what = (lname, dist, desc, small)
        assert np.array_equal(ranks, want), what
        assert np.array_equal(ib[n:] if orep.result_in_aux else ib[:n], want), what
        assert (rep.ncols, rep.result_in_aux, rep.early_exit) == (orep.ncols, orep.result_in_aux, orep.early_exit), what
        if orep.early_exit:  # radix_sort_rank.hpp:52-57
            assert np.array_equal(ib[:n], np.arange(n, dtype=idt)), what


# ---- 64-bit offsets at their natural size for 8-byte keys ------------------------------------------------

N_WIDE = (1 << 30) + 12345


@gpu
@pytest.mark.parametrize("rank_mode", [0, 1], ids=["ticket", "ballot"])
@pytest.mark.parametrize("kind,desc", [(KDF_UNSIGNED, False), (KDF_UNSIGNED, True), (KDF_FLOAT, True)],
                         ids=["u64-asc", "u64-desc", "f64-desc"])
def test_8_byte_keys_above_2_pow_30(rsx, torch, kind, desc, rank_mode):
    """n >= 2^30 switches every pass to 64-bit look-back words and offsets; for 8-byte keys the
    ticket-ranked pass is scatter2_kernel.  Checked by properties: no descent of the derived key and
    the multiset checksum unchanged."""
    src = torch.empty(N_WIDE, dtype=torch.int64, device="cuda")
    rsx.fill_keys(src, seed=29)
    if kind == KDF_FLOAT:
        src = src.view(torch.float64)
    aux = torch.empty_like(src)
    kf = rsx.KeyFunc(kind, desc)
    d0, s0, x0 = rsx.verify(src, kf)
    assert d0 > 0
    rep = rsx.RsxReport()
    try:
        assert rsx.lib().rsx_set_option(b"rank_mode", rank_mode) == 0
        res = rsx.radix_sort(src, aux, None, kf, report=rep)
    finally:
        rsx.lib().rsx_set_option(b"rank_mode", -1)
    d1, s1, x1 = rsx.verify(res, kf)
    assert d1 == 0 and (s1, x1) == (s0, x0)
    assert rep.ncols == 8 and res.data_ptr() == src.data_ptr()


@gpu
def test_rank_sort_u64_indices_above_2_pow_30(rsx, torch):
    """u32 keys (3 live columns, ~64 ties per key) ranked with u64 indices at n > 2^30: ordered by
    (key, original position) and a permutation, in the second half of the index buffer."""
    n = N_WIDE
    keys = torch.empty(n, dtype=torch.int32, device="cuda")
    rsx.fill_keys(keys, seed=31, mask=0x00FFFFFF)
    ib = torch.empty(2 * n, dtype=torch.int64, device="cuda")
    rep = rsx.RsxReport()
    ranks = rsx.radix_sort_rank(keys, ib, n, rsx.KeyFunc(rsx.KDF_UNSIGNED), report=rep)
    assert rep.ncols == 3 and ranks.data_ptr() == ib.data_ptr() + 8 * n

    def key_at(lo, hi):
        return torch.gather(keys, 0, ranks[lo:hi]).to(torch.int64) & 0xFFFFFFFF

    _check_sorted_by_key_then_position(torch, key_at, lambda lo, hi: ranks[lo:hi], n)
    seen = torch.zeros(n, dtype=torch.bool, device="cuda")
    for lo in range(0, n, 1 << 27):
        seen[ranks[lo:lo + (1 << 27)]] = True
    assert bool(seen.all()), "ranks are not a permutation of 0..n-1"
