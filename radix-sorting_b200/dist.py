"""Single-box multi-GPU partitioned radix sort (SURVEY.md section 8e, BASELINE config 5) -- the Python
launcher side.

The algorithm and its host orchestration live in C++ inside librsx.so (csrc/rsx_multi.cu,
`rsx_sort_shard` in include/rsx.h): histogram -> all-gather of the digit counts -> routing of the
top live digit's buckets (or of key ranges for skewed keys) -> fused partition + exchange into the
owners' receive buffers over NVLink (or local partition + all-to-all) -> local LSD sort.  The
concatenation of the ranks' outputs in rank order is bit-identical to `radix_sort` of the
concatenated input.

This module only supplies what a one-process-per-GPU launcher (torchrun) has and a C library has
not: the process group.  It wraps `torch.distributed` all-gather / barrier / all-to-all as the
`rsx_comm` callbacks, allocates the peer-mapped receive buffer with torch symmetric memory, and
calls `rsx_sort_shard`.  (A single process that owns all GPUs calls `rsx_sort_multi` instead, see
tools/radix_multi_b200.cpp.)

tests/test_dist.py runs the same C++ orchestration on CPU over gloo by passing oracle-backed local
primitives (`rsx_shard_ops`); the product path always uses the library's CUDA kernels (ops=None)
and fails without a GPU.
"""
from __future__ import annotations

import ctypes as C
import importlib
import time
from dataclasses import dataclass, field
from typing import Optional

import numpy as np


def _rsx():
    return importlib.import_module("radix-sorting_b200")


def derive_np(records: np.ndarray, L) -> np.ndarray:
    """Vectorised derived keys (uint64) of an (n, record_bytes) uint8 array
    (radix_sort_basic_kdf.hpp:19-46); used by tests to predict key-range destinations."""
    kb = L.key_bytes
    k = np.zeros(records.shape[0], dtype=np.uint64)
    for b in range(kb):
        k |= records[:, L.key_offset + b].astype(np.uint64) << np.uint64(8 * b)
    m = np.uint64((1 << (8 * kb)) - 1) if kb < 8 else np.uint64(0xFFFFFFFFFFFFFFFF)
    top = np.uint64(1 << (8 * kb - 1))
    if L.kdf_kind == 1:
        k ^= top
    elif L.kdf_kind == 2:
        k = np.where(k & top, k ^ m, k ^ top)
    if L.flags & 1:
        k = ~k & m
    return k


def choose_splitters(samples: np.ndarray, world: int):
    """world - 1 ascending derived-key splitters at the quantiles of the pooled samples
    (rsx_multi_splitters)."""
    s = np.ascontiguousarray(samples, dtype=np.uint64)
    out = (C.c_uint64 * (world - 1))()
    st = _rsx().lib().rsx_multi_splitters(s.ctypes.data_as(C.POINTER(C.c_uint64)), s.shape[0], world, out)
    assert st == 0
    return [int(x) for x in out]


def assign_buckets(global_counts: np.ndarray, world: int) -> np.ndarray:
    """Contiguous bucket ranges per rank balancing the counts: owner[b] = rank that receives
    bucket b (the routing table of rsx_multi_route for a one-column histogram)."""
    rsx = _rsx()
    hist = np.zeros((world, 1, 256), dtype=np.uint64)
    hist[0, 0] = np.asarray(global_counts, dtype=np.uint64)
    route = rsx.RsxRoute()
    st = rsx.lib().rsx_multi_route(hist.ctypes.data_as(C.POINTER(C.c_uint64)), world, 1, 0, 1e30, C.byref(route))
    assert st == 0
    return np.array(list(route.owner), dtype=np.int64)


@dataclass
class PartitionInfo:
    routing_column: Optional[int]  # None: nothing routed, -1: key-range routing
    n_out: int
    n_total: int
    imbalance: float
    fused: bool
    seconds: dict = field(default_factory=dict)
    append: bool = False


class _Buffers:
    """Grow-only work buffers per (device, dtype): the peer-mapped receive buffer (torch symmetric
    memory), a plain receive buffer for the all-to-all exchange, and -- when the caller's tensor has
    no slack -- a source copy with capacity."""
    symm = {}   # key -> (tensor, handle), or None once symmetric memory turned out to be unavailable
    gather = {}  # (bytes, world, device) -> staging buffers of the all-gather callback
    plain = {}
    src = {}
    symm_error = None


def _symmetric_recv(capacity_elems, like, group):
    """(tensor, [peer base addresses], handle) of >= capacity elements, or None where symmetric
    memory is unavailable (the exchange then goes through all_to_all_single)."""
    import torch.distributed as dist
    try:
        import torch.distributed._symmetric_memory as symm_mem
    except Exception as e:  # noqa: BLE001
        _Buffers.symm_error = repr(e)
        return None
    key = (like.dtype, like.device.index)
    if key in _Buffers.symm and _Buffers.symm[key] is None:
        return None  # failed before: do not retry on every call
    cur = _Buffers.symm.get(key)
    if cur is None or cur[0].numel() < capacity_elems:
        try:
            t = symm_mem.empty(int(capacity_elems), dtype=like.dtype, device=like.device)
            h = symm_mem.rendezvous(t, group=group if group is not None else dist.group.WORLD)
            cur = (t, h)
        except Exception as e:  # noqa: BLE001  (no fabric / P2P support)
            _Buffers.symm[key] = None
            _Buffers.symm_error = repr(e)
            return None
        _Buffers.symm[key] = cur
    t, h = cur
    return t, [int(p) for p in h.buffer_ptrs], h


def partitioned_sort(keys, kf, group=None, n: Optional[int] = None, ops=None, fused: bool = True,
                     key_range: bool = True, exact: bool = False):
    """Globally sorts the concatenation (in rank order) of every rank's first `n` records of `keys`
    (default: all of it).  Returns (this rank's slice of the sorted sequence, PartitionInfo).
    `keys` is clobbered; tensor capacity beyond `n` is used as working space (a tensor without
    slack costs one extra copy).  Collective: every rank of `group` must call it."""
    import torch
    import torch.distributed as dist
    rsx = _rsx()
    lib = rsx.lib()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = keys.device
    on_gpu = dev.type == "cuda"
    if on_gpu and ops is not None:
        raise ValueError("local primitives may only be substituted on CPU (tests)")
    if not on_gpu and ops is None:
        raise RuntimeError("the partitioned sort runs on CUDA devices; there is no CPU path")
    L = kf.layout(keys.element_size())
    rb = L.record_bytes
    esz = keys.element_size()
    rec_elems = rb // esz
    count = keys.numel() // rec_elems
    n = count if n is None else n
    stream = torch.cuda.current_stream(dev).cuda_stream if on_gpu else 0
    coll_dev = dev if on_gpu else torch.device("cpu")

    # ---- the launcher's collectives as rsx_comm callbacks ------------------------------------------
    state = {"handle": None, "src": None, "recv": None, "err": None}

    def cb_allgather(ctx, send, recv, nbytes):
        try:
            key = (nbytes, world, dev.index if on_gpu else -1)
            bufs = _Buffers.gather.get(key)
            if bufs is None:  # pinned staging + device tensors, reused by every later call
                pin_in = torch.empty(nbytes, dtype=torch.uint8, pin_memory=on_gpu)
                pin_out = torch.empty(world * nbytes, dtype=torch.uint8, pin_memory=on_gpu)
                dev_in = torch.empty(nbytes, dtype=torch.uint8, device=coll_dev) if on_gpu else pin_in
                dev_out = torch.empty(world * nbytes, dtype=torch.uint8, device=coll_dev) if on_gpu else pin_out
                bufs = _Buffers.gather[key] = (pin_in, pin_out, dev_in, dev_out)
            pin_in, pin_out, dev_in, dev_out = bufs
            C.memmove(pin_in.data_ptr(), send, nbytes)
            if on_gpu:
                dev_in.copy_(pin_in, non_blocking=True)
            dist.all_gather_into_tensor(dev_out, dev_in, group=group)
            if on_gpu:
                pin_out.copy_(dev_out, non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()
            C.memmove(recv, pin_out.data_ptr(), world * nbytes)
            return 0
        except Exception as e:  # noqa: BLE001
            state["err"] = e
            return rsx.RSX_ERR_CUDA

    def cb_barrier(ctx):
        try:
            if on_gpu:
                torch.cuda.synchronize(dev)
            if state["handle"] is not None:
                state["handle"].barrier()
            else:
                dist.barrier(group=group)
            return 0
        except Exception as e:  # noqa: BLE001
            state["err"] = e
            return rsx.RSX_ERR_CUDA

    def cb_alltoallv(ctx, send, sbytes, recv, rbytes):
        try:
            by_ptr = {state["src"].data_ptr(): state["src"], state["recv"].data_ptr(): state["recv"]}
            s_t, r_t = by_ptr[send].view(torch.uint8), by_ptr[recv].view(torch.uint8)
            ss, rs = [int(sbytes[d]) for d in range(world)], [int(rbytes[d]) for d in range(world)]
            dist.all_to_all_single(r_t[: sum(rs)], s_t[: sum(ss)], rs, ss, group=group)
            return 0
        except Exception as e:  # noqa: BLE001
            state["err"] = e
            return rsx.RSX_ERR_CUDA

    comm = rsx.RsxComm(rank, world, rsx.ALLGATHER_FN(cb_allgather), rsx.BARRIER_FN(cb_barrier),
                       rsx.ALLTOALLV_FN(cb_alltoallv), None)
    flags = (0 if key_range else rsx.MULTI_NO_KEY_RANGE) | (rsx.MULTI_EXACT if exact else 0)

    capacity = count  # records the caller's tensor can hold
    src = keys
    rep = rsx.RsxMultiReport()
    for attempt in range(3):
        cap_elems = capacity * rec_elems
        symm = _symmetric_recv(cap_elems, keys, group) if (fused and on_gpu) else None
        if fused and on_gpu:  # every rank must take the same branch
            ok = torch.tensor([1 if symm is not None else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
            if not int(ok.item()):
                symm = None
        if symm is not None:
            recv, bases, handle = symm
            peers = (C.c_void_p * world)(*bases)
            state["handle"] = handle
        else:
            key = (keys.dtype, dev.index if on_gpu else -1)
            cur = _Buffers.plain.get(key)
            if cur is None or cur.numel() < cap_elems:
                cur = torch.empty(cap_elems, dtype=keys.dtype, device=dev)
                _Buffers.plain[key] = cur
            recv, peers, state["handle"] = cur, None, None
        state["src"], state["recv"] = src, recv
        res_ptr, n_out = C.c_void_p(), C.c_size_t(0)
        st = lib.rsx_sort_shard(C.byref(comm), C.byref(ops) if ops is not None else None, src.data_ptr(), n, recv.data_ptr(), peers, capacity, C.byref(L),
                                flags | (0 if symm is not None else rsx.MULTI_NO_FUSED), C.byref(res_ptr), C.byref(n_out),
                                C.byref(rep), stream)
        if st == rsx.RSX_ERR_WORKSPACE and attempt < 2:
            # the routed sizes need more room than the tensors have (same verdict on every rank,
            # nothing was moved yet): grow once, with some slack for the next calls
            capacity = max(int(rep.needed_capacity * 1.03) + 1024, capacity + 1)
            skey = (keys.dtype, dev.index if on_gpu else -1)
            cur = _Buffers.src.get(skey)
            if cur is None or cur.numel() < capacity * rec_elems:
                cur = torch.empty(capacity * rec_elems, dtype=keys.dtype, device=dev)
                _Buffers.src[skey] = cur
            cur[: n * rec_elems].copy_(keys.view(-1)[: n * rec_elems])
            src = cur
            continue
        if state["err"] is not None:
            raise state["err"]
        if st != rsx.RSX_OK:
            raise rsx.RsxError(st, "rsx_sort_shard")
        break
    out_t = src if res_ptr.value == src.data_ptr() else recv
    res = out_t.view(-1)[: n_out.value * rec_elems]
    routing = None if (rep.routing_column < 0 and not rep.key_range) else (-1 if rep.key_range else int(rep.routing_column))
    sec = {"histogram+allgather": rep.seconds_histogram, "routing": rep.seconds_routing,
           "partition+exchange": rep.seconds_exchange, "local_sort": rep.seconds_local_sort,
           "exchange": ("fused peer stores (NVLink)" if rep.fused else "all_to_all_single") +
                       (", append mode (sampled routing, no histogram pass)" if rep.append else "") +
                       (", key-range routing" if rep.key_range else "")}
    return res, PartitionInfo(routing, int(n_out.value), int(rep.n_total), float(rep.imbalance), bool(rep.fused), sec,
                              bool(rep.append))


# -------------------------------------------------------------------------------------------------
def bench_partitioned(args, rsx, tname, n_per_gpu, dname, mask, orv, rank, world, dev, sampler=None):
    """bench.py's N > 1 arm: weak scaling, n_per_gpu keys per rank, device-timed, max over ranks."""
    import torch
    import torch.distributed as dist
    tdt = {"u32": torch.int32, "u64": torch.int64, "i32": torch.int32, "i64": torch.int64,
           "f32": torch.float32, "f64": torch.float64}[tname]
    kf = rsx.default_kdf(tdt) if tname[0] != "u" else rsx.KeyFunc(rsx.KDF_UNSIGNED)
    kb = torch.empty(0, dtype=tdt).element_size()
    pristine = torch.empty(n_per_gpu, dtype=tdt, device=dev)
    rsx.fill_keys(pristine, seed=2, start=rank * n_per_gpu, dist=dname, mask=mask, orv=orv)
    _, s0, x0 = rsx.verify(pristine, kf)
    chk0 = torch.tensor([s0 & 0x7FFFFFFFFFFFFFFF, x0 & 0x7FFFFFFFFFFFFFFF, n_per_gpu], dtype=torch.int64, device=dev)
    fused = not getattr(args, "no_fused", False)
    # working tensor with slack: the routed shard sizes differ a little from n_per_gpu
    keys = torch.empty(int(n_per_gpu * 1.04) + 4096, dtype=tdt, device=dev)
    times, last = [], None
    launches0 = 0
    for it in range(args.warmup + args.steps):
        keys[:n_per_gpu].copy_(pristine)
        if it == args.warmup:
            launches0 = rsx.total_kernel_launches()
            if sampler is not None:
                sampler.start()  # nvidia-smi clocks / throttle reasons over the timed steps
        dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res, info = partitioned_sort(keys, kf, n=n_per_gpu, fused=fused)
        e1.record()
        e1.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)  # device time, max over ranks
        if it >= args.warmup:
            times.append(float(ms.item()))
        last = (res, info)
    launches = rsx.total_kernel_launches() - launches0
    clocks = sampler.stop() if sampler is not None else None
    res, info = last
    # verification at full size: every shard ordered, shard boundaries ordered, multiset preserved
    d1, s1, x1 = rsx.verify(res, kf) if info.n_out > 1 else (0, 0, 0)
    def ordered(v):  # unsigned key stored in a signed tensor -> int64 with the same order
        v = v.to(torch.int64)
        return (v & 0xFFFFFFFF) if kb == 4 else (v ^ torch.tensor(-(1 << 63), dtype=torch.int64, device=dev))
    edge = torch.zeros(3, dtype=torch.int64, device=dev)
    if info.n_out:
        edge[0], edge[1], edge[2] = ordered(res.view(-1)[0]), ordered(res.view(-1)[-1]), 1
    edges = [torch.empty_like(edge) for _ in range(world)]
    dist.all_gather(edges, edge)
    nonempty = [e.cpu().tolist() for e in edges if int(e[2])]
    boundaries_ok = all(a[1] <= b[0] for a, b in zip(nonempty, nonempty[1:])) if tname[0] == "u" else True
    # multiset: sum is additive over shards, xor combines with xor
    chk1 = torch.tensor([s1 & 0x7FFFFFFFFFFFFFFF, x1 & 0x7FFFFFFFFFFFFFFF, info.n_out], dtype=torch.int64, device=dev)
    all0 = [torch.empty_like(chk0) for _ in range(world)]
    all1 = [torch.empty_like(chk1) for _ in range(world)]
    dist.all_gather(all0, chk0)
    dist.all_gather(all1, chk1)
    ok_sorted = torch.tensor([int(d1 == 0)], device=dev)
    dist.all_reduce(ok_sorted, op=dist.ReduceOp.MIN)
    n_in = sum(int(a[2]) for a in all0)
    n_outs = [int(a[2]) for a in all1]
    sum_ok = (sum(int(a[0]) for a in all0) - sum(int(a[0]) for a in all1)) % (1 << 63) == 0
    xor0 = xor1 = 0
    for a, b in zip(all0, all1):
        xor0 ^= int(a[1])
        xor1 ^= int(b[1])
    verified = bool(ok_sorted.item()) and n_in == sum(n_outs) and boundaries_ok and sum_ok and xor0 == xor1
    info_t = info  # rsx_sort_shard reports its own per-phase host-clock seconds
    # e2e: every rank's shard starts and ends in pinned HOST memory (H2D + global sort + D2H timed)
    e2e = None
    if not getattr(args, "no_e2e", False):
        h_in = h_out = None
        try:
            h_in = torch.empty(n_per_gpu, dtype=tdt, pin_memory=True)
            h_out = torch.empty(int(n_per_gpu * 1.25) + 1024, dtype=tdt, pin_memory=True)
            ok = 1
        except Exception:  # not enough pinnable host memory for N shards on this box
            ok = 0
        okt = torch.tensor([ok], device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)  # all ranks take the same branch
        if int(okt.item()):
            h_in.copy_(pristine)
            e2e_t = []
            for it in range(1 + args.steps):
                dist.barrier()
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                keys[:n_per_gpu].copy_(h_in, non_blocking=True)
                r_e, info_e = partitioned_sort(keys, kf, n=n_per_gpu, fused=fused)
                h_out[: info_e.n_out].copy_(r_e.view(-1)[: info_e.n_out], non_blocking=True)
                torch.cuda.synchronize(dev)
                dt = torch.tensor([time.perf_counter() - t0], device=dev)
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
                if it:
                    e2e_t.append(float(dt.item()))
            e2e_s = sum(e2e_t) / len(e2e_t)
            e2e = {"value": n_per_gpu * world / e2e_s / 1e9, "unit": "Gkeys/s", "h2d_bytes_per_step": n_per_gpu * kb * world,
                   "d2h_bytes_per_step": n_per_gpu * kb * world, "ms_per_step": e2e_s * 1e3, "steps": len(e2e_t),
                   "note": "per rank: pinned host shard -> device, partitioned global sort, sorted shard -> pinned host; wall clock, max over ranks"}
        else:
            e2e = {"value": None, "unit": "Gkeys/s", "error": "could not pin host memory for every rank's shard"}
        del h_in, h_out
    ms_per_step = sum(times) / len(times)
    n_total = n_per_gpu * world
    value = n_total / (ms_per_step * 1e-3) / 1e9
    single = n_per_gpu * kb * (1 + 2 * kb)  # local LSD sort bytes per GPU
    moved = n_per_gpu * kb * (1 + 2) + single  # + histogram read + partition pass
    return {
        "metric": "Gkeys/s sorted", "value": value, "unit": "Gkeys/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": tname, "data": "synthetic",
        "config": {"workload": f"{args.workload} per GPU, partitioned global sort over {world} GPUs",
                   "keys_total": n_total, "keys_per_gpu": n_per_gpu, "dist": dname, "routing_column": info.routing_column,
                   "imbalance_max_over_mean": max(n_outs) / (n_total / world), "verified": verified,
                   "timing": "CUDA events per rank around partitioned_sort, all_reduce MAX over ranks, mean of steps",
                   "l2": "inputs larger than L2, restored before every step",
                   "phase_seconds_rank0": info_t.seconds, "symm_error": _Buffers.symm_error,
                   "host_orchestration": "C++ rsx_sort_shard (csrc/rsx_multi.cu) with torch.distributed callbacks",
                   "ms_steps": [round(x, 3) for x in times]},
        "roofline": {"bound": "hbm", "kernel": "whole partitioned sort, per GPU", "achieved": moved / (ms_per_step * 1e-3) / 1e9,
                     "peak": None, "unit": "GB/s", "frac": None, "traffic": None,
                     "note": "per-GPU algorithmic HBM bytes (histogram + partition pass + local LSD) over the step time; "
                             "NVLink term: each GPU sends/receives (N-1)/N of its shard",
                     "nvlink_bytes_per_gpu": n_per_gpu * kb * (world - 1) / world},
        "cpu_baseline": None, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
    }
