#!/usr/bin/env python
"""bench.py -- headline benchmark: Gkeys/s sorted on B200, next to the HBM roofline and the
reference's CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference]
                    [--dump-outputs DIR]

One "step" = one complete sort of the workload (histogram + setup + every live scatter pass)
through the C ABI (librsx.so).  The input is restored from a pristine device copy OUTSIDE the
timed region before every step (the reference's own Google-Benchmark loop forgets to do this,
radix_bench.cpp:91-93, SURVEY.md §6); each step is timed with CUDA events on the launch stream.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.

--dump-outputs DIR writes a fixed, seeded sample of what the last timed step returned, per
workload, so that two builds can be compared output for output (see dump_sample).
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

_M64 = (1 << 64) - 1
# name -> (element type, keys per GPU, dist, mask, orv, live passes)
WORKLOADS = {
    "1B-u32-uniform": ("u32", 1_000_000_000, "uniform", _M64, 0, 4),       # BASELINE configs[1] (u32 half)
    "1B-u64-uniform": ("u64", 1_000_000_000, "uniform", _M64, 0, 8),       # BASELINE configs[1] (u64 half)
    "40M-u32-uniform": ("u32", 40_000_000, "uniform", _M64, 0, 4),         # BASELINE configs[0]
    "256M-u32-uniform": ("u32", 256_000_000, "uniform", _M64, 0, 4),       # profiling size (ncu replays)
    "256M-u64-uniform": ("u64", 256_000_000, "uniform", _M64, 0, 8),
    "1B-u32-mask24": ("u32", 1_000_000_000, "uniform", 0x00FFFFFF, 0, 3),  # column skipping, README.md:889-891
    "1B-u32-nibbles": ("u32", 1_000_000_000, "uniform", 0x0F0F0F0F, 0, 4),  # N4: 16 varying bits in 4 live byte columns
    "1B-u64-nibbles": ("u64", 1_000_000_000, "uniform", 0x0F0F0F0F0F0F0F0F, 0, 8),
    "1B-u64-consthi": ("u64", 1_000_000_000, "uniform", 0x000000FFFFFFFFFF, 0xAA00000000000000, 5),
    "500M-f32": ("f32", 500_000_000, "uniform", _M64, 0, 4),               # BASELINE configs[2]
    "500M-i64": ("i64", 500_000_000, "uniform", _M64, 0, 8),
    "2B-u64-uniform": ("u64", 2_000_000_000, "uniform", _M64, 0, 8),       # per-GPU shard of configs[4]
    "2B-u64-zipf": ("u64", 2_000_000_000, "zipf", _M64, 0, 4),             # configs[4], skewed: P(v) ~ 1/v, v < 2^32
    "1B-u32-zipf": ("u32", 1_000_000_000, "zipf", _M64, 0, 4),
    "8B-u64-uniform": ("u64", 8_000_000_000, "uniform", _M64, 0, 8),       # strong-scaling base: 8 B keys on ONE GPU
    "4B-u64-uniform": ("u64", 4_000_000_000, "uniform", _M64, 0, 8),
}
CPU_SAMPLE_KEYS = {4: 256_000_000, 8: 96_000_000}  # bounded CPU sample, ~10-30 s of single-core work


def _torch_dtype(torch, tname):
    return {"u32": torch.int32, "u64": torch.int64, "i32": torch.int32, "i64": torch.int64,
            "f32": torch.float32, "f64": torch.float64}[tname]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()  # the exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


SEED = 2  # every arm sorts the same stream: key i = keygen(SEED, i)


def load_keygen():
    """keygen.py by file path: the reference arm must not import the product package, whose
    __init__ dlopens librsx.so."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("rsx_keygen", os.path.join(ROOT, "radix-sorting_b200", "keygen.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


class CpuReference:
    """The reference's CPU radix_sort (oracle/_ref when present, else the oracle port) on one core --
    the reference is single-threaded by construction.  The sample is the first n keys of the stream
    the GPU arm sorts (same seed, same bytes); both buffers are pre-faulted before the timed call
    (the stock `./radix` malloc path counts the aux page faults, SURVEY.md §3.3)."""

    def __init__(self, tname, n, dist, mask, orv):
        import numpy as np
        import pyoracle
        keygen = load_keygen()
        self.np, self.t, self.n, self.tname, self.dist = np, pyoracle.TYPES[tname], n, tname, dist
        keys = np.empty(n, dtype=f"<u{self.t.key_bytes}")
        CH = 1 << 24
        for s in range(0, n, CH):
            keys[s:s + CH] = keygen.fill(SEED, s, min(CH, n - s), self.t.key_bytes, dist, mask, orv)
        self.src = keys.view(self.t.dtype)
        self.work = np.empty_like(self.src)
        self.aux = np.zeros_like(self.src)
        try:
            os.sched_setaffinity(0, {sorted(os.sched_getaffinity(0))[0]})
        except Exception:
            pass
        if os.path.exists(pyoracle.LIB_REF):
            self.ref, self.kind = pyoracle.Ref(), "reference"
        else:
            self.ref, self.kind = pyoracle.Oracle(), "port"
        self.out = None

    def run(self):
        """One timed radix_sort call; returns seconds.  self.out is the sorted array."""
        import ctypes as C
        np = self.np
        np.copyto(self.work, self.src)
        self.aux[:] = 0
        if self.kind == "reference":
            t0 = time.perf_counter()
            in_aux = self.ref.radix_sort_inplace(self.t, self.work, self.aux)
            dt = time.perf_counter() - t0
        else:
            L = self.t.layout()
            t0 = time.perf_counter()
            resp = self.ref.L.orc_radix_sort(self.work.ctypes.data_as(C.c_void_p), self.aux.ctypes.data_as(C.c_void_p),
                                             self.n, C.byref(L), None, None)
            dt = time.perf_counter() - t0
            in_aux = resp == self.aux.ctypes.data
        self.out = self.aux if in_aux else self.work
        return dt

    def describe(self, seconds, repeats):
        return {"value": self.n / seconds / 1e9, "unit": "Gkeys/s", "cores": 1, "kind": self.kind,
                "sample": f"first {self.n} keys of the {self.tname} stream the GPU arm sorts (seed {SEED}, {self.dist}), "
                          f"one radix_sort call, buffers pre-faulted, best of {repeats}",
                "sample_keys": self.n, "seconds": seconds, "host_cpus": os.cpu_count(),
                "build": ("oracle/_ref: the unmodified reference headers, g++ -O3 -march=x86-64-v3 -funroll-loops (built in "
                          "the CPU container for the GPU box's host, hence not -march=native)")
                if self.kind == "reference" else "oracle/rsx_oracle.c port"}


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    tname, n_full, dist, mask, orv, passes = WORKLOADS[args.workload]
    import pyoracle
    kb = pyoracle.TYPES[tname].key_bytes
    # Each step is a bounded sample: the reference needs ~25-45 s for 1 B u32 keys on one core, and
    # K + W steps must end within a few minutes.  The rate is per key, the sample is stated.
    budget_s = 150.0
    per_key_s = {1: 1 / 150e6, 2: 1 / 80e6, 4: 1 / 40e6, 8: 1 / 12e6}[kb]
    n = int(min(n_full, CPU_SAMPLE_KEYS[kb], max(1 << 22, budget_s / max(1, args.warmup + args.steps) / per_key_s)))
    cpu = CpuReference(tname, n, dist, mask, orv)
    times = []
    for i in range(args.warmup + args.steps):
        dt = cpu.run()
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    val = n / (ms / 1e3) / 1e9
    desc = cpu.describe(ms / 1e3, 1)
    desc["sample"] = f"first {n} of {n_full} {tname} keys per step (seed {SEED}), one radix_sort call per step, mean of steps"
    print(json.dumps({
        "impl": "reference", "metric": "Gkeys/s sorted", "value": val, "unit": "Gkeys/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": tname, "data": "synthetic",
        "config": {"workload": args.workload, "keys": n_full, "keys_per_step": n, "same_config": n == n_full,
                   "note": "reference CPU path, 1 core (single-threaded by construction); each step sorts the first "
                           "keys_per_step keys of the workload's stream (bounded sample; Gkeys/s is a per-key rate)"},
        "cpu_baseline": desc,
        "e2e": {"value": val, "unit": "Gkeys/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def load_traffic(kb):
    """DRAM bytes of one scatter launch from the committed ncu --set full capture (newest round first)."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", name)))["scatter_kernel"]["u32" if kb == 4 else "u64"]
            return tj, name
        except Exception:
            continue
    return None, None


DUMP_SEED = 20261020
DUMP_SAMPLE = 1 << 20  # positions per workload: two workloads of <= 8-byte keys stay under 48 MiB


def dump_sample(out_dir, workload, res):
    """Writes DIR/<workload>_sorted.npy: the key bits of the sorted output at a fixed, seeded sample
    of positions (all of them for small n).  Each 32-bit word is one float64 (exact), an 8-byte key
    gives two columns, low word first: equal arrays mean equal bytes, NaN bit patterns of float
    keys included.  DIR/<workload>_index.npy holds the sampled positions; it carries no output
    and is the same in every build, it only says where each row of _sorted was read."""
    import numpy as np
    import torch
    n = res.numel()
    if n <= DUMP_SAMPLE:
        idx = np.arange(n, dtype=np.int64)
    else:
        idx = np.unique(np.random.default_rng(DUMP_SEED).integers(0, n, size=DUMP_SAMPLE, dtype=np.int64))
    vals = res[torch.from_numpy(idx).to(res.device)].cpu().numpy()
    words = vals.view(np.uint32).reshape(idx.shape[0], -1)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"{workload}_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, f"{workload}_sorted.npy"), words.astype(np.float64))


def bench_single(args, rsx, torch, workload, dev, steps, warmup, do_e2e, do_cpu):
    """One workload on one GPU: device-resident steps (value), per-kernel roofline, optional e2e
    through host buffers and the CPU reference beside it.  Returns the JSON-able dict."""
    import numpy as np
    tname, n, dname, mask, orv, passes = WORKLOADS[workload]
    tdt = _torch_dtype(torch, tname)
    kf = rsx.default_kdf(tdt) if tname[0] != "u" else rsx.KeyFunc(rsx.KDF_UNSIGNED)
    kb = torch.empty(0, dtype=tdt).element_size()

    # three full-size buffers (pristine, src, aux) do not fit for the 8 B-key strong-scaling base:
    # there the input is regenerated in place before every step instead of copied back
    regen = 3 * n * kb > 0.8 * torch.cuda.get_device_properties(dev).total_memory
    src = torch.empty(n, dtype=tdt, device=dev)
    aux = torch.empty_like(src)
    if regen:
        pristine = None

        def restore():
            rsx.fill_keys(src, seed=SEED, dist=dname, mask=mask, orv=orv)
    else:
        pristine = torch.empty_like(src)
        rsx.fill_keys(pristine, seed=SEED, dist=dname, mask=mask, orv=orv)

        def restore():
            src.copy_(pristine)
    restore()
    rsx.reserve(rsx.workspace_bytes(n, kf.layout(kb)))
    rsx.set_profile(True)
    rsx.lib().rsx_set_option(b"rank_mode", args.rank_mode)
    rsx.lib().rsx_set_option(b"scatter_variant", args.variant)
    rank_mode = {0: "ticket", 1: "ballot"}[rsx.lib().rsx_set_option(b"query_rank_mode", 0)]
    d0, s0, x0 = rsx.verify(src, kf)

    def step():
        restore()  # outside the events; also evicts L2 (4-64 GB >> 126 MB)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        rep = rsx.RsxReport()
        e0.record()
        res = rsx.radix_sort(src, aux, None, kf, report=rep)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1), rep, res, rsx.get_profile()

    for _ in range(warmup):
        _, rep, res, _ = step()
    d1, s1, x1 = rsx.verify(res, kf)
    assert d1 == 0 and (s1, x1) == (s0, x0), "warm-up result is not a sorted permutation of the input"
    assert rep.ncols == passes, (rep.ncols, passes)

    sampler = ClockSampler(dev.index or 0)
    torch.cuda.synchronize()
    sampler.start()
    launches0 = rsx.total_kernel_launches()
    times, profs = [], []
    torch.cuda.synchronize()
    for _ in range(steps):
        ms, rep, res, prof = step()
        times.append(ms)
        profs.append(prof)
    torch.cuda.synchronize()
    launches = rsx.total_kernel_launches() - launches0
    clocks = sampler.stop()
    d1, s1, x1 = rsx.verify(res, kf)
    verified = d1 == 0 and (s1, x1) == (s0, x0)
    assert verified, "timed result is not a sorted permutation of the input"
    if args.dump_outputs:
        dump_sample(args.dump_outputs, workload, res)

    ms_per_step = sum(times) / len(times)
    value = n / (ms_per_step * 1e-3) / 1e9

    # ---- roofline of the dominant kernel: the scatter pass (K3) --------------------------------
    peak, peak_src = measured_peak()
    ran = (lambda c: c < rep.compacted_passes) if rep.compacted_passes else (lambda c: (rep.live_mask >> c) & 1)
    pass_ms = [p[2 + c] for p in profs for c in range(kb) if len(p) > 2 + c and p[2 + c] > 0 and ran(c)]
    hist_ms = [p[0] for p in profs if p]
    avg_pass = sum(pass_ms) / len(pass_ms)
    alg_bytes_pass = 2 * n * kb  # read n records + write n records (SURVEY.md §8d: 2K per key per pass)
    achieved = alg_bytes_pass / (avg_pass * 1e-3) / 1e9
    alg_bytes_sort = n * kb * (1 + 2 * passes)
    traffic, traffic_src = None, None
    tj, tname_file = load_traffic(kb)
    if tj:  # DRAM bytes of this kernel from the committed ncu --set full capture, scaled to this n
        traffic = (tj["dram_bytes_read"] + tj["dram_bytes_write"]) * n / tj["keys"]
        traffic_src = (f"dram__bytes_read.sum + dram__bytes_write.sum of one launch at {tj['keys']} keys "
                       f"(profiles/{tname_file}), scaled by n")
    hist_avg = sum(hist_ms) / len(hist_ms)
    roofline = {
        "bound": "hbm", "kernel": "scatter_kernel (K3, one launch per live column)",
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
        "traffic_source": traffic_src,
        "peak_source": peak_src, "alg_bytes_per_launch": alg_bytes_pass, "ms_per_launch": avg_pass,
        "launches_timed": len(pass_ms), "share_of_step": avg_pass * (rep.compacted_passes or passes) / ms_per_step,
        "key_compaction_passes": int(rep.compacted_passes) or None,
        "histogram_kernel": {"ms": hist_avg, "alg_bytes": n * kb, "achieved": n * kb / (hist_avg * 1e-3) / 1e9,
                             "frac": n * kb / (hist_avg * 1e-3) / 1e9 / peak},
        "whole_sort": {"alg_bytes": alg_bytes_sort, "achieved": alg_bytes_sort / (ms_per_step * 1e-3) / 1e9,
                       "frac": alg_bytes_sort / (ms_per_step * 1e-3) / 1e9 / peak,
                       "frac_of_nominal_8TBs": alg_bytes_sort / (ms_per_step * 1e-3) / 1e9 / 8000.0},
    }

    # ---- e2e: the same sort through the C ABI with HOST buffers (H2D + sort + D2H timed) ----------
    e2e = None
    if do_e2e and not regen:
        res_dev = res.clone()  # the device-resident answer, to memcmp the e2e output against
        del src, aux
        torch.cuda.empty_cache()
        h_src = torch.empty(n, dtype=tdt, pin_memory=True)
        h_aux = torch.empty(n, dtype=tdt, pin_memory=True)
        h_pristine = pristine.cpu()
        e2e_steps = steps
        e2e_times = []
        for i in range(1 + e2e_steps):
            h_src.copy_(h_pristine)
            t0 = time.perf_counter()
            res_h = rsx.radix_sort(h_src, h_aux, None, kf)
            dt = time.perf_counter() - t0
            if i:
                e2e_times.append(dt)
        e2e_ok = bool(torch.equal(res_h.to(dev).view(torch.uint8), res_dev.view(torch.uint8)))
        assert e2e_ok, "e2e (host-buffer) result differs from the device-resident result"
        e2e_s = sum(e2e_times) / len(e2e_times)
        e2e = {"value": n / e2e_s / 1e9, "unit": "Gkeys/s", "h2d_bytes_per_step": n * kb, "d2h_bytes_per_step": n * kb,
               "ms_per_step": e2e_s * 1e3, "steps": len(e2e_times), "verified": e2e_ok,
               "note": "rsx_sort on pinned HOST buffers: H2D + sort + D2H inside the timed call (wall clock, mean); the "
                       "three phases are serial (a radix sort needs every key before its first pass), so the two PCIe "
                       "copies are most of it; output memcmp-equal to the device-resident result"}
        del h_src, h_aux, h_pristine, res_dev, res_h
    else:
        del src, aux

    # ---- the CPU reference beside it, on the same bytes, and a memcmp of the two outputs -----------
    cpu = None
    if do_cpu:
        ns = min(n, CPU_SAMPLE_KEYS[kb])
        ref = CpuReference(tname, ns, dname, mask, orv)
        reps = 2
        best = min(ref.run() for _ in range(reps))
        cpu = ref.describe(best, reps)
        # BASELINE.md §3.4: identical bytes.  Sort the same sample on the GPU and memcmp.
        torch.cuda.empty_cache()
        g_src = torch.empty(ns, dtype=tdt, device=dev)
        rsx.fill_keys(g_src, seed=SEED, dist=dname, mask=mask, orv=orv)
        assert g_src[:1 << 20].cpu().numpy().tobytes() == ref.src[:1 << 20].tobytes(), "host and device key streams differ"
        g_res = rsx.radix_sort(g_src, torch.empty_like(g_src), None, kf)
        same = g_res.cpu().numpy().tobytes() == np.ascontiguousarray(ref.out).tobytes()
        assert same, "GPU output differs from the CPU reference's output on the same input"
        cpu["gpu_output_memcmp_equal"] = bool(same)
        del g_src, g_res, ref

    del pristine
    torch.cuda.empty_cache()
    return {
        "metric": "Gkeys/s sorted", "value": value, "unit": "Gkeys/s", "n_gpus": 1, "steps": steps,
        "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": tname, "data": "synthetic",
        "config": {"workload": workload, "keys": n, "key_bytes": kb, "live_passes": passes, "seed": SEED,
                   "dist": dname, "rank_mode": rank_mode, "variant": args.variant, "verified": bool(verified),
                   "cpu_sample_keys": cpu["sample_keys"] if cpu else None,
                   "l2": "inputs (n*key_bytes) larger than L2 and restored by a full-size copy before every step",
                   "timing": "CUDA events around each rsx_sort call on the launch stream, mean of steps",
                   "ms_min": min(times), "ms_max": max(times)},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
        "clocks": clocks,
    }


def run_sweep(args):
    """N2 (SURVEY.md section 8f): the reference's Google-Benchmark sweep, n = 1 .. 40 M (x10) of uint32_t
    keys for radix_sort, radix_sort_rank, std::sort and qsort (radix_bench.cpp:86-138) -- the device
    path (device-resident buffers: CUDA-event time and wall clock of the synchronous call) with the
    reference's CPU path and its two yardsticks timed beside it on one host core.  Input restored
    before every iteration (the reference's loop does not, radix_bench.cpp:91-93).  One JSON line."""
    import ctypes as C
    import numpy as np
    import torch
    import pyoracle
    rsx = importlib.import_module("radix-sorting_b200")
    dev = torch.device("cuda", 0)
    U = rsx.KeyFunc(rsx.KDF_UNSIGNED)
    ref = None
    if os.path.exists(pyoracle.LIB_REF):
        ref = C.CDLL(pyoracle.LIB_REF)
        ref.ref_time_u32.restype = C.c_double
        ref.ref_time_u32.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
    try:
        os.sched_setaffinity(0, {sorted(os.sched_getaffinity(0))[0]})
    except Exception:
        pass
    keygen = load_keygen()
    rows = []
    n = 1
    while n <= 40_000_000:
        pristine = torch.empty(n, dtype=torch.int32, device=dev)
        rsx.fill_keys(pristine, seed=5)
        src, aux = torch.empty_like(pristine), torch.empty_like(pristine)
        ib = torch.empty(2 * n, dtype=torch.int32, device=dev)
        row = {"n": n}
        for name, fn in (("radix_sort", lambda: rsx.radix_sort(src, aux, None, U)),
                         ("radix_sort_rank", lambda: rsx.radix_sort_rank(src, ib, n, U))):
            ev, wall = [], []
            for it in range(12):
                src.copy_(pristine)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0 = time.perf_counter()
                e0.record()
                fn()
                e1.record()
                e1.synchronize()
                t1 = time.perf_counter()
                if it >= 2:
                    ev.append(e0.elapsed_time(e1) * 1e-3)
                    wall.append(t1 - t0)
            row["gpu_" + name] = {"device_us": min(ev) * 1e6, "wall_us": min(wall) * 1e6, "KeyRate_Mkeys_s": n / min(wall) / 1e6}
        if ref is not None:
            h = keygen.fill(5, 0, n, 4).astype(np.uint32)
            assert h[:1000].tobytes() == pristine[:1000].cpu().numpy().tobytes()
            work, haux = np.empty_like(h), np.zeros(2 * n, dtype=np.uint32)
            iters = 5 if n <= 1_000_000 else 2
            for kind, name in enumerate(("radix_sort", "radix_sort_rank", "std_sort", "qsort")):
                if kind == 3 and n > 10_000_000:
                    iters = 1
                sec = ref.ref_time_u32(kind, h.ctypes.data, work.ctypes.data, haux.ctypes.data, n, iters)
                row["cpu_" + name] = {"wall_us": sec * 1e6, "KeyRate_Mkeys_s": n / sec / 1e6}
            row["gpu_over_cpu_radix_sort"] = row["cpu_radix_sort"]["wall_us"] / row["gpu_radix_sort"]["wall_us"]
        rows.append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
        del pristine, src, aux, ib
        n *= 10 if n < 10_000_000 else 4
    crossover = next((r["n"] for r in rows if r.get("gpu_over_cpu_radix_sort", 0) > 1.0), None)
    print(json.dumps({"sweep": "radix_bench.cpp:86-138 on uint32_t keys", "rows": rows,
                      "cpu": "oracle/_ref (unmodified reference headers + std::sort / qsort), 1 core" if ref else None,
                      "device_path_faster_than_cpu_from_n": crossover,
                      "note": "below the crossover the device path is launch-latency-bound and SLOWER than the "
                              "reference on one CPU core; a drop-in caller should keep small arrays on the host"}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sweep", action="store_true", help="the reference's n = 1 .. 40 M sweep (radix_bench.cpp) with CPU columns")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary workloads (u64 / config 5 / zipf sub-lines)")
    ap.add_argument("--no-selftest", action="store_true", help="N > 1: skip the oracle parity run before the timed steps")
    ap.add_argument("--no-fused", action="store_true", help="N > 1: NCCL all_to_all instead of fused peer stores")
    ap.add_argument("--rank-mode", type=int, default=-1, help="-1 auto (hardware probe), 0 ticket, 1 ballot")
    ap.add_argument("--variant", type=int, default=0, help="scatter tuning variant (rsx_scatter.cuh)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of each workload's last timed output to DIR/*.npy "
                         "(one-GPU runs only; refused under torchrun, --impl reference and --sweep)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.sweep or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs applies to the one-GPU timed sort only")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    explicit_workload = args.workload is not None
    if args.workload is None:
        # same per-GPU workload at every N (weak scaling): BASELINE configs[1]; at N > 1 the shards
        # are sorted GLOBALLY (partition + NVLink all-to-all + local LSD) and configs[4]
        # (2 B u64 keys per GPU, uniform and zipf) is measured as extra lines inside the JSON.
        args.workload = "1B-u32-uniform"

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if args.sweep:
        run_sweep(args)
        return

    import torch
    rsx = importlib.import_module("radix-sorting_b200")  # raises if librsx.so is missing: no fallback
    assert torch.cuda.is_available(), "bench.py needs a CUDA device; there is no CPU path"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    if world > 1:
        import copy
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        dsort = importlib.import_module("radix-sorting_b200.dist")
        tname, n, dname, mask, orv, passes = WORKLOADS[args.workload]
        # on-hardware parity of exactly this code path, bytes against the CPU oracle (SURVEY 8e)
        st = None
        if not args.no_selftest:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            st = importlib.import_module("multi_gpu_selftest").selftest(rsx, rank, world, dev)
        result = dsort.bench_partitioned(args, rsx, tname, n, dname, mask, orv, rank, world, dev,
                                         sampler=ClockSampler(local_rank) if rank == 0 else None)
        extras = {}
        if not explicit_workload and not args.no_extra:
            for key, wl in (("config5_u64", "2B-u64-uniform"), ("config5_u64_zipf", "2B-u64-zipf")):
                a2 = copy.copy(args)
                a2.workload, a2.warmup, a2.no_e2e = wl, 3, True
                t2, n2, d2, m2, o2, _ = WORKLOADS[wl]
                torch.cuda.empty_cache()
                r2 = dsort.bench_partitioned(a2, rsx, t2, n2, d2, m2, o2, rank, world, dev,
                                             sampler=ClockSampler(local_rank) if rank == 0 else None)
                extras[key] = {k: r2[k] for k in ("value", "unit", "ms_per_step", "config", "roofline", "steps", "clocks")}
        result.update(extras)
        result["selftest"] = st
        result["config"]["verified"] = bool(result["config"]["verified"] and (st is None or st["passed"]))
        peak, peak_src = measured_peak()
        for r in [result] + list(extras.values()):
            # whole partitioned sort per GPU against the measured HBM peak (the NVLink term is listed beside it)
            r["roofline"].update(peak=peak, peak_source=peak_src, frac=r["roofline"]["achieved"] / peak)
        if rank == 0:
            print(json.dumps(result))
        dist.destroy_process_group()
        return

    out = bench_single(args, rsx, torch, args.workload, dev, args.steps, args.warmup, not args.no_e2e, not args.no_cpu)
    if not explicit_workload and not args.no_extra:
        # the u64 half of BASELINE's "u32/u64" metric, same contract
        r64 = bench_single(args, rsx, torch, "1B-u64-uniform", dev, args.steps, 3, False, False)
        out["u64_1B"] = {k: r64[k] for k in ("value", "unit", "ms_per_step", "steps", "dtype", "config", "roofline",
                                              "gpu_launches", "clocks")}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
