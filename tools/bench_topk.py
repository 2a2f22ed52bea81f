"""Top-k benchmark: rsx_topk / rsx_topk_rank against a full rsx_sort / rsx_sort_rank plus slicing and
against torch.topk(sorted=True), on one GPU.

    python tools/bench_topk.py [--steps 5] [--warmup 2] [--out profiles/r4_topk_1gpu.json] [--only K1,K3]

Workloads (inputs are seeded, generated on the device and larger than the 126 MB L2):
    K1  2^30 int32 uniform, ascending, k = 1 000       K2  K1, k = 1 048 576
    K3  2^30 int64 uniform, ascending, k = 1 000       K4  500 M float32, largest, k = 1 000 000
    K5  2^30 int32 with a 20-bit mask (1 024 copies of every key: the quota path), k = 1 000 000
    K6  K1 as a rank top-k with int64 indices, k = 1 000
    K7  K1, k = n / 4 (a large k)
Every timed call is synchronous and timed with CUDA events on the current stream.  The full sort
restores its input from a pristine copy outside the timing.  Every timed output is checked: top-k
and the sliced sort are byte-equal to the first k of one reference rsx_sort / rsx_sort_rank output,
and torch.topk's values equal them (its order among equal keys is unspecified, so its indices are
checked by the values they point at).  "read_gbps" is the bytes of the read-only passes (the search
passes that ran plus the select) over the whole top-k time, sort of the k records included.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
rsx = importlib.import_module("radix-sorting_b200")


def device_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:  # query only
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in out.split(",")]
    except Exception as e:  # noqa: BLE001 -- recorded, not fatal
        info["power_limit"] = f"unavailable ({e})"
    return info


def expect(cond, msg):
    if not cond:
        raise AssertionError(msg)


def timed(fn, restore, check, steps, warmup):
    """ms per step (CUDA events around fn), with restore() before and check(result) after every step."""
    ms = []
    for i in range(warmup + steps):
        restore()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        check(out)
        if i >= warmup:
            ms.append(a.elapsed_time(b))
    return ms


def summary(ms):
    return {"ms_median": float(np.median(ms)), "ms_min": float(min(ms)), "ms_all": [round(x, 4) for x in ms]}


def workload(name, x, k, kf, rank, steps, warmup, note):
    n = x.numel()
    rb = x.element_size()
    largest = kf.descending
    r = {"workload": name, "input": note, "n": n, "k": k, "dtype": str(x.dtype).replace("torch.", ""),
         "largest": largest, "rank": rank}
    rep = rsx.RsxReport()
    if rank:
        ib = torch.empty(2 * n, dtype=torch.int64, device="cuda")
        want = rsx.radix_sort_rank(x, ib, None, kf)[:k].clone()
        out = torch.empty(k, dtype=torch.int64, device="cuda")
        top = lambda: rsx.radix_topk_rank(x, k, out, kf, report=rep)  # noqa: E731
        full = lambda: rsx.radix_sort_rank(x, ib, None, kf)[:k]  # noqa: E731
        restore = lambda: None  # noqa: E731 -- a rank sort does not write its input
        want_vals = x[want]
    else:
        pristine, aux = x.clone(), torch.empty_like(x)
        want = rsx.radix_sort(x, aux, None, kf)[:k].clone()
        x.copy_(pristine)
        out = torch.empty(k, dtype=x.dtype, device="cuda")
        top = lambda: rsx.radix_topk(x, k, out, kf, report=rep)  # noqa: E731
        full = lambda: rsx.radix_sort(x, aux, None, kf)[:k]  # noqa: E731
        restore = lambda: x.copy_(pristine)  # noqa: E731
        want_vals = want

    def same(label):
        return lambda got: expect(torch.equal(got.view(torch.uint8), want.view(torch.uint8)), f"{name}: {label} differs")

    tms = timed(top, lambda: out.fill_(0), same("rsx_topk"), steps, warmup)
    r["rsx_topk_rank" if rank else "rsx_topk"] = summary(tms)
    r["search_columns"] = rep.ncols
    r["kernel_launches"] = rep.kernel_launches
    read = (rep.ncols + 1) * n * rb
    r["read_only_bytes"] = read
    r["read_gbps"] = read / (float(np.median(tms)) * 1e-3) / 1e9
    sms = timed(full, restore, same("sliced sort"), steps, warmup)
    r["rsx_sort_rank_then_slice" if rank else "rsx_sort_then_slice"] = summary(sms)
    r["topk_over_sort"] = float(np.median(tms)) / float(np.median(sms))
    if not rank:
        x.copy_(pristine)
        del pristine, aux
    else:
        del ib
    torch.cuda.empty_cache()
    try:
        def check_torch(res):
            v, i = res
            expect(torch.equal(v, want_vals), f"{name}: torch.topk values differ")
            expect(torch.equal(x[i], want_vals), f"{name}: torch.topk indices point at other values")
        tt = timed(lambda: torch.topk(x, k, largest=largest, sorted=True), lambda: None, check_torch, steps, warmup)
        r["torch_topk"] = summary(tt)
    except (RuntimeError, torch.cuda.OutOfMemoryError) as e:  # recorded, not fatal
        r["torch_topk"] = {"error": str(e).splitlines()[0][:300]}
        torch.cuda.empty_cache()
    r["outputs_checked"] = True
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_topk_1gpu.json"))
    ap.add_argument("--only", default="", help="comma-separated workload names (K1..K7); default all")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_topk.py needs a CUDA device")
    torch.cuda.set_device(0)
    only = set(args.only.split(",")) if args.only else None
    res = {"device": device_info(), "steps": args.steps, "warmup": args.warmup,
           "rank_mode": rsx.lib().rsx_set_option(b"query_rank_mode", 0),
           "timing": "CUDA events around one synchronous call on the current stream; the full sort's input is restored "
                     "from a pristine copy outside the timing",
           "workloads": []}
    n30 = 1 << 30
    signed = rsx.KeyFunc(rsx.KDF_SIGNED)
    specs = [
        ("K1", torch.int32, n30, 0, 1000, signed, False, "2^30 int32 uniform, ascending"),
        ("K2", torch.int32, n30, 0, 1 << 20, signed, False, "K1, k = 1 048 576"),
        ("K3", torch.int64, n30, 0, 1000, signed, False, "2^30 int64 uniform, ascending"),
        ("K4", torch.float32, 500_000_000, 0, 1_000_000, rsx.KeyFunc(rsx.KDF_FLOAT, True), False,
         "500 M float32 uniform in [-1e6, 1e6), largest"),
        ("K5", torch.int32, n30, 0xFFFFF, 1_000_000, signed, False, "2^30 int32, 20-bit mask (heavy ties)"),
        ("K6", torch.int32, n30, 0, 1000, signed, True, "K1 as a rank top-k, int64 indices"),
        ("K7", torch.int32, n30, 0, n30 // 4, signed, False, "K1, k = n / 4"),
    ]
    for name, dt, n, mask, k, kf, rank, note in specs:
        if only is not None and name not in only:
            continue
        if dt == torch.float32:
            g = torch.Generator(device="cuda").manual_seed(4)
            x = torch.empty(n, dtype=dt, device="cuda").uniform_(-1e6, 1e6, generator=g)
        else:
            x = torch.empty(n, dtype=dt, device="cuda")
            rsx.fill_keys(x, 1, mask=mask if mask else (1 << 64) - 1)
        r = workload(name, x, k, kf, rank, args.steps, args.warmup, note)
        res["workloads"].append(r)
        print(json.dumps(r), flush=True)
        del x
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"device": res["device"], "written": args.out}))


if __name__ == "__main__":
    main()
