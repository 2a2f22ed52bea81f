"""Segmented sort benchmark: rsx_sort_segments / rsx_sort_rank_segments against torch.sort(dim=1)
and against rsx_sort called once per segment, on one GPU.

    python tools/bench_segments.py [--steps 5] [--warmup 2] [--out profiles/r3_segments_1gpu.json]

Workloads (inputs are seeded and larger than the 126 MB L2):
    W1  65 536 segments x 1 024 int32      W2  1 048 576 x 64 int32      W3  4 096 x 16 384 int64
    W4  ragged, ~64 M int32: log-normal lengths, empty segments, some longer than one group
    W5  W1 as a rank sort (segment-relative indices)
Every timed step starts from a pristine device copy of the input (restored outside the timing), is
timed with CUDA events on the current stream (the call is synchronous, so the time includes its host
planning), and its output is checked: W1-W3 / W5 equal torch.sort's values / indices, W4 has no
descent inside a segment, the same multiset checksums as its input and a sample of segments equal
to numpy's sort.  The per-segment loop runs over a prefix of the segments and is extrapolated to
the whole batch; the JSON says so.
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


def summary(ms, n):
    med = float(np.median(ms))
    return {"ms_median": med, "ms_min": float(min(ms)), "ms_all": [round(x, 4) for x in ms], "gkeys_per_s": n / med / 1e6}


def inside_descents(out, offs):
    """Descents of `out` that lie inside a segment (a boundary between segments does not count)."""
    d = out[1:] < out[:-1]
    b = offs[1:-1]
    b = b[(b > 0) & (b < out.numel())]
    d[b - 1] = False
    return int(d.sum())


def loop_prefix(x, offs_h, prefix, steps, warmup):
    """rsx_sort called once per segment over the first `prefix` segments: ms for the prefix."""
    src, aux = torch.empty_like(x), torch.empty_like(x)
    end = int(offs_h[prefix])

    def run():
        for s in range(prefix):
            a, b = int(offs_h[s]), int(offs_h[s + 1])
            if b > a:
                rsx.radix_sort(src[a:b], aux[a:b])
        return None

    def check(_):
        pass  # the per-segment path is rsx_sort itself, pinned by the parity suite

    return timed(run, lambda: src[:end].copy_(x[:end]), check, steps, warmup)


def value_workload(name, x, offs, steps, warmup, prefix, rows=None):
    n = x.numel()
    offs_h = offs.cpu().numpy()
    nseg = len(offs_h) - 1
    src, aux = torch.empty_like(x), torch.empty_like(x)
    want = torch.sort(x.view(rows, -1), dim=1, stable=True).values.reshape(-1) if rows else None
    ck = rsx.verify(x)
    rep = rsx.RsxReport()

    def check(res):
        expect(want is None or torch.equal(res, want), f"{name}: differs from torch.sort")
        expect(inside_descents(res, offs) == 0, f"{name}: a segment is not ordered")
        expect(rsx.verify(res)[1:] == ck[1:], f"{name}: multiset checksum changed")

    ms = timed(lambda: rsx.radix_sort_segments(src, aux, offs, report=rep), lambda: src.copy_(x), check, steps, warmup)
    r = {"workload": name, "n": n, "nseg": nseg, "dtype": str(x.dtype).replace("torch.", ""),
         "segmented": summary(ms, n), "kernel_launches": rep.kernel_launches, "live_columns": rep.ncols,
         "outputs_checked": True}
    if rows:
        xs = x.view(rows, -1)
        tms = timed(lambda: torch.sort(xs, dim=1, stable=True).values, lambda: None,
                    lambda v: expect(torch.equal(v.reshape(-1), want), f"{name}: torch.sort differs"),
                    steps, warmup)
        r["torch_sort_dim1"] = summary(tms, n)
    lms = loop_prefix(x, offs_h, prefix, max(1, steps // 2), 1)
    med = float(np.median(lms))
    r["rsx_sort_loop"] = {"prefix_segments": prefix, "prefix_ms_median": med, "extrapolated": True,
                          "ms_extrapolated": med * nseg / prefix, "gkeys_per_s_extrapolated": n / (med * nseg / prefix) / 1e6}
    return r, src, aux


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_segments_1gpu.json"))
    ap.add_argument("--only", default="", help="comma-separated workload names (W1..W5); default all")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_segments.py needs a CUDA device")
    torch.cuda.set_device(0)
    only = set(args.only.split(",")) if args.only else None
    g = torch.Generator(device="cuda").manual_seed(2024)
    res = {"device": device_info(), "steps": args.steps, "warmup": args.warmup, "rank_mode": rsx.lib().rsx_set_option(b"query_rank_mode", 0),
           "timing": "CUDA events around one synchronous call on the current stream, input restored outside the timing",
           "workloads": []}

    def want(w):
        return only is None or w in only

    def rows_offsets(B, Lr):
        return torch.arange(0, B * Lr + 1, Lr, dtype=torch.int64, device="cuda")

    for name, B, Lr, dt, prefix in [("W1", 65536, 1024, torch.int32, 256), ("W2", 1 << 20, 64, torch.int32, 1024),
                                    ("W3", 4096, 16384, torch.int64, 64)]:
        if not want(name):
            continue
        lo, hi = (-2**31, 2**31 - 1) if dt == torch.int32 else (-2**63, 2**63 - 1)
        x = torch.randint(lo, hi, (B * Lr,), dtype=dt, device="cuda", generator=g)
        r, _, _ = value_workload(name, x, rows_offsets(B, Lr), args.steps, args.warmup, prefix, rows=B)
        res["workloads"].append(r)
        print(json.dumps(r), flush=True)
        del x
        torch.cuda.empty_cache()

    if want("W4"):
        rng = np.random.default_rng(4)
        lengths = []
        while sum(lengths) < 64 << 20:
            ln = rng.lognormal(6.0, 1.6, size=4096).astype(np.int64)
            ln[rng.random(4096) < 0.05] = 0  # empty segments
            lengths.extend(int(v) for v in ln)
        lengths[100:100] = [20000, 250000, 1 << 20]  # longer than one group, into the multi-kernel path
        offs_np = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
        n = int(offs_np[-1])
        x = torch.randint(-2**31, 2**31 - 1, (n,), dtype=torch.int32, device="cuda", generator=g)
        offs = torch.from_numpy(offs_np).cuda()
        r, src, aux = value_workload("W4", x, offs, args.steps, args.warmup, 512)
        out = rsx.radix_sort_segments(src.copy_(x), aux, offs).cpu().numpy()
        xs = x.cpu().numpy()
        sample = sorted(set(rng.integers(0, len(lengths), size=200).tolist()) | {100, 101, 102})
        for s in sample:
            a, b = offs_np[s], offs_np[s + 1]
            expect(np.array_equal(out[a:b], np.sort(xs[a:b], kind="stable")), f"W4 segment {s}")
        r["numpy_checked_segments"] = len(sample)
        r["segments_longer_than_a_group"] = int(sum(1 for v in lengths if v > 13104))
        r["empty_segments"] = int(sum(1 for v in lengths if v == 0))
        r["yardstick"] = "per-segment rsx_sort loop only: torch has no ragged sort"
        res["workloads"].append(r)
        print(json.dumps(r), flush=True)
        del x, src, aux
        torch.cuda.empty_cache()

    if want("W5"):
        B, Lr = 65536, 1024
        x = torch.randint(-2**31, 2**31 - 1, (B * Lr,), dtype=torch.int32, device="cuda", generator=g)
        offs = rows_offsets(B, Lr)
        ib = torch.empty(2 * B * Lr, dtype=torch.int32, device="cuda")
        want_idx = torch.sort(x.view(B, Lr), dim=1, stable=True).indices.to(torch.int32).reshape(-1)
        rep = rsx.RsxReport()

        ms = timed(lambda: rsx.radix_sort_rank_segments(x, ib, offs, report=rep), lambda: ib.fill_(0),
                   lambda r_: expect(torch.equal(r_, want_idx), "W5: indices differ from torch.sort"), args.steps, args.warmup)
        tms = timed(lambda: torch.sort(x.view(B, Lr), dim=1, stable=True).indices, lambda: None,
                    lambda v: expect(torch.equal(v.to(torch.int32).reshape(-1), want_idx), "W5: torch.sort differs"),
                    args.steps, args.warmup)
        r = {"workload": "W5", "n": B * Lr, "nseg": B, "dtype": "int32", "rank": True, "segmented": summary(ms, B * Lr),
             "torch_sort_dim1_indices": summary(tms, B * Lr), "kernel_launches": rep.kernel_launches, "outputs_checked": True}
        res["workloads"].append(r)
        print(json.dumps(r), flush=True)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"device": res["device"], "written": args.out}))


if __name__ == "__main__":
    main()
