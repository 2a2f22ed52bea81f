#!/usr/bin/env python
"""Whole-sort device time per record/payload footprint with the shipped kernel choice
(PreferV2<ES, PL>), verified by descents/checksum (value sorts)."""
import importlib, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
rsx = importlib.import_module("radix-sorting_b200")
dev = torch.device("cuda", 0)
U = rsx.KeyFunc(rsx.KDF_UNSIGNED)

def timed(fn, restore, reps=4):
    best = 1e30
    for r in range(reps):
        restore()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); e1.synchronize()
        if r: best = min(best, e0.elapsed_time(e1))
    return best

rows = []
def report(name, ms, n):
    rows.append({"case": name, "ms": ms, "Gkeys_s": n / ms / 1e6}); print(rows[-1], flush=True)

cases = [("rank u32 keys, u32 idx (4+4)", torch.int32, torch.int32, 1_000_000_000),
         ("rank u64 keys, u64 idx (8+8)", torch.int64, torch.int64, 400_000_000),
         ("rank u64 keys, u32 idx (8+4)", torch.int64, torch.int32, 500_000_000),
         ("rank u32 keys, u64 idx (4+8)", torch.int32, torch.int64, 500_000_000)]
for name, kdt, idt, n in cases:
    keys = torch.empty(n, dtype=kdt, device=dev); rsx.fill_keys(keys, seed=6)
    ib = torch.empty(2 * n, dtype=idt, device=dev)
    ms = timed(lambda: rsx.radix_sort_rank(keys, ib, n, U), lambda: None)
    report(name, ms, n)
    del keys, ib; torch.cuda.empty_cache()
vcases = [("u16 keys (2+0)", torch.int16, 2, 0, 2, 1_000_000_000), ("u8 keys (1+0)", torch.uint8, 1, 0, 1, 1_000_000_000),
          ("rec16 u64 key (16+0)", torch.int64, 16, 0, 8, 400_000_000), ("rec8 u32 key (8+0)", torch.int32, 8, 0, 4, 1_000_000_000),
          ("u32 (4+0)", torch.int32, 4, 0, 4, 1_000_000_000), ("u64 (8+0)", torch.int64, 8, 0, 8, 1_000_000_000)]
for name, tdt, rb, ko, kb, n in vcases:
    elems = n * rb // torch.empty(0, dtype=tdt).element_size()
    pristine = torch.empty(elems, dtype=tdt, device=dev); rsx.fill_keys(pristine, seed=11)
    src, aux = torch.empty_like(pristine), torch.empty_like(pristine)
    kf = rsx.KeyFunc(rsx.KDF_UNSIGNED, False, rb, ko, kb)
    _, s0, x0 = rsx.verify(pristine, kf)
    res = [None]
    def run(): res[0] = rsx.radix_sort(src, aux, None, kf)
    ms = timed(run, lambda: src.copy_(pristine))
    d1, s1, x1 = rsx.verify(res[0], kf)
    assert d1 == 0 and (s1, x1) == (s0, x0), name
    report(name, ms, n)
    del pristine, src, aux; torch.cuda.empty_cache()
json.dump(rows, open(os.path.join(ROOT, "gpurun_out", "footprints.json"), "w"), indent=1)
