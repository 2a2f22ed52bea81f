"""Debug-only: per-phase cycle breakdown of the scatter pass (needs tools/dbg/librsx_dbg.so, built
with -DRSX_PHASE_TIMING).  Not part of the product."""
import ctypes as C, sys, os, importlib
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
pkg_dir = os.path.join(ROOT, "radix-sorting_b200")
# load the debug library in place of the product one
import types
mod = importlib.import_module("radix-sorting_b200")
dbg = C.CDLL(os.path.join(ROOT, "tools", "dbg", "librsx_dbg.so"))
n = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000_000
kb = int(sys.argv[2]) if len(sys.argv) > 2 else 4
dt = torch.int32 if kb == 4 else torch.int64
src = torch.empty(n, dtype=dt, device="cuda"); aux = torch.empty_like(src); pristine = torch.empty_like(src)
mod.fill_keys(pristine, seed=2)
L = mod.RsxLayout(kb, 0, kb, 0, 0)
res = C.c_void_p(); rep = mod.RsxReport()
names = ["load/wait stage", "rank (atoms)", "barrier A", "digit phase", "barrier C", "scatter->smem", "look-back", "barrier D", "write-out", "loop top", "lb rounds", "lb polls", "CTAs"]
for it in range(3):
    src.copy_(pristine)
    out = (C.c_ulonglong * 16)()
    dbg.rsx_dbg_phase(out, 1)
    st = dbg.rsx_sort(C.c_void_p(src.data_ptr()), C.c_void_p(aux.data_ptr()), C.c_size_t(n), C.byref(L), C.byref(res), C.byref(rep), None)
    assert st == 0, st
    dbg.rsx_dbg_phase(out, 0)
tiles_total = None
ctas = out[12]
tot = sum(out[k] for k in range(10))
print(f"n={n} kb={kb} CTAs(sum over {rep.ncols} passes)={ctas}")
for k in range(10):
    print(f"  {names[k]:18s} {out[k]/ctas:12.0f} cyc/CTA  {100*out[k]/tot:5.1f}%")
print(f"  lb rounds {out[10]}  polls {out[11]}")
