"""Per-role cycle counters of the tcgen05 kernel.  Needs a library built with the instrumentation compiled in:
    nvcc ... -DPIO_TC_TIMING=1 ... pio_als.cu   (the default build carries none)
then  PIO_ALS_TC=1 [PIO_ALS_TC_MIN_DEG=...] python tools/tc_timing.py   (TC_NU / TC_NI / TC_NNZ choose the problem size).
The warp -> role map below matches the partition instantiated in pio_als.cu (2 gather, 5 converter warps, 2 teams)."""
import os, sys, ctypes as C
os.environ["PIO_ALS_TC_TIMING"] = "1"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import pio_b200
from pio_b200 import native
nu, ni, nnz, k = int(os.environ.get('TC_NU', 100000)), int(os.environ.get('TC_NI', 20000)), int(os.environ.get('TC_NNZ', 5000000)), 64
du = torch.empty(nnz, dtype=torch.int32, device="cuda"); di = torch.empty_like(du); dr = torch.empty(nnz, dtype=torch.float32, device="cuda")
native.synth_ratings_device(0, nu, ni, nnz, 3, True, 0, du.data_ptr(), di.data_ptr(), dr.data_ptr())
m = native.NativeALS(k, nu, ni, lam=0.01, implicit=True, init_mode=native.INIT_HASH, seed=3)
m.set_ratings_device(du.data_ptr(), di.data_ptr(), dr.data_ptr(), nnz, dedup=1)
m.run(2)
st = m.stats(); print("run ms", st["last_run_ms"], "solve ms", st["last_solve_ms"])
L = native.lib()
buf = np.zeros(148 * 16 * 8, np.int64)
rc = L.pio_als_debug_timing(m._h, buf.ctypes.data_as(C.POINTER(C.c_longlong)), C.c_longlong(buf.size))
t = buf.reshape(148, 16, 8).astype(np.float64)
tot = t[:, :, 7].mean()
print("rc", rc, "(last tc launch = user side) mean kernel cycles per CTA", tot)
np.set_printoptions(precision=1, suppress=True, linewidth=200)
names = {0: ["sched: wait teamdone", "wait tmemfree", "wait full", "build", "mma issue"],
         1: ["gather: advance(desc)", "wait rawempty", "issue bulk copies"],
         2: ["conv: advance(desc)", "wait rawfull", "wait empty", "load raw", "convert+store"],
         4: ["team: wait desc", "wait accfull", "drain", "wait bfull", "team barrier", "dump+solve"]}
for w, nm in ((0, names[0]), (1, names[1]), (2, names[1]), (3, names[2]), (5, names[2]), (7, names[2]), (8, names[4]), (9, names[4]), (12, names[4])):
    pct = t[:, w, :len(nm)].mean(0) / tot * 100
    print(f"warp {w:2d}:", ", ".join(f"{n} {p:.1f}%" for n, p in zip(nm, pct)))
