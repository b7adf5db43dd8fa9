import os, sys, ctypes as C
os.environ["PIO_ALS_TC_DEBUG"] = "1"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import pio_b200
from pio_b200 import native, synth
# tiny problem: 1 item rated by d users; explicit; the item half-step runs first (dst = items)
nu, ni, k = 40, 3, 64
rng = np.random.default_rng(0)
u = np.concatenate([np.arange(10), np.arange(5, 30), np.arange(0, 40)]).astype(np.int32)
i = np.concatenate([np.zeros(10), np.ones(25), np.full(40, 2)]).astype(np.int32)
r = rng.integers(1, 6, u.shape[0]).astype(np.float32)
u0 = synth.synth_init_factors(nu, k, 5, 0)
m = native.NativeALS(k, nu, ni, lam=0.1, implicit=False)
m.set_ratings(u, i, r)
m.set_init(u0)
# run only item half: run(1) does both halves; dump reflects the LAST tc launch (user side). So compare user side: need item factors.
m.run(1)
uf, itf, uh, ih = m.get_factors()
L = native.lib()
ASLOT, KP = 2208, 64
buf = np.zeros(nu * (ASLOT + KP), np.float32)
rc = L.pio_als_debug_dump(m._h, buf.ctypes.data_as(C.POINTER(C.c_float)), C.c_longlong(buf.size))
print("rc", rc)
buf = buf.reshape(nu, ASLOT + KP)
# user side: dst = users (internal order = degree-desc). Expected A for user uu = sum over rated items y y^T (items factors AFTER item half-step)
deg = np.bincount(u, minlength=nu)
order = np.argsort(-deg, kind="stable")
def unpack(a):
    A = np.zeros((64, 64), np.float64)
    for rr in range(64):
        for c in range(rr + 1):
            if rr < 32: v = a[rr * (rr + 1) // 2 + c]
            elif c < 32: v = a[528 + (rr - 32) * 36 + c]
            else: v = a[1680 + (rr - 32) * (rr - 31) // 2 + (c - 32)]
            A[rr, c] = A[c, rr] = v
    return A
for p in range(3):
    uu = order[p]
    sel = np.flatnonzero(u == uu)
    Y = itf[i[sel]].astype(np.float64)
    Aexp = Y.T @ Y
    bexp = (r[sel][:, None] * Y).sum(0)
    A = unpack(buf[p, :ASLOT])
    b = buf[p, ASLOT:]
    print("user", uu, "deg", deg[uu], "A err", np.abs(A - Aexp).max(), "A scale", np.abs(Aexp).max(), "b err", np.abs(b - bexp).max())
    if p == 0:
        np.set_printoptions(precision=4, suppress=True, linewidth=200)
        print("A[0:6,0:6] got\n", A[:6, :6], "\nexp\n", Aexp[:6, :6])
        ratio = A / np.where(np.abs(Aexp) > 1e-9, Aexp, np.nan)
        print("ratio sample", ratio[:4, :4])
        # try to find the pattern: which expected entries equal the got entries
        print("got row0[:12]", A[0, :12]); print("exp row0[:12]", Aexp[0, :12])
        print("got diag[:12]", np.diag(A)[:12]); print("exp diag[:12]", np.diag(Aexp)[:12])
