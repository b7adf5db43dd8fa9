#!/usr/bin/env python
"""bench.py -- ALS iterations/sec and top-k predictions/sec on the BASELINE.json workload (configs[1]: rank 64,
1M users x 100k items, 100M synthetic implicit ratings), B200-native path vs the CPU restatement of the reference.

One "step" = one ALS iteration (item half-step + user half-step) over the whole rating set.
  value    : iterations/sec with ratings + CSR already resident in HBM (CUDA events on the library stream)
  e2e      : iterations/sec through the one-shot C-ABI call pio_als_train with HOST buffers:
             H2D of the COO triplets, ingest (dedup + 2 CSR builds), K iterations, D2H of the factors
  parity   : after the timed region one more iteration runs on the GPU; a sample of its destination rows (strided rows
             plus the heaviest rows of both sides) is recomputed by the CPU oracle from the GPU's own source factors and
             compared; the process exits non-zero above 1e-4
  checksum : CRC of both factor matrices after warm-up + K iterations -- identical at every GPU count
  cpu_baseline / --impl reference : the oracle (C/OpenMP restatement of MLlib ALS) timed on the host's physical cores
             over FULL iterations of the same workload
  topk     : top-k predictions/sec through pio_als_recommend / pio_als_similar with host buffers
See DESIGN.md for the roofline arithmetic.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOADS = {
    # name: (n_users, n_items, nnz, rank, implicit)
    "c2": (1_000_000, 100_000, 100_000_000, 64, True),
    "c3": (10_000_000, 1_000_000, 1_000_000_000, 128, True),
    "c1": (10_000, 1_000, 100_000, 10, False),
    "small": (100_000, 20_000, 5_000_000, 64, True),
    "small128": (200_000, 40_000, 10_000_000, 128, True),
}
LAMBDA, ALPHA, SEED = 0.01, 1.0, 3
PARITY_TOL = 1e-4
DUMP_BYTES = 60_000_000      # --dump-outputs stays below 64 MB including the .npy headers


def algorithmic_work(nu, ni, nnz, k, implicit):
    """BASELINE.md section 4 / SURVEY 8(d): bytes and flops per ALS iteration."""
    b = 16 * nnz + 8 * (nu + ni) * k + 8 * (nu + ni + 2)
    f_solve = 2 * nnz * (k * (k + 1) + 2 * k) + (nu + ni) * (k ** 3 / 3 + 2 * k * k)
    f_gram = (nu + ni) * k * (k + 1) if implicit else 0
    return b, f_solve, f_gram


class ClockSampler:
    """SM clock and throttle reasons sampled WHILE the timed region runs: NVML in a thread every 2 ms (a timed region of a
    few tens of milliseconds at N = 8 is over before a freshly spawned nvidia-smi prints its first line); nvidia-smi -lms
    only if the NVML binding is missing."""

    _BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []
        self.nvml, self.h, self.sm, self.bits, self._stop = None, None, [], 0, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        while True:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                self.bits |= int(reasons(self.h))
            except Exception:
                pass
            if self._stop.wait(0.002):
                return

    def start(self):
        if self.nvml:
            self._stop.clear()
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml:
            self._stop.set()
            self.t.join(timeout=2)
            try:
                mx = float(self.nvml.nvmlDeviceGetMaxClockInfo(self.h, self.nvml.NVML_CLOCK_SM))
            except Exception:
                mx = None
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": mx,
                    "reasons": sorted(v for b, v in self._BITS.items() if self.bits & b), "samples": len(self.sm),
                    "how": "NVML, every 2 ms inside the timed region"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "how": "nvidia-smi -lms 20"}


def traffic_from_profiles(workload):
    """dram__bytes_read+write of ONE launch of the dominant kernel, from the committed ncu --set full capture (null if none)."""
    p = ROOT / "profiles" / "traffic.json"
    try:
        return json.loads(p.read_text())[workload]["dram_bytes_per_launch"]
    except Exception:
        return None


def measured_peaks():
    """HBM GB/s, dense bf16 TFLOP/s (driver-written MEASURED_PEAKS.json), FP32 FFMA TFLOP/s (profiles/peaks_r02.json,
    measured by tools/peaks.cu on this pool; nominal 148 x 128 x 2 x 1.965 GHz otherwise)."""
    hbm, bf16, src = 6650.0, 1590.0, "fallback"
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        hbm, bf16, src = d.get("hbm_gbs", hbm), d.get("bf16_tflops", bf16), "measured"
    fp32, fp32_src = 148 * 128 * 2 * 1.965e9 / 1e12, "nominal 148 SM x 128 lanes x 2 x 1.965 GHz"
    mma_tf32 = dfma = None
    q = ROOT / "profiles" / "peaks_r02.json"
    if q.exists():
        try:
            d = json.loads(q.read_text())
            if d.get("ffma_tflops"):
                fp32, fp32_src = float(d["ffma_tflops"]), "measured (tools/peaks.cu, profiles/peaks_r02.json)"
            mma_tf32 = d.get("mma_sync_tf32_tflops")
            dfma = d.get("dfma_tflops")
        except Exception:
            pass
    return {"hbm": hbm, "bf16": bf16, "src": src, "fp32": fp32, "fp32_src": fp32_src, "mma_tf32": mma_tf32,
            "dfma": dfma or 148 * 64 * 2 * 1.965e9 / 1e12}


# ---------------------------------------------------------------------------------------------------------
# CPU side: the oracle as checker (parity sample) and as reported baseline (full iterations on the host cores)
# ---------------------------------------------------------------------------------------------------------
def physical_cores():
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


def load_oracle():
    """The oracle library, rebuilt with -march=native when gcc is on the box, on the physical cores of the host
    (torchrun exports OMP_NUM_THREADS=1: the explicit oracle_set_num_threads call overrides it)."""
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    from oracle import als_oracle as o
    try:
        import ctypes
        import shutil
        if shutil.which("gcc"):
            # -march=native code must not travel between machines, and the tree may be read-only: build it for this
            # host in a temporary directory on every run (under a second); the loaded library outlives the directory
            import tempfile
            with tempfile.TemporaryDirectory(prefix="pio_oracle_") as tmp:
                so = Path(tmp) / "libals_oracle_native.so"
                subprocess.run(["gcc", "-O3", "-march=native", "-fopenmp", "-fPIC", "-shared", "-fvisibility=hidden",
                                "-o", str(so), str(o._SRC), "-lm"], check=True)
                o._lib = ctypes.CDLL(str(so))
            o._lib.oracle_num_threads.restype = ctypes.c_int
    except Exception:
        pass
    cores = physical_cores()
    o.set_num_threads(cores)
    return o, cores


def build_host_problem(o, nu, ni, k, implicit, coo):
    """Both CSR orientations of the workload on the host, prepared like the GPU ingest (implicit: reduceByKey(_+_))."""
    t0 = time.perf_counter()
    u, i, r = coo
    uptr, ucol, uval = o.csr_build(nu, u, i, r)
    if implicit:
        uptr, ucol, uval = o.csr_dedup_sum(uptr, ucol, uval)
    urow = o.csr_rows(uptr)
    iptr, icol, ival = o.csr_build(ni, ucol, urow, uval)
    return {"nu": nu, "ni": ni, "k": k, "implicit": implicit, "user": (uptr, ucol, uval), "item": (iptr, icol, ival),
            "nnz": int(uptr[-1]), "prep_s": time.perf_counter() - t0}


def cpu_iteration(o, prob, uf, itf, stride=1):
    """One ALS iteration of the oracle in place (YtY, item half-step, YtY, user half-step); stride > 1 solves every
    stride-th destination row only.  Returns seconds."""
    imp = prob["implicit"]
    t0 = time.perf_counter()
    yty = o.gram(uf) if imp else None
    o.half_step(*prob["item"], uf, itf, LAMBDA, imp, ALPHA, yty, 0, prob["ni"], stride)
    yty = o.gram(itf) if imp else None
    o.half_step(*prob["user"], itf, uf, LAMBDA, imp, ALPHA, yty, 0, prob["nu"], stride)
    return time.perf_counter() - t0


def cpu_baseline_steps(o, cores, prob, uf, itf, n_steps, n_warm, budget_s):
    """n_warm + n_steps oracle iterations within about budget_s seconds: full iterations when they fit, otherwise every
    stride-th destination row (>= 25 % of the rows) scaled to a full iteration and flagged as extrapolated."""
    pilot_stride = 16
    t_pilot = cpu_iteration(o, prob, uf, itf, pilot_stride) * pilot_stride      # estimate of one full iteration
    per_step = budget_s / max(1, n_steps + n_warm)
    stride = 1 if t_pilot <= per_step else min(4, int(np.ceil(t_pilot / per_step)))
    secs = []
    for s in range(n_warm + n_steps):
        t = cpu_iteration(o, prob, uf, itf, stride)
        if s >= n_warm:
            secs.append(t)
    it_s = float(np.mean(secs)) * stride if stride > 1 else float(np.mean(secs))
    gram_note = ""
    sample = (f"{n_steps} full iteration(s) over all {prob['nu']} user rows + {prob['ni']} item rows "
              f"({prob['nnz']} ratings), {np.mean(secs):.2f} s each" if stride == 1 else
              f"every {stride}th destination row of each side ({100.0 / stride:.0f} % of the rows, "
              f"{np.mean(secs):.2f} s timed per step), scaled to one iteration")
    out = {"value": 1.0 / it_s, "unit": "iterations/s", "cores": cores, "kind": "port",
           "sample": sample + "; C/OpenMP restatement of MLlib ALS (not Spark), threads bound to physical cores" + gram_note,
           "extrapolated": stride > 1, "sampled_fraction": 1.0 / stride, "seconds_per_step": float(np.mean(secs)),
           "spread": [float(min(secs)), float(max(secs))]}
    return out


def frob_rel(a, b):
    a = a.astype(np.float64)
    b = b.astype(np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def max_row_rel(a, b):
    a = a.astype(np.float64)
    b = b.astype(np.float64)
    nb = np.linalg.norm(b, axis=1)
    d = np.linalg.norm(a - b, axis=1)
    return float((d / np.maximum(nb, 1e-3 * nb.max() + 1e-30)).max())


def parity_sample(o, prob, src_u, new_i, new_u, n_user=2000, n_item=500, n_heavy=50):
    """The last GPU iteration (new_i from src_u, then new_u from new_i) against the oracle on a row sample: strided rows
    plus the heaviest rows of each side (the parts + finish path, the long tensor-core accumulations)."""
    imp = prob["implicit"]
    res = {}
    for side, (ptr, col, val), src, got, n_s in (("item", prob["item"], src_u, new_i, n_item),
                                                 ("user", prob["user"], new_i, new_u, n_user)):
        n = ptr.shape[0] - 1
        deg = np.diff(ptr)
        rows = np.unique(np.concatenate([np.arange(0, n, max(1, n // n_s)), np.argsort(-deg, kind="stable")[:n_heavy]]))
        rows = rows[deg[rows] > 0].astype(np.int32)
        yty = o.gram(src) if imp else None
        want, fails = o.half_step_rows(ptr, col, val, src, rows, LAMBDA, imp, ALPHA, yty)
        res[side] = {"rows": int(rows.shape[0]), "max_ratings_in_a_row": int(deg[rows].max()),
                     "frob_rel": frob_rel(got[rows], want), "max_row_rel": max_row_rel(got[rows], want),
                     "oracle_cholesky_failures": int(fails)}
    worst = max(res["item"]["frob_rel"], res["user"]["frob_rel"])
    return {"frob_rel": worst, "max_rel": max(res["item"]["max_row_rel"], res["user"]["max_row_rel"]),
            "rows": res["item"]["rows"] + res["user"]["rows"], "tolerance": PARITY_TOL, "ok": bool(worst <= PARITY_TOL),
            "item": res["item"], "user": res["user"],
            "how": "GPU iteration W+K+1 recomputed by the CPU oracle (fp64 normal equations) from the GPU's own source "
                   "factors on strided + heaviest destination rows"}


def factor_checksum(uf, itf):
    """64-bit value: CRC32 of the user factor bytes (high word) and of the item factor bytes (low word)."""
    return f"{zlib.crc32(np.ascontiguousarray(uf).view(np.uint8)):08x}{zlib.crc32(np.ascontiguousarray(itf).view(np.uint8)):08x}"


def dump_outputs(out_dir, uf, itf, uh, ih):
    """--dump-outputs: what pio_als_get_factors hands a caller after the timed run (factors and has-flags of both sides)
    as .npy files, so that two builds can be compared output for output.  Both sides keep the same fixed, seeded
    fraction of their rows, chosen to stay under DUMP_BYTES; <side>_rows.npy holds the indices of the rows kept."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    row_bytes = 4 * uf.shape[1] + 4 + 8        # factor row (float32), has-flag (float32), row index (float64)
    frac = min(1.0, DUMP_BYTES / (row_bytes * (uf.shape[0] + itf.shape[0])))
    rng = np.random.default_rng(SEED)
    for side, f, has in (("user", uf, uh), ("item", itf, ih)):
        n = f.shape[0]
        keep = int(n * frac)
        rows = np.arange(n) if keep >= n else np.sort(rng.choice(n, keep, replace=False))
        np.save(out_dir / f"{side}_factors.npy", np.ascontiguousarray(f[rows], np.float32))
        np.save(out_dir / f"{side}_has.npy", has[rows].astype(np.float32))
        np.save(out_dir / f"{side}_rows.npy", rows.astype(np.float64))
    return {"dir": str(out_dir), "rows_fraction": frac}


# ---------------------------------------------------------------------------------------------------------
def reference_arm(args, nu, ni, nnz, k, implicit, config):
    """--impl reference: the reference's CPU algorithm (oracle port of MLlib ALS) on this box's physical cores, same
    workload; every step is a full iteration when W + K of them fit in a few minutes."""
    import pio_b200  # noqa: F401
    from pio_b200 import synth
    o, cores = load_oracle()
    u, i, r = synth.synth_ratings(nu, ni, nnz, seed=SEED, implicit=implicit)
    prob = build_host_problem(o, nu, ni, k, implicit, (u, i, r))
    del u, i, r
    uf = np.ascontiguousarray(np.resize(synth.synth_init_factors(min(nu, 1 << 16), k, SEED, 0), (nu, k)))
    itf = np.ascontiguousarray(np.resize(synth.synth_init_factors(min(ni, 1 << 16), k, SEED, 1), (ni, k)))
    cb = cpu_baseline_steps(o, cores, prob, uf, itf, args.steps, args.warmup, budget_s=240.0)
    v = cb["value"]
    print(json.dumps({"impl": "reference", "metric": "ALS iterations/sec", "value": v, "unit": "iterations/s",
                      "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": 1000.0 * cb["seconds_per_step"], "higher_is_better": True, "scaling": "strong",
                      "vs_baseline": None, "dtype": "f64 accumulate / f32 storage", "data": "synthetic",
                      "config": config, "cpu_baseline": cb, "extrapolated": cb["extrapolated"],
                      "e2e": {"value": v, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def topk_bench(native, o, cores, m, nu, ni, k, uf, itf, uh, ih, peaks, dev):
    """Top-k predictions/sec through the C ABI with host buffers (the second half of BASELINE.json's metric)."""
    out = {}
    rng = np.random.default_rng(SEED)
    # recommendation path (A7/A8): distinct users x top-10 over all items of the trained model
    nq = min(100_000, nu)
    users = rng.permutation(nu)[:nq].astype(np.int32)
    m.recommend(users[:256], 10)   # warm-up
    t0 = time.perf_counter()
    gi, gs, gc = m.recommend(users, 10)
    dt = time.perf_counter() - t0
    ns = min(2000, nq)
    t0 = time.perf_counter()
    oi, os_, oc = o.recommend(uf, uh, itf, ih, users[:ns], 10)
    cpu_dt = time.perf_counter() - t0
    scan_bytes = ni * k * 4
    out["recommend"] = {
        "what": f"pio_als_recommend: {nq} distinct users x top-10 over {ni} items, rank {k}, one call, host buffers",
        "value": nq / dt, "unit": "predictions/s", "seconds": dt,
        "bit_exact_vs_oracle_on_sample": bool(np.array_equal(gi[:ns], oi) and np.array_equal(gs[:ns], os_)),
        "sample_queries_checked": int(ns),
        "cpu_baseline": {"value": ns / cpu_dt, "unit": "predictions/s", "cores": cores, "kind": "port",
                         "sample": f"{ns} of the same queries, fp64 ddot scan + heap (oracle restatement of "
                                   "recommendProducts)"},
        "roofline": {"bound": "fp64", "achieved": 2.0 * nq * ni * k / dt / 1e12, "peak": peaks["dfma"], "unit": "TFLOP/s",
                     "frac": 2.0 * nq * ni * k / dt / 1e12 / peaks["dfma"],
                     "note": "scores are accumulated in fp64 in index order (bit-identical to the JVM's ddot), so the bound "
                             "is the DFMA pipe: one DFMA per (query, item, feature); peak = tools/peaks.cu "
                             "(profiles/peaks_r02.json). Includes the H2D / D2H copies of the call.",
                     "hbm_frac_per_16_queries": nq / 16.0 * scan_bytes / dt / 1e9 / peaks["hbm"]}}
    # similarproduct path (A9, BASELINE.json configs[3]): cosine top-20 over 1 M item vectors (unit-norm Gaussian, rank 64),
    # 10 k queries of 1-5 items, one pio_als_similar_batch call on an imported item-only model
    try:
        from pio_b200 import synth
        n_it, kk, nqs = 1_000_000, 64, 10_000
        big = np.ascontiguousarray(np.resize(synth.synth_init_factors(1 << 16, kk, SEED + 1, 1), (n_it, kk)))
        big *= (1.0 + (np.arange(n_it, dtype=np.float32) % 97)[:, None] / 97.0)      # rows differ although the pattern repeats
        mm = native.NativeALS.from_factors(None, big, None, None, device=dev)
        queries = [rng.integers(0, n_it, rng.integers(1, 6)).astype(np.int32) for _ in range(nqs)]
        mm.similar_batch(queries[:64], 20)
        t0 = time.perf_counter()
        bi, bs, bc = mm.similar_batch(queries, 20)
        dt = time.perf_counter() - t0
        ns2 = 24
        t0 = time.perf_counter()
        ok = True
        for j in range(ns2):
            oi, os_, oc = o.similar(big, None, queries[j], 20)
            ok = ok and np.array_equal(bi[j], oi) and np.array_equal(bs[j], os_)
        cpu_dt = time.perf_counter() - t0
        lat2 = []
        q1 = [q for q in queries if len(q) == 1][:10] or queries[:10]
        for j in range(210):         # ten warm-up calls, then 200 timed ones: one query of one item, top-20
            t0 = time.perf_counter()
            mm.similar(q1[j % len(q1)], 20)
            if j >= 10:
                lat2.append(time.perf_counter() - t0)
        sb = n_it * kk * 4
        nvec = float(sum(len(q) for q in queries))
        out["similar_c4"] = {
            "what": f"pio_als_similar_batch: {nqs} queries of 1-5 items, cosine top-20 over {n_it} item vectors, rank {kk}, "
                    "one call, host buffers",
            "value": nqs / dt, "unit": "predictions/s", "seconds": dt,
            "bit_exact_vs_oracle_on_sample": bool(ok), "sample_queries_checked": ns2,
            "cpu_baseline": {"value": ns2 / cpu_dt, "unit": "predictions/s", "cores": cores, "kind": "port",
                             "sample": f"{ns2} of the same queries (oracle restatement of the similarproduct predict scan)"},
            "roofline": {"bound": "fp64", "achieved": 2.0 * (nvec + nqs / 8.0) * n_it * kk / dt / 1e12, "peak": peaks["dfma"],
                         "unit": "TFLOP/s", "frac": 2.0 * (nvec + nqs / 8.0) * n_it * kk / dt / 1e12 / peaks["dfma"],
                         "note": "fp64 cosine in index order (bit-identical to the reference's loop): one DFMA per (query "
                                 "vector, item, feature) + one per (item, feature) and group of 8 queries for the item norm",
                         "hbm_frac_per_8_queries": nqs / 8.0 * sb / dt / 1e9 / peaks["hbm"]},
            "single_query_ms": float(np.median(lat2) * 1e3), "single_query_p90_ms": float(np.percentile(lat2, 90) * 1e3),
            "single_query_what": "pio_als_similar, one query item, top-20, through the Python binding (ctypes, host buffers): "
                                 "one fused launch, result polled from mapped host memory",
            "single_query_hbm_floor_ms": sb / (peaks["hbm"] * 1e9) * 1e3}
        mm.close()
    except Exception as e:
        out["similar_c4"] = {"error": repr(e)}
    # classification template (A11, BASELINE.json configs[4]): MLlib multinomial NaiveBayes on 10 M labelled points x 3 features
    try:
        n_nb = 10_000_000
        y = rng.integers(0, 4, n_nb).astype(np.int32)
        x = rng.integers(0, 10, (n_nb, 3)).astype(np.float32)
        native.nb_train(y[:1000], x[:1000], 4, 1.0, device=dev)
        t0 = time.perf_counter()
        pi, theta = native.nb_train(y, x, 4, 1.0, device=dev)
        t_tr = time.perf_counter() - t0
        t0 = time.perf_counter()
        lab = native.nb_predict(x, pi, theta, device=dev)
        t_pr = time.perf_counter() - t0
        ns3 = 1_000_000
        t0 = time.perf_counter()
        opi, oth = o.nb_train(y[:ns3], x[:ns3], 4, 1.0)
        cpu_tr = time.perf_counter() - t0
        fpi, fth = o.nb_train(y, x, 4, 1.0)
        out["naive_bayes_c5"] = {
            "what": f"pio_nb_train / pio_nb_predict: {n_nb} labelled points x 3 features, 4 classes, host buffers (H2D inside)",
            "train_rows_per_s": n_nb / t_tr, "train_seconds": t_tr, "predict_rows_per_s": n_nb / t_pr,
            "predict_seconds": t_pr, "bytes": int(x.nbytes + y.nbytes),
            "train_gbs_incl_h2d": (x.nbytes + y.nbytes) / t_tr / 1e9,
            "bit_exact_vs_oracle": bool(np.array_equal(pi, fpi) and np.array_equal(theta, fth) and
                                        np.array_equal(lab[:ns3], o.nb_predict(x[:ns3], fpi, fth))),
            "cpu_baseline": {"value": ns3 / cpu_tr, "unit": "rows/s (train)", "cores": 1, "kind": "port",
                             "sample": f"{ns3} of the same rows, single-threaded restatement of NaiveBayes.train"}}
    except Exception as e:
        out["naive_bayes_c5"] = {"error": repr(e)}
    # single-query latency
    lat = []
    for q in range(210):
        t0 = time.perf_counter()
        m.recommend(users[q:q + 1], 10)
        if q >= 10:
            lat.append(time.perf_counter() - t0)
    out["recommend"]["single_query_ms"] = float(np.median(lat) * 1e3)
    out["recommend"]["single_query_p90_ms"] = float(np.percentile(lat, 90) * 1e3)
    out["recommend"]["single_query_hbm_floor_ms"] = scan_bytes / (peaks["hbm"] * 1e9) * 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("PIO_BENCH_WORKLOAD", "c2"), choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-topk", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the factors of the timed run (a seeded sample of rows, < 64 MB) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    nu, ni, nnz, k, implicit = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl_name = (f"ALS rank={k}, {nu} users x {ni} items, {nnz} synthetic "
               f"{'implicit' if implicit else 'explicit'} ratings")
    config = {"workload": wl_name, "lambda": LAMBDA, "alpha": ALPHA, "seed": SEED,
              "dedup": "sum" if implicit else "none",
              "l2": "inputs (1.6 GB of CSR + 282 MB of factors per iteration at c2) exceed the 126 MB L2",
              "parallelism": (f"rows and input events sharded x{args.gpus}, ratings routed to row owners by NCCL send/recv, "
                              "factor all-gather per half-iteration") if args.gpus > 1 else "1 GPU"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        reference_arm(args, nu, ni, nnz, k, implicit, config)
        return 0

    import torch
    import pio_b200  # noqa: F401
    from pio_b200 import native

    torch.cuda.set_device(local_rank)
    dev = local_rank
    nccl_id = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt = torch.tensor(list(native.nccl_unique_id()), dtype=torch.uint8, device="cuda")
        dist.broadcast(idt, 0)
        nccl_id = bytes(idt.cpu().tolist())

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            torch.cuda.synchronize()

    # ---- inputs resident in HBM ----------------------------------------------------------
    # N > 1: every rank generates and holds only ITS slice of the events (pio_als_set_ratings_coo_sharded_device); the
    # library routes the ratings to the owners of their rows.  No rank holds the full COO.
    per = nnz // world
    ev_lo = rank * per
    ev_hi = nnz if rank == world - 1 else ev_lo + per
    n_loc = ev_hi - ev_lo
    du = torch.empty(n_loc, dtype=torch.int32, device="cuda")
    di = torch.empty(n_loc, dtype=torch.int32, device="cuda")
    dr = torch.empty(n_loc, dtype=torch.float32, device="cuda")
    native.synth_ratings_device(dev, nu, ni, n_loc, SEED, implicit, ev_lo, du.data_ptr(), di.data_ptr(), dr.data_ptr())
    dedup = native.DEDUP_SUM if implicit else native.DEDUP_NONE
    m = native.NativeALS(k, nu, ni, lam=LAMBDA, implicit=implicit, alpha=ALPHA, seed=SEED, device=dev,
                         world_size=world, world_rank=rank, nccl_id=nccl_id, init_mode=native.INIT_HASH)
    m.set_ratings_device(du.data_ptr(), di.data_ptr(), dr.data_ptr(), n_loc, dedup=dedup, sharded=world > 1)
    ingest_ms = m.stats()["last_ingest_ms"]
    nnz_eff = m.stats()["nnz"]
    m.run(max(args.warmup, 0))
    l0 = m.stats()
    sampler = ClockSampler(dev)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    m.run(args.steps)
    barrier()
    wall_s = time.perf_counter() - t0
    clocks = sampler.stop()
    st = m.stats()
    ph = m.phase_ms()
    dev_ms = st["last_run_ms"]
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([dev_ms, st["last_solve_ms"], st["last_gram_ms"], st["last_comm_ms"], wall_s * 1e3,
                          ph["user_solve_ms"], ph["item_solve_ms"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, solve_ms, gram_ms, comm_ms, wall_ms, ph["user_solve_ms"], ph["item_solve_ms"] = t.tolist()
    else:
        solve_ms, gram_ms, comm_ms, wall_ms = st["last_solve_ms"], st["last_gram_ms"], st["last_comm_ms"], wall_s * 1e3
    launches = st["kernel_launches"] - l0["kernel_launches"]
    solve_launches = st["solve_launches"] - l0["solve_launches"]
    value = args.steps / (dev_ms / 1e3)

    # factors after W + K iterations (checksum; source of the parity iteration); then one more iteration for parity
    want_parity = not args.no_parity and nnz <= 200_000_000   # the host-side CSR of a 1 B-rating workload takes minutes
    uf_T = itf_T = uf_T1 = itf_T1 = uh = ih = None
    if rank == 0:
        uf_T, itf_T, uh, ih = m.get_factors()
    checksum = factor_checksum(uf_T, itf_T) if rank == 0 else None
    dumped = dump_outputs(args.dump_outputs, uf_T, itf_T, uh, ih) if args.dump_outputs and rank == 0 else None
    if want_parity:
        m.run(1)
        if rank == 0:
            uf_T1, itf_T1, _, _ = m.get_factors()

    # ---- end to end through the C ABI with host buffers ------------------------------------
    e2e = None
    if not args.no_e2e:
        hu = torch.empty(n_loc, dtype=torch.int32).pin_memory()
        hi = torch.empty(n_loc, dtype=torch.int32).pin_memory()
        hr = torch.empty(n_loc, dtype=torch.float32).pin_memory()
        hu.copy_(du)
        hi.copy_(di)
        hr.copy_(dr)
        out_u = torch.empty((nu, k), dtype=torch.float32).pin_memory() if rank == 0 else None
        out_i = torch.empty((ni, k), dtype=torch.float32).pin_memory() if rank == 0 else None
        m2 = native.NativeALS(k, nu, ni, lam=LAMBDA, implicit=implicit, alpha=ALPHA, seed=SEED, device=dev,
                              world_size=world, world_rank=rank, nccl_id=None if world == 1 else nccl_id_2(native, rank, world),
                              init_mode=native.INIT_HASH)

        def train_call(a, b, c, ou, oi, iters):
            """What a JNI ALS.train binding does: ratings in (this rank's slice), K iterations, factors out (rank 0)."""
            if world == 1:
                m2.train(a, b, c, iters, dedup=dedup, out_user=ou, out_item=oi)
            else:
                m2.set_ratings_sharded(a, b, c, dedup=dedup)
                m2.run(iters)
                if rank == 0:
                    m2.get_factors(out_user=ou, out_item=oi)

        def timed_train(a, b, c, ou, oi):
            barrier()
            t0 = time.perf_counter()
            train_call(a, b, c, ou, oi, args.steps)
            barrier()
            s_ = time.perf_counter() - t0
            if world > 1:
                import torch.distributed as dist
                t = torch.tensor([s_], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                s_ = float(t.item())
            return s_

        ou_np = out_u.numpy() if rank == 0 else None
        oi_np = out_i.numpy() if rank == 0 else None
        train_call(hu.numpy(), hi.numpy(), hr.numpy(), ou_np, oi_np, 1)   # warm-up
        e2e_s = timed_train(hu.numpy(), hi.numpy(), hr.numpy(), ou_np, oi_np)
        st2 = m2.stats()
        # the same call with ordinary pageable arrays (what a JNI caller holding GetPrimitiveArrayCritical arrays passes)
        pu, pi_, pr = (np.array(x.numpy(), copy=True) for x in (hu, hi, hr))
        pou = np.empty((nu, k), np.float32) if rank == 0 else None
        poi = np.empty((ni, k), np.float32) if rank == 0 else None
        e2e_pageable_s = timed_train(pu, pi_, pr, pou, poi)
        del pu, pi_, pr, pou, poi
        h2d_call, d2h_call = 12 * nnz, 4 * (nu + ni) * k + (nu + ni)
        e2e = {"value": args.steps / e2e_s, "unit": "iterations/s", "seconds_per_train_call": e2e_s,
               "iterations_per_call": args.steps,
               "h2d_bytes_per_step": h2d_call / args.steps, "d2h_bytes_per_step": d2h_call / args.steps,
               "h2d_bytes_per_call": h2d_call, "d2h_bytes_per_call": d2h_call,
               "host_memory": "pinned", "value_pageable_host_memory": args.steps / e2e_pageable_s,
               "ingest_ms": st2["last_ingest_ms"], "run_ms": st2["last_run_ms"],
               "note": "one training call = H2D of the COO triplets (N > 1: every rank copies only its 1/N slice, "
                       "pio_als_set_ratings_coo_sharded) + ingest + K iterations + D2H of the factors (rank 0); the copies "
                       "happen once per call, so bytes per step = bytes per call / K"}
        m2.close()
        del hu, hi, hr, out_u, out_i

    if rank != 0:
        return 0

    # ---- roofline of the dominant kernel ------------------------------------------------------
    # One iteration = item half-step + user half-step; each is (YtY) + one solve launch for the rows up to the
    # heavy-row threshold (+ a part launch and a finish launch for longer rows).  The dominant kernel is the solve
    # launch of the slower half-step; its time is the CUDA-event time of that half-step's solve launches (measured
    # inside pio_als_run on the launching stream), its work the algorithmic FLOPs / bytes of that side.
    peaks = measured_peaks()
    hbm_peak, bf16_peak, peak_src = peaks["hbm"], peaks["bf16"], peaks["src"]
    nua = int(uh.sum())
    nia = int(ih.sum())
    b_alg, f_solve, f_gram = algorithmic_work(nua, nia, nnz_eff, k, implicit)
    side_flops = {"user": 2 * nnz_eff * (k * (k + 1) + 2 * k) / 2 + nua * (k ** 3 / 3 + 2 * k * k),
                  "item": 2 * nnz_eff * (k * (k + 1) + 2 * k) / 2 + nia * (k ** 3 / 3 + 2 * k * k)}
    side_bytes = {"user": 8 * nnz_eff + 4 * nua * k + 4 * nia * k, "item": 8 * nnz_eff + 4 * nia * k + 4 * nua * k}
    side_ms = {"user": ph["user_solve_ms"] / args.steps, "item": ph["item_solve_ms"] / args.steps}
    side_kernel = {"user": ph["user_kernel"], "item": ph["item_kernel"]}
    side_tc = {sd: side_kernel[sd] != "fp32" for sd in side_kernel}   # Gramian on tensor cores (tcgen05 or mma.sync)
    kernel_names = {"fp32": "als_solve_kernel (gather + FP32 Gramian + warp Cholesky)",
                    "tcgen05": "tc::als_solve_tc_kernel (tcgen05 split-TF32 Gramian + warp Cholesky)",
                    "mma": "mm::als_solve_mma_kernel (one warp per row: mma.sync 3xTF32 Gramian + warp Cholesky)",
                    "pair": "pr::als_solve_pair_kernel (two rows per warp: mma.sync 3xTF32 Gramian + lockstep Cholesky)"}
    fp32_peak = peaks["fp32"]
    tf32_peak = bf16_peak / 2.0
    split_peak = tf32_peak / 3.0   # an fp32-class product costs three TF32 MMAs (hi*hi + lo*hi + hi*lo)

    def side_obj(sd):
        tf = side_flops[sd] / (side_ms[sd] / 1e3) / 1e12 / max(world, 1)
        gb = side_bytes[sd] / (side_ms[sd] / 1e3) / 1e9 / max(world, 1)
        o_ = {"kernel": kernel_names[side_kernel[sd]] + f", {sd} half-step",
              "ms_per_launch": side_ms[sd], "algorithmic_flops": side_flops[sd], "algorithmic_bytes": side_bytes[sd],
              "achieved_tflops": tf, "achieved_gbs": gb, "frac_of_fp32_fma_peak": tf / fp32_peak,
              "frac_of_hbm_peak": gb / hbm_peak}
        if side_tc[sd]:
            o_["frac_of_split_tf32_tensor_peak"] = tf / split_peak
        return o_

    dom = "user" if side_ms["user"] >= side_ms["item"] else "item"
    other = "item" if dom == "user" else "user"
    d = side_obj(dom)
    roofline = {
        "kernel": d["kernel"],
        "bound": "fp32_fma" if not side_tc[dom] else "tensor",
        "achieved": d["achieved_tflops"], "peak": fp32_peak if not side_tc[dom] else split_peak, "unit": "TFLOP/s",
        "frac": d["achieved_tflops"] / (fp32_peak if not side_tc[dom] else split_peak),
        "frac_of_fp32_fma_peak": d["achieved_tflops"] / fp32_peak,
        "fp32_fma_peak": fp32_peak, "fp32_fma_peak_source": peaks["fp32_src"],
        "mma_sync_tf32_peak_tflops": peaks["mma_tf32"],
        "peak_source": peaks["fp32_src"] if not side_tc[dom] else
                       f"{peak_src} dense bf16 / 2 = tf32 MMA rate, / 3 because an fp32-class product is three TF32 MMAs",
        "ms_per_launch": d["ms_per_launch"],
        "traffic": traffic_from_profiles(args.workload),
        "traffic_unit": "dram bytes of this launch, from the committed ncu --set full capture (profiles/traffic.json)",
        "per_gpu": True,
        "hbm": {"achieved": d["achieved_gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": d["achieved_gbs"] / hbm_peak,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": d["algorithmic_bytes"]},
        "other_half_step": side_obj(other),
        "solve_ms_per_iteration": solve_ms / args.steps, "gram_ms_per_iteration": gram_ms / args.steps,
        "comm_ms_per_iteration": comm_ms / args.steps,
        "launches_per_iteration": solve_launches / max(args.steps, 1),
        "algorithmic_flops_per_iteration": f_solve, "algorithmic_bytes_per_iteration": b_alg,
    }
    out = {"metric": "ALS iterations/sec", "value": value, "unit": "iterations/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "config": config, "clocks": clocks, "gpu_launches": int(launches),
           "wall_ms_per_step": wall_ms / args.steps, "ingest_ms": ingest_ms, "nnz_after_dedup": int(nnz_eff),
           "factor_checksum": checksum,
           "factor_checksum_note": f"crc32(user factors) || crc32(item factors) after {args.warmup}+{args.steps} iterations "
                                   "from the hash initialisation: the same at every GPU count (sharded runs are bit-identical)",
           "roofline": roofline}
    if e2e:
        out["e2e"] = e2e
    if dumped:
        out["dumped_outputs"] = dumped

    rc = 0
    need_host = (want_parity or (not args.no_cpu_baseline and args.gpus == 1) or not args.no_topk)
    if need_host:
        o, cores = load_oracle()
    if want_parity or (not args.no_cpu_baseline and args.gpus == 1):
        del du, di, dr
        torch.cuda.empty_cache()
        fu = torch.empty(nnz, dtype=torch.int32, device="cuda")
        fi = torch.empty(nnz, dtype=torch.int32, device="cuda")
        fr = torch.empty(nnz, dtype=torch.float32, device="cuda")
        native.synth_ratings_device(dev, nu, ni, nnz, SEED, implicit, 0, fu.data_ptr(), fi.data_ptr(), fr.data_ptr())
        coo = (fu.cpu().numpy(), fi.cpu().numpy(), fr.cpu().numpy())
        del fu, fi, fr
        prob = build_host_problem(o, nu, ni, k, implicit, coo)
        del coo
        if want_parity:
            par = parity_sample(o, prob, uf_T, itf_T1, uf_T1)
            par["host_nnz_after_dedup"] = prob["nnz"]
            par["ok"] = bool(par["ok"] and prob["nnz"] == int(nnz_eff))
            out["parity"] = par
            if not par["ok"]:
                rc = 3
        if not args.no_cpu_baseline and args.gpus == 1:
            cu, ci = np.array(uf_T, copy=True), np.array(itf_T, copy=True)
            out["cpu_baseline"] = cpu_baseline_steps(o, cores, prob, cu, ci, n_steps=1, n_warm=0, budget_s=30.0)
        del prob
    if not args.no_topk and args.gpus == 1:
        try:
            # the handle holds the factors of its LAST run: iteration W+K+1 when the parity iteration ran
            cur_u, cur_i = (uf_T1, itf_T1) if want_parity else (uf_T, itf_T)
            out["topk"] = topk_bench(native, o, cores, m, nu, ni, k, cur_u, cur_i, uh, ih, peaks, dev)
        except Exception as e:   # a scoring failure must not hide the training line
            out["topk"] = {"error": repr(e)}
            rc = rc or 4
    print(json.dumps(out))
    return rc


def nccl_id_2(native, rank, world):
    """A second communicator id for the e2e handle (broadcast from rank 0)."""
    import torch
    import torch.distributed as dist
    idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        idt = torch.tensor(list(native.nccl_unique_id()), dtype=torch.uint8, device="cuda")
    dist.broadcast(idt, 0)
    return bytes(idt.cpu().tolist())


if __name__ == "__main__":
    rc = main()
    try:   # leave the torch.distributed group cleanly (no teardown warning after the JSON line)
        import torch.distributed as _dist
        if _dist.is_available() and _dist.is_initialized():
            _dist.destroy_process_group()
    except Exception:
        pass
    sys.exit(rc or 0)
