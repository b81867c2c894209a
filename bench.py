#!/usr/bin/env python
"""bench.py -- headline benchmark of the exact-GP hot path (BASELINE.json metric):
ms to logpdf(fx,y) + posterior(fx,y) at N x D fp64, with the achieved fraction of the tensor roofline of the
trailing update and of the N^3/3 Cholesky rate, next to the reference's CPU LAPACK path timed on the same box.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C4|C2|C4h|C3|C5] [--impl ours|reference] [--n N]
                  [--dump-outputs DIR]

The SAME workload (C4: N = 65 536, D = 64, SqExponential, fp64 -- the configuration BASELINE.json's metric and target are
quoted on; it fits one B200) runs at every --gpus value, so the per-N values form a strong-scaling curve.  At N = 1 the
line also carries C2 (N = 4096, D = 8) as the secondary key "c2".

One "step" = one pass of the hot path through the C ABI of libagp.so:
  fit workloads (C2, C4, C4h): ONE fused fit (Gram + Cholesky -> logpdf, alpha, posterior factor);
  C3: fit (fp32, Matern32 o ARD) + mean_and_var at 10 000 test points;   C5: VFE elbo (streamed over N).
`value` is measured with the inputs resident in HBM (device-pointer mode of the ABI); `e2e` is the same call with pinned
HOST buffers, H2D/D2H inside the timed region.  Device times come from CUDA events recorded by the library on its
launching stream, max over ranks.  The oracle (oracle/agp_ref.py) is used here only as the CPU baseline and as the
out-of-timed-region parity checker.

--dump-outputs DIR writes what the last device-resident timed step returned to its caller as DIR/<name>.npy (logpdf and
alpha; mean and var for C3; elbo and dtc for C5), so two builds can be compared output for output on the same seeded
inputs.  An array too large for the 64 MB budget is replaced by a fixed seeded sample of its entries.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # a benchmark run leaves the tree as it found it (it may be read-only)

WORKLOADS = {  # BASELINE.json configs (SURVEY.md s8d)
    "C2": dict(kind="fit", N=4096, D=8, dtype="f64", kernel="SqExponential", s2=0.1, cfg="C2"),
    "C4": dict(kind="fit", N=65536, D=64, dtype="f64", kernel="SqExponential", s2=0.1, cfg="C4"),
    "C4h": dict(kind="fit", N=32768, D=64, dtype="f64", kernel="SqExponential", s2=0.1, cfg="C4"),
    "C3": dict(kind="fit_predict", N=16384, D=32, M=10000, dtype="f32", kernel="Matern32 o ARDTransform", s2=0.05, cfg="C3"),
    "C5": dict(kind="vfe", N=1000000, D=16, M=8192, dtype="f32", kernel="SqExponential", s2=0.1, cfg="C5"),
}
METRIC = {"fit": "ms to logpdf(fx,y)+posterior(fx,y)", "fit_predict": "ms to logpdf+posterior+mean_and_var(10000 test points)",
          "vfe": "ms to elbo(VFE(f(z)), fx, y)"}
CPU_SUB = 8192  # bounded CPU sample for the cubic workloads (scaled by (N/8192)^3, labelled extrapolated)
DUMP_BYTES = 64 * 10 ** 6  # everything --dump-outputs writes, .npy headers included


def make_inputs(wl, n=None):
    from oracle import agp_ref as ref  # synthetic-input generator only (shared with the parity tests)
    W = WORKLOADS[wl]
    return ref.make_config(W["cfg"], n=n or W["N"])


def wl_string(wl, N, extra=""):
    W = WORKLOADS[wl]
    s = "%s: N=%d D=%d %s %s, sigma2=%g" % (wl, N, W["D"], W["kernel"], "fp64" if W["dtype"] == "f64" else "fp32", W["s2"])
    if W["kind"] == "fit_predict":
        s += ", M=%d test points" % W["M"]
    if W["kind"] == "vfe":
        s += ", M=%d inducing points" % min(W["M"], max(8, N // 8))
    return s + extra


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.dev, self.rows, self.p = dev, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.dev), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        pw = [float(r[3]) for r in self.rows if len(r) >= 9 and r[3].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


def trailing_flops(N, nb=128):
    """algorithmic flops of the outer trailing updates of one factorisation with nb-wide panels: step k applies a
    symmetric rank-K update to the m x m trailing matrix (lower part): 2*K*m(m+1)/2."""
    n_pad = (N + 127) // 128 * 128
    tot, t0 = 0.0, 0
    while t0 < n_pad:
        K = min(nb, n_pad - t0)
        t0 += K
        m = n_pad - t0
        tot += 2.0 * K * m * (m + 1) / 2
    return tot


# ------------------------------------------------------------------------------------------------------------
# CPU side: the reference's own algorithm (oracle port) on the box's host cores
# ------------------------------------------------------------------------------------------------------------
def cpu_step(wl, cfg):
    """One step of the reference's CPU algorithm for the workload (oracle port).  fit: logpdf THEN posterior -- TWO Gram
    builds and TWO LAPACK potrf's, as /root/reference/src/finite_gp_projection.jl:307-308 + src/exact_gpr_posterior.jl:30-31
    do; the Distances.jl (gemm) pairwise formulation the reference executes."""
    from oracle import agp_ref as ref
    kind = WORKLOADS[wl]["kind"]
    old = ref.DEFAULT_METHOD
    ref.DEFAULT_METHOD = "gemm"
    try:
        if kind == "vfe":
            return ref.elbo(cfg["k"], cfg["mean"], cfg["noise"], cfg["X"], cfg["y"], cfg["Z"], cfg["jitter"])
        lp = ref.logpdf(cfg["k"], cfg["mean"], cfg["noise"], cfg["X"], cfg["y"])
        post = ref.posterior(cfg["k"], cfg["mean"], cfg["noise"], cfg["X"], cfg["y"])
        if kind == "fit_predict":
            ref.post_mean_and_var(post, cfg["Xs"], noise_s=cfg["noise"])
        return lp
    finally:
        ref.DEFAULT_METHOD = old


def cpu_sample(wl, n_full):
    """bounded sample of the workload for the CPU arm: (cfg, scale, description)"""
    W = WORKLOADS[wl]
    if W["kind"] == "vfe":  # cost 2 M^2 N: bounded N and M (make_config ties M = min(8192, N / 8)), scaled back
        sub = min(n_full, 20000)
        cfg = make_inputs(wl, n=sub)
        m_sub, m_full = cfg["Z"].shape[0], min(W["M"], max(8, n_full // 8))
        scale = (n_full / sub) * (m_full / m_sub) ** 2
        if scale == 1.0:
            return cfg, 1.0, "full workload"
        return cfg, scale, "N=%d, M=%d sub-sample scaled by (N/%d) x (M/%d)^2 = %.0f (extrapolated, cost 2 M^2 N)" % (sub, m_sub, sub, m_sub, scale)
    if n_full > CPU_SUB:
        cfg = make_inputs(wl, n=CPU_SUB)
        scale = (n_full / CPU_SUB) ** 3
        if W["kind"] == "fit_predict":
            cfg["Xs"] = cfg["Xs"][: max(1, W["M"] * CPU_SUB // n_full)]  # N^2 M term scaled like N^3
        return cfg, scale, "N=%d sub-sample scaled by (N/%d)^3 = %.0f (extrapolated)" % (CPU_SUB, CPU_SUB, scale)
    return make_inputs(wl, n=n_full), 1.0, "full workload (N=%d)" % n_full


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([p.get("num_threads", 1) for p in threadpool_info()] or [os.cpu_count()])
    except Exception:
        return os.cpu_count()


def best_cpu_threads(wl, cfg):
    """OpenBLAS with every hardware thread of a many-core host is often slower than with fewer on these sizes; give
    the CPU arm its best setting: each candidate thread count is run ONCE, the fastest is kept."""
    try:
        from threadpoolctl import threadpool_limits
    except Exception:
        return None, blas_threads()
    cand = sorted({c for c in (8, 16, 32, 64, blas_threads()) if c <= (os.cpu_count() or 8)})
    best, best_c = 1e18, cand[-1]
    for c in cand:
        with threadpool_limits(limits=c):
            t0 = time.perf_counter()
            cpu_step(wl, cfg)
            dt = time.perf_counter() - t0
        if dt < best:
            best, best_c = dt, c
    return threadpool_limits(limits=best_c), best_c


def cpu_baseline(wl, n_full, reps=2):
    cfg, scale, sample = cpu_sample(wl, n_full)
    limiter, cores = best_cpu_threads(wl, cfg)
    best = 1e18
    for _ in range(reps):
        t0 = time.perf_counter()
        cpu_step(wl, cfg)
        best = min(best, time.perf_counter() - t0)
    del limiter
    return {"value": best * 1e3 * scale, "unit": "ms", "cores": cores, "kind": "port",
            "sample": sample + "; reference-faithful step (logpdf then posterior = 2 Gram + 2 potrf) for fit workloads; "
                               "BLAS threads = fastest of {8,16,32,64,all}, best of %d" % reps}


def run_reference(args, wl, n_full):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    W = WORKLOADS[wl]
    cfg, scale, sample = cpu_sample(wl, n_full)
    limiter, cores = best_cpu_threads(wl, cfg)
    for _ in range(args.warmup):
        cpu_step(wl, cfg)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_step(wl, cfg)
    ms = (time.perf_counter() - t0) * 1e3 / args.steps * scale
    del limiter
    line = {"impl": "reference", "metric": METRIC[W["kind"]], "value": ms, "unit": "ms",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": W["dtype"], "data": "synthetic",
            "config": {"workload": wl_string(wl, n_full)},
            "cpu_baseline": {"value": ms, "unit": "ms", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": ms, "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------------------
def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def measure_dgemm_peak(torch, dev):
    """native fp64 reference rate: cuBLAS DGEMM 8192^3 on this box, best of 5 (CUDA events)."""
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def measure_int8_mma_peak(eng, torch, dev, S=7):
    """MEASURED int8 tcgen05 rate of this kernel's own instruction mix: the persistent trailing-update kernel run with
    its operand traffic and epilogue switched off (probe mode 5: every tile still issues all of its tcgen05.mma.kind::i8
    instructions on operands already in shared memory).  TOP/s = executed int8 ops / time, slicing time subtracted."""
    import ctypes as C
    M, K = 16384, 512
    P = torch.randn(K, M, dtype=torch.float64, device=dev)
    Cm = torch.zeros(M, M, dtype=torch.float64, device=dev)
    old = os.environ.get("AGP_OZAKI_EPI")

    def run(ncols):
        best = 1e9
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            eng.check(eng.L.agp_debug_ozaki_syrk(eng.h, C.c_void_p(Cm.data_ptr()), M, C.c_void_p(P.data_ptr()), M, M, ncols, K, S, 1))
            best = min(best, time.perf_counter() - t0)
        return best
    try:
        os.environ["AGP_OZAKI_EPI"] = "5"
        fixed = run(128)
        full = run(M)
    finally:
        if old is None:
            os.environ.pop("AGP_OZAKI_EPI", None)
        else:
            os.environ["AGP_OZAKI_EPI"] = old
    nbi, nbj = M // 128, M // 64
    tiles = sum(min(nbj, 2 * bi + 2) for bi in range(nbi)) - 2  # minus the strip of the `fixed` run (approx.)
    ops = 2.0 * tiles * 128 * 64 * K * (S * (S + 1) // 2)
    del P, Cm
    return ops / max(full - fixed, 1e-9) / 1e12


def ncu_traffic(tag):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel from the committed ncu capture
    under profiles/ (see profiles/README.md), with that launch's algorithmic bytes -- None when no capture is committed."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[tag]
    except Exception:
        return None


class FitProblem:
    """device + pinned-host copies of one workload and the ABI call that is a 'step'"""

    def __init__(self, wl, n, eng, torch, dev, need_post=True):
        import ctypes as C
        from agp_b200 import _cabi as cabi
        self.C, self.cabi, self.eng, self.torch = C, cabi, eng, torch
        W = WORKLOADS[wl]
        self.wl, self.W, self.kind = wl, W, W["kind"]
        cfg = make_inputs(wl, n)
        self.cfg = cfg
        self.np_dt = np.float64 if W["dtype"] == "f64" else np.float32
        self.code = cabi.AGP_F64 if W["dtype"] == "f64" else cabi.AGP_F32
        X = np.ascontiguousarray(cfg["X"], dtype=self.np_dt)  # [N, D] C-order == D x N column-major (ColVecs)
        y = np.ascontiguousarray(cfg["y"], dtype=self.np_dt)
        self.N, self.D = X.shape
        ks = cabi.agp_kernel()
        k = cfg["k"]
        ks.family, ks.variance, ks.linear_c, ks.scale = int(k.family), float(k.variance), 0.0, 1.0
        self.keep = []
        if k.transform == 1:
            ks.transform, ks.scale = 1, float(k.scale)
        elif k.transform == 2:
            ard = np.ascontiguousarray(k.ard, dtype=self.np_dt)
            self.keep.append(ard)
            ks.transform, ks.ard = 2, ard.ctypes.data
        self.ks, self.ms, self.ns = ks, cabi.agp_mean(), cabi.agp_noise()
        self.ns.kind, self.ns.s = 0, float(cfg["noise"].s)
        tdt = torch.float64 if W["dtype"] == "f64" else torch.float32
        self.Xh, self.yh = torch.from_numpy(X).pin_memory(), torch.from_numpy(y).pin_memory()
        self.alpha_h = torch.empty(self.N, dtype=tdt).pin_memory()
        self.Xd, self.yd = self.Xh.to(dev), self.yh.to(dev)
        self.alpha_d = torch.empty(self.N, dtype=tdt, device=dev)
        self.lp = np.zeros(2, dtype=self.np_dt)
        self.h2d = int(X.nbytes + y.nbytes)
        self.d2h = int(self.N * X.itemsize + X.itemsize + 12)
        self.need_post = need_post
        if self.kind == "fit_predict":
            Xs = np.ascontiguousarray(cfg["Xs"], dtype=self.np_dt)
            self.M = Xs.shape[0]
            self.Xsh = torch.from_numpy(Xs).pin_memory()
            self.Xsd = self.Xsh.to(dev)
            self.mu_h, self.var_h = torch.empty(self.M, dtype=tdt).pin_memory(), torch.empty(self.M, dtype=tdt).pin_memory()
            self.mu_d, self.var_d = torch.empty(self.M, dtype=tdt, device=dev), torch.empty(self.M, dtype=tdt, device=dev)
            self.h2d += int(Xs.nbytes)
            self.d2h += int(2 * self.M * Xs.itemsize)
        if self.kind == "vfe":
            Z = np.ascontiguousarray(cfg["Z"], dtype=self.np_dt)
            self.M = Z.shape[0]
            self.Zh = torch.from_numpy(Z).pin_memory()
            self.Zd = self.Zh.to(dev)
            self.js = cabi.agp_noise()
            self.js.kind, self.js.s = 0, float(cfg["jitter"].s)
            self.h2d += int(Z.nbytes)
            self.d2h = 2 * X.itemsize

    def step(self, device_resident, dist=False):
        C, cabi, eng, L = self.C, self.cabi, self.eng, self.eng.L
        eng.set_memspace(cabi.AGP_MEM_DEVICE if device_resident else cabi.AGP_MEM_HOST)
        pick = (lambda d, h: d.data_ptr()) if device_resident else (lambda d, h: h.data_ptr())
        xp, yp, ap = pick(self.Xd, self.Xh), pick(self.yd, self.yh), pick(self.alpha_d, self.alpha_h)
        if self.kind == "vfe":
            rc = L.agp_vfe_elbo(eng.h, self.code, C.byref(self.ks), C.byref(self.ms), C.byref(self.ns), cabi.AGP_POINT_MAJOR,
                                C.c_void_p(xp), self.N, self.D, C.c_void_p(pick(self.Zd, self.Zh)), self.M, C.byref(self.js),
                                C.c_void_p(yp), cabi.ptr(self.lp[0:1]), cabi.ptr(self.lp[1:2]))
            eng.check(rc)
            return eng.timings()
        post = C.c_void_p()
        want_post = self.need_post and not dist
        rc = L.agp_fit(eng.h, self.code, C.byref(self.ks), C.byref(self.ms), C.byref(self.ns), cabi.AGP_POINT_MAJOR,
                       C.c_void_p(xp), self.N, self.D, C.c_void_p(yp), 1, cabi.ptr(self.lp), C.c_void_p(ap),
                       C.byref(post) if want_post else None)
        eng.check(rc)
        t = eng.timings()
        if self.kind == "fit_predict":
            rc = L.agp_post_mean_var(post, cabi.AGP_POINT_MAJOR, C.c_void_p(pick(self.Xsd, self.Xsh)), self.M, None,
                                     C.byref(self.ns), C.c_void_p(pick(self.mu_d, self.mu_h)), C.c_void_p(pick(self.var_d, self.var_h)))
            eng.check(rc)
            t2 = eng.timings()
            t["predict"] = t2["predict"]
            t["total"] = t["total"] + t2["predict"]
        if want_post:
            L.agp_post_free(post)
        return t

    def outputs(self):
        """host copies of what the last device-resident step returned (scalars land in host memory in either mode)"""
        self.torch.cuda.synchronize()
        if self.kind == "vfe":
            return {"elbo": self.lp[0:1].copy(), "dtc": self.lp[1:2].copy()}
        out = {"logpdf": self.lp[0:1].copy(), "alpha": self.alpha_d.cpu().numpy()}
        if self.kind == "fit_predict":
            out["mean"], out["var"] = self.mu_d.cpu().numpy(), self.var_d.cpu().numpy()
        return out


def dump_outputs(outs, d):
    """DIR/<name>.npy per output, within DUMP_BYTES in all; a larger array keeps a fixed seeded sample of its entries"""
    os.makedirs(d, exist_ok=True)
    per = (DUMP_BYTES - 1024 * len(outs)) // len(outs)
    for name, a in outs.items():
        a = np.ascontiguousarray(a).reshape(-1)
        cap = per // a.itemsize
        if a.size > cap:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(d, name + ".npy"), a)


def timed(prob, torch, flush, device_resident, steps, warmup, dist=None):
    eng = prob.eng
    for _ in range(warmup):
        prob.step(device_resident, dist is not None)
    tot = {}
    torch.cuda.synchronize()
    launches0 = eng.launch_count()
    wall = 0.0
    for _ in range(steps):
        flush.zero_()  # L2 flush between timed iterations (outside the event-timed region)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        t = prob.step(device_resident, dist is not None)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        wall += time.perf_counter() - t0
        for k_, v in t.items():
            tot[k_] = tot.get(k_, 0.0) + v
    launches = eng.launch_count() - launches0
    mine = {k_: v / steps for k_, v in tot.items()}
    if dist is not None:
        keys = sorted(mine)
        tt = torch.tensor([mine[k_] for k_ in keys], dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)  # max over ranks, per phase
        mine = dict(zip(keys, tt.tolist()))
    return mine, wall * 1e3 / steps, launches


def parity_check(wl, prob_cls_args, eng, torch, dev, dist=None):
    """out-of-timed-region parity of the BENCHED path against the oracle: the workload itself when N <= 8192, else its
    first 8192 points through the same engine configuration (n_pad >= 8192 keeps the tcgen05 / distributed path)."""
    from oracle import agp_ref as ref
    W = WORKLOADS[wl]
    n_full = prob_cls_args["n"]
    n = min(n_full, CPU_SUB)
    if W["kind"] == "vfe":
        n = min(n_full, 20000)
    p = FitProblem(wl, n, eng, torch, dev)
    p.step(True, dist is not None)
    got = float(p.lp[0])
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    cfg = p.cfg
    tol = 1e-8 if W["dtype"] == "f64" else 1e-4
    old = ref.DEFAULT_METHOD
    ref.DEFAULT_METHOD = "gemm"  # the reference's executed formulation (Distances.jl pairwise)
    try:
        c64 = {k_: (v.astype(np.float64) if isinstance(v, np.ndarray) else v) for k_, v in cfg.items()}
        k64 = cfg["k"]
        if getattr(k64, "ard", None) is not None:
            k64 = ref.KernelSpec(k64.family, k64.variance, k64.transform, k64.scale, np.asarray(k64.ard, dtype=np.float64), k64.linear_c)
        if W["kind"] == "vfe":
            want = ref.elbo(k64, cfg["mean"], cfg["noise"], c64["X"], c64["y"], c64["Z"], cfg["jitter"])
        else:
            want = ref.logpdf(k64, cfg["mean"], cfg["noise"], c64["X"], c64["y"])
    finally:
        ref.DEFAULT_METHOD = old
    return {"quantity": "elbo" if W["kind"] == "vfe" else "logpdf", "n": n, "ours": got, "oracle": float(want),
            "rel_err": float(abs(got - want) / abs(want)), "tol": tol, "ok": bool(abs(got - want) <= tol * abs(want)),
            "oracle_form": "fp64, Distances.jl gemm form", "sample": "full workload" if n == n_full else "first %d points, same engine config" % n}


def fit_roofline(wl, N, eng, torch, dev, prob, flush, args, world=1, dist=None, t_dev=None):
    """roofline of the dominant kernel = the outer trailing update.  Its launches are timed with CUDA events around every
    launch inside the library (profile_kernels = 1); on one GPU the look-ahead schedule overlaps two of them on two
    streams, so that pass runs with look-ahead OFF (serial launches), same inputs, same kernels."""
    peaks = load_peaks()
    cfg0 = eng.get_config()
    W = WORKLOADS[wl]
    if dist is None:
        eng.set_config(lookahead=0, profile_kernels=1)
    else:
        eng.set_config(profile_kernels=1)
    roof_steps = min(args.steps, 3)
    t_serial, _, _ = timed(prob, torch, flush, True, roof_steps, 1, dist)
    eng.set_config(lookahead=cfg0.lookahead, profile_kernels=cfg0.profile_kernels)
    n_pad = (N + 127) // 128 * 128
    nb = cfg0.tile_nb if cfg0.tile_nb > 0 else (512 if n_pad >= 8192 else 128)
    if world > 1:
        n_pad = (N + nb - 1) // nb * nb
    mode = cfg0.fp64_mode if cfg0.fp64_mode >= 0 else (1 if n_pad >= 8192 else 0)
    S_sl = cfg0.ozaki_slices
    tf = trailing_flops(N, nb)
    launches = max(1, n_pad // nb - 1)
    trailing_ms = t_serial.get("trailing", 0.0)  # max over ranks of the per-rank sum of launch durations
    out = {"launches_per_step": launches * world, "alg_flops_per_step": tf, "kernel_ms_per_step": trailing_ms,
           "kernel_ms_per_step_rank_max": trailing_ms, "panel_width": nb,
           "kernel_timing": "CUDA events around each launch%s, %d steps" % (", look-ahead off (serial)" if dist is None else ", max over ranks of the per-rank sum", roof_steps)}
    if W["dtype"] == "f64" and mode == 1:
        pairs = S_sl * (S_sl + 1) // 2
        fp64_eq = tf / world / (trailing_ms * 1e-3) / 1e12 if trailing_ms > 0 else None  # per GPU
        achieved = fp64_eq * pairs if fp64_eq else None  # executed int8 TOP/s per GPU: every fp64 MAC = S(S+1)/2 int8 MACs
        mma_peak = measure_int8_mma_peak(eng, torch, dev, S_sl)
        nominal = 4500.0
        out.update({"bound": "tensor", "kernel": "umma_ozaki_syrk_v2_kernel<%d> (tcgen05.mma.kind::i8, TMA, TMEM; persistent)" % S_sl,
                    "achieved": achieved, "peak": mma_peak, "unit": "TOP/s (int8 tensor, dense, per GPU)",
                    "frac": (achieved / mma_peak) if achieved else None,
                    "peak_source": "MEASURED in this run: the same kernel's tcgen05.mma.kind::i8 instruction stream with operand traffic and "
                                   "epilogue off (operands resident in shared memory), 16384 x 16384 x 512 -- the tensor-pipe ceiling of this "
                                   "instruction mix on this box",
                    "frac_of_2x_bf16_measured": (achieved / (2.0 * peaks["bf16_tflops"])) if (achieved and "bf16_tflops" in peaks) else None,
                    "frac_of_nominal_4500": (achieved / nominal) if achieved else None,
                    "fp64_equivalent_tflops_per_gpu": fp64_eq, "slices": S_sl, "int8_macs_per_fp64_mac": pairs})
    elif W["dtype"] == "f64":
        dgemm = measure_dgemm_peak(torch, dev)
        fp64 = tf / world / (trailing_ms * 1e-3) / 1e12 if trailing_ms > 0 else None
        out.update({"bound": "tensor", "kernel": "gemm_dmma_kernel (DMMA mma.sync.m8n8k4.f64, lower tiles)",
                    "achieved": fp64, "peak": dgemm, "unit": "TFLOP/s (fp64, per GPU)", "frac": (fp64 / dgemm) if fp64 else None,
                    "peak_source": "cuBLAS DGEMM 8192^3 measured in this run (MEASURED_PEAKS.json has no fp64 entry)"})
    else:
        fp32 = tf / world / (trailing_ms * 1e-3) / 1e12 if trailing_ms > 0 else None
        f32_mode = cfg0.fp32_mode if cfg0.fp32_mode >= 0 else (1 if n_pad >= 4096 else 0)
        if f32_mode == 1:  # the same int8-sliced tcgen05 kernel with 4 slices: 10 int8 MACs per fp32 MAC
            S32 = int(os.environ.get("AGP_OZAKI_S32", "4"))
            pairs = S32 * (S32 + 1) // 2
            achieved = fp32 * pairs if fp32 else None
            mma_peak = measure_int8_mma_peak(eng, torch, dev, 7)
            out.update({"bound": "tensor", "kernel": "umma_ozaki_syrk_v3_kernel<%d, ., ., ., float> (tcgen05.mma.kind::i8, fp32 operands in %d slices)" % (S32, S32),
                        "achieved": achieved, "peak": mma_peak, "unit": "TOP/s (int8 tensor, dense, per GPU)",
                        "frac": (achieved / mma_peak) if achieved else None,
                        "peak_source": "MEASURED in this run: the fp64 (7-slice) instance of the same kernel with operand traffic and epilogue off",
                        "frac_of_nominal_4500": (achieved / 4500.0) if achieved else None,
                        "fp32_equivalent_tflops_per_gpu": fp32, "slices": S32, "int8_macs_per_fp32_mac": pairs})
        else:
            ffma_peak = 148 * 128 * 2 * 1.965e9 / 1e12
            out.update({"bound": "fp32 FMA", "kernel": "gemm_simt_kernel (FFMA tiles)", "achieved": fp32, "peak": ffma_peak,
                        "unit": "TFLOP/s (fp32)", "frac": (fp32 / ffma_peak) if fp32 else None,
                        "peak_source": "nominal 148 SMs x 128 FFMA/clk x 2 x 1.965 GHz"})
    tr = ncu_traffic(wl if wl in ("C4", "C4h", "C2", "C3", "C5") else "C4")
    out["traffic"] = tr.get("dram_bytes_per_launch") if tr else None
    out["traffic_detail"] = tr
    if t_dev:
        chol_tf = (N ** 3 / 3.0) / (t_dev["cholesky"] * 1e-3) / 1e12
        out["cholesky_third_n3_tflops"] = chol_tf
    return out


def run_ours(args, wl, n_full):
    import torch
    import agp_b200 as ag

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    W = WORKLOADS[wl]
    if world == 1 and args.gpus > 1:
        print(json.dumps({"metric": METRIC[W["kind"]], "n_gpus": args.gpus,
                          "unavailable": "launch with torchrun --nproc-per-node N (one rank per GPU)"}))
        return
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        from agp_b200.dist import init_distributed_engine
        eng = init_distributed_engine()
        if W["kind"] == "fit_predict":
            if rank == 0:
                print(json.dumps({"metric": METRIC[W["kind"]], "n_gpus": world, "unavailable": "C3 does not shard (N = 16384): replicas only"}))
            return
    else:
        eng = ag.engine()
    prob = FitProblem(wl, n_full, eng, torch, dev)
    N, D = prob.N, prob.D
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    t_dev, wall_dev, launches = timed(prob, torch, flush, True, args.steps, args.warmup, dist)
    if args.dump_outputs and rank == 0:  # before the passes below reuse the problem's buffers
        dump_outputs(prob.outputs(), args.dump_outputs)
    if args.quick:  # development runs (schedule sweeps): device-resident timing only, no e2e / parity / roofline / CPU arm
        if rank == 0:
            sampler.stop()
            print(json.dumps({"quick": True, "n_gpus": world, "workload": wl, "value": t_dev["total"], "unit": "ms",
                              "phases_ms": t_dev, "result": float(prob.lp[0]), "steps": args.steps}))
        return
    t_e2e, wall_e2e, _ = timed(prob, torch, flush, False, args.steps, args.warmup, dist)
    clocks = sampler.stop() if rank == 0 else None
    lp_val = float(prob.lp[0])
    if dist is not None:
        lt = torch.tensor([float(launches)])
        dist.all_reduce(lt)
        launches = int(lt.item())

    parity = None
    try:
        parity = parity_check(wl, {"n": n_full}, eng, torch, dev, dist)
    except Exception as e:  # the parity probe must never take the bench line down
        parity = {"error": repr(e)[:200]}

    roofline = None
    if W["kind"] in ("fit", "fit_predict"):
        roofline = fit_roofline(wl, N, eng, torch, dev, prob, flush, args, world, dist, t_dev)
        if world > 1:
            roofline["whole_job_third_n3_tflops"] = roofline.pop("cholesky_third_n3_tflops", None)
    else:  # VFE: streamed TRSM + SYRK, 2 M^2 N algorithmic flops (reference formulation, SURVEY s8d)
        M = prob.M
        alg = 2.0 * M * M * N + 2.0 * M ** 3 / 3.0
        stream_ms = t_dev.get("predict", 0.0) or t_dev["total"]  # timings[6] = the streamed phase (max over ranks)
        cfg0 = eng.get_config()
        m_pad = (M + 127) // 128 * 128
        f32_mode = cfg0.fp32_mode if cfg0.fp32_mode >= 0 else 1
        tensor = (W["dtype"] == "f32" and f32_mode == 1 and m_pad >= 2048) or (W["dtype"] == "f64" and m_pad >= 8192)
        if tensor:
            S_ = int(os.environ.get("AGP_OZAKI_S32", "4")) if W["dtype"] == "f32" else cfg0.ozaki_slices
            pairs = S_ * (S_ + 1) // 2
            mma_peak = measure_int8_mma_peak(eng, torch, dev, 7)
            ach = 2.0 * M * M * N / world * pairs / (stream_ms * 1e-3) / 1e12  # executed int8 TOP/s per GPU (TRSM + SYRK = M^2 N MACs)
            roofline = {"bound": "tensor", "kernel": "umma_ozaki_syrk_v3_kernel (TRSM rank-512 updates + long-K SYRK accumulate, %d slices)" % S_,
                        "achieved": ach, "peak": mma_peak, "unit": "TOP/s (int8 tensor, dense, per GPU)", "frac": ach / mma_peak,
                        "peak_source": "MEASURED in this run: the 7-slice instance of the same kernel with operand traffic and epilogue off",
                        "frac_of_nominal_4500": ach / 4500.0, "alg_flops_per_step": alg, "kernel_ms_per_step": stream_ms,
                        "fp_equivalent_tflops_whole_job": alg / (t_dev["total"] * 1e-3) / 1e12, "traffic": None,
                        "note": "kernel_ms = the whole streamed phase (cross-Gram, scaling, TRSM, SYRK, reductions), so frac is a lower bound for the kernel"}
        else:
            ffma_peak = 148 * 128 * 2 * 1.965e9 / 1e12 * world
            ach = alg / (t_dev["total"] * 1e-3) / 1e12
            roofline = {"bound": "fp32 FMA", "kernel": "VFE stream on the tile GEMMs", "achieved": ach, "peak": ffma_peak,
                        "unit": "TFLOP/s (whole job)", "frac": ach / ffma_peak, "alg_flops_per_step": alg,
                        "peak_source": "nominal N_gpus x 148 SMs x 128 FMA/clk x 2 x 1.965 GHz", "traffic": None}
    if rank != 0:
        return
    cpu = cpu_baseline(wl, n_full)
    line = {"metric": METRIC[W["kind"]], "value": t_dev["total"], "unit": "ms", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_dev["total"], "higher_is_better": False,
            "scaling": "strong", "vs_baseline": None, "dtype": W["dtype"], "data": "synthetic",
            "config": {"workload": wl_string(wl, N, ", fused fit (1 Gram + 1 Cholesky)" if W["kind"] == "fit" else ""),
                       "l2": "256 MiB flush buffer written between timed iterations",
                       "timer": "CUDA events on the library stream" + (", max over ranks" if world > 1 else ""), "tile": 128,
                       "grid": "1x%d block-column-cyclic, NCCL panel broadcast" % world if world > 1 else "single GPU"},
            "phases_ms": t_dev, "wall_ms_per_step": wall_dev,
            "e2e": {"value": t_e2e["total"], "unit": "ms", "h2d_bytes_per_step": int(prob.h2d * world),
                    "d2h_bytes_per_step": int(prob.d2h * world), "wall_ms_per_step": wall_e2e, "phases_ms": t_e2e},
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks, "parity": parity,
            "result": lp_val}
    if W["kind"] == "fit":
        line["third_n3_tflops"] = (N ** 3 / 3.0) / (t_dev["total"] * 1e-3) / 1e12
    if wl == "C4" and world == 1 and not args.no_c2:
        line["c2"] = secondary_c2(eng, torch, dev, flush, args)
    print(json.dumps(line))


def secondary_c2(eng, torch, dev, flush, args):
    """BASELINE config C2 (N = 4096, D = 8): latency-bound single-GPU case, carried next to the C4 headline"""
    p = FitProblem("C2", None, eng, torch, dev)
    steps = min(args.steps, 20)
    t_dev, _, launches = timed(p, torch, flush, True, steps, 3)
    t_e2e, _, _ = timed(p, torch, flush, False, steps, 3)
    par = None
    try:
        par = parity_check("C2", {"n": 4096}, eng, torch, dev)
    except Exception as e:
        par = {"error": repr(e)[:200]}
    return {"workload": wl_string("C2", 4096), "value": t_dev["total"], "unit": "ms", "e2e": t_e2e["total"], "steps": steps,
            "phases_ms": t_dev, "gpu_launches_per_step": launches / steps, "parity": par,
            "third_n3_tflops": (4096 ** 3 / 3.0) / (t_dev["total"] * 1e-3) / 1e12, "cpu_baseline": cpu_baseline("C2", 4096)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C4", choices=sorted(WORKLOADS))
    ap.add_argument("--n", type=int, default=None, help="override N of the workload (development / shard-sized runs)")
    ap.add_argument("--no-c2", action="store_true", help="skip the secondary C2 measurement on the N=1 C4 line")
    ap.add_argument("--quick", action="store_true", help="development: device-resident timing only (not a bench line)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last device-resident timed step returned as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "ours":
        args.warmup = max(args.warmup, 3)
    wl = args.workload
    n_full = args.n or WORKLOADS[wl]["N"]
    if args.impl == "reference":
        run_reference(args, wl, n_full)
    else:
        run_ours(args, wl, n_full)


if __name__ == "__main__":
    main()
