#!/usr/bin/env python
"""Benchmark of the windowed least-squares spectral estimation hot path (BASELINE.json configs[1]).

workload "cfg2_windowpsd": ls_windowpsd on 2^22 irregular samples, nw=1024 (n=4096, noverlap=2048, K=2047
windows), hanning window, 256 frequencies per window.  One *step* = one full pass over all K windows of one
2^22-sample record.  Multi-GPU: windows shard with no data-path collective -- every rank owns one 2^22-sample
segment (weak scaling, per-GPU work fixed) and only the Nf-long accumulators are all-reduced once per step.

  python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--workload cfg2_windowpsd|cfg3_admm]

Prints ONE JSON line (rank 0).  `value` = windows/s with inputs resident in HBM; `e2e` = the same metric through
the public host-buffer API (H2D of y,t and D2H of the spectrum inside the timed region); `roofline` = the Gram
kernel's FP64 tensor-pipe fraction measured live with CUDA events on the library's stream; `cpu_baseline` = the
oracle's reference-literal algorithm on the host cores for a bounded sample of the same windows.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NSAMP = 1 << 22
NW = 1024
NF = 256
LAMBDA = 1e-10
FP64_PEAK_FILE = os.path.join(ROOT, "profiles", "fp64_peak_r01.json")


def cfg2_config(n):
    """`config` of the JSON line -- identical in the GPU arm and the reference arm (the driver compares them)."""
    return {"workload": "cfg2_windowpsd", "samples_per_gpu": NSAMP, "nw": NW, "n": n, "noverlap": n >> 1,
            "windows_per_gpu": 2 * NW - 1, "freqs": NF, "nreg": 2 * NF - 1, "window": "hanning",
            "l2": "inputs+Gram workspace (4.3 GB/step) larger than L2, no flush needed"}


def make_cfg2(seed=2, nsamp=NSAMP, nw=NW, nf=NF):
    """SURVEY 8(d) cfg2: t=sort(10*U^N), two tones at f[40], f[100] + 0.1 noise, f=(0:nf-1)*2fs/n."""
    rng = np.random.default_rng(seed)
    t = np.sort(10.0 * rng.random(nsamp))
    n = nsamp // nw
    fs = 1.0 / np.mean(np.diff(t))
    f = np.arange(nf, dtype=np.float64) * (2.0 * fs / n)
    y = np.sin(2 * np.pi * f[40] * t) + 0.5 * np.cos(2 * np.pi * f[100] * t + 1.0) + 0.1 * rng.standard_normal(nsamp)
    return t, y, f, n


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        top = sorted(sm)[len(sm) // 2:]  # under-load half
        return {"sm_mhz": statistics.median(top), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


def ncu_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/r02_traffic.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as fh:
            return float(json.load(fh)[kernel]["dram_bytes_per_launch"])
    except Exception:
        return None


def fp64_peak():
    try:
        with open(FP64_PEAK_FILE) as fh:
            d = json.load(fh)
        return float(d["dmma_tflops"]), "profiles/fp64_peak_r01.json (tools/fp64_probe.cu, DMMA.8x8x4 issue peak measured on this pool's B200; MEASURED_PEAKS.json has no FP64 line; cuBLAS DGEMM 8192^3 = %.2f)" % d["dgemm_tflops"]
    except Exception:
        return 37.0, "nominal 37 TFLOP/s (fallback: profiles/fp64_peak_r01.json missing)"


def cpu_baseline_windows(t, y, f, n, nwin, threads=None, mode="literal"):
    """CPU algorithm (oracle) on `nwin` windows of the workload; returns windows/s.  mode="literal" is what the
    reference executes (basis + N-rhs LU per window); mode="gram" is the stronger CPU line SURVEY 8(d) asks for (the
    algorithm the GPU runs -- Gram + Cholesky -- on the host BLAS)."""
    from oracle import lpvs_oracle as o

    W = o.hanning(n)
    hop = n - (n >> 1)
    t0 = time.perf_counter()
    S = np.zeros(len(f))
    for k in range(nwin):
        sl = slice(k * hop, k * hop + n)
        x, _ = o.ls_spectral(y[sl], t[sl], f, W, lam=LAMBDA, mode=mode)
        S += x.real ** 2 + x.imag ** 2
    dt = time.perf_counter() - t0
    return nwin / dt, dt


def blas_threads():
    """Threads the BLAS behind numpy/scipy uses for the CPU arm (north_star: core count AND BLAS thread count)."""
    try:
        from threadpoolctl import threadpool_info

        n = [int(p.get("num_threads", 0)) for p in threadpool_info() if p.get("user_api") == "blas"]
        return max(n) if n else None
    except Exception:
        return None


def make_cfg3(seed=3, N=16384):
    """SURVEY 8(d) cfg3: t=sort(10*U^16384), f=default_freqs(t)[:8192], 5 tones + 0.1 noise."""
    rng = np.random.default_rng(seed)
    t = np.sort(10.0 * rng.random(N))
    fs = 1.0 / np.mean(np.diff(t))
    f = (np.arange(N // 2 + 1) * (fs / N))[: N // 2]
    tones = f[[300, 1200, 2500, 4000, 6000]]
    y = sum(np.sin(2 * np.pi * ft * t + i) for i, ft in enumerate(tones)) + 0.1 * rng.standard_normal(N)
    return t, y, f


def admm_leg(ctx, lp, L, C, rank, world, allsum, allmax, barrier, iters=2000):
    """BASELINE.json configs[2]: ls_sparse_spectral L1 ADMM, N=16384, 8192 freqs (Nreg=16383), lambda=0.1, mu=0.05.
    Fixed iteration count (tol=0) for the throughput figure; every rank runs its own replica (the loop does not
    shard, DESIGN.md section 5), value = sum of per-rank iterations/s."""
    t, y, f = make_cfg3(seed=3 + rank)
    h = C.c_void_p()
    t0 = time.perf_counter()
    ctx.check(ctx.lib.lpvs_admm_create_fourier(ctx.h, y.ctypes.data_as(C.c_void_p), t.ctypes.data_as(C.c_void_p),
                                               len(y), f.ctypes.data_as(C.c_void_p), len(f), None, L.PROX_L1, 0.1,
                                               0.05, None, 0, 0.0, C.byref(h)))
    setup_s = time.perf_counter() - t0
    gms, gl, gfl = ctx.gram_timing()
    solver = lp.ADMM(ctx, h)
    solver.step(100, 0.0)
    barrier()
    solver.step(iters, 0.0)
    ms, bpi = solver.timing()
    barrier()
    solver.free()
    its = iters / (ms * 1e-3)
    its_min = -allmax(-its)
    total = allsum(its)
    # the Float32 instantiation (SURVEY 8f n2): the same problem with the inverse stored in single precision
    f32 = None
    if rank == 0:
        try:
            ctx.set_option(L.OPT_ADMM_M32, 1)
            h32 = C.c_void_p()
            ctx.check(ctx.lib.lpvs_admm_create_fourier(ctx.h, y.ctypes.data_as(C.c_void_p), t.ctypes.data_as(C.c_void_p),
                                                       len(y), f.ctypes.data_as(C.c_void_p), len(f), None, L.PROX_L1, 0.1,
                                                       0.05, None, 0, 0.0, C.byref(h32)))
            ctx.set_option(L.OPT_ADMM_M32, 0)
            s32 = lp.ADMM(ctx, h32)
            s32.step(100, 0.0)
            s32.step(iters, 0.0)
            ms32, bpi32 = s32.timing()
            s32.free()
            f32 = {"iters_per_s": iters / (ms32 * 1e-3), "bytes_per_iter": bpi32,
                   "hbm_gbs": bpi32 * iters / (ms32 * 1e-3) / 1e9,
                   "note": "LPVS_OPT_ADMM_M32: (G+I/mu)^-1 stored in single precision, double accumulation -- what Float32 "
                           "callers of ls_sparse_spectral get"}
        except Exception as e:
            f32 = {"error": repr(e)[:200]}
        finally:
            ctx.set_option(L.OPT_ADMM_M32, 0)
    hbm = 6554.6
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            hbm = float(json.load(fh)["hbm_gbs"])
    except Exception:
        pass
    sharded = None
    if world > 1 and world <= 8:
        # the same problem (rank 0's data on every rank) as ONE problem over all GPUs: device-initiated peer stores over
        # NVLink inside the persistent loop (lpvs_admm_shard_*, DESIGN.md section 5 iii)
        try:
            from lpvspectral_jl_b200 import _dist as D

            t0s, y0s, f0s = make_cfg3(seed=3)
            hs = C.c_void_p()
            rc = ctx.lib.lpvs_admm_create_fourier(ctx.h, y0s.ctypes.data_as(C.c_void_p),
                                                  t0s.ctypes.data_as(C.c_void_p), len(y0s),
                                                  f0s.ctypes.data_as(C.c_void_p), len(f0s), None, L.PROX_L1, 0.1, 0.05,
                                                  None, 0, 0.0, C.byref(hs))
            if allmax(1.0 if rc else 0.0) > 0:  # all ranks agree before any collective of the sharded leg
                if not rc:
                    ctx.lib.lpvs_admm_free(hs)
                raise RuntimeError("sharded ADMM: problem creation failed on some rank")
            ss = D.admm_shard(lp.ADMM(ctx, hs))
            ss.step(100, 0.0)
            barrier()
            ss.step(iters, 0.0)
            ms_s, _ = ss.timing()
            barrier()
            ss.free()
            ms_max = allmax(ms_s)
            sharded = {"iters_per_s": iters / (ms_max * 1e-3), "us_per_iter": ms_max / iters * 1e3,
                       "vs_one_gpu": (iters / (ms_max * 1e-3)) / its_min,
                       "how": "one problem over all GPUs: ONE all-reduce of the partial products per iteration by peer stores "
                              "over NVLink inside the persistent kernel (prox computed redundantly on every rank), max over "
                              "ranks of the device time"}
        except Exception as e:  # never lose the headline line to the optional leg
            sharded = {"error": repr(e)[:200]}
    return {"workload": "cfg3_l1_admm", "nreg": 2 * len(f) - 1, "iters": iters, "iters_per_s": total,
            "iters_per_s_per_gpu_min": its_min, "scaling": "replicas (weak); `sharded` = one problem (strong)",
            "sharded": sharded, "float32_storage": f32, "setup_s": setup_s,
            "gram_tflops": gfl / gms / 1e9,
            "roofline": {"bound": "hbm", "achieved": bpi * its_min / 1e9, "peak": hbm, "unit": "GB/s",
                         "frac": bpi * its_min / 1e9 / hbm, "traffic": ncu_traffic("k_admm_symv"),
                         "traffic_unit": "bytes per iteration (one launch = many iterations)", "kernel": "k_admm_symv",
                         "bytes_per_iter": bpi,
                         "note": "algorithmic bytes = lower-triangle 128x128 blocks of (G+I/mu)^-1 actually streamed"}}


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"])
    except Exception:
        return 6554.6


def fp64_peak_live(torch):
    """cuBLAS DGEMM 8192^3 through torch.matmul, best of 5 after 2 warm-ups, CUDA events -- the method MEASURED_PEAKS.json
    uses for bf16, repeated for FP64 inside this run so the denominator sits under the same clock record."""
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    best = float("inf")
    for i in range(7):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        c = torch.matmul(a, b)
        e1.record()
        e1.synchronize()
        if i >= 2:
            best = min(best, e0.elapsed_time(e1))
    del a, b, c
    torch.cuda.empty_cache()
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def make_cfg1():
    """SURVEY 8(d) cfg1 = BASELINE configs[0]: N=4096 irregular samples, default_freqs(t)[:2048], no weights, lambda=1e-10."""
    rng = np.random.default_rng(1)
    N = 4096
    t = np.sort(10 * rng.random(N))
    y = np.sin(2 * np.pi * 20 * t) + 0.5 * np.cos(2 * np.pi * 55 * t + 1) + 0.1 * rng.standard_normal(N)
    f = (np.arange(N // 2 + 1) * (1.0 / np.mean(np.diff(t)) / N))[:2048]
    return t, y, f


def make_cfg5(nsamp=1 << 24, seed=5):
    """SURVEY 8(d) cfg5 = BASELINE configs[4]: two channels of 2^24 irregular samples, n=4096, 512 freqs at spacing 2 fs / n."""
    rng = np.random.default_rng(seed)
    n = 4096
    t = np.sort(10 * rng.random(nsamp))
    fs = 1.0 / np.mean(np.diff(t))
    f = np.arange(512) * 2 * fs / n
    y = np.sin(2 * np.pi * f[40] * t) + 0.5 * np.cos(2 * np.pi * f[100] * t + 1) + 0.1 * rng.standard_normal(nsamp)
    u = 0.7 * np.roll(y, 5) + 0.5 * rng.standard_normal(nsamp)
    return t, y, u, f, n


def cfg1_leg(ctx, lp, peak):
    """ms per spectrum of BASELINE configs[0] through the host-buffer API (H2D/D2H inside), rank 0 only."""
    t, y, f = make_cfg1()
    best, info, gms, gfl = float("inf"), 0, 0.0, 0.0
    for rep in range(6):
        x, _, info = lp.ls_spectral(y, t, f, ctx=ctx, return_info=True)
        ms = ctx.last_call_ms()
        if rep >= 1 and ms < best:
            best = ms
            gms, _, gfl = ctx.gram_timing()
    nreg, N = 2 * len(f) - 1, len(y)
    flop = N * nreg * (nreg + 1.0) + nreg ** 3 / 3.0 + 2.0 * nreg ** 2  # SURVEY 8(d): Gram + Cholesky + 2 TRSV
    np_ = (len(f) + 63) // 64 * 128
    nr = (N + 127) // 128 * 128
    # the QR-class path (csrc/lsq.cu) really executes: + TRTRI + triangular GEMM + SYRK of Q1 + second Cholesky
    flop_qr = flop + np_ ** 3 / 3.0 + float(nr) * np_ * np_ + (nr + np_ / 2.0) * np_ * (np_ + 1.0) + np_ ** 3 / 3.0
    a = x.real ** 2 + x.imag ** 2
    return {"workload": "cfg1_ls_spectral", "N": N, "freqs": len(f), "nreg": nreg, "lambda": 1e-10,
            "ms_per_spectrum": best, "spectra_per_s": 1e3 / best, "info": int(info),
            "path": "shifted CholeskyQR on the materialised regressor (cond(A)~1e16: the reference's SVD answer, "
                    "tests/test_gpu_rankdef.py)" if info == 2 else "Cholesky + refinement on the synthesised operator",
            "gram_ms": gms, "gram_tflops": gfl / gms / 1e9 if gms else None,
            "roofline": {"bound": "tensor", "unit": "TFLOP/s", "peak": peak,
                         "achieved_survey_flops": flop / best / 1e9, "frac_survey_flops": flop / best / 1e9 / peak,
                         "achieved_executed_flops": (flop_qr if info == 2 else flop) / best / 1e9,
                         "frac_executed_flops": (flop_qr if info == 2 else flop) / best / 1e9 / peak,
                         "flop_survey": flop, "flop_executed": flop_qr if info == 2 else flop},
            "peak_index": int(a.argmax())}


def cfg4_leg(ctx, lp, L, C, iters=2000):
    """BASELINE configs[3]: ls_sparse_spectral_lpv group lasso, N=20000, 64 freqs x Nv=50 (n=6400), lambda=0.1; rank 0 only."""
    from oracle import lpvs_oracle as o

    Y, V, X = o.generate_lpv_signal(20000, seed=4)
    w = 2 * np.pi * np.arange(1, 65) * 0.4
    h = C.c_void_p()
    t0 = time.perf_counter()
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    ctx.check(ctx.lib.lpvs_admm_create_lpv(ctx.h, vp(Y), vp(X), vp(V), len(Y), vp(w), len(w), 50, 0, 1, 0.1, 0.05,
                                           C.byref(h)))
    setup_s = time.perf_counter() - t0
    gms, _, gfl = ctx.gram_timing()
    solver = lp.ADMM(ctx, h)
    solver.step(200, 0.0)
    solver.step(iters, 0.0)
    ms, bpi = solver.timing()
    solver.free()
    its = iters / (ms * 1e-3)
    hbm = hbm_peak()
    return {"workload": "cfg4_group_lasso_lpv", "N": 20000, "freqs": 64, "Nv": 50, "n": 6400, "iters": iters,
            "iters_per_s": its, "us_per_iter": ms / iters * 1e3, "setup_s": setup_s, "gram_tflops": gfl / gms / 1e9,
            "roofline": {"bound": "hbm", "achieved": bpi * its / 1e9, "peak": hbm, "unit": "GB/s",
                         "frac": bpi * its / 1e9 / hbm, "bytes_per_iter": bpi,
                         "note": "algorithmic bytes; the inverse (164 MB lower triangle) is partly L2-resident, so DRAM "
                                 "traffic is lower (profiles/r01c_summary.md)"}}


def cfg4_sharded_leg(ctx, lp, L, C, D, dist, world, allmax, barrier, one_gpu_its, iters=2000):
    """BASELINE configs[3] as ONE problem over the run's N GPUs (exchange 2: all-reduce of the partial products by peer stores,
    group prox computed redundantly on every rank).  Every rank creates the same problem."""
    from oracle import lpvs_oracle as o

    Y, V, X = o.generate_lpv_signal(20000, seed=4)
    w = 2 * np.pi * np.arange(1, 65) * 0.4
    h = C.c_void_p()
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    rc = ctx.lib.lpvs_admm_create_lpv(ctx.h, vp(Y), vp(X), vp(V), len(Y), vp(w), len(w), 50, 0, 1, 0.1, 0.05, C.byref(h))
    if allmax(1.0 if rc else 0.0) > 0:
        if not rc:
            ctx.lib.lpvs_admm_free(h)
        return {"error": "problem creation failed on some rank"}
    ss = D.admm_shard(lp.ADMM(ctx, h))
    ss.step(200, 0.0)
    barrier()
    ss.step(iters, 0.0)
    ms, _ = ss.timing()
    barrier()
    ss.free()
    ms = allmax(ms)
    its = iters / (ms * 1e-3)
    return {"workload": "cfg4_group_lasso_lpv", "n_gpus": world, "iters_per_s": its, "us_per_iter": ms / iters * 1e3,
            "vs_one_gpu": its / one_gpu_its if one_gpu_its else None,
            "how": "one problem over all GPUs: one all-reduce of the partial products per iteration by peer stores over NVLink "
                   "inside the persistent kernel, whole groups per CTA; max over ranks of the device time"}


def cfg5_legs(ctx, lp, L, C, D, torch, dist, rank, world, local, allmax, barrier, peak):
    """BASELINE configs[4] on the run's N GPUs, both forms (SURVEY 8e):
    5a  ls_cohere over K=8191 windows, windows sharded over the ranks (no data-path collective), host buffers;
    5b  the same record as ONE weighted two-channel problem: row-sharded Gram, ONE NCCL all-reduce of the packed Gram
        (timed on its own with CUDA events), then the factorisation on every rank."""
    t, y, u, f, n = make_cfg5()
    NS, Nf = len(t), len(f)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    W = lp.hanning(n)
    hop = n >> 1
    K = lp.window_count(NS, n, hop)
    k0, k1 = D.shard_range(K, rank, world)
    sums = np.zeros(4 * Nf)
    info = C.c_int(0)
    acc = torch.zeros(4 * Nf, dtype=torch.float64, device="cuda")
    out = {}
    best = float("inf")
    gram_ms = gram_fl = 0.0
    for rep in range(3):
        barrier()
        w0 = time.perf_counter()
        ctx.check(ctx.lib.lpvs_ls_window_sums(ctx.h, L.WIN_COHERE, vp(y), vp(u), vp(t), NS, vp(f), Nf, vp(W), n, hop,
                                              LAMBDA, k0, k1, vp(sums), C.byref(info)))
        acc.copy_(torch.from_numpy(sums))
        if world > 1:
            dist.all_reduce(acc)
        coh = lp.window_finalize(L.WIN_COHERE, acc.cpu().numpy(), Nf, K)
        dt = allmax(time.perf_counter() - w0)
        if rep >= 1 and dt < best:
            best = dt
            gram_ms, _, gram_fl = ctx.gram_timing()
    nreg = 2 * Nf - 1
    out["cfg5a"] = {"workload": "cfg5a_ls_cohere", "samples_per_channel": NS, "windows": K, "freqs": Nf, "nreg": nreg,
                    "sharding": "windows [K r/P, K (r+1)/P) per rank, one all-reduce of 4 Nf doubles", "n_gpus": world,
                    "s_per_pass": best, "windows_per_s": K / best,
                    "api": "lpvs_ls_window_sums (host pointers; H2D of this rank's sample range inside)",
                    "gram_tflops_per_gpu": gram_fl / gram_ms / 1e9 if gram_ms else None,
                    "gram_frac": gram_fl / gram_ms / 1e9 / peak if gram_ms else None,
                    "coherence_in_unit_interval": bool(np.all((coh >= 0) & (coh <= 1 + 1e-12)))}
    # the same pass in the opt-in LPVS_PHASE_STRUCTURED_REF mode (Gram matrices from trigonometric sums + half-precision
    # tensor-core correction for the reference's phase rounding): cfg5a's phases (2.6e7 rad) are where that rounding matters
    try:
        coh_default = coh.copy()
        ctx.set_option(L.OPT_PHASE_MODE, L.PHASE_STRUCTURED_REF)
        best_r = float("inf")
        for rep in range(2):
            barrier()
            w0 = time.perf_counter()
            ctx.check(ctx.lib.lpvs_ls_window_sums(ctx.h, L.WIN_COHERE, vp(y), vp(u), vp(t), NS, vp(f), Nf, vp(W), n, hop,
                                                  LAMBDA, k0, k1, vp(sums), C.byref(info)))
            acc.copy_(torch.from_numpy(sums))
            if world > 1:
                dist.all_reduce(acc)
            coh_r = lp.window_finalize(L.WIN_COHERE, acc.cpu().numpy(), Nf, K)
            best_r = min(best_r, allmax(time.perf_counter() - w0))
        out["cfg5a"]["structured_ref_mode"] = {
            "s_per_pass": best_r, "windows_per_s": K / best_r,
            "coherence_rel_l2_vs_default_mode": float(np.linalg.norm(coh_r - coh_default) / np.linalg.norm(coh_default)),
            "coherence_max_abs_diff_vs_default_mode": float(np.abs(coh_r - coh_default).max()),
            "note": "opt-in; the cross-window sums are dominated by a few ill-conditioned windows (cond(A'WA) up to 4.5e7, "
                    "DESIGN.md 1), where both modes carry cond x eps"}
    except Exception as e:  # never lose the line to an extra leg
        out["cfg5a"]["structured_ref_mode"] = {"error": repr(e)[:300]}
    finally:
        ctx.set_option(L.OPT_PHASE_MODE, L.PHASE_AUTO)
    # ---- 5b: row-sharded ----
    Wn = lp.hanning(NS)
    r0, r1 = D.shard_range(NS, rank, world)
    d_t = torch.from_numpy(t[r0:r1]).cuda()
    d_y = torch.from_numpy(y[r0:r1]).cuda()
    d_u = torch.from_numpy(u[r0:r1]).cuda()
    d_W = torch.from_numpy(Wn[r0:r1]).cuda()
    npk = int(ctx.lib.lpvs_packed_size(Nf))
    packed = torch.empty(npk, dtype=torch.float64, device="cuda")
    x = np.empty((2, Nf), dtype=np.complex128)
    p = lambda a: C.c_void_p(a.data_ptr())  # noqa: E731
    res = None
    for rep in range(3):
        barrier()
        w0 = time.perf_counter()
        ctx.check(ctx.lib.lpvs_gram_partial_dev(ctx.h, p(d_y), p(d_u), p(d_t), p(d_W), r1 - r0, vp(f), Nf, p(packed)))
        g_ms = ctx.last_call_ms()
        gk_ms, _, gk_fl = ctx.gram_timing()
        ar_ms = 0.0
        if world > 1:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dist.all_reduce(packed)
            e1.record()
            e1.synchronize()
            ar_ms = e0.elapsed_time(e1)
        ctx.check(ctx.lib.lpvs_solve_packed_dev(ctx.h, p(packed), vp(f), Nf, 2, LAMBDA, vp(x), C.byref(info)))
        s_ms = ctx.last_call_ms()
        wall = allmax(time.perf_counter() - w0)
        cur = dict(wall_s=wall, gram_call_ms=allmax(g_ms), gram_kernel_ms=allmax(gk_ms), allreduce_ms=allmax(ar_ms),
                   solve_ms=allmax(s_ms), flops_rank=gk_fl)
        if rep >= 1 and (res is None or cur["wall_s"] < res["wall_s"]):
            res = cur
    flops = float(NS) * nreg * (nreg + 1.0)
    nbytes = npk * 8
    busbw = (2.0 * (world - 1) / world) * nbytes / (res["allreduce_ms"] * 1e-3) / 1e9 if world > 1 else None
    out["cfg5b_rowsharded"] = {
        "workload": "cfg5b_one_weighted_problem", "rows": NS, "freqs": Nf, "nreg": nreg, "channels": 2, "n_gpus": world,
        "rows_per_gpu": r1 - r0, "ms_total_resident": res["wall_s"] * 1e3, "gram_ms": res["gram_call_ms"],
        "gram_kernel_ms": res["gram_kernel_ms"], "solve_ms": res["solve_ms"],
        "gram_tflops_aggregate": flops / (res["gram_call_ms"] * 1e-3) / 1e12,
        "gram_kernel_frac_per_gpu": res["flops_rank"] / (res["gram_kernel_ms"] * 1e-3) / 1e12 / peak,
        "allreduce": {"bytes": nbytes, "us": res["allreduce_ms"] * 1e3 if world > 1 else None, "busbw_gbs": busbw,
                      "busbw_peak_gbs": 725.0, "frac": busbw / 725.0 if busbw else None,
                      "how": "torch.distributed all_reduce (NCCL, NVLink/NVSwitch) of the packed lower-tile Gram + 2 rhs, "
                             "CUDA events on the launching stream, max over ranks; busbw = 2(P-1)/P bytes/time against the "
                             "725 GB/s measured 8-GPU bus bandwidth"},
        "peak_power_yy": float((x[0].real ** 2 + x[0].imag ** 2).max())}
    # the same problem with the Gram matrix from its trigonometric sums (opt-in LPVS_PHASE_STRUCTURED, exact-phase class) and
    # with the first-order correction to the reference's phase rounding on top (LPVS_PHASE_STRUCTURED_REF: per-sample tables
    # built segment by segment, half-precision tensor-core GEMM over sample splits)
    for key, mode, note in (
            ("structured_mode", L.PHASE_STRUCTURED,
             "opt-in LPVS_PHASE_STRUCTURED: 3 Nf sums over the rows instead of the DMMA Gram; the difference to the default "
             "mode is the reference's phase rounding at phases up to 2.6e7 rad (DESIGN.md 1b / 3a)"),
            ("structured_ref_mode", L.PHASE_STRUCTURED_REF,
             "opt-in LPVS_PHASE_STRUCTURED_REF: the sums + the first-order phase-rounding correction (DESIGN.md 3b): the "
             "default mode's class")):
        try:
            ctx.set_option(L.OPT_PHASE_MODE, mode)
            xs = np.empty((2, Nf), dtype=np.complex128)
            best_s = None
            for rep in range(2):
                barrier()
                w0 = time.perf_counter()
                ctx.check(ctx.lib.lpvs_gram_partial_dev(ctx.h, p(d_y), p(d_u), p(d_t), p(d_W), r1 - r0, vp(f), Nf, p(packed)))
                g_ms = ctx.last_call_ms()
                if world > 1:
                    dist.all_reduce(packed)
                    torch.cuda.synchronize()
                ctx.check(ctx.lib.lpvs_solve_packed_dev(ctx.h, p(packed), vp(f), Nf, 2, LAMBDA, vp(xs), C.byref(info)))
                wall = allmax(time.perf_counter() - w0)
                if best_s is None or wall < best_s[0]:
                    best_s = (wall, allmax(g_ms))
            out["cfg5b_rowsharded"][key] = {
                "ms_total_resident": best_s[0] * 1e3, "gram_ms": best_s[1],
                "rel_l2_vs_default_mode": float(np.linalg.norm(xs - x) / np.linalg.norm(x)), "note": note}
        except Exception as e:  # never lose the headline line to an extra leg
            out["cfg5b_rowsharded"][key] = {"error": repr(e)[:300]}
        finally:
            ctx.set_option(L.OPT_PHASE_MODE, L.PHASE_AUTO)
    del d_t, d_y, d_u, d_W, packed
    torch.cuda.empty_cache()
    return out


def strong_leg(ctx, lp, L, C, D, torch, dist, rank, world, allmax, barrier, one_gpu_ms, steps):
    """BASELINE configs[1] as named: ONE 2^22-sample record, its K=2047 windows split over the ranks, inputs resident."""
    t, y, f, n = make_cfg2()
    K = lp.window_count(len(y), n, -1)
    k0, k1 = D.shard_range(K, rank, world)
    hop = n >> 1
    s0, s1 = k0 * hop, (k1 - 1) * hop + n
    d_t = torch.from_numpy(t[s0:s1]).cuda()
    d_y = torch.from_numpy(y[s0:s1]).cuda()
    W = lp.hanning(n)
    sums = np.zeros(len(f))
    acc = torch.zeros(len(f), dtype=torch.float64, device="cuda")
    info = C.c_int(0)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731

    def step():
        ctx.check(ctx.lib.lpvs_ls_window_sums_dev(ctx.h, L.WIN_PSD, C.c_void_p(d_y.data_ptr()), None,
                                                  C.c_void_p(d_t.data_ptr()), s1 - s0, vp(f), len(f), vp(W), n, hop,
                                                  LAMBDA, 0, k1 - k0, vp(sums), C.byref(info)))
        acc.copy_(torch.from_numpy(sums))
        dist.all_reduce(acc)

    for _ in range(3):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    wall = time.perf_counter() - w0
    ms = allmax(max(e0.elapsed_time(e1), wall * 1e3)) / steps
    S = lp.window_finalize(L.WIN_PSD, acc.cpu().numpy(), len(f), K)
    return {"workload": "cfg2_windowpsd", "scaling": "strong", "n_gpus": world, "windows": K, "ms_per_pass": ms,
            "windows_per_s": K / ms * 1e3, "one_gpu_ms_per_pass": one_gpu_ms, "speedup_vs_one_gpu": one_gpu_ms / ms,
            "peaks": np.argsort(-S)[:2].tolist(),
            "how": "one record, windows [K r/P, K (r+1)/P) per rank, one all-reduce of Nf doubles per pass; max over ranks "
                   "of CUDA-event / wall time; the one-GPU figure is rank 0's resident step on the same record in this run"}


def parity_leg(ctx, lp, L, C, D, torch, dist, rank, world, local, allmax):
    """Sharded paths against this rank's own single-GPU result (what tools/dist_check.py and tools/admm_shard_check.py
    check), once, outside every timed region.  Returns relative errors (max over ranks)."""
    rng = np.random.default_rng(0)
    N = 1 << 18
    t = np.sort(10 * rng.random(N))
    y = np.sin(2 * np.pi * 300 * t) + 0.3 * rng.standard_normal(N)
    u = 0.7 * np.roll(y, 2) + 0.5 * rng.standard_normal(N)
    n = 2048
    f = np.arange(64) * 2.0 / (t[n] - t[0])
    W = lp.hanning(n)
    dev = torch.device("cuda", local)
    rel = lambda a, b: float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))  # noqa: E731
    res, _ = D.ls_window_sharded(L.WIN_PSD, y, None, t, f, n=n, W=W, lam=LAMBDA, ctx=ctx, reduce_device=dev)
    ref, _ = lp.ls_windowpsd(y, t, f, nw=N // n, window_func=lp.hanning, ctx=ctx)
    e_win = rel(res, ref)
    res, _ = D.ls_window_sharded(L.WIN_COHERE, y, u, t, f, n=n, W=W, lam=LAMBDA, ctx=ctx, reduce_device=dev)
    ref, _ = lp.ls_cohere(y, u, t, f, nw=N // n, ctx=ctx)
    e_win = max(e_win, rel(res, ref))
    f2 = np.arange(128) * 40.0
    Wn = 0.5 + rng.random(N)
    xs = D.ls_spectral_rowsharded(y, t, f2, Wn, u=u, lam=LAMBDA, ctx=ctx)
    x1, _ = lp.ls_spectral(y, t, f2, Wn, ctx=ctx)
    e_row = rel(xs[0], x1)
    # ADMM: ONE 4095-unknown L1 problem sharded over the ranks vs the same problem on this GPU alone
    rng = np.random.default_rng(3)
    Na = 4096
    ta = np.sort(10 * rng.random(Na))
    fa = (np.arange(Na // 2 + 1) * (1.0 / np.mean(np.diff(ta)) / Na))[:2048]
    ya = sum(np.cos(2 * np.pi * fa[k] * ta + k) for k in (100, 500, 900)) + 0.1 * rng.standard_normal(Na)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731

    def create(prox=None, pparam=0.1):
        h = C.c_void_p()
        ctx.check(ctx.lib.lpvs_admm_create_fourier(ctx.h, vp(ya), vp(ta), Na, vp(fa), len(fa), None,
                                                   L.PROX_L1 if prox is None else prox, pparam, 0.05, None, 0, 0.0,
                                                   C.byref(h)))
        return lp.ADMM(ctx, h)

    def one_vs_sharded(make, iters, tol):
        one = make()
        one.step(iters, tol)
        x1, z1 = one.get()
        it1 = one.iters
        one.free()
        sh = D.admm_shard(make())
        sh.step(iters, tol)
        dist.barrier()
        xs_, zs_ = sh.get()
        its = sh.iters
        dist.barrier()
        sh.free()
        return max(rel(zs_, z1), rel(xs_, x1)), bool(np.array_equal(zs_ != 0, z1 != 0)) and its == it1

    e_admm, same = one_vs_sharded(create, 600, 1e-9)
    # IndBallL0 (keep the 24 largest): the selection runs redundantly on every rank after the all-reduce
    e_ball, same_ball = one_vs_sharded(lambda: create(L.PROX_BALL_L0, 24.0), 300, 1e-9)
    same = same and same_ball
    # group lasso (ls_sparse_spectral_lpv): ONE 1280-unknown problem (10 blocks of 128 >= 8 ranks) sharded vs this GPU alone
    from oracle import lpvs_oracle as o

    Yg, Vg, Xg = o.generate_lpv_signal(4000, seed=4)
    wg = 2 * np.pi * np.arange(1, 33) * 0.4

    def create_lpv():
        h = C.c_void_p()
        ctx.check(ctx.lib.lpvs_admm_create_lpv(ctx.h, vp(Yg), vp(Xg), vp(Vg), len(Yg), vp(wg), len(wg), 20, 0, 1, 0.1, 0.05,
                                               C.byref(h)))
        return lp.ADMM(ctx, h)

    e_group, same_group = one_vs_sharded(create_lpv, 400, 1e-7)
    same = same and same_group
    out = {"window_sharded": allmax(e_win), "row_sharded": allmax(e_row), "admm_sharded": allmax(e_admm),
           "admm_group_sharded": allmax(e_group), "admm_ball_l0_sharded": allmax(e_ball),
           "admm_same_support_and_iterations": allmax(0.0 if same else 1.0) == 0.0, "bar": 1e-12,
           "how": "every rank compares the sharded result with its own single-GPU result on the same inputs (windowed PSD + "
                  "coherence, row-sharded weighted LS with one NCCL all-reduce, one L1 / IndBallL0 / group-lasso ADMM problem each, sharded by peer stores); "
                  "relative l2, max over ranks"}
    out["ok"] = bool(out["window_sharded"] <= 1e-12 and out["row_sharded"] <= 1e-12 and out["admm_sharded"] <= 1e-12
                     and out["admm_group_sharded"] <= 1e-12 and out["admm_ball_l0_sharded"] <= 1e-12
                     and out["admm_same_support_and_iterations"])
    return out


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle port; Julia is not installed) on host cores."""
    if rank != 0:
        return
    t, y, f, n = make_cfg2()
    nwin = 24
    for _ in range(args.warmup):
        cpu_baseline_windows(t, y, f, n, 2)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_baseline_windows(t, y, f, n, nwin)
    dt = time.perf_counter() - t0
    val = args.steps * nwin / dt
    cores = os.cpu_count()
    line = {
        "impl": "reference", "metric": "windowed LS spectra/sec", "value": val, "unit": "windows/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg2_config(n),
        "cpu_baseline": {"value": val, "unit": "windows/s", "cores": cores, "blas_threads": blas_threads(),
                         "kind": "port",
                         "sample": f"{nwin} of {2 * NW - 1} windows per step, oracle reference-literal mode "
                                   f"(numpy/OpenBLAS, all host threads); Julia is not installed"},
        "e2e": {"value": val, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--cpu-windows", type=int, default=96)
    ap.add_argument("--no-admm", action="store_true", help="skip the cfg3 ADMM leg (extra.admm)")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the other BASELINE configs (extra.cfg1 / cfg4 / cfg5a / cfg5b_rowsharded / strong / parity)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/window_sums.npy (the Nf cross-window sums of "
                         "|x|^2, all-reduced over the ranks) and DIR/psd.npy (the finalised PSD), both float64")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L
    import ctypes as C

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = lp.Context(local)
    # the library enqueues on torch's current stream so torch CUDA events bracket whole steps (kernels + NCCL)
    stream = torch.cuda.Stream()  # an explicit (non-default) stream: the default stream's handle is 0
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)

    # every rank owns one 2^22-sample segment (its own seed): weak scaling, no data-path collective
    t, y, f, n = make_cfg2(seed=2 + rank)
    noverlap = n >> 1
    W = lp.hanning(n)
    K = lp.window_count(NSAMP, n, noverlap)
    # resident inputs (torch owns the allocation; the library takes raw device pointers)
    d_t = torch.from_numpy(t).cuda()
    d_y = torch.from_numpy(y).cuda()
    # pinned host copies for the e2e leg
    h_t = torch.from_numpy(t).pin_memory()
    h_y = torch.from_numpy(y).pin_memory()
    sums = np.zeros(NF)
    info = C.c_int(0)
    fptr, wptr, sptr = f.ctypes.data_as(C.c_void_p), W.ctypes.data_as(C.c_void_p), sums.ctypes.data_as(C.c_void_p)
    acc = torch.zeros(NF, dtype=torch.float64, device="cuda")

    def step_resident():
        ctx.check(ctx.lib.lpvs_ls_window_sums_dev(ctx.h, L.WIN_PSD, C.c_void_p(d_y.data_ptr()), None,
                                                  C.c_void_p(d_t.data_ptr()), NSAMP, fptr, NF, wptr, n, noverlap,
                                                  LAMBDA, 0, K, sptr, C.byref(info)))
        ms = ctx.last_call_ms()
        gms, gl, gfl = ctx.gram_timing()
        if world > 1:  # cross-rank reduction of the accumulators (Nf doubles), then /K_total^2 on the host
            acc.copy_(torch.from_numpy(sums))
            dist.all_reduce(acc)
        return ms, gms, gfl

    def step_e2e():
        ctx.check(ctx.lib.lpvs_ls_window_sums(ctx.h, L.WIN_PSD, C.c_void_p(h_y.data_ptr()), None,
                                              C.c_void_p(h_t.data_ptr()), NSAMP, fptr, NF, wptr, n, noverlap, LAMBDA,
                                              0, K, sptr, C.byref(info)))
        ms = ctx.last_call_ms()
        if world > 1:
            acc.copy_(torch.from_numpy(sums))
            dist.all_reduce(acc)
        return ms

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.check(ctx.lib.lpvs_sync(ctx.h))

    def allsum(v):
        if world == 1:
            return v
        tt = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        return float(tt.item())

    def allmax(v):
        if world == 1:
            return v
        tt = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    # ---- resident leg ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # sampled through warm-up + timed region (same workload), 100 ms period
    for _ in range(args.warmup):
        step_resident()
    launches0 = ctx.launches
    barrier()
    wall0 = time.perf_counter()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    call_ms = gram_ms = gram_fl = 0.0
    for _ in range(args.steps):
        ms, gms, gfl = step_resident()
        call_ms += ms
        gram_ms += gms
        gram_fl += gfl
    ev1.record()
    barrier()
    wall = time.perf_counter() - wall0
    dev_ms = ev0.elapsed_time(ev1)  # CUDA events on the launching stream around exactly K steps
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # before the legs below overwrite `sums`
        last_sums = acc.cpu().numpy() if world > 1 else sums.copy()
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "window_sums.npy"), last_sums)
        np.save(os.path.join(args.dump_outputs, "psd.npy"), lp.window_finalize(L.WIN_PSD, last_sums, NF, world * K))
    launches = ctx.launches - launches0
    one_gpu_ms = allsum(dev_ms / args.steps if rank == 0 else 0.0)  # rank 0's record is make_cfg2()'s default seed
    dev_ms = allmax(dev_ms)
    wall = allmax(wall)
    ms_per_step = dev_ms / args.steps
    value = world * K / (ms_per_step * 1e-3)

    # ---- e2e leg (host buffers through the public C ABI) ----
    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    barrier()
    e2e_steps = max(3, args.steps // 2)
    ew0 = time.perf_counter()
    ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ee0.record()
    for _ in range(e2e_steps):
        step_e2e()
    ee1.record()
    barrier()
    e2e_wall = allmax(time.perf_counter() - ew0)
    e2e_ms = allmax(ee0.elapsed_time(ee1))
    e2e_value = world * K / (max(e2e_ms / e2e_steps, e2e_wall / e2e_steps * 1e3) * 1e-3)

    admm = None
    if not args.no_admm:
        admm = admm_leg(ctx, lp, L, C, rank, world, allsum=lambda v: allsum(v), allmax=allmax, barrier=barrier)

    peak, peak_src = fp64_peak()
    extra = {"admm": admm}
    # The headline runs in the default phase mode (chain_ref: the reference's rounded phase fl(fl(2 pi f) t), 5 extra FP64
    # ops per synthesised element).  For the record: the same step with the mathematically exact phase (LPVS_PHASE_CHAIN),
    # which is faster and closer to the true basis but differs from the REFERENCE by its phase rounding (DESIGN.md 1).
    ctx.set_option(L.OPT_PHASE_MODE, L.PHASE_CHAIN)
    try:
        step_resident()
        barrier()
        x_ms = x_gms = x_gfl = 0.0
        for _ in range(3):
            ms_, gms_, gfl_ = step_resident()
            x_ms, x_gms, x_gfl = x_ms + ms_, x_gms + gms_, x_gfl + gfl_
        barrier()
        extra["exact_phase_mode"] = {"ms_per_step": allmax(x_ms / 3), "gram_ms_per_step": x_gms / 3,
                                     "gram_tflops": x_gfl / (x_gms * 1e-3) / 1e12,
                                     "gram_frac": x_gfl / (x_gms * 1e-3) / 1e12 / peak,
                                     "windows_per_s": world * K / (allmax(x_ms / 3) * 1e-3),
                                     "note": "LPVS_PHASE_CHAIN: not the headline -- parity with the reference needs its "
                                             "phase rounding (tests/test_gpu_baseline_parity.py)"}
    finally:
        ctx.set_option(L.OPT_PHASE_MODE, L.PHASE_AUTO)
    # Opt-in LPVS_PHASE_STRUCTURED: the windows' Gram matrices from their 3 Nf trigonometric sums (Toeplitz + Hankel in the
    # frequency index, csrc/structured.cu) -- the exact-phase accuracy class again, O(n Nf) instead of O(n Nf^2) work.
    ctx.set_option(L.OPT_PHASE_MODE, L.PHASE_STRUCTURED)
    try:
        step_resident()
        barrier()
        x_ms = x_gms = 0.0
        for _ in range(3):
            ms_, gms_, _gfl = step_resident()
            x_ms, x_gms = x_ms + ms_, x_gms + gms_
        barrier()
        extra["structured_mode"] = {"ms_per_step": allmax(x_ms / 3), "gram_stage_ms_per_step": x_gms / 3,
                                    "windows_per_s": world * K / (allmax(x_ms / 3) * 1e-3),
                                    "note": "LPVS_PHASE_STRUCTURED (opt-in, not the headline): Gram stage = sum tables + "
                                            "k_trig_sums + k_gram_fill + k_rhs_from_sums; the rest of the step is the batched "
                                            "Cholesky; exact phase of the ideal grid, tests/test_gpu_structured.py"}
    except Exception as e:  # never lose the headline line to an extra leg
        extra["structured_mode"] = {"error": repr(e)[:300]}
    finally:
        ctx.set_option(L.OPT_PHASE_MODE, L.PHASE_AUTO)
    # Opt-in LPVS_PHASE_STRUCTURED_REF: the same sums plus the first-order correction of G and b for the reference's phase
    # rounding, G += D'B + B'D by a half-precision tensor-core GEMM with eps exact in FP64 (csrc/corr.cu): the default mode's
    # parity class (tests/test_gpu_baseline_parity.py::test_structured_ref_mode_meets_the_default_bars).
    try:
        import numpy as _np

        step_resident()
        sums_default = sums.copy()
        ctx.set_option(L.OPT_PHASE_MODE, L.PHASE_STRUCTURED_REF)
        step_resident()
        sums_ref = sums.copy()
        barrier()
        x_ms = x_gms = 0.0
        for _ in range(3):
            ms_, gms_, _gfl = step_resident()
            x_ms, x_gms = x_ms + ms_, x_gms + gms_
        barrier()
        extra["structured_ref_mode"] = {
            "ms_per_step": allmax(x_ms / 3), "gram_stage_ms_per_step": x_gms / 3,
            "windows_per_s": world * K / (allmax(x_ms / 3) * 1e-3),
            "rel_l2_vs_default_mode": float(_np.linalg.norm(sums_ref - sums_default) / _np.linalg.norm(sums_default)),
            # executed f16 flop: off-diagonal 128-tiles K' = 2 n, diagonal tiles K' = n
            "correction_flop_per_step": float(K) * 2.0 * 128 * 128 * n * ((NF + 63) // 64) ** 2,
            "note": "LPVS_PHASE_STRUCTURED_REF (opt-in, not the headline): structured Gram stage + k_corr_tables (eps exact in "
                    "FP64, once per (column, sample)) + k_gram_corr (f16 mma.sync m16n8k16, f32 accumulation, warp-specialised "
                    "producers / consumers over a 3-stage mbarrier ring) + k_rhs_corr; the reference's phase rounding to first "
                    "order: the default mode's parity class (tests/test_gpu_structured.py, tests/test_gpu_baseline_parity.py)"}
        sm_ = extra.get("structured_mode", {}).get("gram_stage_ms_per_step")
        if sm_:  # tables + k_gram_corr + k_rhs_corr: what the correction adds to the structured Gram stage
            r_ = extra["structured_ref_mode"]
            r_["correction_stage_ms_per_step"] = r_["gram_stage_ms_per_step"] - sm_
            r_["correction_f16_tflops_over_stage"] = r_["correction_flop_per_step"] / (r_["correction_stage_ms_per_step"] * 1e-3) / 1e12
            r_["f16_peaks_tflops"] = {"mma_sync_m16n8k16_issue_peak_this_pool": 554.0, "source": "tools/mma_probe.cu; k_gram_corr "
                                      "alone: profiles/r02_summary.md (14.0 ms = 314 TFLOP/s = 57 %)"}
    except Exception as e:  # never lose the headline line to an extra leg
        extra["structured_ref_mode"] = {"error": repr(e)[:300]}
    finally:
        ctx.set_option(L.OPT_PHASE_MODE, L.PHASE_AUTO)
    parity_ok = True
    if not args.no_extra:
        from lpvspectral_jl_b200 import _dist as D

        peak_live = fp64_peak_live(torch)
        extra["fp64_dgemm_8192_live_tflops"] = peak_live
        if rank == 0:
            for name, fn in (("cfg1", lambda: cfg1_leg(ctx, lp, peak)), ("cfg4", lambda: cfg4_leg(ctx, lp, L, C))):
                try:
                    extra[name] = fn()
                except Exception as e:  # never lose the headline line to an extra leg
                    extra[name] = {"error": repr(e)[:300]}
        barrier()
        extra.update(cfg5_legs(ctx, lp, L, C, D, torch, dist, rank, world, local, allmax, barrier, peak))
        if world > 1:
            one4 = allsum(extra["cfg4"].get("iters_per_s", 0.0) if rank == 0 and isinstance(extra.get("cfg4"), dict) else 0.0)
            extra["cfg4_sharded"] = cfg4_sharded_leg(ctx, lp, L, C, D, dist, world, allmax, barrier, one4)
            extra["strong"] = strong_leg(ctx, lp, L, C, D, torch, dist, rank, world, allmax, barrier, one_gpu_ms,
                                         max(3, args.steps // 2))
            extra["parity"] = parity_leg(ctx, lp, L, C, D, torch, dist, rank, world, local, allmax)
            parity_ok = extra["parity"]["ok"]
        else:
            extra["strong"] = {"workload": "cfg2_windowpsd", "scaling": "strong", "n_gpus": 1,
                               "ms_per_pass": one_gpu_ms, "speedup_vs_one_gpu": 1.0}
            extra["parity"] = {"note": "sharded-path parity is checked at --gpus N > 1"}

    if rank == 0:
        achieved = gram_fl / (gram_ms * 1e-3) / 1e12
        nreg = 2 * NF - 1
        # the CPU baseline is an N=1 figure; at N>1 only a token sample keeps the other ranks from idling in NCCL
        cpu_windows = args.cpu_windows if world == 1 else min(args.cpu_windows, 8)
        cpu_val, cpu_dt = cpu_baseline_windows(t, y, f, n, cpu_windows)
        try:  # second, stronger CPU line (Gram + Cholesky on the host BLAS); never allowed to cost the headline line
            cpu_gram_val, _ = cpu_baseline_windows(t, y, f, n, min(cpu_windows, 48), mode="gram")
        except Exception:
            cpu_gram_val = None
        line = {
            "metric": "windowed LS spectra/sec", "value": value, "unit": "windows/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg2_config(n),
            "timing": {"how": "torch CUDA events on the shared launching stream around exactly K steps (barrier + "
                              "synchronize both sides), max over ranks", "wall_ms_per_step": wall / args.steps * 1e3},
            "e2e": {"value": e2e_value, "unit": "windows/s", "h2d_bytes_per_step": int(2 * NSAMP * 8 + n * 8 + NF * 8),
                    "d2h_bytes_per_step": int(NF * 8), "steps": e2e_steps,
                    "api": "lpvs_ls_window_sums (host pointers, pinned)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "traffic": ncu_traffic("k_gram"), "kernel": "k_gram<GRAM_CHAINREF>",
                         "flops_per_window": float(n) * nreg * (nreg + 1), "windows_per_launch": K,
                         "gram_ms_per_step": gram_ms / args.steps, "gram_share_of_step": gram_ms / call_ms,
                         "peak_source": peak_src, "peak_live": extra.get("fp64_dgemm_8192_live_tflops"),
                         "frac_of_peak_live": (achieved / extra["fp64_dgemm_8192_live_tflops"]
                                               if extra.get("fp64_dgemm_8192_live_tflops") else None),
                         "peak_live_how": "cuBLAS DGEMM 8192^3 via torch.matmul, best of 5, CUDA events, inside this run"},
            "cpu_baseline": {"value": cpu_val, "unit": "windows/s", "cores": os.cpu_count(),
                             "blas_threads": blas_threads(), "kind": "port", "gram_cholesky_value": cpu_gram_val,
                             "sample": f"{cpu_windows} of {K} windows in {cpu_dt:.1f} s, oracle reference-literal "
                                       "mode (N-rhs LU per window, numpy/OpenBLAS all threads)"},
            "clocks": clocks,
            "extra": extra,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if not parity_ok:
        sys.exit(3)  # a sharded path disagreed with the single-GPU result beyond 1e-12: the run is not valid


if __name__ == "__main__":
    main()
