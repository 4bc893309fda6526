#!/usr/bin/env python
"""bench.py - GP fits/sec at N=16384 fp64 (kernel + Cholesky + solve + LML) and Cholesky TFLOP/s.

One "step" = one evaluation of GaussianProcess.compute_likelihood (GPr.py:57-69) on BASELINE
config 2: N = 16384, D = 8 SE-ARD, synthetic targets (SURVEY section 8d recipe).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

* value    : fits/s with X, y resident in HBM (only the 10 hyper-parameters go up and one double
             comes back per step), timed with CUDA events on the launching stream.
* e2e      : the same metric through the drop-in API, GPr.GaussianProcess(...).compute_likelihood(hyp),
             with X and y in pinned HOST memory: every step uploads them and reads the result back.
* roofline : the factorisation stage (>= 99 % of it is the TMA-fed DMMA tile kernel), N^3/3 flops over
             its CUDA-event duration, against the FP64 tensor pipe rate measured in the same run
             (MEASURED_PEAKS.json has no fp64 entry; cuBLAS DGEMM is reported beside it).
* N > 1    : the path shards over independent problems (hyper-parameter vectors): every rank fits its
             own slice, no data-path collective; the scalar likelihoods are all-gathered over NCCL
             after the timed region ("weak" scaling: K fits per GPU).
* --impl reference : the reference's own CPU arithmetic (oracle/gpr_oracle.py, a line-by-line port of
             GPr.py verified bit-for-bit against it) on the host cores, on a bounded sample.
* --dump-outputs DIR : after the timed steps, what they returned in their last step as float64 .npy files:
             DIR/nlml.npy (the device-resident fit of every rank, shape (ranks,)) and DIR/e2e_nlml.npy (rank 0's last
             drop-in call, (1, 1)).  All inputs are seeded, so two builds run with the same arguments can be compared
             output for output.
"""
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

from bench_configs import N_FIT, D_FIT, M_TEST, make_c2, make_c3, make_c4, make_c5, khyp_of  # noqa: E402

METRIC = "GP fits/sec at N=16384 fp64 (kernel+Cholesky+solve+LML)"
WORKLOAD = "GPr N=16384 D=8 SE-ARD fp64 compute_likelihood (BASELINE configs[1])"


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
def cpu_fit_seconds(n, log_hyp, X, y):
    from oracle import gpr_oracle
    t0 = time.perf_counter()
    v = gpr_oracle.nlml(log_hyp, X[:n], y[:n])
    return time.perf_counter() - t0, float(v[0, 0])


_BLAS_LIMIT = None


def use_all_host_cores():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU legs must run on all host cores (SURVEY 8d), so the
    BLAS pool is resized explicitly.  Returns the number of threads in use."""
    global _BLAS_LIMIT
    try:
        from threadpoolctl import threadpool_limits
        _BLAS_LIMIT = threadpool_limits(limits=os.cpu_count() or 1, user_api='blas')
    except Exception:
        pass
    return blas_threads()


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        info = threadpool_info()
        ths = [i.get('num_threads') for i in info if i.get('user_api') == 'blas']
        if ths:
            return int(max(ths))
    except Exception:
        pass
    return os.cpu_count() or 1


def cpu_baseline(budget_s=20.0):
    """The reference's arithmetic (oracle port of GPr.py:57-69) on the host cores, bounded sample."""
    use_all_host_cores()
    X, y, _, lh = make_c2()
    t1024, _ = cpu_fit_seconds(1024, lh, X, y)
    t1024, _ = cpu_fit_seconds(1024, lh, X, y)
    ns = 1024
    for cand in (2048, 4096, 8192):
        if t1024 * (cand / 1024.0) ** 3 <= budget_s:
            ns = cand
    t, _ = cpu_fit_seconds(ns, lh, X, y) if ns > 1024 else (t1024, 0)
    scale = (N_FIT / ns) ** EMPIRICAL_EXPONENT
    return {"value": 1.0 / (t * scale), "unit": "fits/s", "cores": blas_threads(), "kind": "port",
            "sample": "one compute_likelihood at N=%d (first %d points of the workload), %.2f s; scaled x(16384/%d)^%.1f = %.1f "
                      "for N=16384 (empirical exponent from the measured pair in profiles/r02_cpu_full_size.json: a real "
                      "full-size fit takes 72 s on 16 cores; the cubic law of round 1 overshot x3)" % (ns, ns, t, ns, EMPIRICAL_EXPONENT, scale),
            "host_cpus": os.cpu_count(), "other_configs": cpu_other_configs(),
            "measured_full_size": measured_full_size_record()}


def measured_full_size_record():
    """One REAL N=16384 compute_likelihood of the CPU port, measured once on a GPU box's host by
    `bench.py --impl reference --ref-full` (about four minutes: too long for the default run) and kept under profiles/."""
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "r02_cpu_full_size.json")))
        return {k: rec[k] for k in ("value", "unit", "ms_per_step", "cpu_baseline")} | {"source": "profiles/r02_cpu_full_size.json (not measured in this run)"}
    except Exception:
        return None


def cpu_other_configs():
    """Bounded CPU samples of the oracle ports for configs 5, 4 and 3 (SURVEY 8d), a few seconds each."""
    from oracle import gpr_oracle, gppref_oracle, gpc_oracle
    out = {}
    X5, Y5, lhs5 = make_c5()
    t0 = time.perf_counter()
    for l in lhs5[:2]:
        gpr_oracle.nlml(l, X5, Y5)
    t5 = (time.perf_counter() - t0) / 2
    out["c5_sweep_1024x2048"] = {"s_per_problem": t5, "ms_extrapolated": t5 * 1024 * 1e3,
                                 "sample": "2 of the 1024 problems (GPr.py:57-69 port), x512"}
    rng = np.random.default_rng(0)
    n, D, P = 1024, 6, 8192
    x = rng.random((n, D))
    uvi = rng.integers(0, n, (P, 2))
    bad = uvi[:, 0] == uvi[:, 1]
    uvi[bad, 1] = (uvi[bad, 0] + 1) % n
    y = np.where(rng.random(P) < 0.5, 1.0, -1.0).reshape(-1, 1)
    t0 = time.perf_counter()
    gppref_oracle.calc_laplace(x, uvi, y, np.log([0.5] * D + [1.0, 0.1]), max_iter=3)
    t4 = (time.perf_counter() - t0) / 3
    out["c4_gppref"] = {"s_per_iteration_n1024": t4, "ms_per_iteration_n4096_extrapolated": t4 * 64 * 1e3,
                        "sample": "3 iterations of the GPpref.py:112-157 port at n=1024, P=8192; x(4096/1024)^3 per iteration"}
    n, D = 1024, 4
    x = rng.random((n, D))
    yc = np.where(rng.random(n) < 0.5, 1.0, -1.0)
    t0 = time.perf_counter()
    f, lml, st = gpc_oracle.calc_laplace(x, yc, np.log([0.5] * D + [1.0]), max_iter=2, return_state=True)
    t3 = (time.perf_counter() - t0) / max(st["it"], 1)
    out["c3_gpc"] = {"s_per_newton_step_n1024": t3, "ms_per_newton_step_n8192_extrapolated": t3 * 512 * 1e3,
                     "sample": "2 Newton steps of the R&W Alg. 3.1 oracle at N=1024; x(8192/1024)^3 per step"}
    return out


EMPIRICAL_EXPONENT = 2.2   # t(N) of the CPU port between N=4096 (3.4 s) and N=16384 (72.0 s) on a GPU box's 16 host cores
                           # (profiles/r02_cpu_full_size.json): BLAS efficiency grows with N, a cubic law overshoots x3


def run_reference(args, rank, world):
    """The reference's own CPU arithmetic on the host cores: rank 0 only.  Every step is one compute_likelihood at the
    largest N in (1024, 2048, 4096) for which all steps fit ~150 s (a bounded sample of the workload); the factor
    from the sample to the full N=16384 is then MEASURED in the same run by one real full-size fit (about 70 s, 20 GiB)
    unless --no-ref-calibrate (then the empirical exponent above).  --ref-full: every step at the real N=16384."""
    if rank != 0:
        return
    cores = use_all_host_cores()
    X, y, _, lh = make_c2()
    steps, warm = args.steps, args.warmup
    if args.ref_full:
        ns = N_FIT
    else:
        t1024, _ = cpu_fit_seconds(1024, lh, X, y)
        t1024, _ = cpu_fit_seconds(1024, lh, X, y)
        ns = 1024
        for cand in (2048, 4096):
            if t1024 * (cand / 1024.0) ** 3 * (steps + warm) <= 150.0:
                ns = cand
    for _ in range(warm):
        cpu_fit_seconds(ns, lh, X, y)
    t0 = time.perf_counter()
    for _ in range(steps):
        _, v = cpu_fit_seconds(ns, lh, X, y)
    el = time.perf_counter() - t0
    per_sample = el / steps
    calibrated = None
    if ns == N_FIT:
        scale = 1.0
        sample = ("MEASURED: each step = one compute_likelihood of the oracle port of GPr.py:57-69 at the full N=16384, "
                  "%.1f s/step, nlml %.6f" % (per_sample, v))
    else:
        scale = (N_FIT / ns) ** EMPIRICAL_EXPONENT
        how = "empirical exponent %.1f (profiles/r02_cpu_full_size.json)" % EMPIRICAL_EXPONENT
        if not args.no_ref_calibrate:
            try:
                import psutil
                if psutil.virtual_memory().available > 40 * 2 ** 30:
                    t_full, v_full = cpu_fit_seconds(N_FIT, lh, X, y)
                    scale = t_full / per_sample
                    calibrated = {"full_size_fit_s": t_full, "nlml": v_full}
                    how = "factor MEASURED in this run by one real N=16384 fit (%.1f s)" % t_full
            except Exception as exc:      # not enough memory etc.: keep the empirical exponent
                how += "; full-size calibration failed: %r" % (exc,)
        sample = ("each step = one compute_likelihood of the oracle port of GPr.py:57-69 at N=%d (first %d points), "
                  "%.3f s/step measured; scaled x%.1f to N=16384: %s" % (ns, ns, per_sample, scale, how))
    per_fit = per_sample * scale
    val = 1.0 / per_fit
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "fits/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": per_fit * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "n": N_FIT, "d": D_FIT},
            "cpu_baseline": {"value": val, "unit": "fits/s", "cores": cores, "kind": "port", "sample": sample,
                             "host_cpus": os.cpu_count(), "extrapolated": ns != N_FIT and calibrated is None,
                             "calibration": calibrated},
            "e2e": {"value": val, "unit": "fits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), file=RESULT_OUT, flush=True)


# ------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    from gptest_b200 import _lib, GPr

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        # stdout carries exactly one JSON line: whatever NCCL_DEBUG makes NCCL say (its version banner) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    _lib.set_default_device(local_rank)
    h = _lib.default_handle(local_rank)
    h.set_stream(torch.cuda.current_stream().cuda_stream)

    X, y, Z, lh = make_c2()
    steps, warm = args.steps, args.warmup
    # every rank owns its own slice of hyper-parameter vectors (independent fits)
    rng = np.random.default_rng(1000 + rank)
    lhs = lh[None, :] + 0.05 * rng.standard_normal((steps + warm, lh.size))
    lhs[0] = lh
    khs = np.array([khyp_of(l) for l in lhs])

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident arm ----------------
    h.set_train(X, y)
    for i in range(warm):
        h.gpr_nlml(khs[i])
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    l0 = h.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    vals, stage = [], {"kbuild_ms": 0.0, "factor_ms": 0.0, "finish_ms": 0.0, "total_ms": 0.0}
    ev0.record()
    for i in range(steps):
        vals.append(h.gpr_nlml(khs[warm + i]))
        tm = h.timings()
        for k in stage:
            stage[k] += tm[k]
    ev1.record()
    barrier()
    launches = h.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    ms = ev0.elapsed_time(ev1)
    t = torch.tensor([ms], dtype=torch.float64, device='cuda')
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = t.item()
    for k in stage:
        stage[k] /= steps

    # ---------------- end-to-end arm: drop-in API, host buffers ----------------
    Xp = torch.from_numpy(X).pin_memory().numpy()
    yp = torch.from_numpy(y).pin_memory().numpy()
    gp = GPr.GaussianProcess(lh, 0, 0, "SE", "zero", "zero", Xp, yp)
    e_steps = max(3, min(steps, 10))
    for i in range(2):
        gp.compute_likelihood(lhs[i])
    barrier()
    ev0.record()
    for i in range(e_steps):
        out = gp.compute_likelihood(lhs[warm + (i % steps)])
    ev1.record()
    barrier()
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device='cuda')
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = t.item() / e_steps
    assert abs(out[0, 0] - vals[(e_steps - 1) % steps]) <= 1e-9 * abs(out[0, 0])

    # ---------------- gather the scalar likelihoods (the only collective) ----------------
    v = torch.tensor(vals, dtype=torch.float64, device='cuda')
    if dist is not None:
        allv = [torch.empty_like(v) for _ in range(world)]
        dist.all_gather(allv, v)
        v = torch.cat(allv)
    all_vals = v.cpu().numpy()
    if rank == 0 and args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "nlml.npy"), all_vals.reshape(world, steps)[:, -1].astype(np.float64))
        np.save(os.path.join(args.dump_outputs, "e2e_nlml.npy"), np.asarray(out, dtype=np.float64))

    extra = {}
    if rank == 0 and world == 1 and not args.skip_extras:
        extra = single_gpu_extras(h, X, y, Z, lh)
    dmma_peak = h.microbench(0)
    if args.sweep:
        extra["sweep_1024x2048"] = sweep_c5(h, rank, world, dist, torch, dmma_peak)

    if rank == 0:
        fits_per_s = world * steps / (ms_max * 1e-3)
        flops_chol = N_FIT ** 3 / 3.0
        chol_tflops = flops_chol / (stage["factor_ms"] * 1e-3) / 1e12
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("dmma_gemm_dram_bytes_per_launch")
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": fits_per_s, "unit": "fits/s", "n_gpus": world, "steps": steps, "warmup": warm,
            "ms_per_step": ms_max / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "n": N_FIT, "d": D_FIT, "parallelism": "independent fits per GPU (dp%d)" % world,
                       "l2": "working set 2 GiB per fit > 126 MB L2 (no flush needed)", "fits_per_gpu": steps},
            "cholesky_fp64_tflops": chol_tflops,
            "stage_ms": stage,
            "roofline": {"bound": "tensor", "achieved": chol_tflops, "peak": dmma_peak, "unit": "TFLOP/s",
                         "frac": chol_tflops / dmma_peak, "traffic": traffic,
                         "traffic_source": "profiles/traffic.json: one ncu --set full capture of dmma_gemm_nt_kernel at the "
                                           "K=512 trailing-update shape (static file, per launch; not measured in this run)",
                         "frac_vs_cublas": (chol_tflops / extra["cublas_dgemm_8192_tflops"]) if extra.get("cublas_dgemm_8192_tflops") else None,
                         "frac_vs_nominal_40": chol_tflops / 40.0,
                         "kernel": "dmma_gemm_nt_kernel inside the factorisation stage (N^3/3 flop / CUDA-event stage time, panels included)",
                         "peak_source": "FP64 DMMA.8x8x4 pipe rate measured in this run (gpb_microbench); MEASURED_PEAKS.json has no fp64 entry; nominal 37 TFLOP/s",
                         "peak_cublas_dgemm": extra.get("cublas_dgemm_8192_tflops")},
            "roofline_kbuild": {"bound": "hbm", "achieved": extra.get("kxx_full_GBs"), "peak": hbm_peak, "unit": "GB/s",
                                "frac": (extra.get("kxx_full_GBs") / hbm_peak) if extra.get("kxx_full_GBs") else None,
                                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650",
                                "bytes": 8.0 * N_FIT * N_FIT + 8.0 * N_FIT * D_FIT,
                                "variant": "full symmetric matrix (compute_Kxx_matrix, GPr.py:99-103)"},
            "roofline_kbuild_in_path": {"bound": "hbm", "unit": "GB/s", "peak": hbm_peak,
                                        "bytes": 4.0 * N_FIT * (N_FIT + 1) + 8.0 * N_FIT * D_FIT,
                                        "ms": stage["kbuild_ms"],
                                        "achieved": (4.0 * N_FIT * (N_FIT + 1) + 8.0 * N_FIT * D_FIT) / (stage["kbuild_ms"] * 1e-3) / 1e9,
                                        "frac": (4.0 * N_FIT * (N_FIT + 1) + 8.0 * N_FIT * D_FIT) / (stage["kbuild_ms"] * 1e-3) / 1e9 / hbm_peak,
                                        "variant": "lower tiles only - what compute_likelihood's timed path builds (stage kbuild_ms also holds "
                                                   "the point scaling and the y row)"},
            "e2e": {"value": world / (e2e_ms * 1e-3), "unit": "fits/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(X.nbytes + y.nbytes + 8 * (D_FIT + 2)), "d2h_bytes_per_step": 12,
                    "api": "GPr.GaussianProcess.compute_likelihood(hyp), pinned host X/y uploaded every call"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "nlml_first": float(all_vals[0]), "nlml_count": int(all_vals.size),
        }
        line.update(extra)
        if world == 1 and not args.skip_cpu:
            line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line), file=RESULT_OUT, flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def single_gpu_extras(h, X, y, Z, lh):
    """secondary figures of the same run: cuBLAS bar, covariance-assembly bandwidth, predict."""
    import torch
    out = {}
    kh = khyp_of(lh)
    n = 8192
    A = torch.randn(n, n, dtype=torch.float64, device='cuda')
    B = torch.randn(n, n, dtype=torch.float64, device='cuda')
    best = 1e30
    for i in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); C = A @ B.T; e1.record(); torch.cuda.synchronize()
        if i:
            best = min(best, e0.elapsed_time(e1))
    out["cublas_dgemm_8192_tflops"] = 2 * n ** 3 / best / 1e9
    del A, B, C
    K = torch.empty((N_FIT, N_FIT), dtype=torch.float64, device='cuda')
    ts = []
    for i in range(6):
        h.kxx_dev(kh, K.data_ptr())
        if i:
            ts.append(h.timings()["kbuild_ms"])
    out["kxx_full_ms"] = float(np.mean(ts))
    out["kxx_full_GBs"] = (8.0 * N_FIT * N_FIT + 8.0 * N_FIT * D_FIT) / (out["kxx_full_ms"] * 1e-3) / 1e9
    del K
    h.set_train(X, y)
    for i in range(3):
        fz, cov = h.gpr_predict(kh, Z)
    out["fit_predict_ms"] = h.timings()["total_ms"]
    for i in range(2):
        v, g = h.gpr_nlml(kh, want_grad=True)
    tm = h.timings()
    out["fit_grad_ms"] = tm["total_ms"]                       # value + D+2 gradients: N^3 flop (potrf + trtri + U U^T)
    out["fit_grad_tflops"] = float(N_FIT) ** 3 / (tm["total_ms"] * 1e-3) / 1e12
    # four independent hyper-parameter vectors in ONE call (multi-start / grid use): panels of all four share launches
    kh4 = np.array([kh * (1.0 + 0.01 * i) for i in range(4)])
    kh4[:, -1] = kh[-1]
    h.gpr_nlml_batched(kh4)
    t0 = time.perf_counter()
    h.gpr_nlml_batched(kh4)
    out["fits_per_s_batch_of_4"] = 4.0 / (time.perf_counter() - t0)
    # appending 128 points to the stored factor of the first N-128 (gpb_gpr_grow_*) vs the refit above
    h.grow_begin(kh, D_FIT, capacity=N_FIT)
    h.grow_append(X[:N_FIT - 256], y[:N_FIT - 256])
    h.grow_append(X[N_FIT - 256:N_FIT - 128], y[N_FIT - 256:N_FIT - 128])
    t0 = time.perf_counter()
    h.grow_append(X[N_FIT - 128:], y[N_FIT - 128:])
    out["append_128_points_ms"] = (time.perf_counter() - t0) * 1e3
    h.grow_begin(kh, D_FIT, capacity=1)                       # release the stored factor
    out["other_configs"] = other_configs(h)
    peak = h.microbench(0)
    oc = out["other_configs"]
    c3, c4 = oc["c3_gpc_n8192_d4"], oc["c4_gppref_n4096_p32768"]
    f3 = (c3["newton_iters"] + 2) * 8192.0 ** 3 / 3.0          # chol(K) jitter check + one chol(B) per Newton step + the final one
    f4 = 4096.0 ** 3 + c4["iters_reference_semantics"] * 4096.0 ** 3 / 3.0   # potrf + inverse of K, then chol(K^-1 + W) per step
    fp = N_FIT ** 3 / 3.0 + float(N_FIT) ** 2 * M_TEST          # factor + the TRSM of the predictive variance
    out["roofline_configs"] = {
        "peak_tflops": peak, "bound": "tensor",
        "c3_gpc": {"flops": f3, "ms": c3["ms"], "achieved": f3 / (c3["ms"] * 1e-3) / 1e12, "frac": f3 / (c3["ms"] * 1e-3) / 1e12 / peak},
        "c4_gppref": {"flops": f4, "ms": c4["ms"], "achieved": f4 / (c4["ms"] * 1e-3) / 1e12, "frac": f4 / (c4["ms"] * 1e-3) / 1e12 / peak},
        "c2_fit_predict": {"flops": fp, "ms": out["fit_predict_ms"], "achieved": fp / (out["fit_predict_ms"] * 1e-3) / 1e12,
                           "frac": fp / (out["fit_predict_ms"] * 1e-3) / 1e12 / peak},
        "c2_fit_grad": {"flops": float(N_FIT) ** 3, "ms": out["fit_grad_ms"], "achieved": out["fit_grad_tflops"],
                        "frac": out["fit_grad_tflops"] / peak},
        "note": "algorithmic flops (SURVEY 8d) over the wall time of one public call, host setup included",
    }
    return out


def other_configs(h):
    """BASELINE configs 3 and 4 at full size, device time of one call each (recipes: bench_configs.py)."""
    res = {}
    Xc, yc, _, lhc = make_c3()
    D = Xc.shape[1]
    h.set_train(Xc)
    for _ in range(2):
        t0 = time.perf_counter()
        f, lml, iters, trace, jit = h.gpc_laplace(yc, np.r_[np.exp(lhc[:D]), np.exp(lhc[D]) ** 2], link=0, delta_f=1e-6)
        dt = (time.perf_counter() - t0) * 1e3
    Zc = make_c3()[2]
    h.gpc_predict(Zc)
    t0 = time.perf_counter()
    h.gpc_predict(Zc)                                     # R&W Alg. 3.2 from the stored factor: latent mean, variance, probability
    dtp = (time.perf_counter() - t0) * 1e3
    res["c3_gpc_n8192_d4"] = {"ms": dt, "newton_iters": int(iters), "lml": lml, "predict_1024_ms": dtp}
    Xp, uvi, yp, lhp = make_c4()
    D = Xp.shape[1]
    h.set_train(Xp)
    for _ in range(2):
        t0 = time.perf_counter()
        f, lml, iters, trace, jit = h.pref_laplace(uvi, yp, np.r_[np.exp(lhp[:D]), np.exp(lhp[D]) ** 2], sigma=1.0,
                                                   delta_f=1e-6, max_iter=500)
        dt = (time.perf_counter() - t0) * 1e3
    res["c4_gppref_n4096_p32768"] = {"ms": dt, "iters_reference_semantics": int(iters), "ms_per_iter": dt / iters, "lml": lml}
    return res


def sweep_c5(h, rank, world, dist, torch, dmma_peak=None):
    """BASELINE config 5 through the product API: gptest_b200.sweep.sweep_nlml shards the 1024 hyper-parameter vectors
    over the ranks (contiguous slices), every rank uploads (X, y), evaluates its slice with the batched kernels and the
    results are all-gathered over NCCL - all of it INSIDE the timed region (strong scaling)."""
    from gptest_b200 import sweep
    X, Y, lhs = make_c5()
    B = len(lhs)
    sweep.sweep_nlml(X, Y, lhs)        # untimed warm-up with the same shapes (work space, NCCL buffers)
    best, vals = None, None
    for rep in range(2):
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        vals = sweep.sweep_nlml(X, Y, lhs)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device='cuda')
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
        best = ms if best is None else min(best, ms)
    tf = B * 2048 ** 3 / 3.0 / (best * 1e-3) / 1e12
    out = {"problems": B, "n": 2048, "ms": best, "fits_per_s": B / (best * 1e-3), "chol_tflops": tf, "scaling": "strong",
           "api": "gptest_b200.sweep.sweep_nlml (default CUDA evaluator); H2D of (X, y), the batched fits of this rank's slice "
                  "and the NCCL all-gather of the scalar likelihoods are inside the timed region; best of 2",
           "nlml_checksum": float(np.where(np.isfinite(vals), vals, 0.0).sum()), "failed": int((~np.isfinite(vals)).sum())}
    if dmma_peak:
        out["roofline"] = {"bound": "tensor", "achieved": tf, "peak": dmma_peak, "unit": "TFLOP/s", "frac": tf / dmma_peak,
                           "flops": "1024 x N^3/3, N = 2048"}
    return out


RESULT_OUT = sys.stdout


def claim_stdout():
    """stdout carries exactly ONE JSON line.  Libraries write to file descriptor 1 behind Python's back (NCCL's
    version banner under NCCL_DEBUG, whatever NCCL_DEBUG_FILE says on some boxes): from here on descriptor 1 is a
    copy of stderr, and the result line goes to the saved original."""
    global RESULT_OUT
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    RESULT_OUT = os.fdopen(saved, "w")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sweep", action="store_true", default=True, help="also time the 1024 x N=2048 sweep (config 5)")
    ap.add_argument("--no-sweep", dest="sweep", action="store_false")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--ref-full", action="store_true", help="reference arm at the real N=16384 (minutes per step)")
    ap.add_argument("--no-ref-calibrate", action="store_true", help="reference arm: skip the one full-size fit that measures the scale factor")
    ap.add_argument("--skip-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm's sample size depends on the host's speed)")
    claim_stdout()
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
