"""Joint posterior samples of GP regression (gpb_gpr_sample) at the sizes a user of GP_parameter_fit.py meets:
   python tools/gpr_sample_once.py [out.json] [reps]

(a) the C5 points (bench_configs.make_c5: n = 2048, d = 2) with the script's kernel (RBF variance 10, lengthscale 20,
    noise sd 0.25) on the 100 x 100 prediction grid of GP_parameter_fit.py:47-49 (m = 10 000), S = 16 and 1024 draws;
(b) C2 (bench_configs.make_c2: n = 16384, d = 8) with m = 4096 test points and S = 64.
Per case, warm, in one process: the stage times the call reports (CUDA events; median over reps), the flop counts
computed from the shapes (n^3/3 + n^2 m for the factorisation with the test rows, n m^2 for Sigma*, m^3/3 per
factorisation attempt of Sigma*, 2 S m^2 for D = E L^T; padded sizes), the jitter the call chose, the DMMA pipe rate
of the same run (gpb_microbench kind 0), and the GPU name and power limit.  For (a) the same computation in
numpy / scipy on the host's cores (one run, S = 16), and the largest difference of the device's Sigma* from it."""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, '.')
from bench_configs import make_c2, make_c5  # noqa: E402
from gptest_b200 import _lib  # noqa: E402

out = sys.argv[1] if len(sys.argv) > 1 else None
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    name, power, clk = [t.strip() for t in q.split(',')]
    return dict(gpu=name, power_limit=power, max_sm_clock=clk)


def pad(v):
    return -(-v // 128) * 128


def flops(n, m, S, attempts):
    np_, mp, sp = pad(n), pad(m), pad(S)
    return dict(factor_with_rows=np_ ** 3 / 3 + np_ ** 2 * mp, sigma_product=np_ * mp ** 2,
                sigma_factor=attempts * mp ** 3 / 3, draws=2.0 * sp * mp ** 2)


def attempts_of(jitter, sf2):
    return 1 if jitter == 0 else 2 + int(round(np.log10(jitter / sf2))) + 12


h = _lib.Handle(0)


def run(name, X, y, Z, khyp, S):
    h.set_train(X, y)
    rows = []
    for rep in range(reps + 1):                          # rep 0 warms every shape
        t0 = time.perf_counter()
        s, jit = h.gpr_sample(khyp, Z, S, seed=rep)
        wall = (time.perf_counter() - t0) * 1e3
        t = h.timings()
        if rep:
            rows.append(dict(assembly_ms=t['kbuild_ms'], factor_ms=t['factor_ms'], sigma_ms=t['finish_ms'],
                             sampling_ms=t['grad_ms'], total_ms=t['total_ms'], wall_ms=wall))
    med = {k: float(np.median([r[k] for r in rows])) for k in rows[0]}
    n, m = len(X), len(Z)
    att = attempts_of(jit, khyp[-2])
    fl = flops(n, m, S, att)
    total = sum(fl.values())
    r = dict(case=name, n=n, d=X.shape[1], m=m, S=S, jitter=jit, factor_attempts=att, flop=fl, flop_total=total,
             runs=rows, median=med, tflops_overall=total / (med['total_ms'] * 1e-3) / 1e12,
             tflops_sigma_product=fl['sigma_product'] / (med['sigma_ms'] * 1e-3) / 1e12)
    print(json.dumps({k: v for k, v in r.items() if k != 'runs'}), flush=True)
    return r, s


def host_reference(X, y, Z, khyp, S, jitter):
    """Case (a) in numpy / scipy: every stage the device runs, timed on the host."""
    from scipy.linalg import cho_solve, solve_triangular
    from oracle import gpr_oracle
    ell, sf2, sn2 = khyp[:-2], khyp[-2], khyp[-1]
    lh = np.log(np.r_[ell, np.sqrt(sf2), np.sqrt(sn2)])
    t = {}
    t0 = time.perf_counter()
    K = gpr_oracle.kxx(lh, X)
    Ks = gpr_oracle.kxz(lh, X, Z)
    Kzz = gpr_oracle.kxz(lh, Z, Z)
    np.fill_diagonal(Kzz, sf2)
    t['assembly_s'] = time.perf_counter() - t0
    t0 = time.perf_counter()
    L = np.linalg.cholesky(K)
    fz = Ks.T @ cho_solve((L, True), y)
    V = solve_triangular(L, Ks, lower=True)
    t['factor_s'] = time.perf_counter() - t0
    t0 = time.perf_counter()
    Sig = Kzz - V.T @ V
    t['sigma_s'] = time.perf_counter() - t0
    t0 = time.perf_counter()
    Ls = np.linalg.cholesky(Sig + jitter * np.eye(len(Z)))
    E = np.random.default_rng(0).standard_normal((S, len(Z)))
    _ = fz + E @ Ls.T
    t['sampling_s'] = time.perf_counter() - t0
    t['total_s'] = sum(t.values())
    return t, Sig


res = dict(info=gpu_info(), what=__doc__.strip(), host_cpus=os.cpu_count())
h.microbench(0)
res['dmma_peak_tflops'] = h.microbench(0)

X, Y, _ = make_c5()
g = np.linspace(0, 100, 100)
G1, G2 = np.meshgrid(g, g)
Zg = np.column_stack([G1.ravel(), G2.ravel()])
kh_a = np.array([20.0, 20.0, 10.0, 0.25 ** 2])
res['a_S16'], _ = run('a', X, Y, Zg, kh_a, 16)
res['a_S1024'], _ = run('a', X, Y, Zg, kh_a, 1024)
Xc, yc, _, lhc = make_c2()
Zc = make_c2(m=4096)[2]
res['b_S64'], _ = run('b', Xc, yc, Zc, np.r_[np.exp(lhc[:-2]), np.exp(2 * lhc[-2:])], 64)
res['dmma_peak_tflops_after'] = h.microbench(0)

h.set_train(X, Y)
_, cov = h.gpr_predict_full(kh_a, Zg)
ht, Sig = host_reference(X, Y, Zg, kh_a, 16, res['a_S16']['jitter'])
res['a_host'] = dict(ht, max_abs_diff_sigma=float(np.max(np.abs(cov - Sig))), sf2=kh_a[-2])
res['a_host']['host_over_device_S16'] = ht['total_s'] * 1e3 / res['a_S16']['median']['total_ms']
print(json.dumps(res['a_host']), json.dumps(res['info']), 'dmma', res['dmma_peak_tflops'], res['dmma_peak_tflops_after'])
if out:
    with open(out, 'w') as fh:
        json.dump(res, fh, indent=1)
