"""Cost of the classification evidence gradient next to a Newton fit:
   python tools/gpc_grad_once.py [out.json] [reps]

At C3 (bench_configs.make_c3: n = 8192, d = 4) and at n = 4096 (same recipe), warm, in one process: CUDA-event times
of the Newton fit (gpb_gpc_laplace, delta_f = 1e-6, which leaves chol(B) at the mode in place) and of
gpb_gpc_evidence_grad right after it, the stage times the gradient call reports itself, and the rate of its dense
stages - sweep of K W^1/2 through L_B n^3, identity sweep n^3/3, U U^T n^3/3 (n = padded size) - as a fraction of the
DMMA pipe rate measured in the same run (gpb_microbench kind 0)."""
import json
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, '.')
from bench_configs import make_c3  # noqa: E402
from gptest_b200 import _lib  # noqa: E402

out = sys.argv[1] if len(sys.argv) > 1 else None
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clk = [t.strip() for t in q.split(',')]
        return dict(gpu=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:                               # the name from torch at least
        return dict(gpu=torch.cuda.get_device_name(0), power_limit='unknown (%s)' % e)


stream = torch.cuda.Stream()
h = _lib.Handle(0)
h.set_stream(stream.cuda_stream)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    r = fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1), r


def run(n):
    x, y, _, lh = make_c3(n=n)
    d = x.shape[1]
    khyp = np.concatenate([np.exp(lh[:d]), [np.exp(lh[d]) ** 2]])
    h.set_train(x)
    rows = []
    for rep in range(reps + 1):                          # rep 0 warms every shape
        t_fit, (f, lml, iters, trace, jit) = timed(lambda: h.gpc_laplace(y, khyp, link=0, delta_f=1e-6, max_iter=100))
        t_gr, (lml2, g) = timed(h.gpc_evidence_grad)
        st = h.timings()
        if rep:
            rows.append(dict(fit_ms=t_fit, iters=iters, grad_ms=t_gr, grad_dense_ms=st['factor_ms'],
                             grad_rest_ms=st['finish_ms'], grad_refactor_ms=st['kbuild_ms']))
        assert lml2 == lml
    npad = -(-n // 128) * 128
    flops = (1 + 1 / 3 + 1 / 3) * npad ** 3
    med = {k: float(np.median([r[k] for r in rows])) for k in rows[0]}
    return dict(n=n, n_pad=npad, d=d, jitter=jit, lml=lml, grad=g.tolist(), runs=rows, median=med,
                dense_flop=flops, dense_tflops=flops / (med['grad_dense_ms'] * 1e-3) / 1e12,
                grad_over_fit=med['grad_ms'] / med['fit_ms'])


res = dict(info=gpu_info(), what=__doc__.strip())
h.microbench(0)
res['dmma_peak_tflops'] = h.microbench(0)
for n in (4096, 8192):
    r = run(n)
    r['dense_fraction_of_dmma'] = r['dense_tflops'] / res['dmma_peak_tflops']
    res['n%d' % n] = r
    print(json.dumps({k: v for k, v in r.items() if k not in ('runs', 'grad')}), flush=True)
res['dmma_peak_tflops_after'] = h.microbench(0)
print(json.dumps(res['info']), 'dmma', res['dmma_peak_tflops'], res['dmma_peak_tflops_after'])
if out:
    with open(out, 'w') as fh:
        json.dump(res, fh, indent=1)
