"""Same-box A/B of the Laplace and regression entry points of two builds of the library:
   GPB200_LIB=<lib> python tools/laplace_ab.py run OUT_DIR [reps]
   python tools/laplace_ab.py compare A_DIR B_DIR

run: every Laplace entry point on seeded inputs - the preference calls at C4 (bench_configs.make_c4: n = 4096,
P = 32768, d = 6), the classification calls at C3 (make_c3: n = 8192, d = 4), and both at a small odd n (333) - and
every regression entry point: the covariance calls, the likelihood with and without its gradient (n = 333, 2048 and
9000, both sides of the fuse_min_tiles switch), predict, the joint posterior and samples, the batched likelihood with
ragged chunks (batch_chunk 4), the growing training set (thin, split-k and multi-tile appends, a non-positive-definite
append, predict), the dense factorisation hooks, and a preference fit that stays usable across growing-set calls;
the regression calls for each covariance kind (0, 1, 2) that takes one.  Saves
every output to OUT_DIR/outputs.npz and, per call, the launch_count() increment, which timings() slots are non-zero
and the message of a refused call to OUT_DIR/meta.json.  Then CUDA-event times over `reps` warm repeats of the calls
bench.py times (c3_gpc_n8192_d4: the probit fit and predict; c4_gppref_n4096_p32768: the reference-semantics fit) and
of the gradients as tools/gpc_grad_once.py and tools/pref_grad_once.py time them; medians into meta.json.
compare: np.array_equal on every output (NaN equal to NaN), equal launch counts, timing slots and messages; exit status 1
otherwise."""
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench_configs import make_c3, make_c4  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clk = [t.strip() for t in q.split(',')]
        return dict(gpu=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:
        return dict(gpu='unknown', power_limit='unknown (%s)' % e)


def run(out_dir, reps):
    import torch
    from gptest_b200 import _lib
    stream = torch.cuda.Stream()
    h = _lib.Handle(0)
    h.set_stream(stream.cuda_stream)
    outputs, meta = {}, dict(lib=_lib.LIB_PATH, info=gpu_info(), calls={}, times={})

    def call(name, fn):
        l0 = h.launch_count()
        try:
            r = fn()
            err = None
        except (_lib.GpbError, np.linalg.LinAlgError) as e:
            r, err = (), str(e)
        t = list(h.timings().values())
        meta['calls'][name] = dict(launches=h.launch_count() - l0, slots=[i for i, v in enumerate(t) if v != 0],
                                   error=err)
        for i, a in enumerate(r if isinstance(r, tuple) else (r,)):
            outputs['%s/%d' % (name, i)] = np.asarray(a)
        return r

    def timed(name, fn, before=None):
        ts = []
        for rep in range(reps + 1):                     # rep 0 warms every shape
            if before:
                before()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            if rep:
                ts.append(e0.elapsed_time(e1))
        meta['times'][name] = dict(median_ms=float(np.median(ts)), ms=ts)
        print('%-28s %9.3f ms  (%s)' % (name, np.median(ts), ' '.join('%.3f' % t for t in ts)), flush=True)

    def pref_case(tag, n, P):
        x, uvi, y, lh = make_c4(n=n, P=P)
        d = x.shape[1]
        khyp = np.r_[np.exp(lh[:d]), np.exp(lh[d]) ** 2]
        sigma = float(np.exp(lh[-1]))
        rng = np.random.default_rng(n)
        za, zb = rng.random((1024, d)), rng.random((1024, d))
        h.set_train(x)
        fit0 = lambda: h.pref_laplace(uvi, y, khyp, sigma=1.0, delta_f=1e-6, max_iter=500)          # bench.py
        fit1 = lambda: h.pref_laplace(uvi, y, khyp, sigma=sigma, delta_f=1e-9, max_iter=100, grad_mode=1)
        f = call(tag + '/laplace_g0', fit0)[0]
        call(tag + '/evidence_g0', h.pref_evidence)
        call(tag + '/evidence_grad_g0', h.pref_evidence_grad)                     # refused: grad_mode 0
        call(tag + '/predict', lambda: h.pref_predict(za))
        call(tag + '/predict_zb', lambda: h.pref_predict(za, zb))
        call(tag + '/laplace_g1', fit1)
        call(tag + '/evidence_grad', h.pref_evidence_grad)                        # factors G at the mode itself
        call(tag + '/evidence_after_grad', h.pref_evidence)
        call(tag + '/predict_zb_after_grad', lambda: h.pref_predict(za, zb))
        call(tag + '/derivatives_g0', lambda: h.pref_derivatives(uvi, y, f, sigma=1.0, grad_mode=0))
        call(tag + '/derivatives_g1', lambda: h.pref_derivatives(uvi, y, f, sigma=sigma, grad_mode=1))
        K = h.kxx(np.r_[khyp, 0.0]) + 1e-6 * np.eye(n)
        iK = np.linalg.inv(K)
        logdetK = float(np.sum(np.log(np.diag(np.linalg.cholesky(K)))))
        call(tag + '/log_marginal', lambda: h.pref_log_marginal(uvi, y, f, iK, logdetK, sigma=sigma))
        timed(tag + '/fit', fit0)
        timed(tag + '/grad', h.pref_evidence_grad, before=lambda: (fit1(), h.pref_evidence()))

    def gpc_case(tag, n):
        x, y, z, lh = make_c3(n=n)
        d = x.shape[1]
        khyp = np.r_[np.exp(lh[:d]), np.exp(lh[d]) ** 2]
        h.set_train(x)
        for link in (0, 1):
            fit = lambda: h.gpc_laplace(y, khyp, link=link, delta_f=1e-6)                         # bench.py
            call('%s/laplace_link%d' % (tag, link), fit)
            call('%s/predict_link%d' % (tag, link), lambda: h.gpc_predict(z))
            call('%s/evidence_grad_link%d' % (tag, link), h.gpc_evidence_grad)
            call('%s/predict_after_grad_link%d' % (tag, link), lambda: h.gpc_predict(z))
        fit = lambda: h.gpc_laplace(y, khyp, link=0, delta_f=1e-6)
        call(tag + '/laplace_max_iter', lambda: h.gpc_laplace(y, khyp, link=0, delta_f=1e-6, max_iter=1))
        call(tag + '/evidence_grad_max_iter', h.gpc_evidence_grad)                # refused: not converged
        timed(tag + '/fit', fit)
        timed(tag + '/predict', lambda: h.gpc_predict(z), before=fit)
        timed(tag + '/grad', h.gpc_evidence_grad, before=fit)

    def gpr_case(tag, n, d=4, full=True):
        rng = np.random.default_rng(1000 + n)
        x = rng.random((n, d))
        y = np.sin(x @ rng.standard_normal(d)) + 0.1 * rng.standard_normal(n)
        z = rng.random((300, d))
        khyp = np.r_[np.full(d, 0.4), 1.3, 0.01]
        kb = np.c_[rng.uniform(0.2, 0.8, (10, d)), rng.uniform(0.5, 2.0, 10), rng.uniform(0.005, 0.05, 10)]
        h.set_train(x, y)
        for kind in (0, 1, 2):
            t = '%s/k%d/' % (tag, kind)
            call(t + 'nlml', lambda: h.gpr_nlml(khyp, mean=0.1, kind=kind))
            call(t + 'nlml_grad', lambda: h.gpr_nlml(khyp, mean=0.1, want_grad=True, kind=kind))
            if not full:
                continue
            call(t + 'kxx', lambda: h.kxx(khyp, kind=kind))
            call(t + 'kxx_clip', lambda: h.kxx(khyp, flags=1, kind=kind))
            k_dev = torch.empty((n, n), dtype=torch.float64, device='cuda')
            call(t + 'kxx_dev', lambda: (h.kxx_dev(khyp, k_dev.data_ptr(), kind=kind), stream.synchronize(),
                                         k_dev.cpu().numpy())[2])
            call(t + 'kxz', lambda: h.kxz(khyp, z, kind=kind))
            call(t + 'predict', lambda: h.gpr_predict(khyp, z, mean=0.1, kind=kind))
            call(t + 'predict_full', lambda: h.gpr_predict_full(khyp, z, mean=0.1, kind=kind))
            call(t + 'predict_full_noisy', lambda: h.gpr_predict_full(khyp, z, mean=0.1, kind=kind, noisy=True))
            call(t + 'sample', lambda: h.gpr_sample(khyp, z, 64, seed=7, mean=0.1, kind=kind))
            h.set_option('batch_chunk', 4)
            call(t + 'batched', lambda: h.gpr_nlml_batched(kb, mean=0.1, kind=kind))
            call(t + 'batched_grad', lambda: h.gpr_nlml_batched(kb, mean=0.1, want_grad=True, kind=kind))
            h.set_option('batch_chunk', 0)
        if full:
            call(tag + '/sqdist', lambda: h.sqdist(z))

    def grow_case(tag, kind):
        rng = np.random.default_rng(77 + kind)
        d = 3
        x = rng.random((1500, d))
        y = np.cos(x @ rng.standard_normal(d))
        z = rng.random((2500, d))                                # two prediction passes
        h.grow_begin(np.r_[np.full(d, 0.3), 1.1, 0.02], d, 2000, mean=0.05, kind=kind)
        for name, a, b in (('multi', 0, 1100), ('thin_splitk', 1100, 1103), ('thin', 1103, 1108), ('multi2', 1108, 1500)):
            call('%s/k%d/append_%s' % (tag, kind, name), lambda: h.grow_append(x[a:b], y[a:b]))
            call('%s/k%d/predict_%s' % (tag, kind, name), lambda: h.grow_predict(z))
        h.grow_begin(np.r_[np.full(d, 0.3), 1.1, -0.5], d, 100, kind=kind)   # sf2 + sn2 > 0, [[.6, 1.1], [1.1, .6]] is not
        call('%s/k%d/append_one' % (tag, kind), lambda: h.grow_append(x[:1], y[:1]))
        call('%s/k%d/append_not_pd' % (tag, kind), lambda: h.grow_append(x[:1], y[:1]))        # the same point again
        call('%s/k%d/predict_after_not_pd' % (tag, kind), lambda: h.grow_predict(z[:10]))    # refused

    def dense_case(tag):
        rng = np.random.default_rng(5)
        for n in (333, 517):
            a = rng.standard_normal((n, n))
            call('%s/potrf_n%d' % (tag, n), lambda: h.potrf(a @ a.T + n * np.eye(n)))
        a = rng.standard_normal((512, 512))
        spd = torch.zeros((512, 576), dtype=torch.float64, device='cuda')
        spd[:, :512] = torch.from_numpy(a @ a.T + 512 * np.eye(512)).cuda()
        stream.wait_stream(torch.cuda.current_stream())
        call(tag + '/potrf_dev', lambda: (h.potrf_dev(spd.data_ptr(), 512, 576), stream.synchronize(), spd.cpu().numpy())[::2])

    def pref_then_grow(tag):
        x, uvi, y, lh = make_c4(n=333, P=2664)
        d = x.shape[1]
        khyp = np.r_[np.exp(lh[:d]), np.exp(lh[d]) ** 2]
        za = np.random.default_rng(9).random((100, d))
        h.set_train(x)
        call(tag + '/laplace', lambda: h.pref_laplace(uvi, y, khyp, sigma=1.0, delta_f=1e-6, max_iter=500))
        h.grow_begin(np.r_[np.full(d, 0.5), 1.0, 0.01], d, 400)
        call(tag + '/grow_append', lambda: h.grow_append(x[:200], np.sin(x[:200, 0])))
        call(tag + '/grow_predict', lambda: h.grow_predict(za))
        call(tag + '/predict_after_grow', lambda: h.pref_predict(za))

    for kind in (0, 1, 2):
        grow_case('grow', kind)
    dense_case('dense')
    pref_then_grow('pref_grow')
    gpr_case('gpr_n333', 333)
    gpr_case('gpr_n2048', 2048)
    gpr_case('gpr_n9000', 9000, full=False)
    h._kind(0)
    pref_case('pref_n333', 333, 2664)
    gpc_case('gpc_n333', 333)
    pref_case('pref_c4', 4096, 32768)
    gpc_case('gpc_c3', 8192)
    os.makedirs(out_dir, exist_ok=True)
    np.savez(os.path.join(out_dir, 'outputs.npz'), **outputs)
    with open(os.path.join(out_dir, 'meta.json'), 'w') as fh:
        json.dump(meta, fh, indent=1)
    print(json.dumps(meta['info']))


def compare(a_dir, b_dir):
    oa, ob = np.load(os.path.join(a_dir, 'outputs.npz')), np.load(os.path.join(b_dir, 'outputs.npz'))
    ma, mb = (json.load(open(os.path.join(p, 'meta.json'))) for p in (a_dir, b_dir))
    bad = []
    if sorted(oa.files) != sorted(ob.files):
        bad.append('output sets differ: %s' % sorted(set(oa.files) ^ set(ob.files)))
    bad += ['output %s differs' % k for k in sorted(set(oa.files) & set(ob.files))
            if not np.array_equal(oa[k], ob[k], equal_nan=oa[k].dtype.kind in 'fc')]
    bad += ['call %s: %s vs %s' % (k, ma['calls'][k], mb['calls'].get(k)) for k in ma['calls']
            if ma['calls'][k] != mb['calls'].get(k)]
    for k in ma['times']:
        print('%-28s %9.3f %9.3f ms' % (k, ma['times'][k]['median_ms'], mb['times'][k]['median_ms']))
    print('%d outputs, %d calls compared: %s' % (len(oa.files), len(ma['calls']), 'identical' if not bad else 'DIFFERENT'))
    for b in bad:
        print('  ' + b)
    return 1 if bad else 0


if __name__ == '__main__':
    if sys.argv[1] == 'run':
        run(sys.argv[2], int(sys.argv[3]) if len(sys.argv) > 3 else 5)
    else:
        sys.exit(compare(sys.argv[2], sys.argv[3]))
