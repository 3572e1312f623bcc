"""Cost of gradients with respect to the input points, on a C2-style problem (Matern-5/2 + White, points uniform in
[0, 10]^3, one key):

  * lgp_gram_iso_xvjp against lgp_gram_iso_vjp on the same G: n = 20000 with the lower triangle of a symmetric G and b
    (the fused logML route), n = m = 10000 with a dense G (the assembled route);
  * the logML + gradient step at n = 20000: hyperparameters only, against hyperparameters and points;
  * optionally bench.py's step in this tree and in another checkout (--parent-tree), alternated.

  python tools/bench_point_grads.py --out profiles/bench_point_grads_r1.json [--parent-tree DIR]

Times are CUDA events over many launches (kernels) or a host clock around work that ends in a device synchronise
(steps), after a warm-up of the same shapes.  The 3.2 GB G of n = 20000 does not fit the 126 MB L2.  The card's name
and power limit are read in the same run and stored beside the numbers."""
import argparse
import json
import pathlib
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import lsqfitgp_b200 as lgp  # noqa: E402
from lsqfitgp_b200 import _lib, _ops  # noqa: E402

f64 = torch.float64


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        out = f'unknown ({e})'
    return out


def kernel_ms(fn, reps, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def step_s(fn, reps, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t)
    return dict(median=float(np.median(ts)), min=float(np.min(ts)), max=float(np.max(ts)))


DESCS = [dict(kind=_lib.K_MATERNP, term=0, dimmask=7, ipar=2, par0=1e-30, scale_x=1.5, scale_y=1.5, amp=1.0),
         dict(kind=_lib.K_WHITE, term=1, dimmask=7, amp=0.01)]


def kernels(n_sym, n_dense, reps):
    rng = np.random.default_rng(0)
    out = {}
    x = torch.tensor(rng.uniform(0, 10, (3, n_sym)), dtype=f64, device='cuda')
    G = _ops.aligned_empty(n_sym, n_sym, x.device)
    G.normal_()
    b = torch.randn(n_sym, dtype=f64, device='cuda')
    out['symlower'] = dict(
        n=n_sym, gram_iso_vjp_ms=kernel_ms(lambda: _ops.gram_iso_vjp(DESCS, x, G, b), reps),
        gram_iso_xvjp_ms=kernel_ms(lambda: _ops.gram_iso_xvjp(DESCS, x, None, G, b, symlower=True), reps))
    del G
    x = x[:, :n_dense].contiguous()
    y = torch.tensor(rng.uniform(0, 10, (3, n_dense)), dtype=f64, device='cuda')
    G = _ops.aligned_empty(n_dense, n_dense, x.device)
    G.normal_()
    D = _ops.aligned_empty(n_dense, n_dense, x.device)
    tx, ty = torch.randn_like(x), torch.randn_like(y)
    out['dense'] = dict(
        n=n_dense, m=n_dense, gram_iso_vjp_general_ms=kernel_ms(lambda: _ops.gram_iso_vjp_general(DESCS, x, y, G), reps),
        gram_iso_xvjp_ms=kernel_ms(lambda: _ops.gram_iso_xvjp(DESCS, x, y, G), reps),
        gram_iso_jvp_ms=kernel_ms(lambda: _ops.gram_iso_jvp(DESCS, x, y, np.ones((2, 3)), out=D), reps),
        gram_iso_xjvp_ms=kernel_ms(lambda: _ops.gram_iso_xjvp(DESCS, x, y, tx, ty, D, accumulate=True), reps))
    for v in out.values():
        k = [key for key in v if key.startswith('gram_iso_vjp')][0]
        v['xvjp_over_vjp'] = v['gram_iso_xvjp_ms'] / v[k]
    del G, D
    torch.cuda.empty_cache()
    return out


def steps(n, reps):
    rng = np.random.default_rng(1)
    X = rng.uniform(0, 10, (3, n))
    y = np.sin(X[0]) + np.cos(X[1]) * X[2] / 10 + 0.1 * rng.standard_normal(n)
    q0 = torch.tensor([0.0, np.log(1.5), np.log(0.01)], dtype=f64)

    def ml(q, pts):
        k = torch.exp(q[0]) * lgp.Matern(nu=2.5, scale=torch.exp(q[1])) + torch.exp(q[2]) * lgp.White()
        return lgp.GP(k, checkpos=False, checksym=False).addx(pts, 'data').marginal_likelihood({'data': y})

    def hyper_only():
        q = q0.clone().requires_grad_(True)
        return torch.autograd.grad(ml(q, lgp.StructuredArray({'f0': X[0], 'f1': X[1], 'f2': X[2]})), q)

    Xt = torch.tensor(X, dtype=f64, device='cuda')

    def with_points():
        q = q0.clone().requires_grad_(True)
        t = Xt.clone().requires_grad_(True)
        return torch.autograd.grad(ml(q, lgp.StructuredArray({'f0': t[0], 'f1': t[1], 'f2': t[2]})), (q, t))
    # alternate the two, so that drifts of the shared host affect both alike
    a, b = [], []
    for _ in range(reps):
        a.append(step_s(hyper_only, 1)['median'])
        b.append(step_s(with_points, 1)['median'])
    ga, = hyper_only()
    gb, gt = with_points()
    return dict(n=n, hyper_only_s=dict(median=float(np.median(a)), min=min(a), max=max(a)),
                hyper_and_points_s=dict(median=float(np.median(b)), min=min(b), max=max(b)),
                added_ms=1e3 * (float(np.median(b)) - float(np.median(a))),
                hyper_gradient_max_abs_diff=float(torch.max(torch.abs(ga - gb))),
                point_gradient_norm=float(torch.linalg.norm(gt)))


def bench_step(tree, steps_, warmup):
    cmd = [sys.executable, 'bench.py', '--gpus', '1', '--steps', str(steps_), '--warmup', str(warmup), '--no-cpu-baseline']
    out = subprocess.run(cmd, cwd=tree, capture_output=True, text=True, timeout=3000)
    line = [ln for ln in out.stdout.splitlines() if ln.startswith('{')]
    if out.returncode or not line:
        return dict(error=out.stderr[-2000:])
    return json.loads(line[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--n-sym', type=int, default=20000)
    ap.add_argument('--n-dense', type=int, default=10000)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--parent-tree', default=None, help='another checkout (built) whose bench.py step to compare')
    ap.add_argument('--bench-steps', type=int, default=5)
    ap.add_argument('--bench-warmup', type=int, default=3)
    ap.add_argument('--bench-rounds', type=int, default=2)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_point_grads needs a GPU'
    torch.cuda.set_device(0)
    res = dict(card=card(), problem='Matern(nu=2.5) + White, 3 fields, points uniform in [0, 10]^3, one key')
    res['kernels'] = kernels(args.n_sym, args.n_dense, reps=10)
    print(json.dumps(res['kernels']), flush=True)
    res['step'] = steps(args.n_sym, args.reps)
    print(json.dumps(res['step']), flush=True)
    if args.parent_tree:
        torch.cuda.empty_cache()
        runs = []
        for _ in range(args.bench_rounds):
            for name, tree in (('parent', args.parent_tree), ('this', str(ROOT))):
                r = bench_step(tree, args.bench_steps, args.bench_warmup)
                runs.append(dict(tree=name, result=r))
                print(name, json.dumps(r)[:400], flush=True)
        res['bench_py'] = runs
    res['card_after'] = card()
    pathlib.Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    pathlib.Path(args.out).write_text(json.dumps(res, indent=1))


if __name__ == '__main__':
    main()
