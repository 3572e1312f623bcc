"""Cost of the second derivatives of the marginal likelihood on a C2-style problem (Matern-5/2 + White, three
hyperparameters: log amplitude, log scale, log noise amplitude), at n = 5000, 10000, 20000:

  * the gradient step: logML and its gradient (one reverse sweep, the first-order path);
  * the full 3 x 3 Hessian: torch.autograd.functional.hessian through the twice-differentiable nodes;
  * lgp_gram_iso_hvp against lgp_gram_iso_vjp (general kernel, dense G) on the same G.

  python tools/bench_hessian.py --out profiles/bench_hessian_r1.json

Times are CUDA events (kernels) or a host clock around work that ends in a device synchronise (steps), after a warm-up
of the same shapes.  The card's name and power limit are read in the same run and stored beside the numbers."""
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
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def problem(n, seed=0):
    rng = np.random.default_rng(seed)
    X = rng.uniform(0, 10, (n, 3))
    y = np.sin(X[:, 0]) + np.cos(X[:, 1]) * X[:, 2] / 10 + 0.1 * rng.standard_normal(n)
    return lgp.unstructured_to_structured(X, names=['f0', 'f1', 'f2']), y


def objective(xs, y):
    def f(q):
        k = torch.exp(q[0]) * lgp.Matern(nu=2.5, scale=torch.exp(q[1])) + torch.exp(q[2]) * lgp.White()
        return -lgp.GP(k, checkpos=False, checksym=False).addx(xs, 'data').marginal_likelihood({'data': y})
    return f


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sizes', type=int, nargs='+', default=[5000, 10000, 20000])
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', required=True)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_hessian needs a GPU'
    torch.cuda.set_device(0)
    res = dict(card=card(), problem='Matern(nu=2.5) + White, 3 hyperparameters (log amp, log scale, log noise), '
               'points uniform in [0, 10]^3', runs=[])
    q0 = torch.tensor([0.0, np.log(1.5), np.log(0.01)], dtype=f64)
    for n in args.sizes:
        xs, y = problem(n)
        f = objective(xs, y)

        def grad_step():
            q = q0.clone().requires_grad_(True)
            g, = torch.autograd.grad(f(q), q)
            return g

        def hess_step():
            return torch.autograd.functional.hessian(f, q0)
        g = step_s(grad_step, args.reps)
        h = step_s(hess_step, args.reps)
        H = hess_step().numpy()

        # the two contractions on the same dense G, general kernel
        descs = [dict(kind=_lib.K_MATERNP, term=0, dimmask=7, ipar=2, par0=1e-30, scale_x=1.5, scale_y=1.5, amp=1.0),
                 dict(kind=_lib.K_WHITE, term=1, dimmask=7, amp=0.01)]
        xd = torch.tensor(np.stack([xs[k] for k in ('f0', 'f1', 'f2')]), dtype=f64, device='cuda')
        G = _ops.aligned_empty(n, n, xd.device)
        G.normal_()
        tan = np.array([[0.3, -0.7, 0.0], [0.5, 0.0, 0.0]])
        reps = max(2, int(4e9 // (n * n)))
        vjp_ms = kernel_ms(lambda: _ops.gram_iso_vjp_general(descs, xd, xd, G), reps)
        hvp_ms = kernel_ms(lambda: _ops.gram_iso_hvp(descs, xd, xd, G, tan), reps)
        del G
        run = dict(n=n, grad_step_s=dict(zip(('median', 'min', 'max'), g)),
                   hessian_s=dict(zip(('median', 'min', 'max'), h)), hessian=H.tolist(),
                   gram_iso_vjp_general_ms=vjp_ms, gram_iso_hvp_ms=hvp_ms, hvp_over_vjp=hvp_ms / vjp_ms,
                   floor_hessian_gemm_s_at_37tflops=3 * 3 * n ** 3 / 37e12)
        print(json.dumps(run), flush=True)
        res['runs'].append(run)
        torch.cuda.empty_cache()
    res['card_after'] = card()
    pathlib.Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    pathlib.Path(args.out).write_text(json.dumps(res, indent=1))


if __name__ == '__main__':
    main()
