"""Cost of the derivative blocks (lgp_gram_iso_deriv and its VJP) next to the plain Gram kernels, and of one logML +
gradient evaluation with gradient observations against plain observations of the same total size.

  python tools/bench_deriv.py --out result.json

Times are CUDA events around back-to-back launches after a warm-up.  Prints the card name and power limit beside the
numbers; writes one JSON file."""
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


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        out = f'unknown ({e})'
    return out


def events(fn, reps, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def blocks(n, reps):
    rng = np.random.default_rng(0)
    X = torch.from_numpy(rng.uniform(0, 10, (3, n))).cuda()
    Y = torch.from_numpy(rng.uniform(0, 10, (3, n))).cuda()
    out = _ops.aligned_empty(n, n, X.device)
    G = _ops.as_aligned(torch.randn(n, n, dtype=torch.float64, device='cuda'))
    labels = ['f0', 'f1', 'f2']
    rows = []
    for name, k in (('matern52', lgp.Matern(nu=2.5, scale=1.5)), ('expquad', lgp.ExpQuad(scale=1.5))):
        descs, _ = k._descriptor(labels)
        cases = {
            'plain_fast': lambda: _ops.gram_iso(descs, X, Y, out=out),
            'plain_general': lambda: _ops.gram_iso(descs, X, Y, out=out, flags=_lib.GRAM_GENERAL),
            'deriv_x': lambda: _ops.gram_iso_deriv(descs, X, Y, 0, -1, out=out),
            'deriv_xy': lambda: _ops.gram_iso_deriv(descs, X, Y, 0, 1, out=out),
            'plain_general_vjp': lambda: _ops.gram_iso_vjp_general(descs, X, Y, G),
            'deriv_x_vjp': lambda: _ops.gram_iso_deriv_vjp(descs, X, Y, 0, -1, G),
            'deriv_xy_vjp': lambda: _ops.gram_iso_deriv_vjp(descs, X, Y, 0, 1, G),
        }
        for case, fn in cases.items():
            ms = events(fn, reps)
            ent = n * n
            written = 0 if case.endswith('vjp') else 8 * ent
            rows.append(dict(kernel=name, block=case, n=n, ms=ms, entries_per_s=ent / ms * 1e3,
                             GB_per_s_written=written / ms * 1e-6))
            print(f'{name:9s} {case:18s} n=m={n}: {ms:8.3f} ms  {ent / ms * 1e-6:8.2f} Gentries/s  '
                  f'{written / ms * 1e-6:8.1f} GB/s written', flush=True)
    return rows


def logml_step(npts, reps, deriv):
    rng = np.random.default_rng(1)
    X = rng.uniform(0, 10, (npts, 3))
    x = lgp.unstructured_to_structured(X, names=['a', 'b', 'c'])
    if deriv:
        keys = [('f', None), ('da', 'a'), ('db', 'b'), ('dc', 'c')]
    else:
        half = npts // 2
        keys = [('p0', slice(0, half)), ('p1', slice(half, npts))]
    y, gc = {}, {}
    for k, _ in keys:
        m = npts if deriv else npts // 2
        y[k] = rng.standard_normal(m)
    for k1, _ in keys:
        for k2, _ in keys:
            m1, m2 = len(y[k1]), len(y[k2])
            gc[k1, k2] = 0.01 * np.eye(m1) if k1 == k2 else np.zeros((m1, m2))
    theta = torch.tensor([np.log(1.5), 0.0], dtype=torch.float64, requires_grad=True)

    def build():
        k = torch.exp(theta[1]) ** 2 * lgp.Matern(nu=2.5, scale=torch.exp(theta[0]))
        gp = lgp.GP(k, checkpos=False, checksym=False)
        for key, spec in keys:
            gp = gp.addx(x, key, deriv=spec) if deriv else gp.addx(x[spec], key)
        return gp

    def step():
        ml = build().marginal_likelihood(y, gc)
        torch.autograd.grad(ml, theta)

    def gram_only():
        with torch.no_grad():
            build()._assemblecovblocks([k for k, _ in keys])
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) / reps * 1e3
    gms = events(gram_only, reps)
    N = sum(len(v) for v in y.values())
    print(f'logML+grad {"deriv" if deriv else "plain"} N={N}: {ms:.1f} ms/step (assembled Gram blocks alone {gms:.1f} ms)',
          flush=True)
    return dict(case='deriv' if deriv else 'plain', N=N, ms_per_step=ms, gram_assembly_ms=gms)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='bench_deriv.json')
    ap.add_argument('--n', type=int, default=10000)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--points', type=int, default=5000)
    ap.add_argument('--steps', type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_deriv.py needs a GPU')
    dev = card()
    print('card, power limit:', dev, flush=True)
    res = dict(card=dev, blocks=blocks(a.n, a.reps))
    res['steps'] = [logml_step(4 * a.points, a.steps, False), logml_step(a.points, a.steps, True)]
    res['step_ratio'] = res['steps'][1]['ms_per_step'] / res['steps'][0]['ms_per_step']
    print(f"step ratio deriv / plain: {res['step_ratio']:.3f}", flush=True)
    pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    pathlib.Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == '__main__':
    main()
