"""Time the device part of one logML+gradient evaluation (Gram, factor + inverse on two streams, solves, Gram-VJP) at n:
mean of `reps` after a warm-up; prints the separate phases as well.  Env switches (LGP_PANEL_BLOCKS ...) are read once."""
import sys
import numpy as np
import torch
sys.path.insert(0, '.')
from lsqfitgp_b200 import _lib, _ops
n = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 4
fused = not (len(sys.argv) > 3 and sys.argv[3] == 'unfused')
dev = torch.device('cuda:0')
rng = np.random.default_rng(2002)
X = rng.uniform(0, 10, (n, 3))
y = np.sin(X[:, 0]) + np.cos(X[:, 1]) * X[:, 2] / 10 + 0.1 * rng.standard_normal(n)
xd = torch.tensor(np.ascontiguousarray(X.T)).to(dev)
yd = torch.tensor(y).to(dev)
descs = [dict(kind=_lib.K_MATERNP, term=0, dimmask=7, ipar=2, par0=0.0, scale_x=1.5, scale_y=1.5, amp=1.0),
         dict(kind=_lib.K_WHITE, term=1, dimmask=7, amp=0.01)]
K = _ops.aligned_empty(n, n, dev)
side = torch.cuda.Stream(dev)
def step():
    main = torch.cuda.current_stream()
    if fused:
        st, Kinv = _ops.gram_chol_factor(descs, xd, side=side)
    else:
        _ops.gram_iso(descs, xd, xd, out=K, symmetric=True)
        st, Kinv = _ops.chol_factor_inverse(K, side)
    a = _ops.chol_solve(st, yd[:, None], False)
    ldq = _ops.chol_logdet_quad(st, a[:, 0].contiguous())
    b = _ops.chol_solve(st, a, True, inplace=True)
    main.wait_stream(side)
    vjp = _ops.gram_iso_vjp(descs, xd, Kinv, b[:, 0].contiguous())
    return ldq, vjp
def timeit(fn, reps):
    fn(); torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); out = fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.mean(ts)), out
t, (ldq, vjp) = timeit(step, reps)
_ops.gram_iso(descs, xd, xd, out=K, symmetric=True)
tf, st = timeit(lambda: _ops.chol_factor(K), reps)
ti, _ = timeit(lambda: _ops.chol_inverse(st), reps)
print(f'n={n} fused={fused}: step {t:.2f} ms ({n**3/t/1e9:.2f} TF) | factor alone {tf:.2f} | inverse alone {ti:.2f} | logdet {float(ldq[0]):.10g} vjp0 {float(vjp.ravel()[0]):.8g}')
