"""Derivatives with respect to the input points without a GPU: the oracle's dK/dx (oracle/xgrad.py) against complex-step
differentiation (h = 1e-200, exact to rounding) of the oracle's Gram matrix and against mpmath differentiation for the
cores that are not analytic in a complex step (Matern of real order, Cauchy with alpha < 2), the oracle's gradient of
-logML with respect to the points against the complex step of the oracle's -logML, and the columns of points given as
torch tensors, dictionaries of tensors and StructuredArrays of tensors against those of the same numpy points."""
import numpy as np
import pytest
import torch

from lsqfitgp_b200 import _array
from oracle import gp as ogp, xgrad as ox

import mpmath  # noqa: E402

H = 1e-200


def _points(ndim, n, m, seed, s=1.0):
    rng = np.random.default_rng(seed)
    x = rng.uniform(0, 3, (ndim, n)) * s
    y = rng.uniform(0, 3, (ndim, m)) * s
    y[:, :2] = x[:, :2]          # coincident pairs: the derivative is 0 there
    return x, y


def _cs_gram(terms, x, y):
    """ complex step of the oracle's Gram matrix: (dK/dx, dK/dy), each (ndim, n, m); K_ij depends on x only through x_i,
    so one step of a whole field gives the derivative of every entry """
    ndim = x.shape[0]
    dx = np.empty((ndim, x.shape[1], y.shape[1]))
    dy = np.empty_like(dx)
    for d in range(ndim):
        e = np.zeros(x.shape, complex)
        e[d] = 1j * H
        dx[d] = ogp.gram(terms, x + e, y.astype(complex)).imag / H
        e = np.zeros(y.shape, complex)
        e[d] = 1j * H
        dy[d] = ogp.gram(terms, x.astype(complex), y + e).imag / H
    return dx, dy


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


ANALYTIC = {
    'expquad': [(1.3, [dict(kind='expquad', scale=1.7)])],
    'cauchy2': [(0.7, [dict(kind='cauchy', alpha=2, beta=1.4, scale=1.2)])],
    **{f'maternp{p}': [(0.9, [dict(kind='maternp', p=p, scale=1.1)])] for p in (1, 2, 3)},
    'product_partial_dims': [(0.8, [dict(kind='expquad', dims=[0], scale=1.5),
                                    dict(kind='maternp', p=2, dims=[1, 2], scale=0.9)]),
                             (0.3, [dict(kind='cauchy', alpha=2, beta=0.8, dims=[2], scale=2.0)])],
    'scale_loc_pairs': [(1.2, [dict(kind='maternp', p=1, scale=(1.3, 0.9), loc=(0.2, -0.1))]),
                        (0.4, [dict(kind='expquad', scale=(0.7, 1.6), loc=0.3)])],
}


@pytest.mark.parametrize('name', sorted(ANALYTIC))
def test_oracle_xgrad_vs_complex_step(name):
    terms = ANALYTIC[name]
    x, y = _points(3, 9, 7, 1)
    dx, dy = ox.gram_xgrad(terms, x, y)
    cx, cy = _cs_gram(terms, x, y)
    assert _rel(dx, cx) < 1e-14 and _rel(dy, cy) < 1e-14, (_rel(dx, cx), _rel(dy, cy))
    if name != 'scale_loc_pairs':   # coincident pairs (same loc and scale on both sides): exactly 0
        assert np.all(dx[:, :2, :2].diagonal(axis1=1, axis2=2) == 0)


def _mp_core(f, r2):
    kind = f['kind']
    if kind == 'matern':
        nu = mpmath.mpf(f['nu'])
        if r2 == 0:
            return mpmath.mpf(1)
        z = mpmath.sqrt(2 * nu * r2)
        return 2 ** (1 - nu) / mpmath.gamma(nu) * z ** nu * mpmath.besselk(nu, z)
    if kind == 'cauchy':
        a, b = mpmath.mpf(f['alpha']), mpmath.mpf(f['beta'])
        return (1 + r2 ** (a / 2) / b) ** (-b / a)
    if kind == 'expquad':
        return mpmath.exp(-r2 / 2)
    raise KeyError(kind)


def _mp_entry(terms, x, y, i, j):
    """ K_ij as an mpmath function of (x_{.,i}) """
    def k(xi):
        tot = mpmath.mpf(0)
        for amp, factors in terms:
            prod = mpmath.mpf(amp)
            for f in factors:
                dims = range(x.shape[0]) if f.get('dims') is None else f['dims']
                s = mpmath.mpf(f.get('scale', 1.0))
                r2 = sum((xi[d] / s - mpmath.mpf(y[d, j]) / s) ** 2 for d in dims)
                prod *= _mp_core(f, r2)
            tot += prod
        return tot
    return k


REAL_ORDER = {
    **{f'matern{nu}': [(1.1, [dict(kind='matern', nu=nu, scale=1.7)])] for nu in (0.3, 0.7, 1.3, 4.2)},
    **{f'cauchy{a}': [(0.7, [dict(kind='cauchy', alpha=a, beta=1.4, scale=1.3)])] for a in (0.5, 1.0, 1.7)},
    'matern_times_expquad': [(0.6, [dict(kind='matern', nu=1.3, dims=[0, 1], scale=1.2),
                                    dict(kind='expquad', dims=[1], scale=0.8)])],
}


@pytest.mark.parametrize('name', sorted(REAL_ORDER))
def test_oracle_xgrad_vs_mpmath(name):
    terms = REAL_ORDER[name]
    x, y = _points(2, 5, 4, 2)
    dx, _ = ox.gram_xgrad(terms, x, y)
    mpmath.mp.dps = 40
    worst = 0.0
    for i, j in [(0, 2), (2, 3), (3, 1), (4, 0), (1, 3)]:
        k = _mp_entry(terms, x, y, i, j)
        for d in range(x.shape[0]):
            def kd(t, d=d):
                xi = [mpmath.mpf(v) for v in x[:, i]]
                xi[d] = t
                return k(xi)
            ref = float(mpmath.diff(kd, mpmath.mpf(x[d, i])))
            worst = max(worst, abs(dx[d, i, j] - ref) / max(abs(ref), 1e-3))
    assert worst < 1e-12, worst
    # coincident pairs (r = 0, where c' diverges for these orders): 0, the mul0 convention
    assert np.all(dx[:, 0, 0] == 0) and np.all(dx[:, 1, 1] == 0) and np.all(np.isfinite(dx))


MATERN52_WHITE = [(1.3, [dict(kind='maternp', p=2, scale=1.4)]), (0.05, [dict(kind='white')])]


def _cs_logml(terms, X, r, A=None, ycov=None):
    out = np.empty(X.shape)
    for d in range(X.shape[0]):
        for k in range(X.shape[1]):
            Xc = X.astype(complex)
            Xc[d, k] += 1j * H
            out[d, k] = ox.logml(terms, Xc, r, A, ycov).imag / H
    return out


def test_oracle_logml_xgrad_vs_complex_step():
    rng = np.random.default_rng(3)
    X = rng.uniform(0, 5, (2, 20))
    r = rng.standard_normal(20)
    g = ox.logml_xgrad(MATERN52_WHITE, X, r)
    assert _rel(g, _cs_logml(MATERN52_WHITE, X, r)) < 1e-10
    # two keys sharing points (x and x[:k]), a data covariance and a linear map of them
    n, k = 12, 5
    X = rng.uniform(0, 5, (2, n))
    A = np.vstack([np.eye(n), np.eye(n)[:k], 0.5 * np.eye(n)[2:4] + 0.5 * np.eye(n)[6:8]])
    r = rng.standard_normal(len(A))
    ycov = np.diag(rng.uniform(0.1, 0.2, len(A)))
    g = ox.logml_xgrad(MATERN52_WHITE, X, r, A, ycov)
    assert _rel(g, _cs_logml(MATERN52_WHITE, X, r, A, ycov)) < 1e-10
    # the -b b' term matters: without it the gradient is wrong
    Kinv = np.linalg.inv(ogp.gram(MATERN52_WHITE, X, X))
    dx, dy = ox.gram_xgrad(MATERN52_WHITE, X, X)
    wrong = 0.5 * ((Kinv * dx).sum(2) + (Kinv * dy).sum(1))
    assert _rel(wrong, ox.logml_xgrad(MATERN52_WHITE, X, rng.standard_normal(n))) > 1e-3


def test_oracle_fisher_is_expected_hessian_form():
    """ 1/2 tr(K^-1 dK_p K^-1 dK_q) with dK from xjvp: symmetric, positive semidefinite, and equal to the covariance
    of the score, checked against the analytic expectation by a long sample average of the oracle's gradients """
    rng = np.random.default_rng(4)
    X = rng.uniform(0, 4, (1, 10))
    mask = (np.arange(10) % 2).astype(float)[None]
    K = ogp.gram(MATERN52_WHITE, X, X)
    dK = [ox.xjvp(MATERN52_WHITE, X, X, mask, mask)]
    F = ox.fisher(K, dK)
    L = np.linalg.cholesky(K)
    scores = []
    for _ in range(4000):
        r = L @ rng.standard_normal(10)
        scores.append(np.sum(ox.logml_xgrad(MATERN52_WHITE, X, r) * mask))
    assert F.shape == (1, 1) and F[0, 0] > 0
    assert abs(np.var(scores) - F[0, 0]) < 0.1 * F[0, 0]


# ---- points as torch tensors

def test_columns_of_tensors_match_numpy():
    rng = np.random.default_rng(5)
    X = rng.uniform(0, 1, (6, 3))
    t = torch.tensor(X, requires_grad=True)
    for a, b in [(X, t), (X[:, 0], t[:, 0]), (X.astype(np.float32), t.detach().float())]:
        la, da, sa = _array.columns_of(a)
        lb, db, sb = _array.columns_of(b)
        assert la == lb and tuple(sa) == tuple(sb) and np.array_equal(da, db.detach().numpy())
    d_np = {'a': X[:, 0], 'b': X[:, 1:]}
    d_t = {'a': t[:, 0], 'b': t[:, 1:]}
    mixed = {'a': X[:, 0], 'b': t[:, 1:]}
    la, da, sa = _array.columns_of(d_np)
    for d in (d_t, mixed, _array.StructuredArray(d_t)):
        lb, db, sb = _array.columns_of(d)
        assert la == lb and sa == sb and isinstance(db, torch.Tensor) and db.requires_grad
        assert np.array_equal(da, db.detach().numpy())
    sa_np, sa_t = _array.StructuredArray(d_np), _array.StructuredArray(d_t)
    assert sa_np.dtype == sa_t.dtype
    for key in (slice(1, 4), [0, 2, 5]):
        assert np.array_equal(_array.columns_of(sa_np[key])[1], _array.columns_of(sa_t[key])[1].detach().numpy())
    assert np.array_equal(_array.columns_of(sa_np.reshape(2, 3))[1],
                          _array.columns_of(sa_t.reshape(2, 3))[1].detach().numpy())
    # gradients reach the tensor through the columns
    _, db, _ = _array.columns_of(d_t)
    (db * torch.arange(3.0, dtype=torch.float64)[:, None]).sum().backward()
    assert np.array_equal(t.grad.numpy(), np.broadcast_to([0.0, 1.0, 2.0], (6, 3)))
    # numpy points keep their numpy path
    assert isinstance(_array.columns_of(X)[1], np.ndarray) and isinstance(_array.columns_of(d_np)[1], np.ndarray)
    with pytest.raises(TypeError, match='non-real dtype'):
        _array.columns_of(torch.zeros(3, dtype=torch.complex128))
