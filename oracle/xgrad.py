"""Oracle: derivatives of the Gram matrix and of the log marginal likelihood with respect to the input points (NumPy
restatement, float64).

What the reference gets from jax differentiating through the points of `gpfactory` (src/lsqfitgp/_fit.py:687-702).
Per factor, with u = (x - loc_x)/sx, v = (y - loc_y)/sy, D_d = u_d - v_d and r2 = sum_d D_d^2 over its fields,
  dc/dx_{d,i} = 2 c'(r2) D_d / sx,   dc/dy_{d,j} = -2 c'(r2) D_d / sy,
c' the derivative of the core that oracle/iso.py pins (the coefficient of d/d log(scale) = -2 r2 c'), the product
c' D taken as 0 where D = 0 (mul0: c' diverges at r2 = 0 for Maternp p = 0, low-order Matern and Cauchy alpha < 2, where
every D of the factor is 0).  A term is amp * prod_f c_f, differentiated by the product rule.  The derivative block
cov(d_a f(x), f(y)) of oracle/deriv.py is the same dK/dx_a for the kinds it covers.  Terms use the factor format of
oracle/gp.py.
"""

import numpy as np

from . import gp as ogp, iso
from .deriv import mul0


def _pair(v, default):
    if isinstance(v, tuple):
        return tuple(default if w is None else w for w in v)
    return (default, default) if v is None else (v, v)


def factor_dr2(f, x, y):
    """ c'(r2) of a factor (0 for White and Constant) """
    kind = f['kind']
    if kind in ('constant', 'white'):
        return np.zeros((x.shape[1], y.shape[1]))
    r2 = iso.r2(x, y, scale=f.get('scale'), loc=f.get('loc'), dims=f.get('dims'))
    with np.errstate(divide='ignore', invalid='ignore'):
        if kind == 'expquad':
            return iso.expquad_dr2(r2)
        if kind == 'maternp':
            return iso.maternp_dr2(r2, f['p'])
        if kind == 'matern':
            return iso.matern_dr2(r2, f['nu'])
        if kind == 'cauchy':
            return iso.cauchy_dr2(r2, f.get('alpha', 2), f.get('beta', 2))
    raise KeyError(kind)


def factor_xgrad(f, x, y):
    """ (gx, gy), each (ndim, n, m): derivatives of the factor's value with respect to x_{d,i} and y_{d,j} """
    ndim, n, m = x.shape[0], x.shape[1], y.shape[1]
    gx = np.zeros((ndim, n, m))
    gy = np.zeros((ndim, n, m))
    if f['kind'] in ('constant', 'white'):
        return gx, gy
    dims = range(ndim) if f.get('dims') is None else f['dims']
    sx, sy = _pair(f.get('scale'), 1.0)
    lx, ly = _pair(f.get('loc'), 0.0)
    c1 = factor_dr2(f, x, y)
    for d in dims:
        D = (x[d][:, None] - lx) / sx - (y[d][None, :] - ly) / sy
        t = 2 * mul0(c1, D)
        gx[d] = t / sx
        gy[d] = -t / sy
    return gx, gy


def gram_xgrad(terms, x, y):
    """ (dKdx, dKdy), each (ndim, n, m): dK_ij/dx_{d,i} and dK_ij/dy_{d,j} of the kernel `terms` """
    ndim, n, m = x.shape[0], x.shape[1], y.shape[1]
    dx = np.zeros((ndim, n, m))
    dy = np.zeros((ndim, n, m))
    for amp, factors in terms:
        vals = [ogp.factor_value(f, x, y).astype(float) for f in factors]
        for i, f in enumerate(factors):
            others = amp * np.ones((n, m))
            for h, v in enumerate(vals):
                if h != i:
                    others = others * v
            gx, gy = factor_xgrad(f, x, y)
            dx += gx * others
            dy += gy * others
    return dx, dy


def xvjp(terms, x, y, G):
    """ (gx, gy, sx, sy): gx[d, i] = sum_j G_ij dK_ij/dx_{d,i}, gy[d, j] = sum_i G_ij dK_ij/dy_{d,j} (what
    lgp_gram_iso_xvjp computes with a dense G) and the sizes sum |G dK| of each sum """
    dx, dy = gram_xgrad(terms, x, y)
    return ((G * dx).sum(2), (G * dy).sum(1), np.abs(G * dx).sum(2), np.abs(G * dy).sum(1))


def xjvp(terms, x, y, tx, ty):
    """ sum_d tx[d, i] dK_ij/dx_{d,i} + ty[d, j] dK_ij/dy_{d,j} (what lgp_gram_iso_xjvp computes) """
    dx, dy = gram_xgrad(terms, x, y)
    return np.einsum('di,dij->ij', tx, dx) + np.einsum('dj,dij->ij', ty, dy)


def logml(terms, X, r, A=None, ycov=None):
    """ -log ML of data r with covariance A K(X, X) A' + ycov (A = I, ycov = 0 by default): the GP of a set of points
    X, linear maps of it (several keys that select or combine points, addtransf) and an independent data covariance.
    Dtype-generic: complex points X give its complex-step derivatives. """
    K = ogp.gram(terms, X, X)
    if A is not None:
        K = A @ K @ A.T
    if ycov is not None:
        K = K + ycov
    sign, logabs = np.linalg.slogdet(K)   # complex K (complex step): log det = log|det| + i arg(det)
    return 0.5 * (len(r) * np.log(2 * np.pi) + logabs + np.log(sign) + r @ np.linalg.solve(K, r))


def logml_xgrad(terms, X, r, A=None, ycov=None):
    """ gradient of `logml` with respect to the points X, (ndim, n):
      d/dX_{d,k} = 1/2 sum_ij W_ij dK_ij/dX_{d,k},   W = A' (C^-1 - b b') A,  C = A K A' + ycov,  b = C^-1 r,
    which for the symmetric kernel is sum_j W_kj d_1 K(X_k, X_j) (for A = I: sum_j (K^-1 - b b')_kj d_1 K(x_k, x_j)) """
    K = ogp.gram(terms, X, X)
    C = K if A is None else A @ K @ A.T
    if ycov is not None:
        C = C + ycov
    Ci = np.linalg.inv(C)
    Ci = 0.5 * (Ci + Ci.T)
    b = Ci @ r
    W = Ci - np.outer(b, b)
    if A is not None:
        W = A.T @ W @ A
    dx, dy = gram_xgrad(terms, X, X)
    return 0.5 * ((W * dx).sum(2) + (W * dy).sum(1))


def fisher(K, dK):
    """ 1/2 tr(K^-1 dK_p K^-1 dK_q): the Fisher information of zero-mean data with covariance K, dK[p] = dK/dq_p (point
    dependence included, through `xjvp`) """
    Ki = np.linalg.inv(K)
    M = [Ki @ d for d in dK]
    return np.array([[0.5 * np.sum(a * b.T) for b in M] for a in M])
