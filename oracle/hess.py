"""Oracle: second derivatives of the Gram matrix and of the log marginal likelihood with respect to the kernel
hyperparameters (NumPy/SciPy restatement, float64).

Per factor c(u), u the scaled squared distance, lambda = log(scale), beta = Cauchy beta (`core_hess`):
  c, dc/dlambda = -2u c', d2c/dlambda2 = 4u c' + 4u^2 c'', dc/dbeta, d2c/dlambda dbeta, d2c/dbeta2.
A term is amp * prod_f c_f; the hyperparameters of factor f are theta_f = (amp_f, log scale_f, beta_f), amp_f the term's
amplitude on its first factor and 1 on the others (the layout of the Gram kernels' descriptors).  `gram_hessian` gives
dK/dtheta and d2K/dtheta dtheta' by the product rule; `logml_hessian` the exact Hessian of -log ML,
  H_ab = 1/2 tr(K^-1 K_ab) - 1/2 tr(K^-1 K_a K^-1 K_b) - 1/2 b' K_ab b + b' K_a K^-1 K_b b,   b = K^-1 r,
plus the terms of data r that depend on the hyperparameters.  Terms use the factor format of oracle/gp.py.
"""

import numpy as np

from . import gp as ogp, iso
from .deriv import coefs, mul0


def core_hess(kind, u, *, p=None, par0=1e-30, nu=None, alpha=2.0, beta=2.0):
    """ [c, c_l, c_ll, c_b, c_lb, c_bb] at scaled squared distance u (l = log scale, b = Cauchy beta) """
    u = np.asarray(u, dtype=float)
    zero = np.zeros_like(u)
    if kind == 'expquad':
        c = np.exp(-0.5 * u)
        return [c, u * c, (u * u - 2 * u) * c, zero, zero, zero]
    if kind == 'maternp':
        c, _ = coefs('maternp', u, p=p, par0=par0)
        return [c[0], mul0(c[1], -2 * u), mul0(c[1], 4 * u) + mul0(c[2], 4 * u * u), zero, zero, zero]
    if kind == 'matern':
        # u^2 c'' = (nu u / 2) c + (nu - 1) u c' (modified Bessel equation in u): d2c/dlambda2 = 2 nu u (c + 2 c')
        c = iso.matern_core(u, nu)
        c1 = mul0(iso.matern_dr2(u, nu), u)   # u c'
        return [c, -2 * c1, 2 * nu * (u * c + 2 * c1), zero, zero, zero]
    if kind == 'cauchy':
        s = u if alpha == 2 else u ** (alpha / 2)
        B = 1 + s / beta
        c = B ** (-beta / alpha)
        sB = s / B
        l1, l11 = sB, -alpha * sB / B
        lb = (sB / beta - np.log1p(s / beta)) / alpha
        l1b = (sB / beta) ** 2
        lbb = l1b / (alpha * beta)
        return [c, c * l1, c * (l11 + l1 * l1), c * lb, c * (l1b + l1 * lb), c * (lbb + lb * lb)]
    if kind == 'constant':
        return [np.ones_like(u), zero, zero, zero, zero, zero]
    raise KeyError(kind)


def factor_hess(f, x, y):
    """ core_hess of a factor of oracle/gp.py format on the points x (ndim, n), y (ndim, m) """
    kind = f['kind']
    if kind in ('white', 'constant'):
        v = ogp.factor_value(f, x, y).astype(float)
        z = np.zeros_like(v)
        return [v, z, z, z, z, z]
    u = iso.r2(x, y, scale=f.get('scale'), loc=f.get('loc'), dims=f.get('dims'))
    kw = dict(maternp=dict(p=f.get('p'), par0=f.get('par0', 1e-30)), matern=dict(nu=f.get('nu')),
              cauchy=dict(alpha=f.get('alpha', 2), beta=f.get('beta', 2))).get(kind, {})
    return core_hess(kind, u, **kw)


def _factor_derivs(A, h):
    """ first (3) and second (3 x 3) derivatives of A c with respect to (A, log scale, beta) """
    c, cl, cll, cb, clb, cbb = h
    z = np.zeros_like(c)
    d1 = [c, A * cl, A * cb]
    d2 = [[z, cl, cb], [cl, A * cll, A * clb], [cb, A * clb, A * cbb]]
    return d1, d2


def gram_hessian(terms, x, y):
    """ (d1, d2): d1[f][k] = dK/dtheta_{f,k}, d2[(f, k, g, l)] = d2K/dtheta_{f,k} dtheta_{g,l} (missing pairs are 0),
    f, g the factors in descriptor order (terms flattened) """
    d1, d2 = [], {}
    f0 = 0
    for amp, factors in terms:
        vals, fd1, fd2 = [], [], []
        for i, f in enumerate(factors):
            A = amp if i == 0 else 1.0
            h = factor_hess(f, x, y)
            a, b = _factor_derivs(A, h)
            vals.append(A * h[0])
            fd1.append(a)
            fd2.append(b)

        def others(skip):
            out = 1.0
            for i, v in enumerate(vals):
                if i not in skip:
                    out = out * v
            return out
        nf = len(factors)
        for i in range(nf):
            d1.append([fd1[i][k] * others({i}) for k in range(3)])
            for j in range(nf):
                for k in range(3):
                    for l in range(3):
                        if i == j:
                            d2[f0 + i, k, f0 + j, l] = fd2[i][k][l] * others({i})
                        else:
                            d2[f0 + i, k, f0 + j, l] = fd1[i][k] * fd1[j][l] * others({i, j})
        f0 += nf
    return d1, d2


def hvp(terms, x, y, G, tangent):
    """ (out, size): out[f, k] = sum_ij G_ij d/dtheta_{f,k} sum_{g,l} tangent[g, l] dK_ij/dtheta_{g,l} (what
    lgp_gram_iso_hvp computes) and size[f, k] = sum_ij sum_{g,l} |G_ij tangent[g, l] d2K_ij/dtheta_{f,k} dtheta_{g,l}| """
    _, d2 = gram_hessian(terms, x, y)
    nf = len(tangent)
    out = np.zeros((nf, 3))
    size = np.zeros((nf, 3))
    for (f, k, g, l), m in d2.items():
        t = G * m * tangent[g][l]
        out[f, k] += np.sum(t)
        size[f, k] += np.sum(np.abs(t))
    return out, size


def logml_hessian(K, r, dK, d2K, dr=None, d2r=None):
    """ exact Hessian of -log ML = 1/2 (n log 2pi + log det K + r' K^-1 r) with respect to parameters q:
    dK[a] = dK/dq_a, d2K[a][b] = d2K/dq_a dq_b; dr, d2r likewise for data r that depend on q (None: constant) """
    Kinv = np.linalg.inv(K)
    Kinv = 0.5 * (Kinv + Kinv.T)
    b = Kinv @ r
    k = len(dK)
    KiKa = [Kinv @ Ka for Ka in dK]
    H = np.empty((k, k))
    for a in range(k):
        for c in range(k):
            H[a, c] = (0.5 * np.sum(Kinv * d2K[a][c]) - 0.5 * np.sum(KiKa[a] * KiKa[c].T) - 0.5 * b @ d2K[a][c] @ b
                       + b @ dK[a] @ KiKa[c] @ b)
            if dr is not None:
                H[a, c] += (d2r[a][c] @ b + dr[a] @ Kinv @ dr[c] - dr[a] @ KiKa[c] @ b - dr[c] @ KiKa[a] @ b)
    return H
