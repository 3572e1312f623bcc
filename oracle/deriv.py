"""Oracle: derivative blocks of the kernel (NumPy restatement, float64).

cov(d_a f(x), d_b f(y)) = d/dx_a d/dy_b k(x, y) for first derivatives (reference: linop('diff') of the kernel,
src/lsqfitgp/_Kernel/_crosskernel.py, _Kernel/_ops.py, applied by _GP/_elements.py:190-242).  Each factor gives the
hyper-dual number (v, gx, gy, h) of its value and derivatives, a term is their product under the product rule:
  v = c(u), gx = 2 c'(u) D_a / sx, gy = -2 c'(u) D_b / sy, h = -(4 c''(u) D_a D_b + 2 c'(u) delta_ab) / (sx sy),
u = sum_d D_d^2 over the factor's fields, D_d = (x_d - loc_x)/sx - (y_d - loc_y)/sy.  The derivatives with respect to
log(scale) and Cauchy beta differentiate the four numbers once more.  Terms use the factor format of oracle/gp.py.
"""

import numpy as np

from . import gp as ogp, iso


def kvmodx2_hi_ex(ex, x, q):
    poly = 1.0
    for k in reversed(range(q)):
        poly = 1.0 + poly * ((q - k) / ((2 * q - k) * (k + 1))) * 2.0 * x
    return ex * poly


def coefs(kind, u, *, p=None, par0=0.0, beta=2.0):
    """ ([c, c', c'', c'''], [dc/dbeta, dc'/dbeta, dc''/dbeta]) at u (derivatives w.r.t. u) """
    u = np.asarray(u, dtype=float)
    zero = np.zeros_like(u)
    if kind == 'expquad':
        c0 = np.exp(-0.5 * u)
        return [c0, -0.5 * c0, 0.25 * c0, -0.125 * c0], [zero, zero, zero]
    if kind == 'cauchy':
        B = 1.0 + u / beta
        lb = np.log(B)
        c = [B ** (-beta / 2.0)]
        db = []
        hsum = 0.0
        for j in range(4):
            if j > 0:
                c.append(c[j - 1] * (-(0.5 * beta + (j - 1))) / (beta * B))
            if j < 3:
                db.append(c[j] * (hsum - j / beta - 0.5 * lb + (0.5 * beta + j) * u / (beta * beta * B)))
            hsum += 1.0 / (beta + 2.0 * j)
        return c, db
    if kind == 'maternp':
        nu2 = 2 * p + 1
        x = np.sqrt(nu2 * u + par0)
        ex = np.exp(-x)
        c = []
        w = 1.0
        with np.errstate(divide='ignore', invalid='ignore'):
            for j in range(4):
                q = p - j
                if q >= 0:
                    c.append(w * kvmodx2_hi_ex(ex, x, q))
                    if q > 0:
                        w *= -nu2 / (4 * q - 2)
                elif q == -1:
                    c.append(w * nu2 * (-ex / (2.0 * x)))
                elif q == -2:
                    c.append(w * (nu2 * nu2) * (ex * (x + 1.0) / (4.0 * x * x * x)))
                else:
                    c.append(np.full_like(u, np.nan))
        return c, [zero, zero, zero]
    if kind == 'constant':
        return [np.ones_like(u), zero, zero, zero], [zero, zero, zero]
    raise NotImplementedError(kind)


def mul0(c, t):
    """ c * t, 0 where t == 0 (c may be infinite there) """
    with np.errstate(invalid='ignore', over='ignore'):
        return np.where(t == 0, 0.0, c * t)


def _pair(v, default):
    if isinstance(v, tuple):
        return tuple(default if w is None else w for w in v)
    return (default, default) if v is None else (v, v)


def _coef_args(f):
    kind = f['kind']
    if kind == 'matern':
        p = f['nu'] - 0.5
        assert p == int(p) and p >= 1, 'half-integer Matern only'
        return 'maternp', dict(p=int(p), par0=0.0)
    if kind == 'maternp':
        return 'maternp', dict(p=f['p'], par0=1e-30)
    if kind == 'cauchy':
        assert f.get('alpha', 2) == 2
        return 'cauchy', dict(beta=f.get('beta', 2))
    return kind, {}


def factor_hd(f, x, y, a, b):
    """ (q, ql, qb): hyper-dual value of the factor (without amplitude) and its derivatives along log(scale) and beta;
    a, b: field indices of the derivatives on x and y (None for none) """
    n, m = x.shape[1], y.shape[1]
    zero = np.zeros((n, m))
    kind = f['kind']
    dims = list(range(x.shape[0])) if f.get('dims') is None else list(f['dims'])
    ina = a is not None and a in dims and kind != 'constant'
    inb = b is not None and b in dims and kind != 'constant'
    if not (ina or inb):
        v = ogp.factor_value(f, x, y)
        vl = ogp.factor_dlogscale(f, x, y)
        vb = zero
        if kind == 'cauchy':
            u = _u_and_diffs(f, x, y, dims)[0]
            vb = iso.cauchy_dbeta(u, f.get('alpha', 2), f.get('beta', 2))
        return (v, zero, zero, zero), (vl, zero, zero, zero), (vb, zero, zero, zero)
    u, D = _u_and_diffs(f, x, y, dims)
    sx, sy = _pair(f.get('scale'), 1.0)
    ck, kw = _coef_args(f)
    c, db = coefs(ck, u, **kw)
    A = D[a] if ina else zero
    B = D[b] if inb else zero
    delta = 1.0 if (ina and inb and a == b) else 0.0
    W = sx * sy
    AB = A * B
    t2 = mul0(c[2], AB)
    q = (c[0], 2 * c[1] * A / sx, -(2 * c[1] * B / sy), -(4 * t2 + 2 * c[1] * delta) / W)
    ql = (c[1] * (-2 * u),
          -4 * (mul0(c[2], u * A) + c[1] * A) / sx,
          4 * (mul0(c[2], u * B) + c[1] * B) / sy,
          (8 * mul0(c[3], u * AB) + 8 * t2 + 4 * delta * mul0(c[2], u)) / W - 2 * q[3])
    qb = (db[0], 2 * db[1] * A / sx, -(2 * db[1] * B / sy), -(4 * db[2] * AB + 2 * db[1] * delta) / W)
    return q, ql, qb


def _u_and_diffs(f, x, y, dims):
    sx, sy = _pair(f.get('scale'), 1.0)
    lx, ly = _pair(f.get('loc'), 0.0)
    D = {d: (x[d][:, None] - lx) / sx - (y[d][None, :] - ly) / sy for d in dims}
    u = None
    for d in dims:
        u = D[d] ** 2 if u is None else u + D[d] ** 2
    return u, D


def hd_mul(P, Q):
    return (P[0] * Q[0], P[1] * Q[0] + P[0] * Q[1], P[2] * Q[0] + P[0] * Q[2],
            P[3] * Q[0] + (P[1] * Q[2] + P[2] * Q[1]) + P[0] * Q[3])


def _sel(a, b):
    return (a is not None) | ((b is not None) << 1)


def block(terms, x, y, a=None, b=None):
    """ d/dx_a d/dy_b of the kernel (only the derivatives given); a = b = None is the plain Gram matrix """
    if a is None and b is None:
        return ogp.gram(terms, x, y)
    sel = _sel(a, b)
    out = 0.0
    for amp, factors in terms:
        P = None
        for f in factors:
            q = factor_hd(f, x, y, a, b)[0]
            P = q if P is None else hd_mul(P, q)
        out = out + amp * P[sel]
    return out


def block_derivs(terms, x, y, a=None, b=None):
    """ {('amp', ti): d block / d amp_ti, ('logscale', ti, fi): d / d log scale of factor fi of term ti (both scales),
    ('beta', ti, fi): d / d beta} """
    sel = _sel(a, b)
    out = {}
    for ti, (amp, factors) in enumerate(terms):
        hds = [factor_hd(f, x, y, a, b) for f in factors]
        P = None
        for q, _, _ in hds:
            P = q if P is None else hd_mul(P, q)
        out['amp', ti] = P[sel]
        for fi in range(len(factors)):
            O = None
            for h, (q, _, _) in enumerate(hds):
                if h != fi:
                    O = q if O is None else hd_mul(O, q)
            _, ql, qb = hds[fi]
            out['logscale', ti, fi] = amp * (ql if O is None else hd_mul(O, ql))[sel]
            out['beta', ti, fi] = amp * (qb if O is None else hd_mul(O, qb))[sel]
    return out


def joint_cov(terms, parts):
    """ assembled covariance of a list of (points (ndim, n), derivative field index or None) """
    return np.block([[block(terms, xa, xb, da, db) for xb, db in parts] for xa, da in parts])
