"""Oracle: isotropic kernels and kernel algebra (NumPy restatement).

Follows, operation by operation:
  CrossKernel.__new__ linop order scale -> loc -> ... (src/lsqfitgp/_Kernel/_crosskernel.py:167-185):
      on the way in, the input meets `loc` first, then `scale`: u = (x - loc) / scale
      (src/lsqfitgp/_Kernel/_ops.py:292-326), applied to each argument separately;
  IsotropicKernel newcore: r2 = sum over leaf fields of (x_f - y_f)**2, accumulated in field order
      (src/lsqfitgp/_Kernel/_isotropic.py:61-81, src/lsqfitgp/_Kernel/_util.py:74-99);
  cores: ExpQuad _kernels/_basic.py:75; Cauchy :339-343; White :59; Constant :46;
      Maternp _kernels/_matern.py:48-49 + _special/_bessel.py:101-110;
      Matern _kernels/_matern.py:74-76 + _special/_bessel.py:70-82 (scipy.special.kv, as the reference);
  algebra: _Kernel/_alg.py:48-82.
"""

import numpy as np
from scipy import special


def _transform(x, loc, scale):
    """ x: (ndim, n) -> list of per-field arrays after loc then scale """
    out = []
    for f in range(x.shape[0]):
        v = x[f]
        if loc is not None:
            v = v - loc
        if scale is not None:
            v = v / scale
        out.append(v)
    return out


def r2(x, y, *, scale=None, loc=None, dims=None):
    """ squared distance matrix (n, m); x: (ndim, n), y: (ndim, m) """
    sx, sy = scale if isinstance(scale, tuple) else (scale, scale)
    lx, ly = loc if isinstance(loc, tuple) else (loc, loc)
    if dims is not None:
        x = x[list(dims)]
        y = y[list(dims)]
    u = _transform(x, lx, sx)
    v = _transform(y, ly, sy)
    acc = None
    for uf, vf in zip(u, v):
        t = np.square(uf[:, None] - vf[None, :])
        acc = t if acc is None else acc + t
    if acc is None:
        acc = np.zeros((x.shape[1], y.shape[1]))
    return acc


def expquad_core(r2):
    return np.exp(-1 / 2 * r2)


def kvmodx2_hi(x2, p):
    # _special/_bessel.py:101-110
    x = np.sqrt(x2)
    poly = 1
    for k in reversed(range(p)):
        c_kp1_over_ck = (p - k) / ((2 * p - k) * (k + 1))
        poly = 1 + poly * c_kp1_over_ck * 2 * x
    return np.exp(-x) * poly


def kvmodx2(nu, x2, norm_offset=0):
    # _special/_bessel.py:70-82
    x = np.sqrt(x2)
    with np.errstate(all='ignore'):
        normal = 2 / special.gamma(nu + norm_offset) * (x / 2) ** nu * special.kv(nu, x)
    atzero = 1 / np.prod(nu + np.arange(norm_offset))
    atzero = np.where(nu > 0, atzero, 1)
    # for nu > 0 the limit at x -> 0; there x^nu K_nu(x) is 0 * inf in float64 below x ~ 1e-300^(1/nu)
    return np.where((x2 != 0) & ((nu <= 0) | np.isfinite(normal)), normal, atzero)


def maternp_core(r2, p):
    # _kernels/_matern.py:48-49
    r2 = (2 * p + 1) * r2
    return kvmodx2_hi(r2 + 1e-30, p)


def matern_core(r2, nu):
    # _kernels/_matern.py:74-76
    r2 = 2 * np.where(nu, nu, 1) * r2
    return kvmodx2(nu, r2)


def cauchy_core(r2, alpha=2, beta=2):
    # _kernels/_basic.py:339-343
    power = np.where(alpha == 2, r2, r2 ** (alpha / 2))
    return (1 + power / beta) ** (-beta / alpha)


def white(x, y, dims=None):
    # _kernels/_basic.py:59 (prod over fields of x == y)
    if dims is not None:
        x = x[list(dims)]
        y = y[list(dims)]
    acc = None
    for f in range(x.shape[0]):
        t = x[f][:, None] == y[f][None, :]
        acc = t if acc is None else acc * t
    return acc.astype(int)


# derivatives of the cores w.r.t. r2 (what jax's autodiff produces through the custom JVPs)
def expquad_dr2(r2):
    return -1 / 2 * np.exp(-1 / 2 * r2)


def maternp_dr2(r2, p):
    # _special/_bessel.py:112-122 chained with z = (2p+1) r2 + 1e-30
    z = (2 * p + 1) * r2 + 1e-30
    if p == 0:
        x = np.sqrt(z)
        return (2 * p + 1) * (-np.exp(-x) / (2 * x))
    return (2 * p + 1) * (-1 / (p - 1 / 2) * kvmodx2_hi(z, p - 1) / 4)


def matern_dr2(r2, nu):
    # _special/_bessel.py:93-99 chained with z = 2 nu r2
    z = 2 * nu * r2
    return 2 * nu * (-kvmodx2(nu - 1, z, 1) / 4)


def cauchy_dr2(r2, alpha=2, beta=2):
    # d/dr2 (1 + t/beta)^(-beta/alpha), t = r2^(alpha/2): -(1/2) (1 + t/beta)^(-beta/alpha - 1) t / r2; 0 at r2 = 0 for
    # alpha < 2 (where it diverges), as the kernels: it only enters multiplied by r2
    if alpha == 2:
        return -1 / 2 * (1 + r2 / beta) ** (-beta / 2 - 1)
    r2 = np.asarray(r2, dtype=float)
    pos = r2 > 0
    rp = np.where(pos, r2, 1.0)
    t = rp ** (alpha / 2)
    return np.where(pos, -1 / 2 * (1 + t / beta) ** (-beta / alpha - 1) * t / rp, 0.0)


def cauchy_dbeta(r2, alpha=2, beta=2):
    """ d/dbeta (1 + t/beta)^(-beta/alpha), t = r2^(alpha/2).  The two terms cancel to O(t^2) at small t: the result
    is accurate to rounding relative to their size, (1 + t/beta)^(-beta/alpha) t / (alpha beta), not elementwise """
    t = np.where(alpha == 2, r2, r2 ** (alpha / 2))
    base = 1 + t / beta
    return base ** (-beta / alpha) * (-np.log1p(t / beta) / alpha + t / (alpha * beta * base))
