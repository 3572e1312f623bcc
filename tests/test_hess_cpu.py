"""Second hyperparameter derivatives without a GPU: the oracle's per-core second derivatives (oracle/hess.py) against
sympy and against mpmath differentiation, the host build of the kernels' coefficient code (csrc/hess_core.cuh) against
the oracle, the oracle's logML Hessian against differences of its gradient, and the argument checks of
empbayes_fit(method='hessian', covariance='hessian')."""
import ctypes
import pathlib
import subprocess

import numpy as np
import pytest

import lsqfitgp_b200 as lgp
from lsqfitgp_b200 import _lib
from oracle import gp as ogp, hess as oh

ROOT = pathlib.Path(__file__).resolve().parent.parent

sympy = pytest.importorskip('sympy')
import mpmath  # noqa: E402

NAMES = ['c', 'c_l', 'c_ll', 'c_b', 'c_lb', 'c_bb']
U = [1e-9, 1e-4, 0.03, 0.4, 1.0, 2.5, 9.0, 40.0]


def _size(h, u):
    """ magnitude of the terms the coefficients are made of, for absolute tolerances where they cancel """
    return np.abs(h[0]) * (1 + np.abs(u)) ** 2 + np.abs(h[1]) + np.abs(h[3])


# ---- oracle vs sympy (closed forms)

def _sym_core(kind, u, beta, **kw):
    if kind == 'expquad':
        return sympy.exp(-u / 2)
    if kind == 'maternp':
        p = kw['p']
        x = sympy.sqrt((2 * p + 1) * u)
        poly = sympy.Integer(1)
        for k in reversed(range(p)):
            poly = 1 + poly * sympy.Rational(p - k, (2 * p - k) * (k + 1)) * 2 * x
        return sympy.exp(-x) * poly
    if kind == 'cauchy':
        alpha = sympy.Rational(kw['alpha'])
        return (1 + u ** (alpha / 2) / beta) ** (-beta / alpha)
    raise KeyError(kind)


@pytest.mark.parametrize('kind, kw', [('expquad', {}), *[('maternp', dict(p=p)) for p in range(4)],
                                      ('cauchy', dict(alpha=2)), ('cauchy', dict(alpha=1))])
def test_oracle_vs_sympy(kind, kw):
    lam, bet, r2 = sympy.symbols('lam beta r2', positive=True)
    expr = _sym_core(kind, r2 * sympy.exp(-2 * lam), bet, **kw)
    ders = [expr, sympy.diff(expr, lam), sympy.diff(expr, lam, 2), sympy.diff(expr, bet), sympy.diff(expr, lam, bet),
            sympy.diff(expr, bet, 2)]
    beta0 = sympy.Rational(13, 10)
    fns = [sympy.lambdify(r2, d.subs({lam: 0, bet: beta0}), modules='mpmath') for d in ders]
    mpmath.mp.dps = 50
    okw = dict(maternp=dict(p=kw.get('p'), par0=0.0), cauchy=dict(alpha=kw.get('alpha'), beta=1.3)).get(kind, {})
    got = oh.core_hess(kind, np.array(U), **okw)
    size = _size(got, np.array(U))
    for j, fn in enumerate(fns):
        ref = np.array([float(fn(mpmath.mpf(u))) for u in U])
        assert np.all(np.abs(got[j] - ref) <= 1e-13 * (np.abs(ref) + size)), (NAMES[j], got[j], ref)


# ---- oracle vs mpmath differentiation (Bessel and general-alpha cores)

def _mp_core(kind, u, par, beta):
    if kind == 'matern':
        nu = mpmath.mpf(par)
        if u == 0:
            return mpmath.mpf(1)
        x = mpmath.sqrt(2 * nu * u)
        return 2 / mpmath.gamma(nu) * (x / 2) ** nu * mpmath.besselk(nu, x)
    alpha = mpmath.mpf(par)
    return (1 + u ** (alpha / 2) / beta) ** (-beta / alpha)


@pytest.mark.parametrize('kind, par', [('matern', 0.3), ('matern', 0.5), ('matern', 1.3), ('matern', 4.2),
                                       ('cauchy', 0.5), ('cauchy', 1.0), ('cauchy', 2.0)])
def test_oracle_vs_mpmath(kind, par):
    mpmath.mp.dps = 60
    beta0 = mpmath.mpf('0.7')
    u = np.array(U)
    okw = dict(nu=par) if kind == 'matern' else dict(alpha=par, beta=0.7)
    got = oh.core_hess(kind, u, **okw)
    size = _size(got, u)
    for i, ui in enumerate(U):
        R = mpmath.mpf(ui)

        def f(lam, b):
            return _mp_core(kind, R * mpmath.exp(-2 * lam), par, b)
        ref = [f(0, beta0), mpmath.diff(lambda l: f(l, beta0), 0), mpmath.diff(lambda l: f(l, beta0), 0, 2)]
        if kind == 'cauchy':
            ref += [mpmath.diff(lambda b: f(0, b), beta0), mpmath.diff(f, (0, beta0), (1, 1)),
                    mpmath.diff(lambda b: f(0, b), beta0, 2)]
        else:
            ref += [0, 0, 0]
        for j in range(6):
            assert abs(got[j][i] - float(ref[j])) <= 1e-13 * (abs(float(ref[j])) + size[i]), (NAMES[j], ui, got[j][i], ref[j])


def test_matern_half_closed_form():
    """ nu = 1/2 through the Bessel equation reproduces e^-sqrt(u) (u/4 + sqrt(u)/4) for u^2 c'' """
    u = np.array(U)
    h = oh.core_hess('matern', u, nu=0.5)
    x = np.sqrt(u)
    c1 = -np.exp(-x) / (2 * x)
    u2c2 = np.exp(-x) * (u / 4 + x / 4)
    np.testing.assert_allclose(h[2], 4 * u * c1 + 4 * u2c2, rtol=1e-13, atol=1e-15)


# ---- host build of csrc/hess_core.cuh vs the oracle

@pytest.fixture(scope='module')
def host(tmp_path_factory):
    """ oracle/hess_core_host.c (which includes csrc/hess_core.cuh) compiled with g++ into a temporary directory """
    so = tmp_path_factory.mktemp('hess_core_host') / 'libhess_core_host.so'
    subprocess.run(['g++', '-x', 'c++', '-std=c++17', '-O2', '-fPIC', '-shared', '-ffp-contract=off', '-o', str(so),
                    str(ROOT / 'oracle' / 'hess_core_host.c'), '-lm'], check=True)
    lib = ctypes.CDLL(str(so))
    dp = ctypes.POINTER(ctypes.c_double)
    lib.lgp_host_hess_coefs.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double, dp,
                                        ctypes.c_long, dp]
    lib.lgp_host_hess_coefs.restype = ctypes.c_int
    return lib, dp


@pytest.mark.parametrize('kind, p, par0, par1', [
    (_lib.K_EXPQUAD, 0, 0.0, 0.0),
    *[(_lib.K_MATERNP, p, par0, 0.0) for p in (0, 1, 2, 3, 5) for par0 in (0.0, 1e-30)],
    *[(_lib.K_MATERN, 0, nu, 0.0) for nu in (0.0, 0.3, 0.5, 1.3, 4.2)],
    *[(_lib.K_CAUCHY, 0, alpha, beta) for alpha, beta in ((2.0, 0.7), (2.0, 5.0), (1.0, 1.3), (0.5, 3.0))],
    (_lib.K_CONSTANT, 0, 0.0, 0.0),
])
def test_host_coefs_vs_oracle(host, kind, p, par0, par1):
    lib, dp = host
    rng = np.random.default_rng(kind * 100 + p)
    u = np.concatenate([[0.0, 1e-300, 1e-30], 10 ** rng.uniform(-20, 3.3, 100_000)])
    n = u.size
    h = np.empty((n, 6))
    assert lib.lgp_host_hess_coefs(kind, p, par0, par1, u.ctypes.data_as(dp), n, h.ctypes.data_as(dp)) == 0
    name = {_lib.K_EXPQUAD: 'expquad', _lib.K_MATERNP: 'maternp', _lib.K_MATERN: 'matern', _lib.K_CAUCHY: 'cauchy',
            _lib.K_CONSTANT: 'constant'}[kind]
    kw = dict(maternp=dict(p=p, par0=par0), matern=dict(nu=par0), cauchy=dict(alpha=par0, beta=par1)).get(name, {})
    ref = oh.core_hess(name, u, **kw)
    size = _size(ref, u)
    # Matern of real order: the oracle's c, c' come from scipy's kv (AMOS), itself about 1e-14 .. 1e-13 from the exact
    # value for some orders (tests/test_bessel_cpu.py); the closed forms agree to rounding
    bar = 1e-13 if name == 'matern' else 2e-14
    for j in range(6):
        assert np.all(np.isfinite(h[:, j])), NAMES[j]
        err = np.abs(h[:, j] - ref[j])
        bad = err > bar * (np.abs(ref[j]) + size) + 1e-300
        assert not np.any(bad), (NAMES[j], u[bad][:5], h[bad, j][:5], ref[j][bad][:5])


# ---- the oracle's logML Hessian against central differences of its own gradient

def test_logml_hessian_vs_gradient_differences():
    rng = np.random.default_rng(7)
    x = rng.uniform(0, 5, (2, 40))
    r = rng.standard_normal(40)

    def terms(q):   # q = (log amp, log scale, log beta, log noise amp)
        return [(np.exp(q[0]), [dict(kind='cauchy', alpha=1.0, beta=np.exp(q[2]), scale=np.exp(q[1]))]),
                (np.exp(q[3]), [dict(kind='white')])]

    def derivs(q):
        """ dK/dq, d2K/dq2 through oracle.hess.gram_hessian and the chain rule of the exp transforms """
        d1, d2 = oh.gram_hessian(terms(q), x, x)
        # native (descriptor) coordinates: factor 0 (amp, log scale, beta), factor 1 (amp)
        J = {0: (0, 0, np.exp(q[0])), 1: (0, 1, 1.0), 2: (0, 2, np.exp(q[2])), 3: (1, 0, np.exp(q[3]))}
        dK = [J[a][2] * d1[J[a][0]][J[a][1]] for a in range(4)]
        d2K = [[J[a][2] * J[b][2] * d2.get((J[a][0], J[a][1], J[b][0], J[b][1]), np.zeros((40, 40))) for b in range(4)]
               for a in range(4)]
        for a in (0, 2, 3):   # d2/dq2 of exp(q): the first derivative once more
            d2K[a][a] = d2K[a][a] + dK[a]
        return dK, d2K

    def grad(q):
        K = ogp.gram(terms(q), x, x)
        Ki = np.linalg.inv(K)
        b = Ki @ r
        return np.array([0.5 * np.sum(Ki * dK) - 0.5 * b @ dK @ b for dK in derivs(q)[0]])

    q0 = np.array([0.2, 0.1, -0.3, np.log(0.1)])
    dK, d2K = derivs(q0)
    H = oh.logml_hessian(ogp.gram(terms(q0), x, x), r, dK, d2K)
    h = 1e-5
    Hfd = np.stack([(grad(q0 + h * e) - grad(q0 - h * e)) / (2 * h) for e in np.eye(4)])
    np.testing.assert_allclose(H, H.T, rtol=1e-10, atol=1e-10 * np.max(np.abs(H)))
    assert np.max(np.abs(H - Hfd)) < 1e-6 * np.max(np.abs(H))


# ---- empbayes_fit argument checks (raised before any evaluation)

def test_empbayes_method_and_covariance_names():
    hp = {'log(a)': (0.0, 1.0)}
    with pytest.raises(KeyError):
        lgp.empbayes_fit(hp, lambda hp: None, {}, method='hessmod')
    with pytest.raises(KeyError):
        lgp.empbayes_fit(hp, lambda hp: None, {}, covariance='hessmod')
    with pytest.raises(KeyError, match='bogus'):   # 'hessian' is a method: the covariance is checked next
        lgp.empbayes_fit(hp, lambda hp: None, {}, method='hessian', covariance='bogus')
