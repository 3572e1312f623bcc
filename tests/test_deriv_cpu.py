"""Derivative observations without a GPU: `Deriv` parsing, the derivability contract of the kernels, the oracle's
derivative blocks against sympy, and the host build of the kernels' coefficient code (csrc/deriv_core.cuh) against
the oracle."""
import ctypes
import pathlib
import subprocess

import numpy as np
import pytest

import lsqfitgp_b200 as lgp
from lsqfitgp_b200 import _lib
from oracle import deriv as od, gp as ogp

ROOT = pathlib.Path(__file__).resolve().parent.parent


# ---- Deriv

def test_deriv_parsing():
    for empty in (0, None, {}, []):
        d = lgp.Deriv(empty)
        assert not d and d.order == 0 and not d.implicit and list(d) == []
    d = lgp.Deriv(2)
    assert d.implicit and d.order == 2 and list(d) == [(None, 2)]
    assert list(lgp.Deriv('a')) == [('a', 1)] and lgp.Deriv('a').order == 1
    d = lgp.Deriv(['a', 'b', 'a'])
    assert dict(d) == {'a': 2, 'b': 1} and d.order == 3 and not d.implicit
    assert dict(lgp.Deriv({'a': 2, 'c': 0})) == {'a': 2}
    assert lgp.Deriv(lgp.Deriv('a')) == lgp.Deriv({'a': 1})


def test_deriv_errors():
    with pytest.raises(ValueError):
        lgp.Deriv(-1)
    with pytest.raises(ValueError):
        lgp.Deriv({'a': -1})
    with pytest.raises(TypeError):
        lgp.Deriv([1])
    with pytest.raises(TypeError):
        lgp.Deriv({1: 1})
    with pytest.raises(TypeError):
        lgp.Deriv(1.5)


# ---- derivability (checked before any evaluation)

@pytest.mark.parametrize('kern, derivable', [
    (lgp.ExpQuad(), np.inf), (lgp.Constant(), np.inf), (lgp.Cauchy(alpha=2, beta=3), np.inf),
    (lgp.Cauchy(alpha=1), 0), (lgp.Maternp(p=0), 0), (lgp.Maternp(p=3), 3), (lgp.Matern(nu=2.5), 2),
    (lgp.Matern(nu=1.7), 1), (lgp.Matern(nu=0.7), 0), (lgp.White(), 0),
])
def test_derivability_table(kern, derivable):
    f, = kern._terms[0].factors
    assert f.derivable == derivable


def test_linop_diff_errors():
    for k in (lgp.White(), lgp.Cauchy(alpha=1), lgp.Maternp(p=0), lgp.Matern(nu=0.7),
              lgp.BART(splits=lgp.BART.splits_from_coord(np.arange(5.)[:, None]))):
        with pytest.raises(ValueError, match='derivability'):
            k.linop('diff', 1, 0)
    with pytest.raises(ValueError, match='derivability'):
        lgp.Maternp(p=1).linop('diff', 2, 0)
    for spec in (2, ['a', 'b'], {'a': 2}):
        with pytest.raises(NotImplementedError):
            lgp.ExpQuad().linop('diff', spec, 0)
    with pytest.raises(NotImplementedError):
        lgp.Matern(nu=1.7).linop('diff', 1, 0)
    # factors that do not depend on the field impose no limit
    k = lgp.ExpQuad(dim='a') * lgp.White(dim='b') + lgp.Maternp(p=0, dim='b')
    assert k.linop('diff', 'a', 'a')._diff is not None
    with pytest.raises(ValueError):
        k.linop('diff', 'b', 0)
    assert lgp.ExpQuad().linop('diff', 0, None) is not None


# ---- oracle vs sympy

sympy = pytest.importorskip('sympy')
import mpmath  # noqa: E402

X0, X1, X2, Y0, Y1, Y2, S, BETA = sympy.symbols('x0 x1 x2 y0 y1 y2 s beta', real=True)
XS, YS = (X0, X1, X2), (Y0, Y1, Y2)


def _kv_hi(z, p):
    x = sympy.sqrt(z)
    poly = sympy.Integer(1)
    for k in reversed(range(p)):
        poly = 1 + poly * sympy.Rational(p - k, (2 * p - k) * (k + 1)) * 2 * x
    return sympy.exp(-x) * poly


def _sym_factor(f, scale_sym):
    dims = f.get('dims', [0, 1, 2])
    sx, sy = (scale_sym, scale_sym) if not isinstance(f.get('scale'), tuple) else f['scale']
    if f.get('scale') is None:
        sx = sy = 1
    lx, ly = f.get('loc', (0, 0)) if isinstance(f.get('loc'), tuple) else (f.get('loc', 0) or 0,) * 2
    u = sum(((XS[d] - lx) / sx - (YS[d] - ly) / sy) ** 2 for d in dims)
    kind = f['kind']
    if kind == 'expquad':
        return sympy.exp(-u / 2)
    if kind == 'cauchy':
        return (1 + u / BETA) ** (-BETA / 2)
    if kind == 'maternp':
        return _kv_hi((2 * f['p'] + 1) * u + sympy.Float('1e-30', 60), f['p'])
    if kind == 'matern':
        p = int(f['nu'] - 0.5)
        return _kv_hi((2 * p + 1) * u + sympy.Float('1e-40', 120), p)
    if kind == 'constant':
        return sympy.Integer(1)
    raise KeyError(kind)


def _sym_kernel(terms):
    # exact amplitudes: a float amplitude is a 15-digit sympy Float, which caps the precision of the cancellations at
    # coincident points (the Maternp offset 1e-30 makes them cancel to about 15 digits)
    return sum(sympy.Rational(repr(amp)) * _sym_term(fs) for amp, fs in terms)


def _sym_term(factors):
    return sympy.Mul(*[_sym_factor(f, S) for f in factors])


SVAL, BVAL = 1.7, 1.3


def _cases():
    e = lambda **kw: [(1.0, [dict(scale=SVAL, **kw)])]  # noqa: E731
    return {
        'expquad': e(kind='expquad'),
        **{f'maternp{p}': e(kind='maternp', p=p) for p in (1, 2, 3, 4)},
        **{f'matern{nu}': e(kind='matern', nu=nu) for nu in (1.5, 2.5, 3.5)},
        'cauchy': [(1.0, [dict(kind='cauchy', alpha=2, beta=BVAL, scale=SVAL)])],
        'product': [(0.8, [dict(kind='expquad', dims=[0], scale=SVAL), dict(kind='maternp', p=2, dims=[1], scale=SVAL)])],
        'sum_const': [(1.0, [dict(kind='maternp', p=2, scale=SVAL)]), (0.3, [dict(kind='constant')])],
        'loc': [(1.0, [dict(kind='maternp', p=1, scale=SVAL, loc=0.4)])],
        'tuple_scale': [(1.0, [dict(kind='expquad', scale=(1.3, 0.9), loc=(0.2, -0.1))])],
        # both factors depend on field 0: both mixed products of the product rule are non-zero for (0, 0)
        'shared_field': [(0.8, [dict(kind='expquad', dims=[0, 1], scale=SVAL),
                                dict(kind='cauchy', alpha=2, beta=BVAL, dims=[0, 2], scale=SVAL)])],
        # the differentiated field 2 is the second slot of the factor
        'dims02': [(1.3, [dict(kind='maternp', p=2, dims=[0, 2], scale=SVAL)])],
        # the second term does not depend on field 0; its Cauchy factor does not depend on field 1 either but carries
        # scale and beta
        'indep_term': [(1.0, [dict(kind='maternp', p=1, dims=[0, 1], scale=SVAL)]),
                       (0.4, [dict(kind='expquad', dims=[1], scale=SVAL),
                              dict(kind='cauchy', alpha=2, beta=BVAL, dims=[2], scale=SVAL)])],
    }


NEW_CASES = ('shared_field', 'dims02', 'indep_term')


def _points():
    rng = np.random.default_rng(5)
    x = rng.uniform(-1, 1, (3, 4))
    y = np.concatenate([x[:, :2], rng.uniform(-1, 1, (3, 2))], axis=1)  # two exactly coincident pairs
    return x, y


def _sym_eval(expr, x, y, subs_extra):
    mpmath.mp.dps = 110
    fn = sympy.lambdify((*XS, *YS, S, BETA), expr, modules='mpmath')
    out = np.empty((x.shape[1], y.shape[1]))
    for i in range(x.shape[1]):
        for j in range(y.shape[1]):
            out[i, j] = float(fn(*[mpmath.mpf(v) for v in (*x[:, i], *y[:, j])], mpmath.mpf(SVAL), mpmath.mpf(BVAL)))
    return out


def _sym_block(expr, a, b):
    if a is not None:
        expr = sympy.diff(expr, XS[a])
    if b is not None:
        expr = sympy.diff(expr, YS[b])
    return expr


@pytest.mark.parametrize('name', list(_cases()))
@pytest.mark.parametrize('a, b', [(0, None), (None, 1), (0, 0), (0, 1)])
def test_oracle_vs_sympy(name, a, b):
    _check_oracle_vs_sympy(name, a, b)


@pytest.mark.parametrize('name', NEW_CASES)
@pytest.mark.parametrize('a, b', [(2, None), (None, 2), (2, 2), (1, 2)])
def test_oracle_vs_sympy_field2(name, a, b):
    _check_oracle_vs_sympy(name, a, b)


def _check_oracle_vs_sympy(name, a, b):
    terms = _cases()[name]
    x, y = _points()
    expr = _sym_block(_sym_kernel(terms), a, b)
    ref = _sym_eval(expr, x, y, {})
    got = od.block(terms, x, y, a, b)
    assert np.all(np.isfinite(got))
    np.testing.assert_allclose(got, ref, rtol=1e-13, atol=1e-13 * np.max(np.abs(ref)))
    if isinstance(terms[0][1][0].get('scale'), tuple):
        return
    ders = od.block_derivs(terms, x, y, a, b)
    # d / d log s of the factor scales (every factor of every term has scale s here, or none)
    dl = sum(v for key, v in ders.items() if key[0] == 'logscale' and terms[key[1]][1][key[2]].get('scale'))
    ref_l = _sym_eval(S * sympy.diff(expr, S), x, y, {})
    np.testing.assert_allclose(dl, ref_l, rtol=1e-12, atol=1e-12 * max(np.max(np.abs(ref_l)), 1e-300))
    if any(f['kind'] == 'cauchy' for _, fs in terms for f in fs):
        ref_b = _sym_eval(sympy.diff(expr, BETA), x, y, {})
        db = sum(v for key, v in ders.items() if key[0] == 'beta')
        np.testing.assert_allclose(db, ref_b, rtol=1e-12, atol=1e-12 * max(np.max(np.abs(ref_b)), 1e-300))
    if name in NEW_CASES:
        for ti, (_, fs) in enumerate(terms):
            ref_a = _sym_eval(_sym_block(_sym_term(fs), a, b), x, y, {})
            np.testing.assert_allclose(ders['amp', ti], ref_a, rtol=1e-12, atol=1e-12 * max(np.max(np.abs(ref_a)), 1e-300))


@pytest.mark.parametrize('kind, kw, anchor', [
    ('expquad', {}, 1.0), ('cauchy', dict(alpha=2, beta=0.7), 1.0),
    ('matern', dict(nu=1.5), 3.0), ('matern', dict(nu=2.5), 5 / 3), ('matern', dict(nu=3.5), 7 / 5),
])
def test_r0_anchors(kind, kw, anchor):
    s = 1.3
    x = np.array([[0.3, -0.2]])
    K = od.block([(1.0, [dict(kind=kind, scale=s, **kw)])], x, x, 0, 0)
    np.testing.assert_allclose(np.diag(K), anchor / s ** 2, rtol=1e-15)


# ---- hyperparameter derivatives of the plain cores (oracle.gp.factor_dlogscale, oracle.deriv.block_derivs) vs mpmath

def _mp_core(kind, r2, nu=None, alpha=None, beta=None):
    if kind == 'matern':
        if r2 == 0:
            return mpmath.mpf(1)
        x = mpmath.sqrt(2 * nu * r2)
        return 2 / mpmath.gamma(nu) * (x / 2) ** nu * mpmath.besselk(nu, x)
    return (1 + r2 ** (alpha / 2) / beta) ** (-beta / alpha)


# squared distances (before the scale 1.7): 0, tiny, moderate and large
_R2 = [0.0, 1e-300, 1e-200, 1e-30, 1e-12, 1e-6, 0.01, 0.3, 1.0, 2.5, 10.0, 60.0]


@pytest.mark.parametrize('kind, kw', [('matern', dict(nu=0.3)), ('matern', dict(nu=1.3)), ('matern', dict(nu=4.2)),
                                      ('cauchy', dict(alpha=1.3, beta=0.7)), ('cauchy', dict(alpha=0.5, beta=3.0)),
                                      ('cauchy', dict(alpha=2, beta=1.3))])
def test_dlogscale_and_dbeta_vs_mpmath(kind, kw):
    """ d/d log(scale) of every core and d/d beta of Cauchy of any alpha, on plain (underived) blocks, against mpmath
    differentiation to 40 digits (working precision 360 digits: 1 + t / beta and the Bessel series cancel the digits
    of tiny t) """
    s = 1.7
    x = np.sqrt(np.array(_R2))[None, :]
    y = np.zeros((1, 1))
    f = dict(kind=kind, scale=s, **kw)
    got_l = ogp.factor_dlogscale(f, x, y)[:, 0]
    ders = od.block_derivs([(1.0, [f])], x, y)
    np.testing.assert_array_equal(ders['logscale', 0, 0][:, 0], got_l)
    mpmath.mp.dps = 360
    mkw = {k: mpmath.mpf(v) for k, v in kw.items()}
    for i, r2 in enumerate(_R2):
        R = mpmath.mpf(r2) / mpmath.mpf(s) ** 2
        ref = mpmath.diff(lambda ls: _mp_core(kind, R * mpmath.exp(-2 * ls), **mkw), 0) if r2 else 0
        assert abs(got_l[i] - float(ref)) <= 1e-13 * max(abs(float(ref)), 1e-300) + 1e-300, (r2, got_l[i], ref)
        if kind == 'cauchy':
            kb = dict(mkw)
            del kb['beta']
            ref_b = mpmath.diff(lambda b: _mp_core(kind, R, beta=b, **kb), mkw['beta'])
            got_b = ders['beta', 0, 0][i, 0]
            # d/dbeta = c (t / (alpha beta B) - log(B) / alpha), B = 1 + t/beta: the two terms cancel to O(t^2)
            t = float(R / mpmath.mpf(s) ** 2) ** (kw['alpha'] / 2)
            size = t / (kw['alpha'] * kw['beta'])
            assert abs(got_b - float(ref_b)) <= 1e-13 * (abs(float(ref_b)) + size) + 1e-300, (r2, got_b, ref_b)


# ---- host build of csrc/deriv_core.cuh vs the oracle

@pytest.fixture(scope='module')
def host(tmp_path_factory):
    """ oracle/deriv_core_host.c (which includes csrc/deriv_core.cuh) compiled with g++ into a temporary directory """
    so = tmp_path_factory.mktemp('deriv_core_host') / 'libderiv_core_host.so'
    subprocess.run(['g++', '-x', 'c++', '-std=c++17', '-O2', '-fPIC', '-shared', '-ffp-contract=off', '-o', str(so),
                    str(ROOT / 'oracle' / 'deriv_core_host.c'), '-lm'], check=True)
    lib = ctypes.CDLL(str(so))
    dp = ctypes.POINTER(ctypes.c_double)
    lib.lgp_host_deriv_coefs.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double, dp,
                                         ctypes.c_long, dp, dp]
    return lib, dp


@pytest.mark.parametrize('kind, p, par0, beta', [
    (_lib.K_EXPQUAD, 0, 0.0, 0.0), (_lib.K_CAUCHY, 0, 2.0, 0.7), (_lib.K_CAUCHY, 0, 2.0, 5.0),
    *[(_lib.K_MATERNP, p, par0, 0.0) for p in (1, 2, 3, 4) for par0 in (0.0, 1e-30)],
])
def test_host_coefs_vs_oracle(host, kind, p, par0, beta):
    lib, dp = host
    rng = np.random.default_rng(kind * 10 + p)
    u = np.concatenate([[0.0, 1e-300, 1e-30], 10 ** rng.uniform(-20, 3.3, 100_000)])
    n = u.size
    c = np.empty((n, 4))
    db = np.empty((n, 3))
    lib.lgp_host_deriv_coefs(kind, p, par0, beta, u.ctypes.data_as(dp), n, c.ctypes.data_as(dp), db.ctypes.data_as(dp))
    name = {_lib.K_EXPQUAD: 'expquad', _lib.K_CAUCHY: 'cauchy', _lib.K_MATERNP: 'maternp'}[kind]
    kw = dict(p=p, par0=par0) if name == 'maternp' else dict(beta=beta) if name == 'cauchy' else {}
    rc, rdb = od.coefs(name, u, **kw)
    # the products the kernels form: c, c' alone; c'' with a factor u (D_a D_b <= u), c''' with u^2 (u D_a D_b)
    weights = [1.0, 1.0, u, u * u]
    for j in range(4):
        got = od.mul0(c[:, j], weights[j]) if j >= 2 else c[:, j]
        ref = od.mul0(rc[j], weights[j]) if j >= 2 else rc[j]
        assert np.all(np.isfinite(got)), j
        np.testing.assert_allclose(got, ref, rtol=2e-15, atol=1e-300)
    for j in range(3):
        # d/dbeta is c^(j) times a sum of terms that cancel near its zero: the tolerance scales with those terms
        scale = 1.0
        if name == 'cauchy':
            scale = 1 + j / beta + np.abs(np.log1p(u / beta)) + (0.5 * beta + j) * u / (beta * (beta + u))
        assert np.all(np.abs(db[:, j] - rdb[j]) <= 2e-15 * np.abs(rdb[j]) + 1e-300 + 2e-15 * np.abs(c[:, j]) * scale), j
    if kind == _lib.K_MATERNP and par0 == 0.0:
        np.testing.assert_allclose(-2 * c[0, 1], (2 * p + 1) / (2 * p - 1), rtol=1e-15)
