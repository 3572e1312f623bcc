"""Derivative observations and predictions on the GPU (lgp_gram_iso_deriv and its VJP / JVP) against the NumPy
oracle (oracle/deriv.py), finite differences of the plain Gram kernel and the GP-level oracle."""
import numpy as np
import pytest
import torch

import lsqfitgp_b200 as lgp
from lsqfitgp_b200 import _ops
from oracle import deriv as od, gp as ogp

pytestmark = pytest.mark.gpu

S = 1.7
KERNELS = {
    'expquad': (lambda: lgp.ExpQuad(scale=S), [(1.0, [dict(kind='expquad', scale=S)])]),
    **{f'maternp{p}': (lambda p=p: lgp.Maternp(p=p, scale=S), [(1.0, [dict(kind='maternp', p=p, scale=S)])])
       for p in (1, 2, 3, 4)},
    **{f'matern{nu}': (lambda nu=nu: lgp.Matern(nu=nu, scale=S), [(1.0, [dict(kind='matern', nu=nu, scale=S)])])
       for nu in (1.5, 2.5, 3.5)},
    'cauchy': (lambda: lgp.Cauchy(alpha=2, beta=1.3, scale=S), [(1.0, [dict(kind='cauchy', alpha=2, beta=1.3, scale=S)])]),
    'product': (lambda: 0.8 * lgp.ExpQuad(scale=S, dim='a') * lgp.Maternp(p=2, scale=S, dim='b'),
                [(0.8, [dict(kind='expquad', dims=[0], scale=S), dict(kind='maternp', p=2, dims=[1], scale=S)])]),
    'sum_const': (lambda: lgp.Maternp(p=2, scale=S) + 0.3, [(1.0, [dict(kind='maternp', p=2, scale=S)]),
                                                            (0.3, [dict(kind='constant')])]),
    'loc': (lambda: lgp.Maternp(p=1, scale=S, loc=0.4), [(1.0, [dict(kind='maternp', p=1, scale=S, loc=0.4)])]),
    'tuple_scale': (lambda: lgp.ExpQuad(scale=(1.3, 0.9), loc=(0.2, -0.1)),
                    [(1.0, [dict(kind='expquad', scale=(1.3, 0.9), loc=(0.2, -0.1))])]),
}


def _pts(n, seed, dup=0):
    rng = np.random.default_rng(seed)
    X = rng.uniform(-2, 2, (n, 2))
    if dup:
        X[:dup] = X[n - dup:]
    return X


def _sa(X):
    return lgp.unstructured_to_structured(X, names=['a', 'b'])


def _nwerr(got, ref):
    return np.max(np.abs(got - ref)) / np.max(np.abs(ref))


@pytest.mark.parametrize('name', list(KERNELS))
@pytest.mark.parametrize('da, db', [('a', None), (None, 'b'), ('a', 'a'), ('a', 'b')])
def test_linop_diff_vs_oracle(name, da, db):
    mk, terms = KERNELS[name]
    X, Y = _pts(150, 1, dup=10), _pts(130, 2)
    Y[:5] = X[:5]                                             # coincident pairs
    got = mk().linop('diff', da or 0, db or 0)(_sa(X)[:, None], _sa(Y)[None, :])
    fa = {'a': 0, 'b': 1, None: None}
    ref = od.block(terms, X.T.copy(), Y.T.copy(), fa[da], fa[db])
    assert np.all(np.isfinite(got))
    assert _nwerr(got, ref) < 1e-13
    # central differences of the plain GPU Gram
    if name != 'tuple_scale' and (da is None or db is None):
        k = mk()
        h = 1e-5
        shift = np.zeros(2)
        shift[fa[da or db]] = h
        if da:
            fd = (k(_sa(X + shift)[:, None], _sa(Y)[None, :]) - k(_sa(X - shift)[:, None], _sa(Y)[None, :])) / (2 * h)
        else:
            fd = (k(_sa(X)[:, None], _sa(Y + shift)[None, :]) - k(_sa(X)[:, None], _sa(Y - shift)[None, :])) / (2 * h)
        assert _nwerr(got, fd) < 1e-6


@pytest.mark.parametrize('name', ['expquad', 'maternp1', 'matern2.5', 'cauchy', 'product', 'sum_const'])
@pytest.mark.parametrize('field', ['a', 'b'])
def test_symmetric_mode_bit_identical(name, field):
    mk, _ = KERNELS[name]
    k = mk()
    X = _pts(300, 3, dup=7)
    labels = ['a', 'b']
    xd = torch.from_numpy(X.T.copy()).cuda()
    f = labels.index(field)
    gen = k._gram_device(xd, xd.clone(), labels, dfields=(f, f)).cpu().numpy()
    sym = k._gram_device(xd, xd, labels, symmetric=True, dfields=(f, f)).cpu().numpy()
    assert np.array_equal(gen, sym)
    assert np.array_equal(sym, sym.T)
    assert np.all(np.isfinite(np.diag(sym)))


def _gp_parts(n=60, seed=11):
    X = _pts(n, seed)
    x = _sa(X)
    return X, x


def test_prior_joint_vs_oracle():
    X, x = _gp_parts()
    mk, terms = KERNELS['matern2.5']
    gp = lgp.GP(mk()).addx(x, 'f').addx(x, 'dfa', deriv='a').addx(x[:30], 'dfb', deriv='b')
    cov = gp.prior(raw=True)
    Xt = X.T.copy()
    parts = [('f', Xt, None), ('dfa', Xt, 0), ('dfb', Xt[:, :30], 1)]
    for r, xr, ar in parts:
        for c, xc, ac in parts:
            ref = od.block(terms, xr, xc, ar, ac)
            assert _nwerr(cov[r, c], ref) < 1e-13, (r, c)


def test_pred_derivatives_vs_oracle():
    X, x = _gp_parts(80, 12)
    mk, terms = KERNELS['expquad']
    rng = np.random.default_rng(4)
    y = np.sin(X[:, 0]) * np.cos(X[:, 1])
    noise = 1e-4 * np.eye(80)
    gp = lgp.GP(mk()).addx(x, 'f').addx(x[:20], 'dfa', deriv='a').addx(x[:20], 'dfb', deriv='b')
    mean, cov = gp.predfromdata({'f': y}, ['dfa', 'dfb'], {('f', 'f'): noise}, raw=True)
    Xt = X.T.copy()
    Kxx = od.block(terms, Xt, Xt) + noise
    parts = [(Xt[:, :20], 0), (Xt[:, :20], 1)]
    Kxs = np.concatenate([od.block(terms, Xt, xs, None, b) for xs, b in parts], axis=1)
    Kss = od.joint_cov(terms, parts)
    m_o, c_o = ogp.pred(Kxx, Kxs, Kss, y)
    m = np.concatenate([mean['dfa'], mean['dfb']])
    c = np.block([[cov['dfa', 'dfa'], cov['dfa', 'dfb']], [cov['dfb', 'dfa'], cov['dfb', 'dfb']]])
    assert _nwerr(m, m_o) < 1e-9 and _nwerr(c, c_o) < 1e-9
    # values from derivative data plus one value
    yd = rng.standard_normal(20)
    gp2 = lgp.GP(mk()).addx(x[:20], 'd', deriv='a').addx(x[:1], 'v').addx(x[20:40], 'out')
    mean2, cov2 = gp2.predfromdata({'d': yd, 'v': [0.3]}, 'out', raw=True)
    inp = [(Xt[:, :20], 0), (Xt[:, :1], None)]
    Kxx2 = od.joint_cov(terms, inp)
    Kxs2 = np.concatenate([od.block(terms, xi, Xt[:, 20:40], ai, None) for xi, ai in inp], axis=0)
    m2, c2 = ogp.pred(Kxx2, Kxs2, od.block(terms, Xt[:, 20:40], Xt[:, 20:40]), np.concatenate([yd, [0.3]]))
    assert _nwerr(mean2, m2) < 1e-9 and _nwerr(cov2, c2) < 1e-9


def test_sin_predicts_cos():
    x = np.linspace(0, 2 * np.pi, 40)
    gp = lgp.GP(lgp.ExpQuad(scale=1.0)).addx(x, 'f').addx(x[5:-5], 'df', deriv=1)
    mean = gp.predfromdata({'f': np.sin(x)}, 'df', raw=True)[0]
    assert np.max(np.abs(mean - np.cos(x[5:-5]))) < 1e-3


def _ml_setup():
    X = _pts(70, 21)
    x = _sa(X)
    rng = np.random.default_rng(8)
    y = {'f': rng.standard_normal(70), 'dfa': rng.standard_normal(25), 'dfb': rng.standard_normal(25)}
    Xt = X.T.copy()
    parts = [(Xt, None), (Xt[:, :25], 0), (Xt[:, 25:50], 1)]
    noise = {k: 0.01 * np.eye(len(v)) for k, v in y.items()}
    return x, y, parts, noise


def _terms(theta):
    amp, s, beta = np.exp(theta)
    return [(amp ** 2, [dict(kind='cauchy', alpha=2, beta=beta, scale=s)])]


def _oracle_ml(theta, parts, yv, noise):
    K = od.joint_cov(_terms(theta), parts) + noise
    return ogp.logml(K, yv)


def _gp_ml(theta_t, x, y, noise, keys=('f', 'dfa', 'dfb')):
    amp, s, beta = torch.exp(theta_t)
    k = amp ** 2 * lgp.Cauchy(alpha=2, beta=beta, scale=s)
    gp = lgp.GP(k, checkpos=False, checksym=False).addx(x, 'f').addx(x[:25], 'dfa', deriv='a') \
        .addx(x[25:50], 'dfb', deriv='b')
    gc = {(a, b): (noise[a] if a == b else np.zeros((len(y[a]), len(y[b])))) for a in keys for b in keys}
    return gp.marginal_likelihood({k_: y[k_] for k_ in keys}, gc)


def test_marginal_likelihood_and_gradient_vs_oracle():
    x, y, parts, noise = _ml_setup()
    theta = np.array([0.1, np.log(1.2), np.log(1.7)])
    tt = torch.tensor(theta, dtype=torch.float64, requires_grad=True)
    ml = _gp_ml(tt, x, y, noise)
    g, = torch.autograd.grad(ml, tt)
    yv = np.concatenate([y['f'], y['dfa'], y['dfb']])
    nz = np.diag(np.concatenate([np.diag(noise[k]) for k in ('f', 'dfa', 'dfb')]))
    ref = _oracle_ml(theta, parts, yv, nz)
    assert abs(float(ml.detach()) - ref) / abs(ref) < 1e-9
    h = 1e-5
    fd = np.array([(_oracle_ml(theta + h * e, parts, yv, nz) - _oracle_ml(theta - h * e, parts, yv, nz)) / (2 * h)
                   for e in np.eye(3)])
    assert np.max(np.abs(g.numpy() - fd)) / np.max(np.abs(fd)) < 1e-6
    with torch.no_grad():
        v = _gp_ml(torch.tensor(theta), x, y, noise)
    assert abs(v - ref) / abs(ref) < 1e-9


@pytest.mark.parametrize('da, db', [(0, -1), (-1, 1), (0, 0), (0, 1)])
def test_vjp_jvp_adjoint(da, db):
    """ <G, JVP(t)> = <t, VJP(G)>: the reverse- and forward-mode kernels differentiate the same block """
    k = 1.3 * lgp.Maternp(p=2, scale=0.8, dim='a') * lgp.Cauchy(alpha=2, beta=1.4, scale=1.1) + 0.4 * lgp.ExpQuad(scale=0.7)
    descs, _ = k._descriptor(['a', 'b'])
    X, Y = _pts(200, 31, dup=4), _pts(170, 32)
    Y[:3] = X[:3]
    xd, yd = torch.from_numpy(X.T.copy()).cuda(), torch.from_numpy(Y.T.copy()).cuda()
    G = _ops.as_aligned(torch.from_numpy(np.random.default_rng(3).standard_normal((200, 170))).cuda())
    vjp = _ops.gram_iso_deriv_vjp(descs, xd, yd, da, db, G).cpu().numpy()
    rng = np.random.default_rng(9)
    for _ in range(3):
        t = rng.standard_normal((len(descs), 3))
        D = _ops.gram_iso_deriv_jvp(descs, xd, yd, da, db, t)
        lhs = float((G * D).sum())
        rhs = float((t * vjp).sum())
        assert abs(lhs - rhs) / max(abs(lhs), np.max(np.abs(t * vjp))) < 1e-12


def test_single_derivative_key_takes_assembled_path():
    X = _pts(90, 41)
    x = _sa(X)
    y = np.random.default_rng(2).standard_normal(90)

    def ml(split):
        th = torch.tensor([0.2, np.log(0.3)], dtype=torch.float64, requires_grad=True)
        k = torch.exp(th[0]) * lgp.ExpQuad(scale=torch.exp(th[1]))
        gp = lgp.GP(k, checkpos=False, checksym=False)
        if split:
            gp = gp.addx(x[:40], 'd1', deriv='a').addx(x[40:], 'd2', deriv='a')
            v = gp.marginal_likelihood({'d1': y[:40], 'd2': y[40:]})
        else:
            v = gp.addx(x, 'd', deriv='a').marginal_likelihood({'d': y})
        return float(v.detach()), torch.autograd.grad(v, th)[0].numpy()
    v1, g1 = ml(False)
    v2, g2 = ml(True)
    assert abs(v1 - v2) / abs(v2) < 1e-12
    assert np.max(np.abs(g1 - g2)) / np.max(np.abs(g2)) < 1e-12
    with torch.no_grad():
        gp = lgp.GP(lgp.ExpQuad(scale=0.3)).addx(x, 'd', deriv='a')
        gp2 = lgp.GP(lgp.ExpQuad(scale=0.3)).addx(x[:40], 'd1', deriv='a').addx(x[40:], 'd2', deriv='a')
        assert abs(gp.marginal_likelihood({'d': y}) - gp2.marginal_likelihood({'d1': y[:40], 'd2': y[40:]})) \
            < 1e-12 * abs(gp2.marginal_likelihood({'d1': y[:40], 'd2': y[40:]}))


@pytest.mark.parametrize('method, forward', [('gradient', False), ('gradient', True), ('fisher', False)])
def test_empbayes_fit_gradient_enhanced(method, forward):
    X = np.linspace(0, 6, 25)
    rng = np.random.default_rng(6)
    y = {'f': np.sin(X) + 0.05 * rng.standard_normal(25), 'df': np.cos(X) + 0.05 * rng.standard_normal(25)}
    gc = {('f', 'f'): 0.0025 * np.eye(25), ('df', 'df'): 0.0025 * np.eye(25),
          ('f', 'df'): np.zeros((25, 25)), ('df', 'f'): np.zeros((25, 25))}
    hyperprior = {'log(s)': (0.0, 1.0), 'log(a)': (0.0, 1.0)}

    def gpfactory(hp):
        return lgp.GP(hp['a'] ** 2 * lgp.ExpQuad(scale=hp['s']), checkpos=False, checksym=False) \
            .addx(X, 'f').addx(X, 'df', deriv=1)
    fit = lgp.empbayes_fit(hyperprior, gpfactory, (y, gc), raises=False, method=method, forward=forward)
    Xt = X[None, :]
    noise = 0.0025 * np.eye(50)
    yv = np.concatenate([y['f'], y['df']])

    def obj(p):
        s, a = np.exp(p)
        terms = [(a ** 2, [dict(kind='expquad', scale=s)])]
        K = od.joint_cov(terms, [(Xt, None), (Xt, 0)]) + noise
        return -ogp.logml(K, yv) + 0.5 * (2 * np.log(2 * np.pi) + p @ p)
    p = fit.minresult.x
    h = 1e-5
    fdg = np.array([(obj(p + h * e) - obj(p - h * e)) / (2 * h) for e in np.eye(2)])
    assert np.max(np.abs(fdg)) < 1e-4, fdg


def test_error_semantics():
    x = _sa(_pts(10, 1))
    for k in (lgp.White(), lgp.Cauchy(alpha=1), lgp.Maternp(p=0),
              lgp.BART(splits=lgp.BART.splits_from_coord(_pts(10, 1)))):
        with pytest.raises(ValueError):
            lgp.GP(k).addx(x, 'd', deriv='a')
    for spec in ({'a': 2}, ['a', 'b']):
        with pytest.raises(NotImplementedError):
            lgp.GP(lgp.ExpQuad()).addx(x, 'd', deriv=spec)
    with pytest.raises(ValueError):
        lgp.GP(lgp.ExpQuad()).addx(x, 'd', deriv=1)           # implicit on structured points
    with pytest.raises(ValueError):
        lgp.GP(lgp.ExpQuad()).addx(np.arange(3.), 'd', deriv='a')   # named on unstructured points
    with pytest.raises(ValueError):
        lgp.GP(lgp.ExpQuad()).addx(x, 'd', deriv='c')
    with pytest.raises(ValueError):
        lgp.GP(lgp.Maternp(p=1)).addx(np.arange(3.), 'd', deriv=2)
