"""Second derivatives on the GPU: the second-order Gram contraction (lgp_gram_iso_hvp) against the exact oracle
(oracle/hess.py), the Hessian of the marginal likelihood through the public API (torch.autograd.functional.hessian over
twice-differentiable autograd nodes) against the oracle's exact logML Hessian, the unchanged first order under
create_graph, empbayes_fit(method='hessian', covariance='hessian'), and the refusals of second derivatives the library
does not implement.

Bars: a contraction within 1e-12 sum |G (tangent . d2K)| of the oracle per output (atomicAdd order varies the last
bits); logML Hessians within 1e-9 of the oracle normwise."""
import numpy as np
import pytest
import torch

import lsqfitgp_b200 as lgp
from lsqfitgp_b200 import _lib, _ops
from oracle import gp as ogp, hess as oh

pytestmark = pytest.mark.gpu

f64 = torch.float64
KIND = {'expquad': _lib.K_EXPQUAD, 'maternp': _lib.K_MATERNP, 'matern': _lib.K_MATERN, 'cauchy': _lib.K_CAUCHY,
        'white': _lib.K_WHITE, 'constant': _lib.K_CONSTANT}


def _pair(v, default):
    return v if isinstance(v, tuple) else (default if v is None else v,) * 2


def descs_of(terms, ndim):
    """ C-ABI descriptors of a kernel in the oracle's format (oracle/gp.py); Maternp carries its offset as par0 """
    out = []
    for ti, (amp, factors) in enumerate(terms):
        for fi, f in enumerate(factors):
            dims = range(ndim) if f.get('dims') is None else f['dims']
            sx, sy = _pair(f.get('scale'), 1.0)
            lx, ly = _pair(f.get('loc'), 0.0)
            d = dict(kind=KIND[f['kind']], term=ti, dimmask=0 if f['kind'] == 'constant' else sum(1 << k for k in dims),
                     scale_x=sx, scale_y=sy, loc_x=lx, loc_y=ly, amp=amp if fi == 0 else 1.0)
            if f['kind'] == 'maternp':
                d.update(ipar=f['p'], par0=f.get('par0', 1e-30))
            elif f['kind'] == 'matern':
                d.update(par0=f['nu'])
            elif f['kind'] == 'cauchy':
                d.update(par0=f.get('alpha', 2), par1=f.get('beta', 2))
            out.append(d)
    return out


def dev(a):
    return torch.tensor(np.ascontiguousarray(a), dtype=f64, device='cuda')


def points(ndim, n, m, s, seed):
    """ coincident pairs, a duplicated point and a far point, in units of the scale s """
    rng = np.random.default_rng(seed)
    x = rng.uniform(0, 4, (ndim, n))
    y = rng.uniform(0, 4, (ndim, m))
    k = min(n, m, 3)
    y[:, :k] = x[:, :k]
    if n >= 8:
        x[:, 5] = x[:, 6]
        x[:, 7] = x[:, 1] + 40.0
    return x * s, y * s


# ---- lgp_gram_iso_hvp against the oracle

S = 1.7
CASES = {
    'expquad': [(1.3, [dict(kind='expquad', scale=S)])],
    **{f'maternp{p}_par0{z}': [(0.9, [dict(kind='maternp', p=p, par0=z, scale=S)])] for p in range(4) for z in (0.0, 1e-30)},
    **{f'matern{nu}': [(1.1, [dict(kind='matern', nu=nu, scale=S)])] for nu in (0.0, 0.3, 1.3, 4.2)},
    **{f'cauchy{a}': [(0.7, [dict(kind='cauchy', alpha=a, beta=1.4, scale=S)])] for a in (0.5, 1.0, 2.0)},
    'product': [(0.8, [dict(kind='expquad', dims=[0], scale=S), dict(kind='cauchy', alpha=1.3, beta=0.9, dims=[1, 2],
                                                                      scale=1.3),
                       dict(kind='maternp', p=2, par0=0.0, dims=[0, 2], scale=2.1)])],
    'loc_tuple_scale': [(1.2, [dict(kind='maternp', p=1, par0=1e-30, scale=(1.3, 0.9), loc=(0.2, -0.1))]),
                        (0.4, [dict(kind='matern', nu=0.7, scale=S, loc=0.3)])],
    'loc': [(1.2, [dict(kind='maternp', p=1, par0=1e-30, scale=1.3, loc=0.2)]),
            (0.4, [dict(kind='matern', nu=0.7, scale=S, loc=0.3), dict(kind='expquad', dims=[2], scale=0.8)])],
}


def _extras(terms):
    return terms + [(0.05, [dict(kind='white')]), (0.3, [dict(kind='constant')])]


def _check_hvp(terms, x, y, G, tan, got, what):
    ref, size = oh.hvp(terms, x, y, G, tan)
    assert np.all(np.isfinite(got)), what
    bad = np.abs(got - ref) > 1e-12 * size + 1e-300
    assert not np.any(bad), (what, got, ref, size)


@pytest.mark.parametrize('name', list(CASES))
def test_hvp_vs_oracle(name):
    """ every kind, with White and Constant terms, dense G at n != m and tile edges, and symmetric G (lower triangle
    and b) on the diagonal block, each with random and unit tangents """
    terms = _extras(CASES[name])
    descs = descs_of(terms, 3)
    nf = len(descs)
    rng = np.random.default_rng(len(name))
    tangents = [rng.standard_normal((nf, 3)), rng.standard_normal((nf, 3)), np.eye(3 * nf)[1].reshape(nf, 3)]
    for n, m in [(1, 1), (63, 64), (65, 129), (130, 97)]:
        x, y = points(3, n, m, S, n + m)
        G = rng.standard_normal((n, m))
        Gd = _ops.as_aligned(dev(G))
        for t, tan in enumerate(tangents):
            got = _ops.gram_iso_hvp(descs, dev(x), dev(y), Gd, tan).cpu().numpy()
            _check_hvp(terms, x, y, G, tan, got, f'{name} dense {n}x{m} tangent {t}')
    if any(isinstance(f.get(k), tuple) for _, fs in terms for f in fs for k in ('scale', 'loc')):
        return   # different transforms of x and y: K(x, x) is not symmetric, the symmetric form does not apply
    for n in (1, 64, 65, 130):
        x, _ = points(3, n, 1, S, n)
        A = rng.standard_normal((n, n))
        Gs = A + A.T
        b = rng.standard_normal(n)
        low = np.tril(Gs) + np.triu(np.full((n, n), np.nan), 1)   # the upper triangle must not be read
        for t, tan in enumerate(tangents):
            got = _ops.gram_iso_hvp(descs, dev(x), None, _ops.as_aligned(dev(low)), tan, b=dev(b),
                                    symlower=True).cpu().numpy()
            _check_hvp(terms, x, x, Gs - np.outer(b, b), tan, got, f'{name} symlower n={n} tangent {t}')


def test_hvp_symmetry():
    """ out_a with tangent e_b equals out_b with tangent e_a: the columns of the Hessian of sum G K """
    terms = _extras(CASES['product'] + CASES['cauchy1.0'])
    descs = descs_of(terms, 3)
    nf = len(descs)
    x, y = points(3, 97, 130, S, 3)
    G = np.random.default_rng(4).standard_normal((97, 130))
    Gd = _ops.as_aligned(dev(G))
    cols = np.stack([_ops.gram_iso_hvp(descs, dev(x), dev(y), Gd, e.reshape(nf, 3)).cpu().numpy().reshape(-1)
                     for e in np.eye(3 * nf)], axis=1)
    _, size = oh.hvp(terms, x, y, G, np.ones((nf, 3)))
    bar = 1e-12 * np.max(size)
    assert np.max(np.abs(cols - cols.T)) <= bar, np.max(np.abs(cols - cols.T))


# ---- Hessian of the marginal likelihood through the public API

def _logml_derivs(terms_of, q, x, spec):
    """ (K, dK, d2K) at q from the oracle's derivatives in the descriptor coordinates; terms_of(q) builds the oracle
    kernel, spec[a] = (factor, k, c, how): the hyperparameter k of the factor is exp(c q_a) (how = 'exp': an amplitude
    or beta) or q_a itself (how = 'lin': a log scale) """
    terms = terms_of(q)
    d1, d2 = oh.gram_hessian(terms, x, x)
    n = x.shape[1]
    zero = np.zeros((n, n))
    # d theta / d q: c theta for theta = exp(c q); the native amplitude and beta derivatives are taken at theta
    jac = [c * np.exp(c * q[a]) if how == 'exp' else 1.0 for a, (f, k, c, how) in enumerate(spec)]
    dK = [jac[a] * d1[f][k] for a, (f, k, c, how) in enumerate(spec)]
    d2K = [[jac[a] * jac[b] * d2.get((fa, ka, fb, kb), zero) for b, (fb, kb, _, _) in enumerate(spec)]
           for a, (fa, ka, _, _) in enumerate(spec)]
    for a, (f, k, c, how) in enumerate(spec):
        if how == 'exp':
            d2K[a][a] = d2K[a][a] + c * dK[a]
    return ogp.gram(terms, x, x), dK, d2K


def _struct(X):
    return lgp.unstructured_to_structured(X.T.copy(), names=[f'f{i}' for i in range(X.shape[0])])


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


def test_logml_hessian_fused_route():
    """ one key, plain points, kernel-only covariance: the fused Gram -> Chol node """
    rng = np.random.default_rng(11)
    n = 300
    X = rng.uniform(0, 10, (2, n))
    y = rng.standard_normal(n)
    q0 = torch.tensor([0.3, 0.5, np.log(0.2)], dtype=f64)

    def f(q):
        k = torch.exp(q[0]) * lgp.Maternp(p=2, scale=torch.exp(q[1])) + torch.exp(q[2]) * lgp.White()
        return -lgp.GP(k, checkpos=False, checksym=False, epsrel=0).addx(_struct(X), 'a').marginal_likelihood({'a': y})
    H = torch.autograd.functional.hessian(f, q0).numpy()

    def terms_of(q):
        return [(np.exp(q[0]), [dict(kind='maternp', p=2, scale=np.exp(q[1]))]), (np.exp(q[2]), [dict(kind='white')])]
    spec = [(0, 0, 1.0, 'exp'), (0, 1, 1.0, 'lin'), (1, 0, 1.0, 'exp')]
    K, dK, d2K = _logml_derivs(terms_of, q0.numpy(), X, spec)
    Ho = oh.logml_hessian(K, y, dK, d2K)
    assert _rel(H, Ho) <= 1e-9, (H, Ho)


def test_logml_hessian_assembled_route():
    """ two keys and a given covariance: Gram blocks assembled with torch.cat, one shared scale tensor in two factors,
    Cauchy beta as a hyperparameter """
    rng = np.random.default_rng(12)
    n1, n2 = 130, 97
    X1, X2 = rng.uniform(0, 6, (2, n1)), rng.uniform(0, 6, (2, n2))
    y1, y2 = rng.standard_normal(n1), rng.standard_normal(n2)
    C1 = 0.1 * np.eye(n1) + 0.02
    C2 = 0.2 * np.eye(n2)
    q0 = torch.tensor([0.2, 0.4, -0.3], dtype=f64)

    def f(q):
        s = torch.exp(q[1])
        k = (torch.exp(q[0]) * lgp.ExpQuad(scale=s, dim='f0') * lgp.Cauchy(alpha=1.0, beta=torch.exp(q[2]), scale=s)
             + 0.3)
        gp = lgp.GP(k, checkpos=False, checksym=False, epsrel=0).addx(_struct(X1), 'a').addx(_struct(X2), 'b')
        return -gp.marginal_likelihood({'a': y1, 'b': y2}, {('a', 'a'): C1, ('b', 'b'): C2, ('a', 'b'): np.zeros((n1, n2)),
                                                              ('b', 'a'): np.zeros((n2, n1))})
    H = torch.autograd.functional.hessian(f, q0).numpy()

    X = np.concatenate([X1, X2], axis=1)

    def terms_of(q):
        s = np.exp(q[1])
        return [(np.exp(q[0]), [dict(kind='expquad', scale=s, dims=[0]), dict(kind='cauchy', alpha=1.0, beta=np.exp(q[2]),
                                                                              scale=s)]),
                (0.3, [dict(kind='constant')])]
    # the shared scale: d/dq1 = d/dlog scale of factor 0 + of factor 1
    q = q0.numpy()
    d1, d2 = oh.gram_hessian(terms_of(q), X, X)
    N = X.shape[1]
    Z = np.zeros((N, N))
    a0, b0 = np.exp(q[0]), np.exp(q[2])
    dK = [a0 * d1[0][0], d1[0][1] + d1[1][1], b0 * d1[1][2]]
    g = lambda *k: d2.get(k, Z)  # noqa: E731
    d2K = [[a0 * a0 * g(0, 0, 0, 0) + dK[0], a0 * (g(0, 0, 0, 1) + g(0, 0, 1, 1)), a0 * b0 * g(0, 0, 1, 2)],
           [None, g(0, 1, 0, 1) + g(0, 1, 1, 1) + g(1, 1, 0, 1) + g(1, 1, 1, 1), b0 * (g(0, 1, 1, 2) + g(1, 1, 1, 2))],
           [None, None, b0 * b0 * g(1, 2, 1, 2) + dK[2]]]
    for a in range(3):
        for c in range(a):
            d2K[a][c] = d2K[c][a]
    Cy = np.block([[C1, np.zeros((n1, n2))], [np.zeros((n2, n1)), C2]])
    Ho = oh.logml_hessian(ogp.gram(terms_of(q), X, X) + Cy, np.concatenate([y1, y2]), dK, d2K)
    assert _rel(H, Ho) <= 1e-9, (H, Ho)


def test_logml_hessian_data_depend_on_hyperparameter():
    """ the data minus a mean that depends on a hyperparameter: the r-terms of the Hessian (fused route) """
    rng = np.random.default_rng(13)
    n = 200
    X = rng.uniform(0, 8, (1, n))
    t = rng.uniform(-1, 1, n)
    y = rng.standard_normal(n) + 0.7 * t
    q0 = torch.tensor([0.1, 0.3, np.log(0.5)], dtype=f64)
    td = torch.tensor(t, dtype=f64)

    def f(q):
        k = torch.exp(q[0]) * lgp.ExpQuad(scale=torch.exp(q[1])) + 0.1 * lgp.White()
        r = torch.tensor(y, dtype=f64) - torch.exp(q[2]) * td
        return -lgp.GP(k, checkpos=False, checksym=False, epsrel=0).addx(_struct(X), 'a').marginal_likelihood({'a': r})
    H = torch.autograd.functional.hessian(f, q0).numpy()

    q = q0.numpy()

    def terms_of(q):
        return [(np.exp(q[0]), [dict(kind='expquad', scale=np.exp(q[1]))]), (0.1, [dict(kind='white')])]
    K, dK2, d2K2 = _logml_derivs(terms_of, q[:2], X, [(0, 0, 1.0, 'exp'), (0, 1, 1.0, 'lin')])
    Z = np.zeros((n, n))
    dK = dK2 + [Z]
    d2K = [row + [Z] for row in d2K2] + [[Z, Z, Z]]
    z = np.zeros(n)
    dr = [z, z, -np.exp(q[2]) * t]
    d2r = [[z, z, z], [z, z, z], [z, z, -np.exp(q[2]) * t]]
    Ho = oh.logml_hessian(K, y - np.exp(q[2]) * t, dK, d2K, dr, d2r)
    assert _rel(H, Ho) <= 1e-9, (H, Ho)


def test_first_order_unchanged_under_create_graph():
    """ the gradient built for a second differentiation equals the ordinary one (fused and assembled routes) """
    rng = np.random.default_rng(14)
    X = rng.uniform(0, 10, (2, 257))
    y = rng.standard_normal(257)
    for two_keys in (False, True):
        q = torch.tensor([0.3, 0.5, np.log(0.2)], dtype=f64, requires_grad=True)

        def ml():
            k = torch.exp(q[0]) * lgp.Matern(nu=1.3, scale=torch.exp(q[1])) + torch.exp(q[2]) * lgp.White()
            gp = lgp.GP(k, checkpos=False, checksym=False)
            if two_keys:
                gp = gp.addx(_struct(X[:, :100]), 'a').addx(_struct(X[:, 100:]), 'b')
                return gp.marginal_likelihood({'a': y[:100], 'b': y[100:]})
            return gp.addx(_struct(X), 'a').marginal_likelihood({'a': y})
        g0, = torch.autograd.grad(ml(), q)
        g1, = torch.autograd.grad(ml(), q, create_graph=True)
        assert g1.requires_grad
        np.testing.assert_allclose(g1.detach().numpy(), g0.numpy(), rtol=1e-13, atol=0)


# ---- empbayes_fit(method='hessian', covariance='hessian')

def test_empbayes_fit_hessian_vs_gradient_fisher_and_oracle():
    rng = np.random.default_rng(3005)
    n = 300
    X3 = rng.uniform(0, 100, (n, 2))
    K3 = ogp.gram([(1.3 ** 2, [dict(kind='expquad', scale=8.0)])], X3.T.copy(), X3.T.copy())
    y3 = np.linalg.cholesky(K3 + 1e-10 * np.eye(n)) @ rng.standard_normal(n) + 0.2 * rng.standard_normal(n)
    x3 = lgp.unstructured_to_structured(X3, names=['a', 'b'])
    mean = np.array([np.log(3), 0.0, np.log(0.1)])
    hyperprior = {'log(ell)': (mean[0], 1.0), 'log(sf)': (mean[1], 1.0), 'log(sn)': (mean[2], 1.0)}

    def gpfactory(hp):
        k = hp['sf'] ** 2 * lgp.ExpQuad(scale=hp['ell']) + hp['sn'] ** 2 * lgp.White()
        return lgp.GP(k, checkpos=False, checksym=False, epsrel=0).addx(x3, 'data')
    fitg = lgp.empbayes_fit(hyperprior, gpfactory, {'data': y3}, raises=False)
    fitf = lgp.empbayes_fit(hyperprior, gpfactory, {'data': y3}, raises=False, method='fisher')
    fith = lgp.empbayes_fit(hyperprior, gpfactory, {'data': y3}, method='hessian', covariance='hessian')
    assert fith._ncalls['hess'] >= 1
    for other in (fitg, fitf):
        assert np.max(np.abs(fith.minresult.x - other.minresult.x)) < 1e-4
        assert abs(fith.minresult.fun - other.minresult.fun) / abs(other.minresult.fun) < 1e-8

    # the oracle's Hessian of -logML + p.p/2 at the optimum, p = whitened parameters (prior sdev 1: q = mean + p)
    q = mean + fith.minresult.x

    def terms_of(q):
        return [(np.exp(2 * q[1]), [dict(kind='expquad', scale=np.exp(q[0]))]), (np.exp(2 * q[2]), [dict(kind='white')])]
    spec = [(0, 1, 1.0, 'lin'), (0, 0, 2.0, 'exp'), (1, 0, 2.0, 'exp')]
    K, dK, d2K = _logml_derivs(terms_of, q, X3.T.copy(), spec)
    Ho = oh.logml_hessian(K, y3, dK, d2K) + np.eye(3)
    cov = np.array([[fith.pcov[a, b] for b in hyperprior] for a in hyperprior])
    assert _rel(cov, np.linalg.inv(Ho)) <= 1e-8


# ---- refusals

def test_second_order_refusals():
    rng = np.random.default_rng(15)
    n = 60
    X = rng.uniform(0, 5, (2, n))
    y = rng.standard_normal(n)

    def check(make, match):
        q = torch.tensor([0.9, 1.6, 0.3], dtype=f64, requires_grad=True)
        g, = torch.autograd.grad(make(q), q)   # the first order still works
        assert torch.all(torch.isfinite(g))
        with pytest.raises(NotImplementedError, match=match):
            torch.autograd.functional.hessian(make, q.detach())

    splits = lgp.BART.splits_from_coord(X.T)

    def bart(q):
        k = q[2] ** 2 * lgp.BART(splits=splits, alpha=q[0], beta=q[1], maxd=4, reset=2) + 0.3 * lgp.White()
        return lgp.GP(k, checkpos=False, checksym=False).addx(_struct(X), 'a').marginal_likelihood({'a': y})
    check(bart, 'BART')

    def deriv(q):
        k = torch.exp(q[2]) * lgp.ExpQuad(scale=q[1])
        gp = (lgp.GP(k, checkpos=False, checksym=False).addx(_struct(X[:, :30]), 'a')
              .addx(_struct(X[:, 30:]), 'd', deriv='f0'))
        noise = {('a', 'a'): 0.1 * np.eye(30), ('d', 'd'): 0.1 * np.eye(n - 30), ('a', 'd'): np.zeros((30, n - 30)),
                 ('d', 'a'): np.zeros((n - 30, 30))}
        return gp.marginal_likelihood({'a': y[:30], 'd': y[30:]}, noise)
    check(deriv, 'derivative observations')

    k = torch.tensor(1.3, dtype=f64, requires_grad=True) * lgp.ExpQuad()
    gp = lgp.GP(k, solver='chol-dist', checkpos=False, checksym=False).addx(_struct(X), 'a')
    with pytest.raises(NotImplementedError, match='chol-dist'):
        gp.marginal_likelihood({'a': y})
