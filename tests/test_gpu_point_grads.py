"""Gradients with respect to the input points on the GPU: the point-VJP and point-JVP of the Gram build
(lgp_gram_iso_xvjp, lgp_gram_iso_xjvp) against the exact oracle (oracle/xgrad.py), their argument checks, the gradient
of the marginal likelihood with respect to points given as torch tensors through the public API (fused one-key route,
assembled route, BART), empbayes_fit with a `gpfactory` that shifts points by a hyperparameter, and the refusals.

Bars: a VJP output within 1e-12 sum_j |G_ij dK_ij| of the oracle (atomicAdd order varies the last bits), a JVP matrix
within 1e-13 normwise, the adjoint identity to 1e-12, logML gradients within 1e-9 of the oracle normwise."""
import numpy as np
import pytest
import torch

import lsqfitgp_b200 as lgp
from lsqfitgp_b200 import _lib, _ops
from oracle import gp as ogp, xgrad as ox

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


def points(ndim, n, m, seed):
    """ coincident pairs across x and y and a duplicated point within x """
    rng = np.random.default_rng(seed)
    x = rng.uniform(0, 4, (ndim, n))
    y = rng.uniform(0, 4, (ndim, m))
    k = min(n, m, 3)
    y[:, :k] = x[:, :k]
    if n >= 8:
        x[:, 5] = x[:, 6]
    return x, y


S = 1.7
CASES = {
    'expquad': [(1.3, [dict(kind='expquad', scale=S)])],
    **{f'maternp{p}': [(0.9, [dict(kind='maternp', p=p, scale=S)])] for p in range(4)},
    **{f'matern{nu}': [(1.1, [dict(kind='matern', nu=nu, scale=S)])] for nu in (0.3, 1.3, 4.2)},
    **{f'cauchy{a}': [(0.7, [dict(kind='cauchy', alpha=a, beta=1.4, scale=S)])] for a in (0.5, 1.0, 2.0)},
    'white_constant': [(0.5, [dict(kind='white')]), (0.3, [dict(kind='constant')]),
                       (0.8, [dict(kind='expquad', scale=S)])],
    'product_partial_dims': [(0.8, [dict(kind='expquad', dims=[0], scale=S),
                                    dict(kind='cauchy', alpha=1.3, beta=0.9, dims=[1, 2], scale=1.3),
                                    dict(kind='maternp', p=2, dims=[0, 2], scale=2.1)]),
                             (0.4, [dict(kind='matern', nu=0.7, dims=[1], scale=S)])],
    'loc': [(1.2, [dict(kind='maternp', p=1, scale=1.3, loc=0.2)]),
            (0.4, [dict(kind='matern', nu=0.7, scale=S, loc=0.3), dict(kind='expquad', dims=[2], scale=0.8)])],
}
# a kernel with different scales / locs for the two arguments is not symmetric: dense G only
PAIRS = {'scale_loc_pairs': [(1.2, [dict(kind='maternp', p=1, scale=(1.3, 0.9), loc=(0.2, -0.1))]),
                             (0.4, [dict(kind='expquad', scale=(0.7, 1.6), loc=(0.3, 0.1))])]}


def _check(got, ref, size, what):
    err = np.abs(got - ref)
    bar = 1e-12 * size + 1e-300
    assert np.all(np.isfinite(got)), what
    assert np.all(err <= bar), (what, float(np.max(err / bar)))


@pytest.mark.parametrize('nm', [(1, 5), (63, 65), (64, 1), (65, 129)])
@pytest.mark.parametrize('name', sorted({**CASES, **PAIRS}))
def test_xvjp_dense_vs_oracle(name, nm):
    terms = {**CASES, **PAIRS}[name]
    n, m = nm
    x, y = points(3, n, m, 11 + n + m)
    G = np.random.default_rng(n * m).standard_normal((n, m))
    gx, gy = _ops.gram_iso_xvjp(descs_of(terms, 3), dev(x), dev(y), dev(G))
    rx, ry, sx, sy = ox.xvjp(terms, x, y, G)
    _check(gx.cpu().numpy(), rx, sx, 'gx')
    _check(gy.cpu().numpy(), ry, sy, 'gy')
    # one side only
    gx1, gy1 = _ops.gram_iso_xvjp(descs_of(terms, 3), dev(x), dev(y), dev(G), need_y=False)
    assert gy1 is None
    _check(gx1.cpu().numpy(), rx, sx, 'gx alone')


def _sym_case(n, seed):
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((n, n))
    Gfull = A + A.T
    b = rng.standard_normal(n)
    buf = np.tril(Gfull) + np.triu(np.full((n, n), np.nan), 1)   # the upper triangle must never be read
    return Gfull, b, buf


@pytest.mark.parametrize('n', [1, 63, 64, 65, 129])
@pytest.mark.parametrize('name', sorted(CASES))
def test_xvjp_symlower_vs_oracle(name, n):
    terms = CASES[name]
    x, _ = points(3, n, n, 5 + n)
    Gfull, b, buf = _sym_case(n, n)
    Gs = Gfull - np.outer(b, b)
    got, gy = _ops.gram_iso_xvjp(descs_of(terms, 3), dev(x), None, dev(buf), dev(b), symlower=True)
    assert gy is None
    dx, dy = ox.gram_xgrad(terms, x, x)
    ref = (Gs * dx).sum(2) + (Gs * dy).sum(1)
    size = np.abs(Gs * dx).sum(2) + np.abs(Gs * dy).sum(1)
    _check(got.cpu().numpy(), ref, size, 'symlower')


@pytest.mark.parametrize('ndim', [1, 32])
def test_xvjp_many_fields(ndim):
    """ 32 fields: 4 accumulators of 64 doubles per slot need more than the 48 KiB default of shared memory """
    terms = [(0.9, [dict(kind='maternp', p=2, scale=4.0)]),
             (0.5, [dict(kind='expquad', dims=list(range(0, ndim, 3)), scale=3.0),
                    dict(kind='cauchy', alpha=1.5, beta=1.1, dims=list(range(ndim // 2 + 1)), scale=2.5)])]
    n, m = 65, 70
    x, y = points(ndim, n, m, ndim)
    G = np.random.default_rng(1).standard_normal((n, m))
    gx, gy = _ops.gram_iso_xvjp(descs_of(terms, ndim), dev(x), dev(y), dev(G))
    rx, ry, sx, sy = ox.xvjp(terms, x, y, G)
    _check(gx.cpu().numpy(), rx, sx, 'gx')
    _check(gy.cpu().numpy(), ry, sy, 'gy')
    Gfull, b, buf = _sym_case(n, 2)
    got, _ = _ops.gram_iso_xvjp(descs_of(terms, ndim), dev(x), None, dev(buf), dev(b), symlower=True)
    Gs = Gfull - np.outer(b, b)
    dx, dy = ox.gram_xgrad(terms, x, x)
    _check(got.cpu().numpy(), (Gs * dx).sum(2) + (Gs * dy).sum(1), np.abs(Gs * dx).sum(2) + np.abs(Gs * dy).sum(1),
           'symlower')
    if ndim == 32:   # fields 31.. of the partial factors: only the first factor depends on them
        assert np.any(gx.cpu().numpy()[-1] != 0)


@pytest.mark.parametrize('kind', ['maternp0', 'cauchy1'])
def test_duplicated_points_mul0(kind):
    """ coincident points where c' diverges at r = 0 (Maternp p = 0 without offset, Cauchy alpha = 1): finite, and the
    coincident pairs contribute exactly 0 """
    f = dict(kind='maternp', p=0, par0=0.0, scale=S) if kind == 'maternp0' else dict(kind='cauchy', alpha=1.0,
                                                                                    beta=1.2, scale=S)
    terms = [(1.0, [f])]
    x = np.array([[0.5, 0.5, 1.0, 0.5, 2.0]])
    G = np.ones((5, 5))
    gx, gy = _ops.gram_iso_xvjp(descs_of(terms, 1), dev(x), dev(x), dev(G))
    gx, gy = gx.cpu().numpy(), gy.cpu().numpy()
    assert np.all(np.isfinite(gx)) and np.all(np.isfinite(gy))
    # only the pairs with a different point count: the reference zeroes the coincident ones (mul0)
    rx, ry, sx, _ = ox.xvjp([(1.0, [dict(f, par0=1e-30) if kind == 'maternp0' else f])], x, x, G)
    _check(gx, rx, sx, 'gx')
    Ginv = np.eye(5)
    got, _ = _ops.gram_iso_xvjp(descs_of(terms, 1), dev(x), None, dev(Ginv), None, symlower=True)
    assert np.all(got.cpu().numpy() == 0)   # a diagonal G: only the r = 0 entries, exactly 0


@pytest.mark.parametrize('name', ['expquad', 'maternp0', 'maternp2', 'matern1.3', 'cauchy0.5', 'cauchy2.0',
                                  'product_partial_dims', 'scale_loc_pairs', 'white_constant'])
def test_xjvp_vs_oracle_and_adjoint(name):
    terms = {**CASES, **PAIRS}[name]
    n, m = 70, 65
    x, y = points(3, n, m, 3)
    rng = np.random.default_rng(9)
    tx, ty = rng.standard_normal((3, n)), rng.standard_normal((3, m))
    descs = descs_of(terms, 3)
    ref = ox.xjvp(terms, x, y, tx, ty)
    D = _ops.aligned_empty(n, m, 'cuda')
    _ops.gram_iso_xjvp(descs, dev(x), dev(y), dev(tx), dev(ty), D, accumulate=False)
    scale = max(np.max(np.abs(ref)), 1e-300)
    assert np.max(np.abs(D.cpu().numpy() - ref)) <= 1e-13 * scale
    # accumulate onto an existing matrix, one side only
    base = rng.standard_normal((n, m))
    D2 = _ops.as_aligned(dev(base))
    _ops.gram_iso_xjvp(descs, dev(x), dev(y), None, dev(ty), D2, accumulate=True)
    ref2 = base + ox.xjvp(terms, x, y, 0 * tx, ty)
    assert np.max(np.abs(D2.cpu().numpy() - ref2)) <= 1e-13 * max(np.max(np.abs(ref2)), 1.0)
    # adjoint identity <xjvp(t), G> = <t, xvjp(G)>
    G = rng.standard_normal((n, m))
    gx, gy = _ops.gram_iso_xvjp(descs, dev(x), dev(y), dev(G))
    lhs = float(torch.sum(D * dev(G)))
    rhs = float(torch.sum(dev(tx) * gx) + torch.sum(dev(ty) * gy))
    dx, dy = ox.gram_xgrad(terms, x, y)
    size = np.sum(np.abs(G * (np.einsum('di,dij->ij', tx, dx) + np.einsum('dj,dij->ij', ty, dy)))) + 1e-300
    assert abs(lhs - rhs) <= 1e-12 * size


def test_argument_errors_are_returned():
    lib = _lib.load()
    terms = CASES['expquad']
    facs = _ops.make_factors(descs_of(terms, 2))
    x = dev(np.ones((2, 8)))
    G = dev(np.ones((8, 8)))
    gx = dev(np.full((2, 8), 7.0))
    gy = dev(np.full((2, 8), 7.0))
    D = dev(np.full((8, 8), 7.0))
    st = _lib.stream_ptr()
    p = _lib.ptr

    def xv(**kw):
        a = dict(nf=1, ndim=2, ldx=8, n=8, m=8, ldg=8, sym=0, gx=gx, gy=gy, ldgx=8, ldgy=8, G=G)
        a.update(kw)
        return lib.lgp_gram_iso_xvjp(st, facs, a['nf'], a['ndim'], p(x), a['ldx'], a['n'], p(x), 8, a['m'], p(a['G']),
                                     a['ldg'], None, a['sym'], p(a['gx']), a['ldgx'], p(a['gy']), a['ldgy'])
    assert xv(sym=1, m=7) == -1          # symlower needs n == m
    assert xv(sym=1) == -1               # ... and gy NULL
    assert xv(gx=None, gy=None) == -1    # nothing to compute
    assert xv(ldx=7) == -1
    assert xv(ldgx=7) == -1
    assert xv(G=None) == -1
    assert xv(n=0) == -1
    assert xv(nf=0) == -1
    assert xv(ndim=33) == -1
    bad = _ops.make_factors([dict(kind=17, term=0, dimmask=1)])
    assert lib.lgp_gram_iso_xvjp(st, bad, 1, 2, p(x), 8, 8, p(x), 8, 8, p(G), 8, None, 0, p(gx), 8, p(gy), 8) == -4
    assert lib.lgp_gram_iso_xjvp(st, facs, 1, 2, p(x), 8, 8, p(x), 8, 8, p(gx), 8, None, 0, p(D), 7, 0) == -1
    assert lib.lgp_gram_iso_xjvp(st, facs, 1, 2, p(x), 8, 8, p(x), 8, 8, p(gx), 7, None, 0, p(D), 8, 0) == -1
    assert lib.lgp_gram_iso_xjvp(st, bad, 1, 2, p(x), 8, 8, p(x), 8, 8, p(gx), 8, None, 0, p(D), 8, 0) == -4
    torch.cuda.synchronize()
    for t in (gx, gy, D):
        assert torch.all(t == 7.0)       # nothing was launched


# ---- public API

MAT52_WHITE = [(1.3, [dict(kind='maternp', p=2, scale=1.4)]), (0.05, [dict(kind='white')])]


def _kernel(th=None):
    if th is None:
        return 1.3 * lgp.Maternp(p=2, scale=1.4) + 0.05 * lgp.White()
    return 1.3 * lgp.Maternp(p=2, scale=torch.exp(th)) + 0.05 * lgp.White()


def _gp(k):
    return lgp.GP(k, checkpos=False, checksym=False, epsrel=0)


def _struct(t):
    return lgp.StructuredArray({'a': t[0], 'b': t[1]})


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


@pytest.mark.parametrize('device', ['cuda', 'cpu'])
def test_logml_point_gradient_fused_route(device):
    rng = np.random.default_rng(21)
    n = 150
    X = rng.uniform(0, 6, (2, n))
    y = rng.standard_normal(n)
    t = torch.tensor(X, dtype=f64, device=device, requires_grad=True)
    ml = _gp(_kernel()).addx(_struct(t), 'k').marginal_likelihood({'k': y})
    g, = torch.autograd.grad(ml, t)
    ref = -ox.logml_xgrad(MAT52_WHITE, X, y)
    assert g.device.type == device and _rel(g.cpu().numpy(), ref) < 1e-9
    # points and hyperparameters together equal each alone
    th = torch.tensor(np.log(1.4), dtype=f64, requires_grad=True)
    gp = _gp(_kernel(th)).addx(_struct(t), 'k')
    gt, gth = torch.autograd.grad(gp.marginal_likelihood({'k': y}), (t, th))
    gth_alone, = torch.autograd.grad(_gp(_kernel(th)).addx(_struct(X), 'k').marginal_likelihood({'k': y}), th)
    assert _rel(gt.cpu().numpy(), g.cpu().numpy()) < 1e-13
    assert abs(float(gth - gth_alone)) <= 1e-13 * abs(float(gth_alone))
    # numpy points: the same value as tensor points
    ml_np = _gp(_kernel()).addx(_struct(X), 'k').marginal_likelihood({'k': y})
    assert abs(float(ml) - ml_np) <= 1e-13 * abs(ml_np)


def test_logml_point_gradient_assembled_route():
    """ two keys sharing one tensor (x and x[:k]), an addtransf of the first, a given covariance """
    rng = np.random.default_rng(22)
    n, k = 90, 30
    X = rng.uniform(0, 6, (2, n))
    M = np.zeros((2, n))
    M[0, 3], M[0, 8], M[1, 10] = 0.5, 0.5, 1.0
    A = np.vstack([np.eye(n), np.eye(n)[:k], M])
    sizes = [n, k, 2]
    ycov = np.diag(rng.uniform(0.05, 0.1, n + k + 2))
    r = rng.standard_normal(n + k + 2)
    keys = ['a', 'b', 'c']
    offs = np.cumsum([0] + sizes)
    given = {kk: r[offs[i]:offs[i + 1]] for i, kk in enumerate(keys)}
    givencov = {(ki, kj): ycov[offs[i]:offs[i + 1], offs[j]:offs[j + 1]] for i, ki in enumerate(keys)
                for j, kj in enumerate(keys)}
    t = torch.tensor(X, dtype=f64, device='cuda', requires_grad=True)

    def ml(t, th=None):
        gp = _gp(_kernel(th)).addx(_struct(t), 'a').addx(_struct(t[:, :k]), 'b').addtransf({'a': M}, 'c')
        return gp.marginal_likelihood(given, givencov)
    g, = torch.autograd.grad(ml(t), t)
    ref = -ox.logml_xgrad(MAT52_WHITE, X, r, A, ycov)
    assert _rel(g.cpu().numpy(), ref) < 1e-9
    th = torch.tensor(np.log(1.4), dtype=f64, requires_grad=True)
    gt, gth = torch.autograd.grad(ml(t, th), (t, th))
    gth_alone, = torch.autograd.grad(ml(X, th), th)
    assert _rel(gt.cpu().numpy(), g.cpu().numpy()) < 1e-13
    assert abs(float(gth - gth_alone)) <= 1e-13 * abs(float(gth_alone))


def test_logml_point_gradient_with_bart():
    """ BART depends on the points only through bin indices: its part of the point gradient is 0 """
    rng = np.random.default_rng(23)
    n = 120
    X = rng.uniform(0, 6, (2, n))
    y = rng.standard_normal(n)
    splits = lgp.BART.splits_from_coord(X.T)
    kb = 0.7 * lgp.BART(splits=splits)
    t = torch.tensor(X, dtype=f64, device='cuda', requires_grad=True)
    ke = 1.1 * lgp.ExpQuad(scale=1.6) + 0.05 * lgp.White()
    g, = torch.autograd.grad(_gp(ke + kb).addx(_struct(t), 'k').marginal_likelihood({'k': y}), t)
    Kb = _gp(kb).addx(_struct(X), 'k').prior('k', raw=True)
    ref = -ox.logml_xgrad([(1.1, [dict(kind='expquad', scale=1.6)]), (0.05, [dict(kind='white')])], X, y, ycov=Kb)
    assert _rel(g.cpu().numpy(), ref) < 1e-9


def test_points_with_integer_dtype_and_no_grad_unchanged():
    """ tensors that do not require grad take the value-only path and give what numpy points give """
    rng = np.random.default_rng(24)
    X = np.stack([rng.permutation(60), rng.integers(0, 20, 60)])   # distinct points: White is exact equality
    y = rng.standard_normal(60)
    a = _gp(_kernel()).addx(_struct(X), 'k').marginal_likelihood({'k': y})
    b = _gp(_kernel()).addx(_struct(torch.tensor(X, device='cuda')), 'k').marginal_likelihood({'k': y})
    assert a == b


def _delay_problem():
    rng = np.random.default_rng(31)
    n = 80
    T = np.sort(rng.uniform(0, 10, n))
    mask = (np.arange(n) % 2).astype(float)
    Xtrue = T + 0.7 * mask
    K = ogp.gram(MAT52_WHITE, Xtrue[None], Xtrue[None])
    y = np.linalg.cholesky(K) @ rng.standard_normal(n)
    hyperprior = {'log(scale)': (np.log(1.4), 0.5), 'delay': (0.5, 0.5)}

    def gpfactory(hp):
        x = torch.tensor(T, dtype=f64) + hp['delay'] * torch.tensor(mask, dtype=f64)
        k = 1.3 * lgp.Maternp(p=2, scale=hp['scale']) + 0.05 * lgp.White()
        return _gp(k).addx(x, 'k')

    def oracle_objective(p):
        """ the objective of empbayes_fit with the oracle's -logML (complex-friendly in p) """
        ls = np.log(1.4) + 0.5 * p[0]
        delay = 0.5 + 0.5 * p[1]
        terms = [(1.3, [dict(kind='maternp', p=2, scale=np.exp(ls))]), (0.05, [dict(kind='white')])]
        X = (T + delay * mask)[None]
        return ox.logml(terms, X, y) + 0.5 * (2 * np.log(2 * np.pi) + p @ p), terms, X
    return hyperprior, gpfactory, {'k': y}, oracle_objective, mask


def test_empbayes_fit_delay_gradient_fisher_and_oracle():
    hyperprior, gpfactory, data, oobj, mask = _delay_problem()
    fg = lgp.empbayes_fit(hyperprior, gpfactory, data, method='gradient', covariance='fisher', raises=False)
    ff = lgp.empbayes_fit(hyperprior, gpfactory, data, method='fisher', raises=False)
    xg, xf = fg.minresult.x, ff.minresult.x
    assert np.max(np.abs(xg - xf)) < 1e-4, (xg, xf)
    assert abs(fg.minresult.fun - ff.minresult.fun) < 1e-8
    # stationary point of the oracle's objective (complex step in p)
    h = 1e-200
    grad = np.array([oobj(xg + 1j * h * e)[0].imag / h for e in np.eye(2)])
    assert np.max(np.abs(grad)) < 1e-5, grad
    assert abs(oobj(xg)[0].real - fg.minresult.fun) < 1e-9 * abs(fg.minresult.fun)
    # the Fisher matrix at the optimum (plus the prior precision) against the oracle's, dK/dp by complex step
    _, terms, X = oobj(xg)
    K = ogp.gram(terms, X, X)
    dK = []
    for e in np.eye(2):
        _, tc, Xc = oobj(xg + 1j * h * e)
        dK.append(ogp.gram(tc, Xc, Xc).imag / h)
    F = ox.fisher(K, dK) + np.eye(2)
    got = np.linalg.inv(np.asarray(fg._pcov_p))
    assert _rel(got, F) < 1e-9
    # the delay part of dK is the oracle's point JVP
    assert _rel(dK[1], 0.5 * ox.xjvp(terms, X, X, mask[None], mask[None])) < 1e-12


# ---- refusals

def test_refusals():
    rng = np.random.default_rng(41)
    X = rng.uniform(0, 5, 30)
    y = rng.standard_normal(30)
    t = torch.tensor(X, dtype=f64, requires_grad=True)
    # a point gradient through a derivative-observation block, on either side
    kd = lgp.ExpQuad(scale=1.3)
    for make in (lambda: lgp.GP(kd, checkpos=False).addx(t, 'a').addx(X[:5] + 0.1, 'd', deriv=1),
                 lambda: lgp.GP(kd, checkpos=False).addx(X, 'a').addx(t[:5] + 0.1, 'd', deriv=1)):
        ml = make().marginal_likelihood({'a': y, 'd': np.zeros(5)})
        with pytest.raises(NotImplementedError, match='derivative-observation block'):
            torch.autograd.grad(ml, t)
    # second derivatives involving the points: fused and assembled routes, functional.hessian
    k = lgp.ExpQuad(scale=1.3) + 0.1 * lgp.White()
    for make in (lambda u: _gp(k).addx(u, 'a').marginal_likelihood({'a': y}),
                 lambda u: _gp(k).addx(u, 'a').addx(u[:4] * 1.1, 'b').marginal_likelihood({'a': y, 'b': y[:4]})):
        g, = torch.autograd.grad(make(t), t, create_graph=True)
        with pytest.raises(NotImplementedError, match='second derivatives with respect to the points'):
            torch.autograd.grad(g.sum(), t)
        with pytest.raises(NotImplementedError, match='second derivatives with respect to the points'):
            torch.autograd.functional.hessian(make, t)
    hyperprior, gpfactory, data, _, _ = _delay_problem()
    with pytest.raises(NotImplementedError, match='second derivatives with respect to the points'):
        lgp.empbayes_fit(hyperprior, gpfactory, data, method='hessian')
    # the distributed solver keeps refusing all derivatives
    with pytest.raises(NotImplementedError, match='chol-dist'):
        lgp.GP(k, solver='chol-dist', checkpos=False).addx(t, 'a').marginal_likelihood({'a': y})
