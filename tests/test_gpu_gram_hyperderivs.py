"""Hyperparameter derivatives of the Gram kernels against the exact float64 oracle (oracle/deriv.py::block_derivs).

Covers the reverse-mode (VJP) and forward-mode (JVP) kernels of plain Gram blocks (general, device-descriptor and fused
symmetric forms) and of derivative blocks, the public logML gradient and Fisher matrix with derivative observations,
and descriptors whose staged coordinates need more than 48 KiB of shared memory.

Bars: a contraction sum_ij G_ij dK_ij must be within 1e-12 sum_ij |G_ij dK_ij| of the oracle (atomicAdd order varies
the last bits); a JVP matrix within 1e-13 of the oracle normwise and 1e-12 elementwise (atol 1e-13 max |ref|)."""
import numpy as np
import pytest
import torch

import lsqfitgp_b200 as lgp
from lsqfitgp_b200 import _lib, _ops
from oracle import deriv as od, gp as ogp

pytestmark = pytest.mark.gpu

KIND = {'expquad': _lib.K_EXPQUAD, 'maternp': _lib.K_MATERNP, 'matern': _lib.K_MATERN, 'cauchy': _lib.K_CAUCHY,
        'white': _lib.K_WHITE, 'constant': _lib.K_CONSTANT}


# ---- kernel specifications: a list of terms (amp, [factor, ...]) in the oracle's format (oracle/gp.py), translated
# into the descriptors of the C ABI.  Maternp with par0 = 0 is the library's half-integer Matern: the oracle calls it
# 'matern' in derivative blocks (oracle/deriv.py::_coef_args).

def _pair(v, default):
    return v if isinstance(v, tuple) else (default if v is None else v,) * 2


def descs_of(terms, ndim):
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


def oracle_terms(terms, deriv=False):
    """ the oracle's spelling: par0 dropped; Maternp with par0 = 0 becomes the half-integer Matern in derivative blocks """
    out = []
    for amp, factors in terms:
        fs = []
        for f in factors:
            f = {k: v for k, v in f.items() if k != 'par0'} | (
                dict(kind='matern', nu=f['p'] + 0.5) if deriv and f['kind'] == 'maternp' and f.get('par0') == 0.0 else {})
            fs.append(f)
        out.append((amp, fs))
    return out


def derivs_per_factor(terms, x, y, a=None, b=None, deriv=False):
    """ [(dK/d amp_f, dK/d log scale_f, dK/d par1_f) for every factor f in descriptor order] from the oracle """
    ders = od.block_derivs(oracle_terms(terms, deriv), x, y, a, b)
    out = []
    for ti, (amp, factors) in enumerate(terms):
        for fi, f in enumerate(factors):
            # amp of the descriptor: the term's amplitude on the first factor, 1 on the others
            d_amp = ders['amp', ti] if fi == 0 else amp * ders['amp', ti]
            d_par1 = ders['beta', ti, fi] if f['kind'] == 'cauchy' else np.zeros_like(d_amp)
            out.append((d_amp, ders['logscale', ti, fi], d_par1))
    return out


def check_contraction(got, G, dK_list, what):
    got = np.asarray(got)
    for f, dks in enumerate(dK_list):
        for k, dK in enumerate(dks):
            ref = float(np.sum(G * dK))
            bar = 1e-12 * float(np.sum(np.abs(G * dK)))
            assert abs(got[f, k] - ref) <= bar, (what, f, k, got[f, k], ref, bar)


def check_matrix(got, ref, what, nw=1e-13):
    scale = float(np.max(np.abs(ref))) if ref.size else 0.0
    assert np.all(np.isfinite(got)), what
    assert float(np.max(np.abs(got - ref))) <= nw * scale, (what, float(np.max(np.abs(got - ref))), scale)
    np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-13 * scale, err_msg=what)


def jvp_ref(dK_list, tan):
    return sum(tan[f, k] * dK for f, dks in enumerate(dK_list) for k, dK in enumerate(dks))


def points(ndim, n, m, s, seed, *, off=0.0):
    """ (x, y) in units of the scale s: coincident pairs x_i = y_i, a duplicated point within x, a point 40 scales away
    (ExpQuad underflows to 0 against every other point), all shifted by `off` scales from the origin """
    rng = np.random.default_rng(seed)
    x = rng.uniform(0, 4, (ndim, n))
    y = rng.uniform(0, 4, (ndim, m))
    k = min(n, m, 3)
    y[:, :k] = x[:, :k]
    if n >= 8:
        x[:, 5] = x[:, 6]
        x[:, 7] = x[:, 1] + 40.0
    return (x + off) * s, (y + off) * s


def dev(a):
    return torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device='cuda')


# ---- plain Gram VJP / JVP

def _plain_cases():
    cases = {
        'expquad': [(1.3, [dict(kind='expquad')])],
        **{f'maternp{p}_par0{z}': [(0.9, [dict(kind='maternp', p=p, par0=z)])] for p in range(5) for z in (0.0, 1e-30)},
        **{f'matern{nu}': [(1.1, [dict(kind='matern', nu=nu)])] for nu in (0.3, 1.3, 4.2)},
        'cauchy2': [(0.7, [dict(kind='cauchy', alpha=2, beta=1.4)])],
        'cauchy1.3': [(0.7, [dict(kind='cauchy', alpha=1.3, beta=0.8)])],
    }
    return cases


PLAIN = _plain_cases()


def _scaled(terms, s, loc=None):
    """ every factor that has a scale gets `s` (and `loc`) """
    return [(amp, [f | (dict(scale=s) | ({} if loc is None else dict(loc=loc)) if f['kind'] not in ('white', 'constant')
                        else {}) for f in fs]) for amp, fs in terms]


def _with_extras(terms, white, const):
    out = list(terms)
    if white:
        out.append((0.05, [dict(kind='white')]))
    if const:
        out.append((0.3, [dict(kind='constant')]))
    return out


def _run_plain(terms, x, y, tag=''):
    ndim = x.shape[0]
    descs = descs_of(terms, ndim)
    xd, yd = dev(x), dev(y)
    n, m = x.shape[1], y.shape[1]
    rng = np.random.default_rng(n * 1000 + m)
    G = rng.standard_normal((n, m))
    dK = derivs_per_factor(terms, x, y)
    check_contraction(_ops.gram_iso_vjp_general(descs, xd, yd, _ops.as_aligned(dev(G))).cpu().numpy(), G, dK,
                      'vjp_general' + tag)
    devpar = _ops.devpar_of(descs, 'cuda')
    check_contraction(_ops.gram_iso_vjp_dev(descs, devpar, xd, yd, _ops.as_aligned(dev(G))).cpu().numpy(), G, dK,
                      'vjp_dev' + tag)
    tan = rng.standard_normal((len(descs), 3))
    ref = jvp_ref(dK, tan)
    check_matrix(_ops.gram_iso_jvp(descs, xd, yd, tan).cpu().numpy(), ref, 'jvp' + tag)
    check_matrix(_ops.gram_iso_jvp_dev(descs, devpar, xd, yd, dev(tan)).cpu().numpy(), ref, 'jvp_dev' + tag)


def _run_sym(terms, x, tag=''):
    """ the symmetric VJP with the rank-one term (fast path where the kernel is in its family, else the general
    kernel): sum_ij (Gsym - b b')_ij dK_ij, Gsym given by its lower triangle """
    descs = descs_of(terms, x.shape[0])
    n = x.shape[1]
    rng = np.random.default_rng(n + 17)
    A = rng.standard_normal((n, n))
    Gs = A + A.T
    bvec = rng.standard_normal(n)
    low = np.tril(Gs) + np.triu(np.full((n, n), np.nan), 1)   # the upper triangle must not be read
    xd = dev(x)
    got = _ops.gram_iso_vjp(descs, xd, _ops.as_aligned(dev(low)), dev(bvec)).cpu().numpy()
    dK = derivs_per_factor(terms, x, x)
    check_contraction(got, Gs - np.outer(bvec, bvec), dK, 'vjp_sym' + tag)
    got = _ops.gram_iso_vjp_dev(descs, _ops.devpar_of(descs, 'cuda'), xd, xd, _ops.as_aligned(dev(low)), b=dev(bvec),
                                symlower=True).cpu().numpy()
    check_contraction(got, Gs - np.outer(bvec, bvec), dK, 'vjp_dev_sym' + tag)


SHAPES = [(1, 1), (1, 65), (63, 64), (64, 64), (65, 129), (333, 257)]
SYM_N = [1, 64, 65, 130, 333]


@pytest.mark.parametrize('name', list(PLAIN))
def test_plain_vjp_jvp_shapes(name):
    """ every kind at every shape, with a White and a Constant term """
    terms = _with_extras(_scaled(PLAIN[name], 1.7), True, True)
    for n, m in SHAPES:
        x, y = points(3, n, m, 1.7, n + m)
        _run_plain(terms, x, y, tag=f' {n}x{m}')
    for n in SYM_N:
        x, _ = points(3, n, 1, 1.7, n)
        _run_sym(terms, x, tag=f' n={n}')


@pytest.mark.parametrize('name', list(PLAIN))
@pytest.mark.parametrize('scale', [1e-3, 1.0, 1e3])
@pytest.mark.parametrize('white, const', [(False, False), (True, False), (False, True)])
def test_plain_vjp_jvp_combinations(name, scale, white, const):
    """ scales far from 1, loc != 0, points far from the origin, with and without White / Constant """
    terms = _with_extras(_scaled(PLAIN[name], scale, loc=0.3 * scale), white, const)
    x, y = points(2, 130, 70, scale, 3, off=100.0)
    _run_plain(terms, x, y)
    _run_sym(terms, x)
    # unequal scales and locations of the two arguments (general kernels only)
    terms = _with_extras([(amp, [f | dict(scale=(scale, 1.3 * scale), loc=(0.2 * scale, -0.1 * scale))
                                 for f in fs]) for amp, fs in PLAIN[name]], white, const)
    x, y = points(2, 65, 129, scale, 4)
    _run_plain(terms, x, y)


PRODUCTS = {
    # overlapping fields {0, 1} and {1, 2}
    'overlap': [(1.2, [dict(kind='expquad', dims=[0, 1], scale=0.9),
                       dict(kind='cauchy', alpha=2, beta=2.5, dims=[1, 2], scale=1.6)])],
    # disjoint fields, three factors, loc
    'disjoint3': [(0.8, [dict(kind='maternp', p=2, par0=0.0, dims=[0], scale=1.1, loc=0.4),
                         dict(kind='matern', nu=1.3, dims=[1], scale=0.7),
                         dict(kind='cauchy', alpha=1.3, beta=0.6, dims=[2], scale=2.0)])],
    'sum_of_products': [(0.6, [dict(kind='expquad', dims=[0], scale=0.5),
                               dict(kind='maternp', p=1, par0=1e-30, dims=[0, 2], scale=1.9)]),
                        (0.4, [dict(kind='cauchy', alpha=2, beta=0.9, dims=[1, 2], scale=1.2)]),
                        (0.05, [dict(kind='white')]), (0.3, [dict(kind='constant')])],
}


@pytest.mark.parametrize('name', list(PRODUCTS))
def test_plain_vjp_jvp_products(name):
    terms = PRODUCTS[name]
    for n, m in SHAPES:
        x, y = points(3, n, m, 1.0, 7 * n + m)
        _run_plain(terms, x, y, tag=f' {n}x{m}')
    for n in SYM_N:
        x, _ = points(3, n, 1, 1.0, n + 5)
        _run_sym(terms, x, tag=f' n={n}')


# ---- derivative blocks

S = 1.7
DERIV = {
    'expquad': [(1.0, [dict(kind='expquad', scale=S)])],
    **{f'maternp{p}': [(1.0, [dict(kind='maternp', p=p, scale=S)])] for p in (1, 2, 3, 4)},
    **{f'matern{p + 0.5}': [(1.0, [dict(kind='maternp', p=p, par0=0.0, scale=S)])] for p in (1, 2, 3)},
    'cauchy': [(1.0, [dict(kind='cauchy', alpha=2, beta=1.3, scale=S)])],
    'tuple_scale': [(1.2, [dict(kind='expquad', scale=(1.3, 0.9), loc=(0.2, -0.1))])],
    # both factors depend on field 0 (both mixed products of the product rule are non-zero for (0, 0))
    'shared_field': [(0.8, [dict(kind='expquad', dims=[0, 1], scale=S),
                            dict(kind='cauchy', alpha=2, beta=1.3, dims=[0, 2], scale=1.1)])],
    # field 2 is the second slot of the factor
    'dims02': [(1.3, [dict(kind='maternp', p=2, dims=[0, 2], scale=S)])],
    # the second term does not depend on field 0; its Cauchy factor carries scale and beta without depending on field 1
    'indep_term': [(1.0, [dict(kind='maternp', p=1, dims=[0, 1], scale=S)]),
                   (0.4, [dict(kind='expquad', dims=[1], scale=0.8),
                          dict(kind='cauchy', alpha=2, beta=1.3, dims=[2], scale=1.4)])],
    # a factor over the differentiated field next to a Constant term, times a Matern of real order that does not depend
    # on it
    'mixed': [(0.9, [dict(kind='expquad', dims=[0, 2], scale=1.2, loc=0.3),
                     dict(kind='matern', nu=1.3, dims=[1], scale=0.8)]),
              (0.3, [dict(kind='constant')])],
}
SELECTIONS = [(0, None), (None, 2), (2, 2), (0, 2)]


def _sentinel_out(n, m):
    """ (n, m) aligned view at column offset 2 of a wider buffer filled with a sentinel (as _assemblecovblocks writes
    blocks into the joint matrix), and the buffer """
    buf = torch.full((max(n, 1), m + 6), -7.25e300, dtype=torch.float64, device='cuda')
    return buf[:n, 2:2 + m], buf


def _check_sentinel(buf, m, what):
    edge = torch.cat([buf[:, :2], buf[:, 2 + m:]], dim=1)
    assert bool(torch.all(edge == -7.25e300)), what


def _run_deriv(terms, x, y, a, b, tag=''):
    descs = descs_of(terms, x.shape[0])
    xd, yd = dev(x), dev(y)
    n, m = x.shape[1], y.shape[1]
    aa, bb = -1 if a is None else a, -1 if b is None else b
    ref = od.block(oracle_terms(terms, True), x, y, a, b)
    out, buf = _sentinel_out(n, m)
    _ops.gram_iso_deriv(descs, xd, yd, aa, bb, out=out)
    check_matrix(out.cpu().numpy(), ref, 'deriv value' + tag)
    _check_sentinel(buf, m, 'deriv value sentinel' + tag)
    rng = np.random.default_rng(n * 7 + m)
    dK = derivs_per_factor(terms, x, y, a, b, deriv=True)
    G = rng.standard_normal((n, m))
    check_contraction(_ops.gram_iso_deriv_vjp(descs, xd, yd, aa, bb, _ops.as_aligned(dev(G))).cpu().numpy(), G, dK,
                      'deriv vjp' + tag)
    tan = rng.standard_normal((len(descs), 3))
    out, buf = _sentinel_out(n, m)
    _ops.gram_iso_deriv_jvp(descs, xd, yd, aa, bb, tan, out=out)
    check_matrix(out.cpu().numpy(), jvp_ref(dK, tan), 'deriv jvp' + tag)
    _check_sentinel(buf, m, 'deriv jvp sentinel' + tag)


@pytest.mark.parametrize('name', list(DERIV))
@pytest.mark.parametrize('a, b', SELECTIONS)
def test_deriv_blocks_vs_oracle(name, a, b):
    terms = DERIV[name]
    for n, m in SHAPES:
        x, y = points(3, n, m, 1.0, 3 * n + m)
        _run_deriv(terms, x, y, a, b, tag=f' {n}x{m}')


@pytest.mark.parametrize('name', list(DERIV))
@pytest.mark.parametrize('field', [0, 2])
def test_deriv_blocks_symmetric_mode(name, field):
    """ symmetric mode (x is y, same field on both sides) against the oracle, not only against the general mode """
    terms = DERIV[name]
    if any(isinstance(f.get('scale'), tuple) or isinstance(f.get('loc'), tuple) for _, fs in terms for f in fs):
        pytest.skip('the symmetric mode needs equal scales and locations of the two arguments')
    descs = descs_of(terms, 3)
    for n in SYM_N:
        x, _ = points(3, n, 1, 1.0, n + 1)
        xd = dev(x)
        ref = od.block(oracle_terms(terms, True), x, x, field, field)
        out, buf = _sentinel_out(n, n)
        _ops.gram_iso_deriv(descs, xd, xd, field, field, out=out, symmetric=True)
        got = out.cpu().numpy()
        check_matrix(got, ref, f'symmetric n={n}')
        assert np.array_equal(got, got.T)
        _check_sentinel(buf, n, f'symmetric sentinel n={n}')


# ---- public API with derivative observations, exact dK

def _sa(X, names):
    return lgp.unstructured_to_structured(X, names=names)


def _joint(blocks_fn, parts):
    return np.block([[blocks_fn(xr, ar, xc, ac) for xc, ac in parts] for xr, ar in parts])


def _joint_derivs(terms, parts, keys):
    """ {key: assembled dK} for the oracle keys of block_derivs """
    rows = []
    for xr, ar in parts:
        row = []
        for xc, ac in parts:
            ders = od.block_derivs(terms, xr, xc, ar, ac) if (ar is not None or ac is not None) else \
                od.block_derivs(terms, xr, xc)
            row.append(ders)
        rows.append(row)
    return {k: np.block([[rows[i][j][k] for j in range(len(parts))] for i in range(len(parts))]) for k in keys}


API_KERNELS = {
    'maternp2': (lambda th: torch.exp(th[0]) * lgp.Maternp(p=2, scale=torch.exp(th[1])),
                 lambda th: [(np.exp(th[0]), [dict(kind='maternp', p=2, scale=np.exp(th[1]))])],
                 lambda th: [[('amp', 0)], [('logscale', 0, 0)]]),
    'matern2.5': (lambda th: torch.exp(th[0]) * lgp.Matern(nu=2.5, scale=torch.exp(th[1])),
                  lambda th: [(np.exp(th[0]), [dict(kind='matern', nu=2.5, scale=np.exp(th[1]))])],
                  lambda th: [[('amp', 0)], [('logscale', 0, 0)]]),
    'product': (lambda th: torch.exp(th[0]) * lgp.ExpQuad(scale=torch.exp(th[1]), dim='a')
                * lgp.Cauchy(alpha=2, beta=torch.exp(th[2]), scale=torch.exp(th[3])),
                lambda th: [(np.exp(th[0]), [dict(kind='expquad', dims=[0], scale=np.exp(th[1])),
                                             dict(kind='cauchy', alpha=2, beta=np.exp(th[2]), scale=np.exp(th[3]))])],
                lambda th: [[('amp', 0)], [('logscale', 0, 0)], [('beta', 0, 1)], [('logscale', 0, 1)]]),
}


def _api_data():
    rng = np.random.default_rng(8)
    X = rng.uniform(-2, 2, (60, 2))
    y = {'f': rng.standard_normal(60), 'dfa': rng.standard_normal(25), 'dfb': rng.standard_normal(20)}
    Xt = X.T.copy()
    parts = [(Xt, None), (Xt[:, :25], 0), (Xt[:, 25:45], 1)]
    return X, y, parts


@pytest.mark.parametrize('name', list(API_KERNELS))
def test_marginal_likelihood_gradient_exact(name):
    mk, mkterms, mkkeys = API_KERNELS[name]
    th0 = {'maternp2': [0.1, 0.2], 'matern2.5': [-0.2, 0.3], 'product': [0.1, 0.4, 0.3, 0.2]}[name]
    X, y, parts = _api_data()
    x = _sa(X, ['a', 'b'])
    tt = torch.tensor(th0, dtype=torch.float64, requires_grad=True)
    gp = lgp.GP(mk(tt), checkpos=False, checksym=False).addx(x, 'f').addx(x[:25], 'dfa', deriv='a') \
        .addx(x[25:45], 'dfb', deriv='b')
    noise = {k: 0.01 * np.eye(len(v)) for k, v in y.items()}
    gc = {(p, q): (noise[p] if p == q else np.zeros((len(y[p]), len(y[q])))) for p in y for q in y}
    ml = gp.marginal_likelihood(y, gc)
    g, = torch.autograd.grad(ml, tt)
    terms = mkterms(np.array(th0))
    K = od.joint_cov(terms, parts) + 0.01 * np.eye(105)
    yv = np.concatenate([y['f'], y['dfa'], y['dfb']])
    ref = ogp.logml(K, yv)
    assert abs(float(ml.detach()) - ref) <= 1e-9 * abs(ref)
    Kinv = np.linalg.inv(K)
    bvec = Kinv @ yv
    groups = mkkeys(th0)
    keys = [k for grp in groups for k in grp]
    dKs = _joint_derivs(terms, parts, keys)
    ref_g = []
    for grp in groups:
        dK = sum(dKs[k] for k in grp)
        if grp[0][0] == 'amp':
            dK = np.exp(th0[0]) * dK                 # d amp / d log amp
        if grp[0][0] == 'beta':
            dK = np.exp(th0[2]) * dK                 # d beta / d log beta
        ref_g.append(-0.5 * np.sum(Kinv * dK) + 0.5 * bvec @ dK @ bvec)
    ref_g = np.array(ref_g)
    assert np.max(np.abs(g.numpy() - ref_g)) <= 1e-9 * np.max(np.abs(ref_g)), (g.numpy(), ref_g)


def test_fisher_matrix_exact():
    X = np.linspace(0, 6, 25)
    rng = np.random.default_rng(6)
    y = {'f': np.sin(X) + 0.05 * rng.standard_normal(25), 'df': np.cos(X) + 0.05 * rng.standard_normal(25)}
    gc = {('f', 'f'): 0.0025 * np.eye(25), ('df', 'df'): 0.0025 * np.eye(25),
          ('f', 'df'): np.zeros((25, 25)), ('df', 'f'): np.zeros((25, 25))}
    hyperprior = {'log(s)': (0.0, 1.0), 'log(a)': (0.0, 1.0)}

    def gpfactory(hp):
        return lgp.GP(hp['a'] ** 2 * lgp.Maternp(p=2, scale=hp['s']), checkpos=False, checksym=False) \
            .addx(X, 'f').addx(X, 'df', deriv=1)
    fit = lgp.empbayes_fit(hyperprior, gpfactory, (y, gc), raises=False, method='fisher')
    p = fit.minresult.x
    s, a = np.exp(p)
    terms = [(a ** 2, [dict(kind='maternp', p=2, scale=s)])]
    Xt = X[None, :]
    parts = [(Xt, None), (Xt, 0)]
    K = od.joint_cov(terms, parts) + 0.0025 * np.eye(50)
    dKs = _joint_derivs(terms, parts, [('logscale', 0, 0), ('amp', 0)])
    dK = [dKs['logscale', 0, 0], 2 * a ** 2 * dKs['amp', 0]]     # d / d log s, d / d log a
    Kinv = np.linalg.inv(K)
    F = np.array([[0.5 * np.sum((Kinv @ di) * (Kinv @ dj).T) for dj in dK] for di in dK])
    got = np.asarray(fit.minresult.hess) - np.eye(2)
    assert np.max(np.abs(got - F)) <= 1e-9 * np.max(np.abs(F)), (got, F)


# ---- descriptor width across the 48 KiB shared-memory limit

NW, MW = 130, 70


def _wide_terms(slots):
    """ 1-3 factors over up to 32 fields with `slots` participating fields in all; every factor covers field 5, at
    different slot positions """
    sizes = [32] * ((slots - 1) // 32) + [slots - 32 * ((slots - 1) // 32)]
    kinds = [dict(kind='expquad', scale=2.0), dict(kind='cauchy', alpha=2, beta=1.5, scale=2.5),
             dict(kind='maternp', p=2, scale=3.0)]
    others = [d for d in range(32) if d != 5]
    return [(0.9, [kinds[i] | dict(dims=sorted([5] + [others[(7 * i + k) % 31] for k in range(sz - 1)]))
                   for i, sz in enumerate(sizes)])]


def _wide_points(seed):
    rng = np.random.default_rng(seed)
    x = rng.uniform(0, 1, (32, NW))
    y = rng.uniform(0, 1, (32, MW))
    y[:, :3] = x[:, :3]
    return x, y


@pytest.mark.parametrize('slots', list(range(40, 51)) + [96])
def test_wide_descriptor_general_kernels(slots):
    terms = _wide_terms(slots)
    assert sum(len(f['dims']) for f in terms[0][1]) == slots
    descs = descs_of(terms, 32)
    x, y = _wide_points(slots)
    xd, yd = dev(x), dev(y)
    # values
    ref = ogp.gram(terms, x, y)
    check_matrix(_ops.gram_iso(descs, xd, yd).cpu().numpy(), ref, 'gram')
    devpar = _ops.devpar_of(descs, 'cuda')
    check_matrix(_ops.gram_iso_dev(descs, devpar, xd, yd).cpu().numpy(), ref, 'gram_dev')
    # VJP / JVP, host and device descriptors, general and symmetric lower-triangle forms
    _run_plain(terms, x, y)
    _run_sym(terms, x)
    # derivative blocks (value, VJP, JVP) and the symmetric derivative value
    for a, b in [(5, None), (None, 5), (5, 5), (5, 31)]:
        _run_deriv(terms, x, y, a, b, tag=f' ({a}, {b})')
    ref = od.block(terms, x, x, 5, 5)
    check_matrix(_ops.gram_iso_deriv(descs, xd, xd, 5, 5, symmetric=True).cpu().numpy(), ref, 'deriv symmetric')


FAST_KINDS = {'expquad': dict(kind='expquad'), 'cauchy': dict(kind='cauchy', alpha=2, beta=1.5),
              'matern1.3': dict(kind='matern', nu=1.3)}


@pytest.mark.parametrize('kind', list(FAST_KINDS))
@pytest.mark.parametrize('white_raw', [False, True])
def test_wide_fast_path(kind, white_raw):
    """ a * K(scale=s) + w * White() over nd = 20 ... 32 fields: the fast Gram kernels (symmetric and rectangular), the
    fused symmetric VJP and the fused Gram + factorisation; White compares raw coordinates when s != 1 """
    s = 2.5 if white_raw else 1.0
    rng = np.random.default_rng(11)
    for nd in range(20, 33):
        terms = [(1.3, [FAST_KINDS[kind] | dict(scale=s)]), (0.1, [dict(kind='white')])]
        descs = descs_of(terms, nd)
        x = rng.uniform(0, 1, (nd, NW)) * s
        x[:, 5] = x[:, 6]
        y = rng.uniform(0, 1, (nd, MW)) * s
        y[:, :3] = x[:, :3]
        xd, yd = dev(x), dev(y)
        Kref = ogp.gram(terms, x, x)
        K = _ops.gram_iso(descs, xd, xd, symmetric=True)
        check_matrix(K.cpu().numpy(), Kref, f'gram sym nd={nd}')
        check_matrix(_ops.gram_iso(descs, xd, yd).cpu().numpy(), ogp.gram(terms, x, y), f'gram rect nd={nd}')
        _run_sym(terms, x, tag=f' nd={nd}')
        # factorisation: without the duplicated point, which makes the matrix singular
        x[:, 5] = rng.uniform(0, 1, nd) * s
        xd = dev(x)
        Kref = ogp.gram(terms, x, x)
        K = _ops.gram_iso(descs, xd, xd, symmetric=True)
        L2 = _ops.chol_get_factor(_ops.chol_factor(K, epsrel=0.0)).cpu().numpy()
        Lref = np.linalg.cholesky(Kref)
        assert np.max(np.abs(L2 - Lref)) <= 1e-11 * np.max(np.abs(Lref)), nd
        st = _ops.gram_chol_factor(descs, xd, epsrel=0.0)
        if st is not None:      # (the fused build declines inputs whose tiles do not fit three CTAs per SM)
            assert int(st.info.item()) == 0
            L1 = _ops.chol_get_factor(st).cpu().numpy()
            assert np.max(np.abs(L1 - Lref)) <= 1e-11 * np.max(np.abs(Lref)), nd


def test_wide_public_api_logml_gradient():
    """ the fused logML node on 25 fields, ExpQuad with a scale plus White: its backward pass is the fused symmetric
    VJP with raw White coordinates """
    rng = np.random.default_rng(25)
    nd, n = 25, 300
    X = rng.uniform(0, 1, (n, nd))
    yv = rng.standard_normal(n)
    th = np.array([0.2, np.log(2.0), np.log(0.05)])
    tt = torch.tensor(th, dtype=torch.float64, requires_grad=True)
    kern = torch.exp(tt[0]) * lgp.ExpQuad(scale=torch.exp(tt[1])) + torch.exp(tt[2]) * lgp.White()
    gp = lgp.GP(kern, checkpos=False, checksym=False).addx(_sa(X, [f'f{i}' for i in range(nd)]), 'x')
    ml = gp.marginal_likelihood({'x': yv})
    g, = torch.autograd.grad(ml, tt)
    terms = [(np.exp(th[0]), [dict(kind='expquad', scale=np.exp(th[1]))]), (np.exp(th[2]), [dict(kind='white')])]
    val, grad = ogp.logml_and_grad(terms, X.T.copy(), yv, [('amp', 0), ('logscale', 0, 0), ('amp', 1)])
    ref_g = -np.array([grad[0] * np.exp(th[0]), grad[1], grad[2] * np.exp(th[2])])
    assert abs(float(ml.detach()) + val) <= 1e-9 * abs(val)
    assert np.max(np.abs(g.numpy() - ref_g)) <= 1e-9 * np.max(np.abs(ref_g)), (g.numpy(), ref_g)


def test_too_many_slots_is_unsupported_and_leaves_no_error():
    terms97 = [(1.0, [dict(kind='expquad', dims=list(range(32))), dict(kind='expquad', dims=list(range(32))),
                      dict(kind='expquad', dims=list(range(32))), dict(kind='expquad', dims=[0])])]
    x, y = _wide_points(97)
    xd, yd = dev(x), dev(y)
    G = _ops.as_aligned(dev(np.ones((NW, MW))))
    calls = [lambda d: _ops.gram_iso(d, xd, yd), lambda d: _ops.gram_iso_vjp_general(d, xd, yd, G),
             lambda d: _ops.gram_iso_jvp(d, xd, yd, np.zeros((len(d), 3))),
             lambda d: _ops.gram_iso_deriv(d, xd, yd, 0, 0),
             lambda d: _ops.gram_iso_deriv_vjp(d, xd, yd, 0, -1, G),
             lambda d: _ops.gram_iso_deriv_jvp(d, xd, yd, -1, 0, np.zeros((len(d), 3))),
             lambda d: _ops.gram_iso_dev(d, _ops.devpar_of(d, 'cuda'), xd, yd)]
    d97 = descs_of(terms97, 32)
    d96 = descs_of(_wide_terms(96), 32)
    for call in calls:
        with pytest.raises(RuntimeError, match=_lib.ERRORS[-4]):
            call(d97)
        call(d96)          # the next call on the stream succeeds: no error is left behind
        torch.cuda.synchronize()
    check_matrix(_ops.gram_iso(d96, xd, yd).cpu().numpy(), ogp.gram(_wide_terms(96), x, y), 'gram 96 after 97')
