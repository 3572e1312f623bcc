"""Parity against golden vectors produced by executing the REFERENCE'S OWN SOURCE under the numpy stand-in for jax
(oracle/refshim.py, tests/golden/gen_reference_vectors.py -> tests/golden/reference_vectors.npz):
lgp.GP.marginal_likelihood / predfromdata(raw=True), every supported kernel's Gram block, _linalg.Chol with value,
forward gradient and Fisher matrix, BART preprocessing and correlation.

  * not gpu: the oracle restatement against the file (pins the oracle to the reference's code, not to a re-reading of it);
  * gpu: the CUDA path (public API and C ABI) against the same file.  Tolerances of BASELINE.json north_star: Gram 1e-13
    relative (2e-13 for Matern of non-half-integer order: AMOS's own accuracy, tests/test_bessel_cpu.py), logML and
    posterior mean 1e-9."""
import pathlib

import numpy as np
import pytest

from oracle import gp as ogp, decomp as odecomp, bart as obart

GOLD = pathlib.Path(__file__).resolve().parent / 'golden' / 'reference_vectors.npz'
NAMES = ['f0', 'f1', 'f2']


@pytest.fixture(scope='module')
def vec():
    return dict(np.load(GOLD))


# kernel name -> oracle terms
GRAM_TERMS = {
    'expquad': [(1.0, [dict(kind='expquad', scale=1.5)])],
    'expquad_loc': [(3.0, [dict(kind='expquad', scale=0.3, loc=1.0)])],
    'maternp0': [(1.0, [dict(kind='constant'), dict(kind='maternp', p=0, scale=2.0)])],
    'maternp1': [(1.0, [dict(kind='maternp', p=1, scale=2.0)])],
    'maternp2': [(1.0, [dict(kind='maternp', p=2, scale=2.0)])],
    'maternp3': [(1.0, [dict(kind='maternp', p=3, scale=2.0)])],
    'matern05': [(1.0, [dict(kind='matern', nu=0.5, scale=2.0)])],
    'matern25': [(1.0, [dict(kind='matern', nu=2.5, scale=2.0)])],
    'matern03': [(1.0, [dict(kind='matern', nu=0.3, scale=2.0)])],
    'matern13': [(1.0, [dict(kind='matern', nu=1.3, scale=2.0)])],
    'matern42': [(1.0, [dict(kind='matern', nu=4.2, scale=2.0)])],
    'ratquad': [(1.0, [dict(kind='cauchy', alpha=2, beta=3.0, scale=1.5)])],
    'cauchy13': [(1.0, [dict(kind='cauchy', alpha=1.3, beta=0.7, scale=4.0)])],
    'white_sum': [(2.0, [dict(kind='expquad', scale=1.5)]), (0.01, [dict(kind='white')]), (0.25, [dict(kind='constant')])],
    'product': [(2.0, [dict(kind='cauchy', alpha=2, beta=3.0, dims=[0]), dict(kind='expquad', scale=0.7, dims=[1])])],
}
GP_TERMS = {
    'c2': [(1.0, [dict(kind='matern', nu=2.5, scale=1.5)]), (0.01, [dict(kind='white')])],
    'c2nu13': [(1.3, [dict(kind='matern', nu=1.3, scale=1.5)]), (0.01, [dict(kind='white')])],
    'c3': [(1.44, [dict(kind='expquad', scale=2.0)]), (0.01, [dict(kind='white')])],
    'rq': [(0.8, [dict(kind='cauchy', alpha=2, beta=3.0, scale=1.5)]), (0.01, [dict(kind='white')])],
}
BART_VARIANTS = {
    'd0': dict(maxd=0), 'd1': dict(maxd=1), 'd2': dict(maxd=2), 'd4r2': dict(maxd=4, reset=2),
    'd2g': dict(maxd=2, gamma=0.3, intercept=False), 'd10': dict(maxd=10, reset=[2, 4, 6, 8], gamma=1),
    'd6w': dict(maxd=6, reset=[2, 4], weights=np.array([1., 0., 2., 3., 0.5])),
}


def relerr(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    den = np.abs(b).clip(1e-300)
    return float(np.max(np.abs(a - b) / den))


# ------------------------------------------------------------------------------------------------ CPU tier
def test_oracle_gram_matches_reference(vec):
    A, B = vec['gram_A'].T.copy(), vec['gram_B'].T.copy()
    for name, terms in GRAM_TERMS.items():
        K = ogp.gram(terms, A, B)
        assert relerr(K, vec['gram_' + name]) <= 1e-15, name       # same formulas, same libm: identical or a few ulp


# Tolerances of the factorisation-level comparisons below leave room for another CPU model's BLAS kernels (cond * eps);
# on the machine that wrote the file the oracle and the reference agree to 0-2 ulp on every one of these numbers.
def test_oracle_gp_matches_reference(vec):
    rng = np.random.default_rng(1001)
    x = np.sort(rng.uniform(0, 100, 1000))
    y = np.sin(x / 3) + 0.1 * rng.standard_normal(1000)
    xp = np.linspace(-5, 105, 500)
    terms = [(1.0, [dict(kind='expquad', scale=3)])]
    Kxx, Kxs, Kss = ogp.gram(terms, x[None], x[None]), ogp.gram(terms, x[None], xp[None]), ogp.gram(terms, xp[None], xp[None])
    ycov = 0.01 * np.eye(1000)
    assert abs(ogp.logml(Kxx, y, ycov) - vec['c1_logml']) <= 1e-10 * abs(vec['c1_logml'])
    m, c = ogp.pred(Kxx, Kxs, Kss, y, ycov)
    assert relerr(m, vec['c1_mean']) <= 1e-9
    assert np.max(np.abs(np.diag(c) - vec['c1_cov_diag'])) <= 1e-10
    X, y2, Xs = vec['c2_X'], vec['c2_y'], vec['c2_Xs']
    for tag, terms in GP_TERMS.items():
        K = ogp.gram(terms, X.T.copy(), X.T.copy())
        assert relerr(K[:5], vec[tag + '_prior_rows']) <= 4e-16, tag
        assert abs(ogp.logml(K, y2) - vec[tag + '_logml']) <= 1e-10 * abs(vec[tag + '_logml']), tag
        Kxs = ogp.gram(terms, X.T.copy(), Xs.T.copy())      # (the White term lives on every key of the GP)
        Kss = ogp.gram(terms, Xs.T.copy(), Xs.T.copy())
        m, c = ogp.pred(K, Kxs, Kss, y2)
        assert np.max(np.abs(m - vec[tag + '_mean'])) <= 1e-9 * np.max(np.abs(vec[tag + '_mean'])), tag
        assert np.max(np.abs(c - vec[tag + '_cov'])) <= 1e-10, tag


@pytest.mark.parametrize('nn', [10, 64])
def test_oracle_chol_matches_reference(vec, nn):
    g = lambda k: vec[f'chol{nn}_{k}']
    dec = odecomp.Chol(g('K'))
    assert abs(dec.eps - float(g('eps'))) <= 1e-13 * float(g('eps'))   # (row sums: summation order may differ by CPU)
    val, _, gradfwd, fisher, _ = dec.minus_log_normal_density(g('r'), dK=g('dK'), dr=g('dr'), value=True, gradfwd=True,
                                                             fisher=True)
    assert abs(val - float(g('value'))) <= 1e-12 * abs(float(g('value')))
    np.testing.assert_allclose(gradfwd, g('gradfwd'), rtol=1e-10)
    np.testing.assert_allclose(fisher, g('fisher'), rtol=1e-10)
    dK, dr, v = g('dK'), g('dr'), g('vec')
    _, gradrev, _, _, fishvec = dec.minus_log_normal_density(
        g('r'), dK_vjp=lambda G: np.einsum('ij,ijk->k', G, dK), dr_vjp=lambda x: x @ dr, dK_jvp_vec=dK @ v, dr_jvp_vec=dr @ v,
        gradrev=True, fishvec=True)
    np.testing.assert_allclose(gradrev, g('gradrev'), rtol=1e-10)
    np.testing.assert_allclose(fishvec, g('fishvec'), rtol=1e-10)
    np.testing.assert_allclose(gradrev, g('gradfwd'), rtol=1e-9)      # the two modes agree (reference test :241-261)
    np.testing.assert_allclose(fishvec, g('fisher') @ v, rtol=1e-9)
    np.testing.assert_allclose(dec.ginv_linear(g('A')), g('ginv_linear'), rtol=1e-10, atol=1e-15)
    np.testing.assert_allclose(dec.ginv_quad(g('A')), g('ginv_quad'), rtol=1e-10, atol=1e-15)
    np.testing.assert_allclose(dec.pinv_bilinear(g('A'), g('r')), g('pinv_bilinear'), rtol=1e-10, atol=1e-15)
    np.testing.assert_allclose(dec.correlate(g('r')), g('correlate'), rtol=1e-10)
    np.testing.assert_allclose(dec.pinv_correlate(g('r')), g('pinv_correlate'), rtol=1e-10)


def test_oracle_bart_matches_reference(vec):
    length, splits = obart.splits_from_coord(vec['bart_X'])
    assert np.array_equal(length, vec['bart_length']) and np.array_equal(splits, vec['bart_splits'])
    idx = obart.indices_from_coord(vec['bart_X'], (length, splits))
    assert np.array_equal(idx, vec['bart_idx'])
    for name, kw in BART_VARIANTS.items():
        c = obart.gram(length, idx, idx, **kw)
        ref = vec['bart_corr_' + name]
        assert np.max(np.abs(c - ref) / np.spacing(np.abs(ref))) <= 32, name   # the reference's own bar between its two paths


def test_oracle_bart_recipe_matches_reference(vec):
    X5, y5 = vec['c4_X'], vec['c4_y']
    length, splits = obart.splits_from_coord(X5)
    idx = obart.indices_from_coord(X5, (length, splits))
    K = 1.3 ** 2 * obart.gram(length, idx, idx, maxd=10, reset=[2, 4, 6, 8]) + 0.25 * np.eye(len(y5)) + 0.49
    assert relerr(K, vec['c4_prior']) <= 1e-14
    assert abs(ogp.logml(K, y5, epsrel=0) - vec['c4_logml']) <= 1e-10 * abs(vec['c4_logml'])


# ------------------------------------------------------------------------------------------------ GPU tier
def _structured(lgp, X):
    return lgp.unstructured_to_structured(np.ascontiguousarray(X), names=NAMES)


@pytest.mark.gpu
def test_cuda_gram_matches_reference(vec):
    import lsqfitgp_b200 as lgp
    A, B = vec['gram_A'], vec['gram_B']
    xa, xb = _structured(lgp, A), _structured(lgp, B)
    kernels = {
        'expquad': lgp.ExpQuad(scale=1.5),
        'expquad_loc': 3.0 * lgp.ExpQuad(scale=0.3, loc=1.0),
        'maternp0': lgp.Constant() * lgp.Maternp(p=0, scale=2.0),
        'maternp1': lgp.Maternp(p=1, scale=2.0),
        'maternp2': lgp.Maternp(p=2, scale=2.0),
        'maternp3': lgp.Maternp(p=3, scale=2.0),
        'matern05': lgp.Matern(nu=0.5, scale=2.0),
        'matern25': lgp.Matern(nu=2.5, scale=2.0),
        'matern03': lgp.Matern(nu=0.3, scale=2.0),
        'matern13': lgp.Matern(nu=1.3, scale=2.0),
        'matern42': lgp.Matern(nu=4.2, scale=2.0),
        'ratquad': lgp.Cauchy(alpha=2, beta=3.0, scale=1.5),
        'cauchy13': lgp.Cauchy(alpha=1.3, beta=0.7, scale=4.0),
        'white_sum': 2.0 * lgp.ExpQuad(scale=1.5) + 0.01 * lgp.White() + 0.25,
        'product': lgp.Cauchy(alpha=2, beta=3.0, dim='f0') * (2.0 * lgp.ExpQuad(scale=0.7, dim='f1')),
    }
    for name, k in kernels.items():
        K = k(xa.reshape(-1, 1), xb.reshape(1, -1))
        tol = 2e-13 if name in ('matern03', 'matern13', 'matern42') else 1e-13
        assert relerr(K, vec['gram_' + name]) <= tol, name


@pytest.mark.gpu
def test_cuda_gp_matches_reference(vec):
    import lsqfitgp_b200 as lgp
    rng = np.random.default_rng(1001)
    x = np.sort(rng.uniform(0, 100, 1000))
    y = np.sin(x / 3) + 0.1 * rng.standard_normal(1000)
    xp = np.linspace(-5, 105, 500)
    gp = lgp.GP(lgp.ExpQuad(scale=3), checkpos=False).addx(x, 'data').addx(xp, 'pred')
    ycov = {('data', 'data'): 0.01 * np.eye(1000)}
    ml = gp.marginal_likelihood({'data': y}, ycov)
    assert abs(ml - vec['c1_logml']) <= 1e-9 * abs(vec['c1_logml'])
    m, c = gp.predfromdata({'data': y}, 'pred', ycov, raw=True)
    assert relerr(m, vec['c1_mean']) <= 1e-9
    assert np.max(np.abs(np.diag(c) - vec['c1_cov_diag'])) <= 1e-9
    assert np.max(np.abs(c[::25, ::25] - vec['c1_cov_sub'])) <= 1e-9
    X, y2, Xs = vec['c2_X'], vec['c2_y'], vec['c2_Xs']
    kernels = {'c2': 1.0 ** 2 * lgp.Matern(nu=2.5, scale=1.5) + 0.1 ** 2 * lgp.White(),
               'c2nu13': 1.3 * lgp.Matern(nu=1.3, scale=1.5) + 0.1 ** 2 * lgp.White(),
               'c3': 1.2 ** 2 * lgp.ExpQuad(scale=2.0) + 0.1 ** 2 * lgp.White(),
               'rq': 0.8 * lgp.Cauchy(alpha=2, beta=3.0, scale=1.5) + 0.1 ** 2 * lgp.White()}
    for tag, kern in kernels.items():
        gp = lgp.GP(kern, checkpos=False).addx(_structured(lgp, X), 'data').addx(_structured(lgp, Xs), 'pred')
        ml = gp.marginal_likelihood({'data': y2})
        assert abs(ml - vec[tag + '_logml']) <= 1e-9 * abs(vec[tag + '_logml']), tag
        m, c = gp.predfromdata({'data': y2}, 'pred', raw=True)
        assert np.max(np.abs(m - vec[tag + '_mean'])) <= 1e-9 * np.max(np.abs(vec[tag + '_mean'])), tag
        assert np.max(np.abs(c - vec[tag + '_cov'])) <= 1e-9, tag
        tol = 2e-13 if tag == 'c2nu13' else 1e-13
        assert relerr(gp.prior('data', raw=True)[:5], vec[tag + '_prior_rows']) <= tol, tag


@pytest.mark.gpu
@pytest.mark.parametrize('nn', [10, 64])
def test_cuda_chol_matches_reference(vec, nn):
    import lsqfitgp_b200 as lgp
    g = lambda k: vec[f'chol{nn}_{k}']
    dec = lgp._linalg.Chol(g('K'))
    assert abs(dec.eps - float(g('eps'))) <= 1e-13 * float(g('eps'))
    val, _, gradfwd, fisher, _ = dec.minus_log_normal_density(g('r'), dK=g('dK'), dr=g('dr'), value=True, gradfwd=True,
                                                             fisher=True)
    assert abs(val - float(g('value'))) <= 1e-9 * abs(float(g('value')))
    np.testing.assert_allclose(gradfwd, g('gradfwd'), rtol=1e-9, atol=1e-9 * np.abs(g('gradfwd')).max())
    np.testing.assert_allclose(fisher, g('fisher'), rtol=1e-9, atol=1e-9 * np.abs(g('fisher')).max())
    dK, dr, v = g('dK'), g('dr'), g('vec')
    _, gradrev, _, _, fishvec = dec.minus_log_normal_density(
        g('r'), dK_vjp=lambda G: np.einsum('ij,ijk->k', np.asarray(G), dK), dr_vjp=lambda x: np.asarray(x) @ dr,
        dK_jvp_vec=dK @ v, dr_jvp_vec=dr @ v, gradrev=True, fishvec=True)
    np.testing.assert_allclose(gradrev, g('gradrev'), rtol=1e-9, atol=1e-9 * np.abs(g('gradrev')).max())
    np.testing.assert_allclose(fishvec, g('fishvec'), rtol=1e-9, atol=1e-9 * np.abs(g('fishvec')).max())
    np.testing.assert_allclose(dec.ginv_linear(g('A')), g('ginv_linear'), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(dec.ginv_quad(g('A')), g('ginv_quad'), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(dec.pinv_bilinear(g('A'), g('r')), g('pinv_bilinear'), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(dec.correlate(g('r')), g('correlate'), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(dec.pinv_correlate(g('r')), g('pinv_correlate'), rtol=1e-9, atol=1e-12)


@pytest.mark.gpu
def test_cuda_bart_matches_reference(vec):
    import lsqfitgp_b200 as lgp
    X4 = vec['bart_X']
    length, splits = lgp.BART.splits_from_coord(X4)
    assert np.array_equal(length, vec['bart_length']) and np.array_equal(splits, vec['bart_splits'])
    idx = lgp.BART.indices_from_coord(X4, (length, splits))
    assert np.array_equal(idx, vec['bart_idx'])
    xi = lgp.unstructured_to_structured(idx.astype(np.int32), names=[f'c{i}' for i in range(5)])
    for name, kw in BART_VARIANTS.items():
        kb = lgp.BART(splits=(length, splits), indices=True, **kw)
        K = lgp.GP(kb, checkpos=False, checksym=False).addx(xi, 't').prior('t', raw=True)
        assert relerr(K, vec['bart_corr_' + name]) <= 1e-13, name


@pytest.mark.gpu
def test_cuda_bart_recipe_matches_reference(vec):
    """ config C4 recipe through the public API exactly as the reference's bayestree.bart builds it """
    import lsqfitgp_b200 as lgp
    X5, y5 = vec['c4_X'], vec['c4_y']
    n = len(y5)
    sp = lgp.BART.splits_from_coord(X5)
    idx = lgp.BART.indices_from_coord(X5, sp)
    xi = lgp.unstructured_to_structured(idx.astype(np.int32), names=[f'c{i}' for i in range(5)])
    kb = lgp.BART(splits=sp, indices=True, maxd=10, reset=[2, 4, 6, 8])
    gp = (lgp.GP(1.3 ** 2 * kb, checkpos=False, checksym=False, epsrel=0)
          .addx(xi, 'trainmean').addcov(0.5 ** 2 * np.eye(n), 'trainnoise').addcov(0.7 ** 2, 'mean')
          .addtransf({'trainmean': 1, 'trainnoise': 1, 'mean': 1}, 'train'))
    assert relerr(gp.prior('train', raw=True), vec['c4_prior']) <= 1e-13
    ml = gp.marginal_likelihood({'train': y5})
    assert abs(ml - vec['c4_logml']) <= 1e-9 * abs(vec['c4_logml'])


@pytest.mark.gpu
def test_cuda_multikey_gp_matches_reference(vec):
    """ several keys, addtransf, data on two keys with given covariances, predfromdata on a list of keys, predfromfit:
    the reference's GP orchestration (_GP/_elements.py:248-649, _compute.py:138-322) against this one """
    import lsqfitgp_b200 as lgp
    g = lambda k: vec['mk_' + k]
    gp = (lgp.GP(1.5 * lgp.ExpQuad(scale=2.0) + 0.05 * lgp.Maternp(p=1, scale=0.7), checkpos=False)
          .addx(g('xa'), 'a').addx(g('xb'), 'b').addtransf({'a': g('Ta'), 'b': g('Tb')}, 'c'))
    pr = gp.prior(['a', 'c'], raw=True)
    np.testing.assert_allclose(pr['a', 'c'], g('prior_ac'), rtol=1e-12, atol=1e-13)
    np.testing.assert_allclose(pr['c', 'c'], g('prior_cc'), rtol=1e-12, atol=1e-12)
    ml = gp.marginal_likelihood({'c': g('yc'), 'a': g('ya')}, {('c', 'c'): g('ccov'), ('a', 'a'): 0.01 * np.eye(25),
                                                              ('c', 'a'): np.zeros((7, 25)), ('a', 'c'): np.zeros((25, 7))})
    assert abs(ml - float(g('logml'))) <= 1e-9 * abs(float(g('logml')))
    m, c = gp.predfromdata({'c': g('yc')}, ['a', 'b'], {('c', 'c'): g('ccov')}, raw=True)
    np.testing.assert_allclose(m['a'], g('mean_a'), rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(m['b'], g('mean_b'), rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(c['a', 'b'], g('cov_ab'), rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(c['b', 'b'], g('cov_bb'), rtol=1e-9, atol=1e-10)
    m, c = gp.predfromfit({'c': g('yc')}, 'b', {('c', 'c'): g('ccov')}, raw=True)
    np.testing.assert_allclose(m, g('fit_mean_b'), rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(c, g('fit_cov_bb'), rtol=1e-9, atol=1e-10)


@pytest.mark.gpu
def test_cuda_input_formats_match_reference(vec):
    """ fields with a shape, `dim=` selecting such a field, unstructured inputs with broadcasting, integer inputs """
    import lsqfitgp_b200 as lgp
    xs = np.zeros(20, dtype=[('a', float), ('b', float, 3)])
    ys = np.zeros(15, dtype=xs.dtype)
    xs['a'], xs['b'], ys['a'], ys['b'] = vec['fmt_xa'], vec['fmt_xb'], vec['fmt_ya'], vec['fmt_yb']
    K = lgp.Matern(nu=1.5, scale=1.3)(xs[:, None], ys[None, :])
    assert relerr(K, vec['fmt_shaped']) <= 1e-13
    K = lgp.ExpQuad(scale=0.9, dim='b')(xs[:, None], ys[None, :])
    assert relerr(K, vec['fmt_dim_b']) <= 1e-13
    K = (lgp.ExpQuad(dim='a') * lgp.Cauchy(beta=2.0, dim='b'))(xs[:, None], ys[None, :])
    assert relerr(K, vec['fmt_dim_a_times_b']) <= 1e-13
    K = lgp.Maternp(p=2, scale=0.8, loc=0.5)(vec['fmt_u'][:, None], vec['fmt_v'][None, :])
    assert relerr(K, vec['fmt_plain']) <= 1e-13
    K = (2 * lgp.ExpQuad(scale=3) + lgp.White())(np.arange(6)[:, None], np.arange(4, 9)[None, :])
    assert relerr(K, vec['fmt_int']) <= 1e-13
