"""GPU parity of the BART path added in round 2: chained bracket stages (reset patterns that do not fold into one
`repeat` sequence, reference _kernels/_bart.py:447-455), symmetric evaluation, alpha / beta gradients through the
public API in reverse and forward mode (the kernels themselves are checked in test_gpu_bart_exact.py), and the
`bayestree.bart` recipe (reference bayestree/_bart.py:147-240) fitted end to end against the oracle's objective."""
import numpy as np
import pytest
import torch
from scipy import optimize, stats

import lsqfitgp_b200 as lgp
from lsqfitgp_b200 import _ops
from oracle import gp as ogp, bart as obart

pytestmark = pytest.mark.gpu
DEV = 'cuda'


def _data(n, seed=4004, p=6):
    rng = np.random.default_rng(seed)
    X = np.concatenate([rng.standard_normal((n, p - 2)), rng.integers(0, 3, (n, 2)).astype(float)], axis=1)
    splits = lgp.BART.splits_from_coord(X)
    idx = lgp.BART.indices_from_coord(X, splits)
    return X, splits, idx


def _dev_idx(idx):
    return torch.tensor(np.ascontiguousarray(idx.T.astype(np.int32)), device=DEV)


@pytest.mark.parametrize('kw', [dict(maxd=3, reset=[1]), dict(maxd=6, reset=[1, 2, 4]),
                                dict(maxd=7, reset=[2, 3, 5], intercept=False, gamma=0.4),
                                dict(maxd=4, reset=[2], weights=np.r_[1., 0., 2., 0.5, 1., 3.]),
                                dict(maxd=10, reset=[2, 4, 6, 8])])
def test_chained_stages_and_symmetry_vs_oracle(kw):
    X, splits, idx = _data(333)
    xi = lgp.unstructured_to_structured(idx.astype(np.int32), names=[f'c{i}' for i in range(idx.shape[1])])
    kb = lgp.BART(splits=splits, indices=True, **kw)
    gp = lgp.GP(kb, checkpos=False, checksym=False).addx(xi, 'a').addx(xi[:70], 'b')
    pr = gp.prior(['a', 'b'], raw=True)
    Ko = obart.gram(splits[0], idx, idx, **kw)
    assert np.max(np.abs(pr['a', 'a'] - Ko) / np.abs(Ko)) < 1e-13
    assert np.max(np.abs(pr['a', 'b'] - Ko[:, :70]) / np.abs(Ko[:, :70])) < 1e-13
    assert np.array_equal(pr['a', 'a'], pr['a', 'a'].T)
    # the symmetric evaluation (lower tiles mirrored) is bit-identical to the general one
    spec = kb._bart[0]
    widths, nrows, rows, drows, gamma = spec.stages()
    w = np.ones(idx.shape[1]) if kw.get('weights') is None else kw['weights']
    ix = _dev_idx(idx)
    Ks = _ops.gram_bart_stages(splits[0], w, widths, nrows, rows, drows, gamma, 1.0, ix, ix, symmetric=True)
    Kg = _ops.gram_bart_stages(splits[0], w, widths, nrows, rows, drows, gamma, 1.0, ix, ix.clone(), symmetric=False)
    assert torch.equal(Ks, Kg)


def test_alpha_beta_gradient_through_api():
    """ d logML / d (alpha, beta, amplitude) by torch.autograd through lgp_gram_bart_vjp against
    -1/2 tr(K^-1 dK) + 1/2 b' dK b, b = K^-1 y, with dK from the oracle's complex-step derivatives (the derivatives the
    reference gets by tracing _bart.py with JAX): one folded width-3 stage on 6 columns, and chained stages on 17
    columns of which one has weight 0 """
    w17 = np.r_[np.ones(9), 0.0, np.linspace(0.5, 2, 7)]
    for p, kw in ((6, dict(maxd=10, reset=[2, 4, 6, 8])), (17, dict(maxd=6, reset=[1, 2, 4], weights=w17))):
        X, splits, idx = _data(240, seed=21, p=p)
        n = len(idx)
        xi = lgp.unstructured_to_structured(idx.astype(np.int32), names=[f'c{i}' for i in range(idx.shape[1])])
        y = np.random.default_rng(5).standard_normal(n)
        t0 = np.array([0.9, 1.6, 1.2])
        th = torch.tensor(t0, dtype=torch.float64, requires_grad=True)
        kb = th[2] ** 2 * lgp.BART(splits=splits, indices=True, alpha=th[0], beta=th[1], **kw)
        gp = (lgp.GP(kb, checkpos=False, checksym=False, epsrel=0).addx(xi, 'f').addcov(0.3 * np.eye(n), 'e')
              .addtransf({'f': 1, 'e': 1}, 'y'))
        ml = gp.marginal_likelihood({'y': y})
        g, = torch.autograd.grad(ml, th)
        Kb, dKa, dKb = obart.gram_derivs(splits[0], idx, idx, alpha=t0[0], beta=t0[1], **kw)
        Ko = t0[2] ** 2 * Kb + 0.3 * np.eye(n)
        assert abs(float(ml.detach()) - ogp.logml(Ko, y, epsrel=0)) <= 1e-9 * abs(ogp.logml(Ko, y, epsrel=0)), p
        Ki = np.linalg.inv(Ko)
        b = Ki @ y
        want = np.array([-0.5 * np.sum(Ki * dK) + 0.5 * b @ dK @ b
                         for dK in (t0[2] ** 2 * dKa, t0[2] ** 2 * dKb, 2 * t0[2] * Kb)])
        assert np.max(np.abs(g.numpy() - want)) <= 1e-9 * np.max(np.abs(want)), (p, g.numpy(), want)


def test_empbayes_fit_fisher_bart():
    """ method='fisher' on a BART GP runs the BART forward mode (lgp_gram_bart_stages with derivatives, through the
    Gram JVP of the public API): amplitude and noise fitted in log space, alpha = sigmoid(za) and beta = exp(zb) mapped
    by torch ops.  minresult.hess - I equals the oracle's 1/2 tr(K^-1 dK_i K^-1 dK_j) (prior sdev 1: identity
    jacobian), with dK/dp_i by complex step through the parameter maps and the BART correlation """
    X, splits, idx = _data(200, seed=31)
    n = len(idx)
    xi = lgp.unstructured_to_structured(idx.astype(np.int32), names=[f'c{i}' for i in range(idx.shape[1])])
    rng = np.random.default_rng(32)
    y = np.sin(X[:, 0]) + 0.5 * X[:, 4] + 0.3 * rng.standard_normal(n)
    hyperprior = {'log(amp)': (0.0, 1.0), 'log(noise)': (np.log(0.3), 1.0), 'za': (1.0, 1.0), 'zb': (0.5, 1.0)}
    bkw = dict(maxd=10, reset=[2, 4, 6, 8])

    def gpfactory(hp):
        k = hp['amp'] ** 2 * lgp.BART(splits=splits, indices=True, alpha=torch.sigmoid(hp['za']),
                                      beta=torch.exp(hp['zb']), **bkw) + hp['noise'] ** 2 * lgp.White()
        return lgp.GP(k, checkpos=False, checksym=False).addx(xi, 'data')
    fit = lgp.empbayes_fit(hyperprior, gpfactory, {'data': y}, raises=False, method='fisher')
    mean = np.array([v[0] for v in hyperprior.values()])

    def Kof(pv):
        la, ln, za, zb = mean + pv
        Kb = obart.gram(splits[0], idx, idx, alpha=1 / (1 + np.exp(-za)), beta=np.exp(zb), **bkw)
        return np.exp(2 * la) * Kb + np.exp(2 * ln) * np.eye(n)
    x = fit.minresult.x
    h = 1e-200
    Ki = np.linalg.inv(Kof(x))
    A = [Ki @ (Kof(x + 1j * h * e).imag / h) for e in np.eye(4)]
    fo = np.array([[0.5 * np.sum(a * b.T) for b in A] for a in A])
    assert np.max(np.abs(fit.minresult.hess - np.eye(4) - fo)) <= 1e-9 * np.max(np.abs(fo)), (fit.minresult.hess, fo)


def test_bayestree_bart_fit_vs_oracle():
    """ the bayestree.bart recipe end to end (hyperprior on alpha, beta, log k, log sigma2; epsrel=0; l-bfgs-b) at n = 300:
    the optimum found on the GPU is a stationary point of the ORACLE's objective, with the same objective value, and the
    oracle's own minimisation from the prior mean lands on it (reference tests/test_fit.py:142-176: atol 1e-5). """
    rng = np.random.default_rng(4006)
    n, p = 300, 5
    X = rng.standard_normal((n, p))
    y = np.sin(2 * X[:, 0]) + 0.5 * X[:, 1] * (X[:, 2] > 0) + 0.3 * rng.standard_normal(n)
    fit = lgp.bayestree.bart(X, y, fitkw=dict(minkw=dict(method='l-bfgs-b', options=dict(maxiter=300, ftol=1e-14,
                                                                                        gtol=1e-8))))
    res = fit.fit.minresult
    splits = lgp.BART.splits_from_coord(X)
    idx = lgp.BART.indices_from_coord(X, splits)
    ymin, ymax = y.min(), y.max()
    mu_mu, ksm = (ymax + ymin) / 2, (ymax - ymin) / 2
    s2pm = np.mean((y - y.mean()) ** 2)
    mean = np.array([0.0, 0.0, np.log(2), np.log(s2pm)])
    sd = np.array([1.0, 1.0, 2.0, 2.0])

    def hp_of(pv):
        z = mean + sd * pv
        alpha = stats.beta.ppf(stats.norm.cdf(z[0]), 2, 1)
        beta = stats.invgamma.ppf(stats.norm.cdf(z[1]), 1) if z[1] < 0 else stats.invgamma.isf(stats.norm.cdf(-z[1]), 1)
        return alpha, beta, np.exp(z[2]), np.exp(z[3])

    def obj(pv):
        alpha, beta, k, s2 = hp_of(pv)
        Ko = (ksm / k) ** 2 * obart.gram(splits[0], idx, idx, alpha=alpha, beta=beta, maxd=10, reset=[2, 4, 6, 8]) \
            + s2 * np.eye(n) + ksm ** 2
        return -ogp.logml(Ko, y - mu_mu, epsrel=0) + 0.5 * (4 * np.log(2 * np.pi) + pv @ pv)
    x = res.x
    assert abs(res.fun - obj(x)) <= 1e-9 * abs(obj(x))
    h = 1e-5
    g_or = np.array([(obj(x + e) - obj(x - e)) / (2 * h) for e in h * np.eye(4)])
    assert np.max(np.abs(g_or)) < 2e-4, g_or          # stationary point of the oracle objective (FD noise ~1e-5)
    ro = optimize.minimize(obj, np.zeros(4), method='l-bfgs-b', options=dict(maxiter=300, ftol=1e-15, gtol=1e-9))
    assert abs(ro.fun - res.fun) <= 1e-8 * abs(ro.fun)
    assert np.max(np.abs(ro.x - x)) < 1e-3
    # fitted attributes and prediction API
    a, b = fit.alpha[0], fit.beta[0]
    ao, bo, ko, s2o = hp_of(x)
    assert a == pytest.approx(ao, rel=1e-12) and b == pytest.approx(bo, rel=1e-10)
    assert fit.meansdev[0] == pytest.approx(ksm / ko, rel=1e-12) and fit.sigma[0] == pytest.approx(np.sqrt(s2o), rel=1e-12)
    m, c = fit.pred()
    Kf = (ksm / ko) ** 2 * obart.gram(splits[0], idx, idx, alpha=ao, beta=bo, maxd=10, reset=[2, 4, 6, 8])
    m_o, c_o = ogp.pred(Kf + s2o * np.eye(n) + ksm ** 2, Kf, Kf, y - mu_mu, epsrel=0)   # 'trainmean': the latent f only
    np.testing.assert_allclose(m, m_o + mu_mu, rtol=1e-8, atol=1e-9)
    Xt = rng.standard_normal((40, p))
    mt, ct = fit.pred(x_test=Xt, error=True)
    assert mt.shape == (40,) and ct.shape == (40, 40) and np.all(np.diag(ct) > s2o * 0.99)
    assert 'BART fit' in repr(fit)
    # CUDA-event phase timers of the fit (reference _fit.py:410-442,775-794)
    t = fit.fit.times
    assert set(t) == {'gp&cov', 'decomp', 'likelihood', 'other'} and all(v >= 0 for v in t.values())
    assert t['gp&cov'] > 0 and t['decomp'] > 0 and t['likelihood'] > 0


def test_c4_size_fit_step_timing():
    """ one objective + gradient evaluation of the recipe at the BASELINE configs[3] size (n = 5000, p = 10) runs and is
    finite; its timing is reported by tools/bench_configs.py """
    rng = np.random.default_rng(4004)
    n = 5000
    X = np.concatenate([rng.standard_normal((n, 8)), rng.integers(0, 2, (n, 2)).astype(float)], axis=1)
    y = rng.standard_normal(n)
    splits = lgp.BART.splits_from_coord(X)
    idx = lgp.BART.indices_from_coord(X, splits)
    xi = lgp.unstructured_to_structured(idx.astype(np.int32), names=[f'c{i}' for i in range(10)])
    th = torch.tensor([0.95, 2.0, 1.1, 0.5], dtype=torch.float64, requires_grad=True)
    kb = th[2] ** 2 * lgp.BART(splits=splits, indices=True, alpha=th[0], beta=th[1], maxd=10, reset=[2, 4, 6, 8])
    gp = (lgp.GP(kb, checkpos=False, checksym=False, checkfinite=False, epsrel=0).addx(xi, 'trainmean')
          .addcov(torch.diag((th[3] * torch.ones(n, dtype=torch.float64)).to(DEV)), 'trainnoise').addcov(0.49, 'mean')
          .addtransf({'trainmean': 1, 'trainnoise': 1, 'mean': 1}, 'train'))
    ml = gp.marginal_likelihood({'train': y})
    g, = torch.autograd.grad(ml, th)
    assert np.isfinite(float(ml.detach())) and np.all(np.isfinite(g.numpy())) and np.all(g.numpy() != 0)
