"""Golden vectors produced by EXECUTING THE REFERENCE'S OWN SOURCE (/root/reference/src/lsqfitgp) under the numpy stand-in
for jax of oracle/refshim.py (jax, jaxlib and gvar are not installable in this image).  Run in the build container:

    PYTHONPATH=. python tests/golden/gen_reference_vectors.py        # writes tests/golden/reference_vectors.npz

What runs is the reference's code: lgp.GP.marginal_likelihood / predfromdata(raw=True) (_GP/_compute.py), the kernel
classes (_kernels/_basic.py, _matern.py, _bart.py with _Kernel/*), _linalg/_decomp.py Chol.  What stands in for JAX:
numpy for jax.numpy, scipy LAPACK for jax.scipy.linalg, python loops for lax.scan / fori_loop.  tests/test_reference_vectors.py
checks the oracle (and, on the GPU, the CUDA path) against the file."""
import pathlib
import sys
import warnings

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[2]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
OUT = pathlib.Path(__file__).resolve().parent / 'reference_vectors.npz'


def structured(X, names):
    x = np.zeros(len(X), dtype=[(n, float) for n in names])
    for i, n in enumerate(names):
        x[n] = X[:, i]
    return x


def generate():
    from oracle import refshim
    warnings.simplefilter('ignore')
    GPm, basic, matern, bartm, decomp = refshim.load_reference('_GP', '_kernels._basic', '_kernels._matern',
                                                               '_kernels._bart', '_linalg._decomp')
    GP = GPm.GP
    out = {}

    # ---- config C1 at full size: ExpQuad 1-D n=1000, data covariance 0.01 I, 500 prediction points (SURVEY 8d)
    rng = np.random.default_rng(1001)
    x = np.sort(rng.uniform(0, 100, 1000))
    y = np.sin(x / 3) + 0.1 * rng.standard_normal(1000)
    xp = np.linspace(-5, 105, 500)
    gp = GP(basic.ExpQuad(scale=3), checkpos=False).addx(x, 'data').addx(xp, 'pred')
    ycov = {('data', 'data'): 0.01 * np.eye(1000)}
    out['c1_logml'] = float(gp.marginal_likelihood({'data': y}, ycov))
    m, c = gp.predfromdata({'data': y}, 'pred', ycov, raw=True)
    out['c1_mean'] = np.asarray(m)
    out['c1_cov_diag'] = np.diag(np.asarray(c)).copy()
    out['c1_cov_sub'] = np.asarray(c)[::25, ::25].copy()

    # ---- config C2 at n=400: sf^2 Matern(nu=2.5, scale=ell) + sn^2 White on 3 fields; logML, posterior mean at 20 points
    rng = np.random.default_rng(2002)
    n = 400
    X = rng.uniform(0, 10, (n, 3))
    y2 = np.sin(X[:, 0]) + np.cos(X[:, 1]) * X[:, 2] / 10 + 0.1 * rng.standard_normal(n)
    Xs = rng.uniform(0, 10, (20, 3))
    names = ['f0', 'f1', 'f2']
    for tag, kern in [('c2', 1.0 ** 2 * matern.Matern(nu=2.5, scale=1.5) + 0.1 ** 2 * basic.White()),
                      ('c2nu13', 1.3 * matern.Matern(nu=1.3, scale=1.5) + 0.1 ** 2 * basic.White()),
                      ('c3', 1.2 ** 2 * basic.ExpQuad(scale=2.0) + 0.1 ** 2 * basic.White()),
                      ('rq', 0.8 * basic.Cauchy(alpha=2, beta=3.0, scale=1.5) + 0.1 ** 2 * basic.White())]:
        gp = GP(kern, checkpos=False).addx(structured(X, names), 'data').addx(structured(Xs, names), 'pred')
        out[tag + '_logml'] = float(gp.marginal_likelihood({'data': y2}))
        m, c = gp.predfromdata({'data': y2}, 'pred', raw=True)
        out[tag + '_mean'] = np.asarray(m)
        out[tag + '_cov'] = np.asarray(c)
        out[tag + '_prior_rows'] = np.asarray(gp.prior('data', raw=True))[:5].copy()
    out['c2_X'], out['c2_y'], out['c2_Xs'] = X, y2, Xs

    # ---- Gram blocks of every supported kernel (rectangular, 3 fields)
    rng = np.random.default_rng(11)
    A = rng.uniform(0, 10, (40, 3))
    B = rng.uniform(0, 10, (30, 3))
    B[3] = A[5]   # a coincident point (White, r2 == 0)
    out['gram_A'], out['gram_B'] = A, B
    xa, xb = structured(A, names), structured(B, names)
    kernels = {
        'expquad': basic.ExpQuad(scale=1.5),
        'expquad_loc': 3.0 * basic.ExpQuad(scale=0.3, loc=1.0),
        'maternp0': basic.Constant() * matern.Maternp(p=0, scale=2.0),
        'maternp1': matern.Maternp(p=1, scale=2.0),
        'maternp2': matern.Maternp(p=2, scale=2.0),
        'maternp3': matern.Maternp(p=3, scale=2.0),
        'matern05': matern.Matern(nu=0.5, scale=2.0),
        'matern25': matern.Matern(nu=2.5, scale=2.0),
        'matern03': matern.Matern(nu=0.3, scale=2.0),
        'matern13': matern.Matern(nu=1.3, scale=2.0),
        'matern42': matern.Matern(nu=4.2, scale=2.0),
        'ratquad': basic.Cauchy(alpha=2, beta=3.0, scale=1.5),
        'cauchy13': basic.Cauchy(alpha=1.3, beta=0.7, scale=4.0),
        'white_sum': 2.0 * basic.ExpQuad(scale=1.5) + 0.01 * basic.White() + 0.25,
        'product': basic.Cauchy(alpha=2, beta=3.0, dim='f0') * (2.0 * basic.ExpQuad(scale=0.7, dim='f1')),
    }
    for name, k in kernels.items():
        out['gram_' + name] = np.asarray(k(xa[:, None], xb[None, :]))

    # ---- input formats: a field with a shape (reduced with a sum over its last axis, _Kernel/_util.py:74-99), `dim=` on it,
    # unstructured 1-D inputs with broadcasting, integer inputs
    rng = np.random.default_rng(12)
    xs_ = np.zeros(20, dtype=[('a', float), ('b', float, 3)])
    ys_ = np.zeros(15, dtype=xs_.dtype)
    xs_['a'], xs_['b'] = rng.uniform(0, 5, 20), rng.uniform(0, 5, (20, 3))
    ys_['a'], ys_['b'] = rng.uniform(0, 5, 15), rng.uniform(0, 5, (15, 3))
    out['fmt_xa'], out['fmt_xb'], out['fmt_ya'], out['fmt_yb'] = xs_['a'], xs_['b'], ys_['a'], ys_['b']
    out['fmt_shaped'] = np.asarray(matern.Matern(nu=1.5, scale=1.3)(xs_[:, None], ys_[None, :]))
    out['fmt_dim_b'] = np.asarray(basic.ExpQuad(scale=0.9, dim='b')(xs_[:, None], ys_[None, :]))
    out['fmt_dim_a_times_b'] = np.asarray((basic.ExpQuad(dim='a') * basic.Cauchy(beta=2.0, dim='b'))(xs_[:, None], ys_[None, :]))
    u1, v1 = rng.uniform(0, 5, 12), rng.uniform(0, 5, 9)
    out['fmt_u'], out['fmt_v'] = u1, v1
    out['fmt_plain'] = np.asarray(matern.Maternp(p=2, scale=0.8, loc=0.5)(u1[:, None], v1[None, :]))
    ui, vi = np.arange(6), np.arange(4, 9)
    out['fmt_int'] = np.asarray((2 * basic.ExpQuad(scale=3) + basic.White())(ui[:, None], vi[None, :]))

    # ---- Chol (reference tests/linalg/test_decomp.py matrices) with value, forward gradient and Fisher matrix
    from scipy import stats
    rng = np.random.default_rng(5)
    for nn in (10, 64):
        O = stats.ortho_group.rvs(nn, random_state=rng)
        K = (O * (1 + 1e-3 + np.cos(0.3 + np.arange(nn)))) @ O.T
        K = (K + K.T) / 2
        K = K * np.outer(np.exp(rng.uniform(-3, 3, nn)), np.ones(nn))      # unequal scales: exercises the equilibration
        K = (K + K.T) / 2 + 50 * np.diag(np.exp(rng.uniform(-3, 3, nn)))
        r = rng.standard_normal(nn)
        Amat = rng.standard_normal((nn, 3))
        dK = rng.standard_normal((nn, nn, 2))
        dK = dK + dK.transpose(1, 0, 2)
        dr = rng.standard_normal((nn, 2))
        dec = decomp.Chol(K)
        val, _, gradfwd, fisher, _ = dec.minus_log_normal_density(r, dK=dK, dr=dr, value=True, gradfwd=True, fisher=True)
        out[f'chol{nn}_K'], out[f'chol{nn}_r'], out[f'chol{nn}_A'] = K, r, Amat
        out[f'chol{nn}_dK'], out[f'chol{nn}_dr'] = dK, dr
        out[f'chol{nn}_eps'] = float(dec.eps)
        out[f'chol{nn}_value'] = float(val)
        out[f'chol{nn}_gradfwd'] = np.asarray(gradfwd)
        out[f'chol{nn}_fisher'] = np.asarray(fisher)
        # reverse-mode assembly (_decomp.py:505-512) and Fisher-vector product (:560-582) with explicit callbacks
        vecv = rng.standard_normal(2)
        _, gradrev, _, _, fishvec = dec.minus_log_normal_density(
            r, dK_vjp=lambda G: np.einsum('ij,ijk->k', np.asarray(G), dK), dr_vjp=lambda g: np.asarray(g) @ dr,
            dK_jvp_vec=dK @ vecv, dr_jvp_vec=dr @ vecv, gradrev=True, fishvec=True)
        out[f'chol{nn}_vec'] = vecv
        out[f'chol{nn}_gradrev'] = np.asarray(gradrev)
        out[f'chol{nn}_fishvec'] = np.asarray(fishvec)
        out[f'chol{nn}_ginv_linear'] = np.asarray(dec.ginv_linear(Amat))
        out[f'chol{nn}_ginv_quad'] = np.asarray(dec.ginv_quad(Amat))
        out[f'chol{nn}_pinv_bilinear'] = np.asarray(dec.pinv_bilinear(Amat, r))
        out[f'chol{nn}_correlate'] = np.asarray(dec.correlate(r))
        out[f'chol{nn}_pinv_correlate'] = np.asarray(dec.pinv_correlate(r))

    # ---- BART: preprocessing and correlation variants (reference _kernels/_bart.py)
    rng = np.random.default_rng(4004)
    nb = 30
    X4 = np.concatenate([rng.standard_normal((nb, 4)), rng.integers(0, 2, (nb, 1)).astype(float)], axis=1)
    length, splits = bartm.BART.splits_from_coord(X4)
    idx = np.asarray(bartm.BART.indices_from_coord(X4, (length, splits)))
    out['bart_X'], out['bart_length'], out['bart_splits'], out['bart_idx'] = X4, np.asarray(length), np.asarray(splits), idx
    variants = {
        'd0': dict(maxd=0), 'd1': dict(maxd=1), 'd2': dict(maxd=2), 'd4r2': dict(maxd=4, reset=2),
        'd2g': dict(maxd=2, gamma=0.3, intercept=False), 'd10': dict(maxd=10, reset=[2, 4, 6, 8], gamma=1),
        'd6w': dict(maxd=6, reset=[2, 4], weights=np.array([1., 0., 2., 3., 0.5])),
    }
    for name, kw in variants.items():
        out['bart_corr_' + name] = np.asarray(bartm.BART.correlation(np.asarray(length), idx[:, None, :], idx[None, :, :],
                                                                     altinput=True, **kw))
    # ---- multi-key GP: two sets of points, a linear transformation of both, data on the transformed key and on one set;
    # predfromdata on several keys, predfromfit with a given covariance, prior blocks (_GP/_elements.py, _compute.py)
    rng = np.random.default_rng(77)
    xa_, xb_ = np.sort(rng.uniform(0, 10, 25)), np.sort(rng.uniform(0, 10, 18))
    Ta, Tb = rng.standard_normal((7, 25)), rng.standard_normal((7, 18))
    yc, ya = rng.standard_normal(7), rng.standard_normal(25)
    R = rng.standard_normal((7, 7))
    ccov = R @ R.T / 7 + 0.1 * np.eye(7)
    gp = (GP(1.5 * basic.ExpQuad(scale=2.0) + 0.05 * matern.Maternp(p=1, scale=0.7), checkpos=False)
          .addx(xa_, 'a').addx(xb_, 'b').addtransf({'a': Ta, 'b': Tb}, 'c'))
    out['mk_xa'], out['mk_xb'], out['mk_Ta'], out['mk_Tb'] = xa_, xb_, Ta, Tb
    out['mk_yc'], out['mk_ya'], out['mk_ccov'] = yc, ya, ccov
    pr = gp.prior(['a', 'c'], raw=True)
    out['mk_prior_ac'], out['mk_prior_cc'] = np.asarray(pr['a', 'c']), np.asarray(pr['c', 'c'])
    out['mk_logml'] = float(gp.marginal_likelihood({'c': yc, 'a': ya}, {('c', 'c'): ccov, ('a', 'a'): 0.01 * np.eye(25),
                                                                         ('c', 'a'): np.zeros((7, 25)), ('a', 'c'): np.zeros((25, 7))}))
    m, c = gp.predfromdata({'c': yc}, ['a', 'b'], {('c', 'c'): ccov}, raw=True)
    out['mk_mean_a'], out['mk_mean_b'] = np.asarray(m['a']), np.asarray(m['b'])
    out['mk_cov_ab'], out['mk_cov_bb'] = np.asarray(c['a', 'b']), np.asarray(c['b', 'b'])
    m, c = gp.predfromfit({'c': yc}, 'b', {('c', 'c'): ccov}, raw=True)
    out['mk_fit_mean_b'], out['mk_fit_cov_bb'] = np.asarray(m), np.asarray(c)

    # ---- config C4 recipe (bayestree.bart, reference bayestree/_bart.py:187-227): lambda^2 BART + sigma^2 I + k^2 through
    # addx / addcov / addtransf of the reference's GP, epsrel = 0
    rng = np.random.default_rng(4005)
    nr = 40
    X5 = np.concatenate([rng.standard_normal((nr, 4)), rng.integers(0, 2, (nr, 1)).astype(float)], axis=1)
    sp = bartm.BART.splits_from_coord(X5)
    idx5 = np.asarray(bartm.BART.indices_from_coord(X5, sp))
    xi = np.zeros(nr, dtype=[(f'c{i}', 'i4') for i in range(5)])
    for i in range(5):
        xi[f'c{i}'] = idx5[:, i]
    y5 = rng.standard_normal(nr)
    lam, sig, kk = 1.3, 0.5, 0.7
    kb = bartm.BART(splits=sp, indices=True, maxd=10, reset=[2, 4, 6, 8])
    gp = (GP(lam ** 2 * kb, checkpos=False, checksym=False, epsrel=0)
          .addx(xi, 'trainmean').addcov(sig ** 2 * np.eye(nr), 'trainnoise').addcov(kk ** 2, 'mean')
          .addtransf({'trainmean': 1, 'trainnoise': 1, 'mean': 1}, 'train'))
    out['c4_X'], out['c4_y'] = X5, y5
    out['c4_logml'] = float(gp.marginal_likelihood({'train': y5}))
    out['c4_prior'] = np.asarray(gp.prior('train', raw=True))
    return out


if __name__ == '__main__':
    vec = generate()
    np.savez_compressed(OUT, **vec)
    print(f'wrote {OUT} ({OUT.stat().st_size / 1024:.0f} KiB, {len(vec)} arrays)')
    for k in ('c1_logml', 'c2_logml', 'c2nu13_logml', 'c3_logml', 'rq_logml', 'chol10_eps', 'chol64_value'):
        print(k, vec[k])
