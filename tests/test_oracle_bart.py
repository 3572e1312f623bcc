"""Pin the BART oracle (reference tests/kernels/test_bart.py restated): the fast closed-form path against the
independent recursive implementation `_correlation_old` (test_altinput :332-353), exactness cases (:105-133),
intercept / pnt identities (:283-301), splits (:268-271), and the C restatement."""
import ctypes
import pathlib

import numpy as np
import pytest

from oracle import bart

rng0 = np.random.default_rng(202307302223)
plist = [1, 5]
SCASES = sum([[
    (*rng0.integers(0, 4, (3, p)), rng0.integers(1, 10, p)),
    (*np.zeros((3, p), int), rng0.integers(1, 10, p)),
    (np.zeros(p, int), np.pad([1], (0, p - 1)), np.zeros(p, int), rng0.integers(1, 10, p)),
    (rng0.integers(0, 10, p), (np.arange(p) == rng0.integers(p)).astype(int), rng0.integers(0, 10, p),
     rng0.integers(1, 10, p)),
] for p in plist], [])
smark = pytest.mark.parametrize('sb,sbw,sa,w', SCASES)
ALPHAS = [0.0, 1.0, 0.01, 0.5, 0.95]
BETAS = [0.0, 1.0, 2.0, 5.5]


@pytest.mark.parametrize('md,reset', [(0, None), (1, None), (2, None), (2, [1]), (3, None), (3, [1, 2]), (4, None),
                                      (4, [2]), (4, [1, 2, 3])])
@smark
def test_altinput(sb, sbw, sa, w, md, reset, rng):
    """ fast index-based path == old count-based recursion (reference :332-353) """
    if md >= 3 and max(sb.max(), sbw.max(), sa.max()) > 4 and reset is None:
        pytest.skip('exponential recursion too slow in pure python')
    for a in ALPHAS[:3] + ALPHAS[4:]:
        for b in BETAS[:3]:
            for u in (0.0, 1.0):
                kw = dict(alpha=a, beta=b, gamma=u, maxd=md, reset=reset, weights=w)
                c1 = bart.correlation(sb, sbw, sa, altinput=False, **kw)
                n = sb + sbw + sa
                ix, iy = sb, sb + sbw
                swap = rng.integers(0, 2, size=ix.shape, dtype=bool)
                ix, iy = np.where(swap, iy, ix), np.where(swap, ix, iy)
                c2 = bart.correlation(n, ix, iy, altinput=True, **kw)
                np.testing.assert_allclose(c1, c2, rtol=1e-15, atol=2e-15)


@pytest.mark.parametrize('md', range(5))
def test_corr_1(md, rng):
    for p in plist:
        for u in (0.0, 0.4, 1.0):
            n = rng.integers(0, 10, p)
            ix = rng.integers(0, n + 1)
            reset = [2] if md == 4 else None
            c = bart.correlation(n, ix, ix, alpha=0.7, beta=1.3, gamma=u, maxd=md, reset=reset)
            assert c == 1
            c = bart.correlation(n, ix, rng.integers(0, n + 1), alpha=0.7, beta=1.3, gamma=u, maxd=md, reset=reset,
                                 weights=np.zeros(p))
            assert c == 1
    empty = np.array([], int)
    assert bart.correlation(empty, empty, empty) == 1


def test_pnt_and_intercept():
    n, ix, iy = np.array([9, 11]), np.array([1, 2]), np.array([4, 3])
    alpha, beta = 0.9, 1.6
    c1 = bart.correlation(n, ix, iy, alpha=alpha, beta=beta, maxd=2)
    c2 = bart.correlation(n, ix, iy, pnt=[alpha, alpha / 2 ** beta, alpha / 3 ** beta])
    np.testing.assert_allclose(c1, c2, rtol=1e-15)
    c3 = bart.correlation(n, ix, iy, alpha=alpha, beta=beta, maxd=2, intercept=False)
    np.testing.assert_allclose(c1, c3 * alpha + (1 - alpha), rtol=1e-15)


def test_bounds_and_monotonicity(rng):
    p = 5
    n = rng.integers(1, 10, p)
    ix, iy = rng.integers(0, n + 1, (2, 30, p))
    prev_lo = prev_up = None
    for md in range(3):
        lo = bart.correlation(n, ix, iy, gamma=0, maxd=md)
        up = bart.correlation(n, ix, iy, gamma=1, maxd=md)
        assert np.all(lo >= -1e-15) and np.all(up <= 1 + 1e-15) and np.all(lo <= up + 1e-15)
        if md:
            assert np.all(lo >= prev_lo - 1e-15) and np.all(up <= prev_up + 1e-15)
        prev_lo, prev_up = lo, up


def test_hash_equals_exact(rng):
    """ the reference detects equal points by fasthash64 (_bart.py:675-678); equality test is equivalent """
    p = 4
    n = rng.integers(1, 6, p)
    ix = rng.integers(0, n + 1, (40, p)).astype(np.int64)
    iy = ix.copy()
    iy[::3] = rng.integers(0, n + 1, (len(iy[::3]), p))
    kw = dict(maxd=4, reset=2)
    c1 = bart.correlation(n, ix, iy, use_hash=True, **kw)
    c2 = bart.correlation(n, ix, iy, use_hash=False, **kw)
    assert np.array_equal(c1, c2)


def test_splits_and_indices(rng):
    x = np.repeat(np.arange(10 * 2.).reshape(-1, 2), 2, axis=0)
    length, splits = bart.splits_from_coord(x)
    assert np.all(length == 9)  # reference test_duplicates
    X = rng.standard_normal((50, 3))
    length, splits = bart.splits_from_coord(X)
    assert np.all(length == 49) and splits.shape == (49, 3)
    idx = bart.indices_from_coord(X, (length, splits))
    for j in range(3):
        assert np.array_equal(np.sort(idx[:, j]), np.arange(50))  # every point in its own bin
    # symmetric positive semidefinite Gram
    K = bart.gram(length, idx, idx, maxd=10, reset=[2, 4, 6, 8])
    np.testing.assert_allclose(K, K.T, rtol=0, atol=1e-15)
    assert np.linalg.eigvalsh(K).min() > -1e-10
    assert np.all(np.diag(K) == 1)


def test_fold_brackets():
    # maxd=10, reset=[2,4,6,8] folds into one bracket of 5 rows of width 3, deepest first (SURVEY A.5)
    pnt = bart.make_pnt(0.95, 2, 10)
    stages = bart.fold_brackets(pnt, [2, 4, 6, 8])
    assert len(stages) == 1
    probs, repeat = stages[0]
    assert repeat == 5
    rows = probs.reshape(5, 3)
    np.testing.assert_array_equal(rows[:, 0], [1, 1, 1, 1, pnt[0]])
    np.testing.assert_array_equal(rows[:, 1:].ravel(), pnt[[9, 10, 7, 8, 5, 6, 3, 4, 1, 2]])


def test_c_restatement(rng):
    so = pathlib.Path(bart.__file__).resolve().parent / 'liboracle_c.so'
    if not so.exists():
        pytest.skip('oracle/liboracle_c.so not built')
    lib = ctypes.CDLL(str(so))
    f = lib.oracle_bart_pair_w3
    f.restype = ctypes.c_double
    i64p = ctypes.POINTER(ctypes.c_int64)
    dp = ctypes.POINTER(ctypes.c_double)
    f.argtypes = [ctypes.c_int, i64p, i64p, i64p, dp, dp, ctypes.c_int, ctypes.c_double]
    p = 6
    n = rng.integers(0, 50, p).astype(np.int64)
    w = np.array([1., 2., 0., 1., 0.5, 3.])
    pnt = bart.make_pnt(0.95, 2, 10)
    (probs, repeat), = bart.fold_brackets(pnt, [2, 4, 6, 8])
    rows = np.ascontiguousarray(probs.reshape(repeat, 3))
    for _ in range(200):
        ix = rng.integers(0, n + 1).astype(np.int64)
        iy = rng.integers(0, n + 1).astype(np.int64) if rng.random() < 0.9 else ix.copy()
        c_np = bart.correlation(n, ix, iy, maxd=10, reset=[2, 4, 6, 8], weights=w, gamma=0.7)
        c_c = f(p, n.ctypes.data_as(i64p), ix.ctypes.data_as(i64p), iy.ctypes.data_as(i64p), w.ctypes.data_as(dp),
                rows.ctypes.data_as(dp), repeat, 0.7)
        assert abs(c_np - c_c) <= 1e-14 * abs(c_np)


def _cs(f, x, h=1e-200):
    """ complex-step derivative Im f(x + ih) / h """
    return np.imag(f(x + 1j * h)) / h


@pytest.mark.parametrize('md,reset', [(1, None), (2, None), (3, [1]), (4, [2])])
def test_complex_step_closed_forms_vs_old_recursion(md, reset, rng):
    """ d/dalpha and d/dbeta by complex step through the closed forms (altinput) == the same through the independent
    older implementation: the complex-step oracle of gram_derivs does not inherit an error of one formulation """
    for _ in range(4):
        p = int(rng.integers(1, 7))
        n = rng.integers(0, 25, p)
        ix, iy = rng.integers(0, n + 1, (2, 40, p))
        iy[:5] = ix[:5]                     # coinciding points
        w = rng.uniform(0.2, 3, p)
        w[rng.random(p) < 0.25] = 0.0
        nm, n0, npl = np.minimum(ix, iy), np.abs(ix - iy), n - np.maximum(ix, iy)
        alpha, beta, gamma = rng.uniform(0.1, 1), rng.uniform(0, 4), rng.choice([0.0, 1.0, rng.uniform()])
        kw = dict(gamma=gamma, maxd=md, reset=reset, weights=w)

        def new(a, b):
            return bart.correlation(n, ix, iy, alpha=a, beta=b, **kw)

        def old(a, b):
            return bart.correlation(nm, n0, npl, alpha=a, beta=b, altinput=False, **kw)
        for d1, d2 in [(_cs(lambda a: new(a, beta), alpha), _cs(lambda a: old(a, beta), alpha)),
                       (_cs(lambda b: new(alpha, b), beta), _cs(lambda b: old(alpha, b), beta))]:
            assert np.max(np.abs(d1 - d2)) <= 1e-14 * np.max(np.abs(d2)), (np.max(np.abs(d1 - d2)), np.max(np.abs(d2)))
            assert np.all(d1[:5] == 0)


def test_gram_derivs_vs_central_differences(rng):
    """ sanity of gram_derivs' complex step against central differences of the real oracle """
    n = rng.integers(0, 30, 6)
    ix, iy = rng.integers(0, n + 1, (2, 30, 6))
    kw = dict(maxd=10, reset=[2, 4, 6, 8], gamma=0.6)
    alpha, beta, h = 0.9, 1.7, 1e-5
    K, dKa, dKb = bart.gram_derivs(n, ix, iy, alpha=alpha, beta=beta, **kw)
    assert K.dtype == dKa.dtype == dKb.dtype == float
    assert np.array_equal(K, bart.gram(n, ix, iy, alpha=alpha, beta=beta, **kw))
    fa = (bart.gram(n, ix, iy, alpha=alpha + h, beta=beta, **kw) - bart.gram(n, ix, iy, alpha=alpha - h, beta=beta, **kw))
    fb = (bart.gram(n, ix, iy, alpha=alpha, beta=beta + h, **kw) - bart.gram(n, ix, iy, alpha=alpha, beta=beta - h, **kw))
    np.testing.assert_allclose(dKa, fa / (2 * h), rtol=1e-7, atol=1e-9)
    np.testing.assert_allclose(dKb, fb / (2 * h), rtol=1e-7, atol=1e-9)
