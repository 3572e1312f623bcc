"""CPU accuracy test of the product's per-pair BART arithmetic (lsqfitgp_b200/csrc/bart_core.cuh, compiled for the host
by oracle/Makefile into oracle/libbart_core_host.so) against the oracle restatement of the reference
(oracle/bart.py <- src/lsqfitgp/_kernels/_bart.py:301-455,628-757): value (including the staged-reciprocal divisions and
the index-selected digamma lookups), chained stages for reset patterns that do not fold into one bracket sequence, the
alpha / beta duals of the `repeat` scan against the oracle's complex-step derivatives (exact to rounding), and the
derivative rows `drows` of _BartSpec.stages() against the complex step of the bracket folding."""
import ctypes
import pathlib

import numpy as np
import pytest

from lsqfitgp_b200._kernels import _BartSpec
from oracle import bart as obart

LIB = pathlib.Path(__file__).resolve().parents[1] / 'oracle' / 'libbart_core_host.so'


def _lib():
    if not LIB.exists():
        pytest.skip('oracle/libbart_core_host.so not built (make -C oracle)')
    lib = ctypes.CDLL(str(LIB))
    ip, dp = ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_double)
    lib.lgp_host_bart_pairs.argtypes = [ctypes.c_int, ip, dp, ctypes.c_int, ip, ip, dp, dp, ctypes.c_double, ip, ip,
                                        ctypes.c_long, dp]
    lib.lgp_host_bart_pairs.restype = ctypes.c_int
    return lib


def host_pairs(nsplits, w, spec, ix, iy):
    lib = _lib()
    widths, nrows, rows, drows, gamma = spec.stages()
    nsplits = np.ascontiguousarray(nsplits, dtype=np.int32)
    w = np.ascontiguousarray(w, dtype=np.float64)
    ix = np.ascontiguousarray(ix, dtype=np.int32)
    iy = np.ascontiguousarray(iy, dtype=np.int32)
    rows = np.ascontiguousarray(rows, dtype=np.float64)
    out = np.empty((len(ix), 3))
    ip, dp = ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_double)
    dr = np.ascontiguousarray(drows, dtype=np.float64) if drows is not None else None
    lib.lgp_host_bart_pairs(len(nsplits), nsplits.ctypes.data_as(ip), w.ctypes.data_as(dp), len(widths),
                            np.ascontiguousarray(widths, dtype=np.int32).ctypes.data_as(ip),
                            np.ascontiguousarray(nrows, dtype=np.int32).ctypes.data_as(ip), rows.ctypes.data_as(dp),
                            dr.ctypes.data_as(dp) if dr is not None else None, float(gamma), ix.ctypes.data_as(ip),
                            iy.ctypes.data_as(ip), len(ix), out.ctypes.data_as(dp))
    return out


def _problem(rng, p, npairs, nmax):
    nsplits = rng.integers(0, nmax + 1, p)
    ix = np.stack([rng.integers(0, n + 1, npairs) for n in nsplits], axis=1)
    iy = np.stack([rng.integers(0, n + 1, npairs) for n in nsplits], axis=1)
    same = rng.random(npairs) < 0.15       # coinciding points and partially coinciding coordinates
    iy[same] = ix[same]
    part = rng.random((npairs, p)) < 0.3
    iy[part] = ix[part]
    return nsplits, ix, iy


CASES = [  # (maxd, reset, intercept, weights?)
    (10, [2, 4, 6, 8], True, False),   # bayestree.bart: one stage, width 3, repeat 5
    (2, None, True, False),
    (1, None, True, True),
    (0, None, True, False),
    (3, [1], True, False),             # does not fold: width-3 stage feeding a width-2 stage
    (6, [1, 2, 4], True, True),
    (7, [2, 3, 5], False, False),
    (5, [1, 2, 3, 4], True, False),
    (4, [2], False, True),
]


@pytest.mark.parametrize('maxd,reset,intercept,weighted', CASES)
def test_value_matches_oracle(maxd, reset, intercept, weighted):
    rng = np.random.default_rng(hash((maxd, intercept, weighted)) % 2 ** 32)
    p = 6
    nsplits, ix, iy = _problem(rng, p, 400, 40)
    w = rng.uniform(0.2, 3, p) if weighted else np.ones(p)
    if weighted:
        w[2] = 0.0          # a masked covariate
    alpha, beta, gamma = 0.93, 1.6, 0.7
    spec = _BartSpec(1.0, (nsplits, None), True, alpha, beta, maxd, gamma, None, intercept, w, reset)
    got = host_pairs(nsplits, w, spec, ix, iy)[:, 0]
    want = obart.correlation(nsplits, ix, iy, alpha=alpha, beta=beta, gamma=gamma, maxd=maxd, intercept=intercept,
                             weights=w, reset=reset)
    np.testing.assert_allclose(got, want, rtol=2e-14, atol=0)
    assert np.all(got[np.all(ix == iy, axis=1)] == 1.0)


def test_large_split_counts_value():
    """ continuous covariates: thousands of splits per dimension, as in BASELINE configs[3] """
    rng = np.random.default_rng(44)
    p = 10
    nsplits = np.r_[np.full(8, 4999), 1, 1]
    ix = np.stack([rng.integers(0, n + 1, 300) for n in nsplits], axis=1)
    iy = np.stack([rng.integers(0, n + 1, 300) for n in nsplits], axis=1)
    w = np.ones(p)
    spec = _BartSpec(1.0, (nsplits, None), True, 0.95, 2, 10, 1, None, True, None, [2, 4, 6, 8])
    got = host_pairs(nsplits, w, spec, ix, iy)[:, 0]
    want = obart.correlation(nsplits, ix, iy, alpha=0.95, beta=2, gamma=1, maxd=10, reset=[2, 4, 6, 8])
    np.testing.assert_allclose(got, want, rtol=2e-14, atol=0)


@pytest.mark.parametrize('maxd,reset,intercept,weighted', CASES)
def test_alpha_beta_duals_match_complex_step(maxd, reset, intercept, weighted):
    """ value and alpha / beta duals against the oracle's complex-step derivatives (exact to rounding), over covariate
    counts, split counts from 3 to 4999 and (alpha, beta, gamma) including gamma = 0, alpha = 1 and beta = 0 """
    for p in (1, 5, 9, 17):
        for nmax in (3, 40, 4999):
            rng = np.random.default_rng([maxd, p, nmax])
            nsplits, ix, iy = _problem(rng, p, 200, nmax)
            w = rng.uniform(0.2, 3, p) if weighted else np.ones(p)
            if weighted and p > 2:
                w[2] = 0.0      # a masked covariate
            for alpha, beta, gamma in ((0.9, 1.8, 0.6), (1.0, 0.0, 1.0), (0.3, 4.0, 0.0)):
                spec = _BartSpec(1.0, (nsplits, None), True, alpha, beta, maxd, gamma, None, intercept, w, reset)
                got = host_pairs(nsplits, w, spec, ix, iy)
                want = obart.correlation_derivs(nsplits, ix, iy, alpha=alpha, beta=beta, gamma=gamma, maxd=maxd,
                                                intercept=intercept, weights=w, reset=reset)
                what = (p, nmax, alpha, beta, gamma)
                assert np.max(np.abs(got[:, 0] - want[0])) <= 1e-14, what
                for k in (1, 2):
                    ref = want[k]
                    assert np.max(np.abs(got[:, k] - ref)) <= 2e-14 * np.max(np.abs(ref)), (what, k)
                eq = np.all(np.where(w != 0, ix == iy, True), axis=1)
                assert np.all(got[eq, 0] == 1) and np.all(got[eq, 1] == 0) and np.all(got[eq, 2] == 0), what


@pytest.mark.parametrize('maxd,reset,intercept,weighted', CASES)
def test_stage_drows_match_complex_step(maxd, reset, intercept, weighted):
    """ _BartSpec.stages(): rows == the oracle's bracket folding, and drows == the complex step of make_pnt followed by
    the folding; the entries the folding fixes to 1 (and pnt_0 without intercept) have derivative exactly 0 """
    alpha, beta, h = 0.87, 1.9, 1e-200
    spec = _BartSpec(1.0, (np.ones(3), None), True, alpha, beta, maxd, 0.5, None, intercept, None, reset)
    widths, nrows, rows, drows, gamma = spec.stages()

    def folded(a, b):
        pnt = obart.make_pnt(a, b, maxd)
        if not intercept:
            pnt[0] = 1
        out = []
        for probs, repeat in obart.fold_brackets(pnt, reset):
            r = probs.reshape(repeat or 1, -1)
            out.append(np.concatenate([r, np.ones((len(r), 3 - r.shape[1]))], axis=1))
        return np.concatenate(out)
    assert np.array_equal(rows, folded(alpha, beta))
    for k, ref in enumerate([folded(alpha + 1j * h, beta).imag / h, folded(alpha, beta + 1j * h).imag / h]):
        np.testing.assert_allclose(drows[k], ref, rtol=1e-15, atol=0, err_msg=str(k))
        assert np.all(drows[k][ref == 0] == 0)
    assert np.all(drows[:, rows == 1] == 0)
