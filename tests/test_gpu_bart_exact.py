"""The BART Gram kernels (lgp_gram_bart_stages, lgp_gram_bart_vjp, lgp_gram_bart) and their alpha / beta derivatives
against the exact float64 oracle: oracle/bart.py::gram_derivs takes dK/dalpha and dK/dbeta by complex step, which is
exact to rounding and shares nothing with the kernel's dual numbers or the host-side `drows`.

Covers every <NEED2, NEED3> instantiation, tile edges (64 x 64 tiles), more than one 8-covariate chunk (both passes
restage), zero-weight compaction that moves covariates between chunks, 0 and 4999 splits, indices at 0 and n_k, the
symmetric mode, the scalar store path, NULL outputs, strided index arrays, p = 0, the single-bracket entry point, the
digamma table and the rejected configurations.

Bars: K within 1e-13 elementwise relative where gamma > 0 and 1e-14 max|K| normwise; dK within 1e-13 max|ref| normwise
and 1e-12 |ref| + 1e-13 max|ref| elementwise; a contraction sum_ij G_ij dK_ij within 1e-12 sum_ij |G_ij dK_ij| (the
atomicAdd order varies the last bits)."""
import functools

import numpy as np
import pytest
import torch
from scipy import special

from lsqfitgp_b200 import _lib, _ops
from lsqfitgp_b200._kernels import _BartSpec
from oracle import bart as obart

pytestmark = pytest.mark.gpu
DEV = 'cuda'
AMP, ALPHA, BETA = 1.3, 0.9, 1.7

# bracket layouts: all four <NEED2, NEED3> kernel instantiations, a folded `repeat` scan, no intercept, gamma 0 and 1
STAGES = {
    'w1': dict(maxd=0, gamma=0.4),                          # width 1
    'w2': dict(maxd=1, gamma=0.4),                          # width 2
    'w3': dict(maxd=2, gamma=0.4),                          # width 3
    'w3w2': dict(maxd=3, reset=[1], gamma=0.4),             # width 3 feeding width 2
    'rep5': dict(maxd=10, reset=[2, 4, 6, 8]),              # one width-3 stage of 5 rows, gamma 1
    'noint': dict(maxd=6, reset=[1, 2, 4], intercept=False, gamma=0.7),
    'g0': dict(maxd=3, reset=[1], gamma=0.0),
}
SHAPES = [(1, 1), (1, 65), (63, 64), (64, 64), (65, 129), (129, 65), (200, 333)]
SYM_N = [1, 64, 65, 129, 200]


def problem(p, nzero, n, m, seed):
    """ p active covariates among p + nzero columns (the zero-weight ones spread out, so the kernel's compacted
    covariate k is not column k and covariates change chunk); column 0 has 0 splits, column 1 4999; indices 0 and n_k
    in every column on both sides; coinciding points, points that differ only in a zero-weight column, points that
    differ in one active column only.  Returns (nsplits, w, X (n, cols), Y (m, cols), same), same: pairs whose
    correlation is exactly 1 (K = amp, dK = 0) """
    rng = np.random.default_rng(seed)
    cols = p + nzero
    zero = np.linspace(0, cols, nzero + 2)[1:-1].astype(int)
    w = rng.uniform(0.3, 2.5, cols)
    w[zero] = 0.0
    active = np.flatnonzero(w)
    nsplits = rng.integers(1, 60, cols)
    if len(active) > 2:
        nsplits[active[0]] = 0
    nsplits[active[min(1, len(active) - 1)]] = 4999
    X = rng.integers(0, nsplits + 1, (n, cols))
    Y = rng.integers(0, nsplits + 1, (m, cols))
    if n > 1:
        X[0], X[-1] = 0, nsplits
    if m > 1:
        Y[0], Y[-1] = nsplits, 0
    if n >= 8 and m >= 8:
        Y[2] = X[2]                                  # coinciding
        Y[3] = X[3]
        if nzero:
            Y[3, zero[0]] = (X[3, zero[0]] + 1) % (nsplits[zero[0]] + 1)     # differs in a masked column only
        Y[4] = X[4]
        k = active[-1]
        Y[4, k] = (X[4, k] + 1) % (nsplits[k] + 1)   # differs in one active column only
        X[6] = X[5]                                  # a duplicated point within x
    same = np.all(np.where(w != 0, X[:, None, :] == Y[None, :, :], True), axis=-1)
    return nsplits, w, X, Y, same


def dev_idx(A, pad=0):
    """ (cols, rows) int32 device tensor; pad > 0: a view with leading dimension rows + pad """
    t = torch.zeros((A.shape[1], A.shape[0] + pad), dtype=torch.int32, device=DEV)
    t[:, :A.shape[0]] = torch.tensor(A.T.astype(np.int32), device=DEV)
    return t[:, :A.shape[0]]


def spec_of(w, nsplits, kw, alpha=ALPHA, beta=BETA):
    s = _BartSpec(AMP, (nsplits, None), True, alpha, beta, kw['maxd'], kw.get('gamma', 1.0), None,
                  kw.get('intercept', True), w, kw.get('reset'))
    return s.stages()


@functools.lru_cache(maxsize=None)
def ref_case(p, nzero, n, m, seed, stage, sym=False):
    """ the problem and AMP * (K, dK/dalpha, dK/dbeta) from the oracle, cached per case """
    nsplits, w, X, Y, same = problem(p, nzero, n, m, seed)
    if sym:
        Y, same = X, np.all(np.where(w != 0, X[:, None, :] == X[None, :, :], True), axis=-1)
    kw = STAGES[stage]
    K, dKa, dKb = obart.gram_derivs(nsplits, X, Y, alpha=ALPHA, beta=BETA, weights=w, **kw)
    return nsplits, w, X, Y, same, AMP * K, AMP * dKa, AMP * dKb


def check_K(got, ref, gamma, what):
    scale = float(np.max(np.abs(ref)))
    assert np.all(np.isfinite(got)), what
    assert float(np.max(np.abs(got - ref))) <= 1e-14 * scale, (what, float(np.max(np.abs(got - ref))), scale)
    if gamma > 0:   # (without intercept, points separated by every split have correlation exactly 0)
        nz = ref != 0
        assert float(np.max(np.abs(got - ref)[nz] / np.abs(ref[nz]))) <= 1e-13, what


def check_dK(got, ref, what):
    scale = float(np.max(np.abs(ref)))
    assert np.all(np.isfinite(got)), what
    assert float(np.max(np.abs(got - ref))) <= 1e-13 * scale, (what, float(np.max(np.abs(got - ref))), scale)
    np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-13 * scale, err_msg=what)


def check_all(out, ref, same, gamma, what):
    K, dKa, dKb = (t.cpu().numpy() for t in out)
    check_K(K, ref[0], gamma, what + ' K')
    check_dK(dKa, ref[1], what + ' dKa')
    check_dK(dKb, ref[2], what + ' dKb')
    assert np.all(K[same] == AMP) and np.all(dKa[same] == 0) and np.all(dKb[same] == 0), what


def run(nsplits, w, st, ix, iy, **kw):
    widths, nrows, rows, drows, gamma = st
    return _ops.gram_bart_stages(nsplits, w, widths, nrows, rows, drows, gamma, AMP, ix, iy, **kw)


def vjp(nsplits, w, st, ix, iy, G, **kw):
    widths, nrows, rows, drows, gamma = st
    return _ops.gram_bart_vjp(nsplits, w, widths, nrows, rows, drows, gamma, AMP, ix, iy, G, **kw).cpu().numpy()


# ---- forward matrices against the oracle

@pytest.mark.parametrize('shape', SHAPES, ids=[f'{n}x{m}' for n, m in SHAPES])
@pytest.mark.parametrize('stage', list(STAGES))
def test_derivs_vs_oracle(stage, shape):
    """ 9 active covariates of 11 columns (two chunks; zero weights shift the compacted covariates) """
    n, m = shape
    nsplits, w, X, Y, same, *ref = ref_case(9, 2, n, m, 11, stage)
    st = spec_of(w, nsplits, STAGES[stage])
    ix, iy = dev_idx(X), dev_idx(Y)
    out = run(nsplits, w, st, ix, iy, deriv=True)
    check_all(out, ref, same, st[4], f'{stage} {shape}')
    # the value-only kernel computes the same K bit for bit
    assert torch.equal(run(nsplits, w, st, ix, iy), out[0])


@pytest.mark.parametrize('p', [1, 7, 8, 9, 16, 17, 64])
@pytest.mark.parametrize('stage', ['w2', 'w3w2', 'rep5'])
def test_active_covariates_vs_oracle(stage, p):
    """ 1 to 64 active covariates: one chunk, a full chunk, a chunk plus one, two full chunks, the limit B_MAX_P; 10
    columns with two zero weights for p = 8 """
    nzero = 2 if p in (8, 64) else 1
    nsplits, w, X, Y, same, *ref = ref_case(p, nzero, 65, 129, 100 + p, stage)
    st = spec_of(w, nsplits, STAGES[stage])
    out = run(nsplits, w, st, dev_idx(X), dev_idx(Y), deriv=True)
    check_all(out, ref, same, st[4], f'{stage} p={p}')


@pytest.mark.parametrize('n', SYM_N)
@pytest.mark.parametrize('stage', ['w1', 'w2', 'w3', 'w3w2', 'rep5'])
def test_symmetric_derivs(stage, n):
    """ the symmetric mode (lower tiles evaluated, mirrored through shared memory) is bit-identical to the general mode
    for K, dKa and dKb, and matches the oracle """
    nsplits, w, X, _, same, *ref = ref_case(17, 2, n, n, 7, stage, sym=True)
    st = spec_of(w, nsplits, STAGES[stage])
    ix = dev_idx(X)
    outs = run(nsplits, w, st, ix, ix, deriv=True, symmetric=True)
    outg = run(nsplits, w, st, ix, ix.clone(), deriv=True)
    for a, b in zip(outs, outg):
        assert torch.equal(a, b)
    check_all(outs, ref, same, st[4], f'sym {stage} n={n}')


# ---- the C ABI directly: NULL outputs, scalar stores, strided index arrays

def abi_stages(nsplits, w, st, ix, n, iy, m, K, ldk, dKa, dKb, ldd, flags=0):
    """ lgp_gram_bart_stages with raw pointers (ints) and leading dimensions; returns the status """
    widths, nrows, rows, drows, gamma = st
    args, keep, nsplits = _ops._bart_cargs(nsplits, w, widths, nrows, rows, drows)
    psi = _ops.digamma_table(int(nsplits.max()) + 2, DEV)
    return _lib.load().lgp_gram_bart_stages(_lib.stream_ptr(), *args, float(gamma), AMP, _lib.ptr(psi), _lib.ptr(ix),
                                            ix.stride(0), n, _lib.ptr(iy), iy.stride(0), m, K, ldk, dKa, dKb, ldd, flags)


@pytest.mark.parametrize('stage', ['w2', 'w3w2', 'rep5'])
def test_abi_output_variants(stage):
    n, m = 65, 129
    nsplits, w, X, Y, same, *ref = ref_case(9, 2, n, m, 11, stage)
    st = spec_of(w, nsplits, STAGES[stage])
    ix, iy = dev_idx(X), dev_idx(Y)
    Kr, dKar, dKbr = run(nsplits, w, st, ix, iy, deriv=True)
    check_all((Kr, dKar, dKbr), ref, same, st[4], stage)
    sentinel = 7.25

    def buf(ld, off):
        """ (n, m) view at `off` doubles into a (n, ld) buffer full of the sentinel """
        b = torch.full((n * ld + 2,), sentinel, dtype=torch.float64, device=DEV)
        return b, b[off:off + n * ld].view(n, ld)[:, :m]

    def intact(b, view):
        """ everything outside the window `view` of buffer `b` still holds the sentinel """
        mask = torch.ones_like(b, dtype=torch.bool)
        off = view.data_ptr() - b.data_ptr()
        ld = view.stride(0)
        rows, cols = view.shape
        idx = off // 8 + (torch.arange(rows, device=DEV)[:, None] * ld + torch.arange(cols, device=DEV)[None, :])
        mask[idx.reshape(-1)] = False
        return bool(torch.all(b[mask] == sentinel))
    # derivatives without K, and one derivative at a time (even ld, aligned: vector stores)
    for which in ('both', 'a', 'b'):
        ba, va = buf(m + 1, 0)
        bb, vb = buf(m + 1, 0)
        pa = va.data_ptr() if which in ('both', 'a') else None
        pb = vb.data_ptr() if which in ('both', 'b') else None
        assert abi_stages(nsplits, w, st, ix, n, iy, m, None, 0, pa, pb, m + 1) == 0
        if pa:
            assert torch.equal(va, dKar) and intact(ba, va), which
        else:
            assert bool(torch.all(ba == sentinel)), which
        if pb:
            assert torch.equal(vb, dKbr) and intact(bb, vb), which
        else:
            assert bool(torch.all(bb == sentinel)), which
    # scalar stores: an odd leading dimension, or an 8-byte offset from 16-byte alignment (K and dK separately)
    for ldk, offk, ldd, offd in ((m, 0, m + 1, 0), (m + 1, 1, m + 1, 0), (m + 1, 0, m + 2, 0), (m + 1, 0, m + 1, 1)):
        bk, vk = buf(ldk, offk)
        ba, va = buf(ldd, offd)
        bb, vb = buf(ldd, offd)
        assert abi_stages(nsplits, w, st, ix, n, iy, m, vk.data_ptr(), ldk, va.data_ptr(), vb.data_ptr(), ldd) == 0
        for v, r, b in ((vk, Kr, bk), (va, dKar, ba), (vb, dKbr, bb)):
            assert torch.equal(v, r) and intact(b, v), (ldk, offk, ldd, offd)
    # symmetric mode with the scalar stores of the direct tile and the mirrored one
    nsplits, w, Xs, _, _, *refs = ref_case(9, 2, n, n, 11, stage, sym=True)
    ixs = dev_idx(Xs)
    Ks = run(nsplits, w, st, ixs, ixs, deriv=True, symmetric=True)
    bk, vk = buf(n, 1)
    vk = vk[:, :n]
    ba, va = buf(n + 2, 0)
    va = va[:, :n]
    assert abi_stages(nsplits, w, st, ixs, n, ixs, n, vk.data_ptr(), n, None, va.data_ptr(), n + 2,
                      _lib.BART_SYMMETRIC) == 0
    assert torch.equal(vk, Ks[0]) and torch.equal(va, Ks[2])
    assert intact(bk, vk) and intact(ba, va)         # the mirrored stores stay inside the (n, n) window
    # index arrays with a leading dimension larger than the number of points (padding never read)
    ixp, iyp = dev_idx(X, pad=5), dev_idx(Y, pad=3)
    ixp.as_strided((ixp.shape[0], 5), (ixp.stride(0), 1), ixp.shape[1]).fill_(-7)
    K2 = _ops.aligned_empty(n, m, DEV)
    dKa2, dKb2 = _ops.aligned_empty(n, m, DEV), _ops.aligned_empty(n, m, DEV)
    assert abi_stages(nsplits, w, st, ixp, n, iyp, m, K2.data_ptr(), K2.stride(0), dKa2.data_ptr(), dKb2.data_ptr(),
                      dKa2.stride(0)) == 0
    assert torch.equal(K2, Kr) and torch.equal(dKa2, dKar) and torch.equal(dKb2, dKbr)


# ---- reverse mode

@pytest.mark.parametrize('stage', ['w1', 'w2', 'w3', 'w3w2', 'rep5', 'noint'])
def test_vjp_vs_oracle(stage):
    """ lgp_gram_bart_vjp against sum G * {K / amp, dKa, dKb} formed in float64 from the oracle's matrices: a dense G,
    and the symlower form (lower triangle of a symmetric G minus b b^T, weights 2 off the diagonal, NaN above) """
    n, m = 65, 129
    nsplits, w, X, Y, _, K, dKa, dKb = ref_case(17, 2, n, m, 13, stage)
    st = spec_of(w, nsplits, STAGES[stage])
    gen = np.random.default_rng(5)
    G = gen.standard_normal((n, m))
    got = vjp(nsplits, w, st, dev_idx(X), dev_idx(Y), _ops.as_aligned(torch.tensor(G, device=DEV)))
    for k, dK in enumerate((K / AMP, dKa, dKb)):
        ref = float(np.sum(G * dK))
        assert abs(got[k] - ref) <= 1e-12 * float(np.sum(np.abs(G * dK))), (stage, k, got[k], ref)
    # symmetric
    nsplits, w, Xs, _, _, Ks, dKas, dKbs = ref_case(17, 2, 129, 129, 13, stage, sym=True)
    A = gen.standard_normal((129, 129))
    Gs = A + A.T
    b = gen.standard_normal(129)
    low = np.tril(Gs) + np.triu(np.full_like(Gs, np.nan), 1)      # the upper triangle must not be read
    ixs = dev_idx(Xs)
    got = vjp(nsplits, w, st, ixs, ixs, _ops.as_aligned(torch.tensor(low, device=DEV)),
              b=torch.tensor(b, device=DEV), symlower=True)
    Gf = Gs - np.outer(b, b)
    for k, dK in enumerate((Ks / AMP, dKas, dKbs)):
        ref = float(np.sum(Gf * dK))
        assert abs(got[k] - ref) <= 1e-12 * float(np.sum(np.abs(Gf * dK))), (stage, 'sym', k, got[k], ref)


# ---- no active covariate, the single-bracket entry point, the digamma table

@pytest.mark.parametrize('cols', [0, 3])
def test_no_active_covariate(cols):
    """ p = 0, or every weight 0: correlation identically 1, so K = amp, dK = 0, and the VJP is sum w (G - b b^T) """
    n, m = 70, 131
    rng = np.random.default_rng(9)
    nsplits, w = np.full(cols, 5), np.zeros(cols)
    X, Y = rng.integers(0, 6, (n, cols)), rng.integers(0, 6, (m, cols))
    st = spec_of(w, nsplits, STAGES['rep5'])
    ix, iy = dev_idx(X), dev_idx(Y)
    K, dKa, dKb = run(nsplits, w, st, ix, iy, deriv=True)
    assert bool(torch.all(K == AMP)) and bool(torch.all(dKa == 0)) and bool(torch.all(dKb == 0))
    assert bool(torch.all(run(nsplits, w, st, ix, iy) == AMP))
    G = rng.standard_normal((n, m))
    got = vjp(nsplits, w, st, ix, iy, _ops.as_aligned(torch.tensor(G, device=DEV)))
    assert abs(got[0] - G.sum()) <= 1e-12 * np.abs(G).sum() and got[1] == 0 and got[2] == 0
    A = rng.standard_normal((n, n))
    Gs, b = A + A.T, rng.standard_normal(n)
    low = np.tril(Gs) + np.triu(np.full_like(Gs, np.nan), 1)
    got = vjp(nsplits, w, st, ix, ix, _ops.as_aligned(torch.tensor(low, device=DEV)), b=torch.tensor(b, device=DEV),
              symlower=True)
    Gf = Gs - np.outer(b, b)
    assert abs(got[0] - Gf.sum()) <= 1e-12 * np.abs(Gf).sum() and got[1] == 0 and got[2] == 0


@pytest.mark.parametrize('stage', ['w1', 'w2', 'w3', 'rep5'])
def test_single_bracket_entry_vs_oracle(stage):
    """ lgp_gram_bart (one stage, rows of `width` probabilities) """
    nsplits, w, X, Y, same, K, _, _ = ref_case(9, 2, 65, 129, 17, stage)
    st = spec_of(w, nsplits, STAGES[stage])
    widths, nrows, rows, _, gamma = st
    assert len(widths) == 1
    got = _ops.gram_bart(nsplits, w, rows[:, :widths[0]], gamma, AMP, dev_idx(X), dev_idx(Y)).cpu().numpy()
    check_K(got, K, gamma, stage)
    assert np.all(got[same] == AMP)


def test_digamma_table():
    """ lgp_bart_digamma_table (long-double recurrence) against scipy's digamma within 2 ulp up to k = 2e5 """
    length = 200_001
    psi = np.empty(length)
    _ops.check(_lib.load().lgp_bart_digamma_table(psi.ctypes.data_as(_lib.c_double_p), length), 'digamma table')
    k = np.arange(1, length, dtype=float)
    ref = special.digamma(k)
    assert psi[0] == -np.inf
    assert np.max(np.abs(psi[1:] - ref) / np.spacing(np.abs(ref))) <= 2


# ---- rejections

def test_unsupported_configurations_leave_no_error():
    """ 65 active covariates, 17 rows or 9 stages: LGP_ERR_UNSUPPORTED from both entry points, and the next call on
    the stream succeeds """
    nsplits, w, X, Y, same, *ref = ref_case(64, 2, 65, 129, 100 + 64, 'rep5')
    ix, iy = dev_idx(X), dev_idx(Y)
    G = _ops.as_aligned(torch.ones((65, 129), dtype=torch.float64, device=DEV))
    good = spec_of(w, nsplits, STAGES['rep5'])
    w65 = w.copy()
    w65[np.flatnonzero(w == 0)[0]] = 1.0                     # 65 of the 66 columns active
    r17 = np.ones((17, 3))
    bad = [(w65, good), (w, (np.array([3]), np.array([17]), r17, np.zeros((2, 17, 3)), 1.0)),
           (w, (np.ones(9, np.int32), np.ones(9, np.int32), r17[:9], np.zeros((2, 9, 3)), 1.0))]
    for wb, sb in bad:
        for call in (lambda: run(nsplits, wb, sb, ix, iy, deriv=True), lambda: run(nsplits, wb, sb, ix, iy),
                     lambda: vjp(nsplits, wb, sb, ix, iy, G)):
            with pytest.raises(RuntimeError, match=_lib.ERRORS[-4]):
                call()
            check_all(run(nsplits, w, good, ix, iy, deriv=True), ref, same, 1.0, 'after a rejection')
            torch.cuda.synchronize()
