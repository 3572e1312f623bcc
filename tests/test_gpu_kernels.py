"""GPU parity: low-level C-ABI kernels (GEMM, Cholesky pipeline, Gram) against the oracle / NumPy.
Tolerances: Gram entries 1e-13 relative (north_star), factor/solves 1e-10, logdet/eps 1e-12."""
import numpy as np
import pytest
import scipy.linalg as sl
import torch

from lsqfitgp_b200 import _lib, _ops
from oracle import gp as ogp, decomp as odecomp

pytestmark = pytest.mark.gpu


def dev():
    return torch.device('cuda:0')


def relerr(a, b):
    return float((a - b).abs().max() / b.abs().max())


# (grids below one CTA per SM run the 32x32 latency tiles, larger ones the 64x64 throughput tiles: both are covered)
@pytest.mark.parametrize('M,N,K', [(128, 128, 128), (300, 200, 150), (257, 129, 77), (1, 1, 1), (64, 640, 33),
                                   (1024, 512, 2048), (1100, 900, 130), (1537, 1025, 50)])
@pytest.mark.parametrize('akm', [True, False])
@pytest.mark.parametrize('bkm', [True, False])
def test_dgemm_layouts(M, N, K, akm, bkm):
    g = torch.Generator(device='cpu').manual_seed(M * 7 + N * 3 + K)
    Aop = torch.randn(M, K, generator=g, dtype=torch.float64).to(dev())
    Bop = torch.randn(N, K, generator=g, dtype=torch.float64).to(dev())
    C0 = torch.randn(M, N, generator=g, dtype=torch.float64).to(dev())
    A = _ops.as_aligned(Aop if akm else Aop.T.contiguous())
    B = _ops.as_aligned(Bop if bkm else Bop.T.contiguous())
    C = _ops.as_aligned(C0.clone())
    _ops.dgemm(A, B, C, a_kmajor=akm, b_kmajor=bkm, M=M, N=N, K=K, alpha=-1.0)
    assert relerr(C, C0 - Aop @ Bop.T) < 1e-13
    _ops.dgemm(A, B, C, a_kmajor=akm, b_kmajor=bkm, M=M, N=N, K=K, alpha=2.0, flags=_lib.GEMM_BETA0)
    assert relerr(C, 2 * (Aop @ Bop.T)) < 1e-13


def test_dgemm_flags():
    M, K = 384, 200
    g = torch.Generator(device='cpu').manual_seed(5)
    Aop = torch.randn(M, K, generator=g, dtype=torch.float64).to(dev())
    C0 = torch.randn(M, M, generator=g, dtype=torch.float64).to(dev())
    A = _ops.as_aligned(Aop)
    C = _ops.as_aligned(C0.clone())
    _ops.dgemm(A, A, C, a_kmajor=True, b_kmajor=True, M=M, N=M, K=K, alpha=-1.0, flags=_lib.GEMM_LOWER)
    ref = C0 - Aop @ Aop.T
    assert relerr(torch.tril(C), torch.tril(ref)) < 1e-13
    assert torch.equal(torch.triu(C, 1), torch.triu(C0, 1))  # strictly upper part untouched, bit for bit
    L = torch.tril(torch.randn(M, M, generator=g, dtype=torch.float64)).to(dev())
    X = torch.randn(M, 130, generator=g, dtype=torch.float64).to(dev())
    Y = _ops.aligned_empty(M, 130, dev())
    _ops.dgemm(_ops.as_aligned(L), _ops.as_aligned(X), Y, a_kmajor=True, b_kmajor=False, M=M, N=130, K=M,
               flags=_lib.GEMM_BETA0 | _lib.GEMM_A_LOWER_K)
    assert relerr(Y, L @ X) < 1e-13
    _ops.dgemm(_ops.as_aligned(L), _ops.as_aligned(X), Y, a_kmajor=False, b_kmajor=False, M=M, N=130, K=M,
               flags=_lib.GEMM_BETA0 | _lib.GEMM_A_UPPER_K)
    assert relerr(Y, L.T @ X) < 1e-13


@pytest.mark.parametrize('M', [384, 1500])  # latency tiles / throughput tiles of the lower-triangular enumeration
def test_dgemm_lower_both_tile_configurations(M):
    K = 136
    g = torch.Generator(device='cpu').manual_seed(M)
    Aop = torch.randn(M, K, generator=g, dtype=torch.float64).to(dev())
    C0 = torch.randn(M, M, generator=g, dtype=torch.float64).to(dev())
    C = _ops.as_aligned(C0.clone())
    _ops.dgemm(_ops.as_aligned(Aop), _ops.as_aligned(Aop), C, a_kmajor=True, b_kmajor=True, M=M, N=M, K=K, alpha=-1.0,
               flags=_lib.GEMM_LOWER)
    assert relerr(torch.tril(C), torch.tril(C0 - Aop @ Aop.T)) < 1e-13
    assert torch.equal(torch.triu(C, 1), torch.triu(C0, 1))


@pytest.mark.parametrize('t', [128, 256, 1024])
def test_tile_potrf_leaf_against_torch(t):
    """The 128x128 leaf (Cholesky factor + its inverse in one CTA, csrc/chol_leaf3.cuh) through lgp_tile_potrf: factor,
    inverted diagonal blocks, diagonal, zeros above the diagonal, failure index.  The strict upper triangle of the input
    is scratch and must be ignored."""
    lib = _lib.load()
    K = spd(t, 11 + t).to(dev())
    L = torch.linalg.cholesky(K)
    A = _ops.as_aligned(K + torch.triu(torch.full_like(K, 3.0), 1))
    invd = torch.full((t // 128, 128, 128), 7.0, dtype=torch.float64, device=dev())
    dvec = torch.zeros(t + 5, dtype=torch.float64, device=dev())
    info = torch.full((1,), 2**31 - 1, dtype=torch.int32, device=dev())
    rc = lib.lgp_tile_potrf(_lib.stream_ptr(), _lib.ptr(A), A.stride(0), t, _lib.ptr(invd), _lib.ptr(dvec), _lib.ptr(info), 5)
    torch.cuda.synchronize()
    assert rc == 0 and int(info.item()) == 2**31 - 1
    assert relerr(torch.tril(A), L) < 1e-12
    assert relerr(dvec[5:], torch.diagonal(L)) < 1e-13
    for b in range(t // 128):
        blk = slice(128 * b, 128 * (b + 1))
        assert torch.equal(torch.triu(A[blk, blk], 1), torch.zeros(128, 128, dtype=torch.float64, device=dev()))
        Xb = torch.linalg.inv(L[blk, blk])
        assert relerr(invd[b], Xb) < 1e-11
        assert torch.equal(torch.triu(invd[b], 1), torch.zeros(128, 128, dtype=torch.float64, device=dev()))
    # first failing pivot (global, 1-based): column 70 of the second block if there is one
    j = 70 + (128 if t > 128 else 0)
    Kb = K.clone()
    Kb[j, j] = -1.0
    A = _ops.as_aligned(Kb)
    info.fill_(2**31 - 1)
    lib.lgp_tile_potrf(_lib.stream_ptr(), _lib.ptr(A), A.stride(0), t, _lib.ptr(invd), _lib.ptr(dvec), _lib.ptr(info), 5)
    torch.cuda.synchronize()
    assert int(info.item()) == 5 + j + 1


def test_dgemm_rejects_misaligned():
    A = torch.zeros(9, 9, dtype=torch.float64, device=dev())
    with pytest.raises(RuntimeError, match='misaligned'):
        _ops.dgemm(A, A, A.clone(), a_kmajor=True, b_kmajor=True, M=9, N=9, K=9)


def spd(n, seed):
    g = torch.Generator(device='cpu').manual_seed(seed)
    x = torch.rand(n, 2, generator=g, dtype=torch.float64) * 10
    d2 = ((x[:, None, :] - x[None, :, :]) ** 2).sum(-1)
    return 1.7 * torch.exp(-0.5 * d2 / 1.5 ** 2) + 0.05 * torch.eye(n, dtype=torch.float64)


@pytest.mark.parametrize('n', [1, 2, 10, 127, 128, 129, 300, 640, 1000, 2500])
def test_chol_pipeline_vs_oracle(n):
    Kc = spd(n, n)
    st = _ops.chol_factor(Kc.to(dev()))
    assert int(st.info.item()) == 0
    do = odecomp.Chol(Kc.numpy())
    Lr = do._L
    Lg = _ops.chol_get_factor(st).cpu().numpy()
    assert np.abs(Lg - Lr).max() / np.abs(Lr).max() < 1e-12
    assert np.all(np.triu(Lg, 1) == 0)
    sc = st.scalars().cpu().numpy()
    assert abs(sc[1] * sc[3] - do.eps) / do.eps < 1e-14          # eps: same Gershgorin bound, bit-level
    ld = np.sum(np.log(np.diag(Lr)))
    assert abs(sc[4] - ld) / max(1, abs(ld)) < 1e-12
    g = torch.Generator(device='cpu').manual_seed(n)
    for m in (1, 3, 130):
        B = torch.randn(n, m, generator=g, dtype=torch.float64)
        x1 = _ops.chol_solve(st, B.to(dev()), False).cpu().numpy()
        r1 = sl.solve_triangular(Lr, B.numpy(), lower=True)
        assert np.abs(x1 - r1).max() / np.abs(r1).max() < 1e-10
        x2 = _ops.chol_solve(st, B.to(dev()), True).cpu().numpy()
        r2 = sl.solve_triangular(Lr.T, B.numpy(), lower=False)
        assert np.abs(x2 - r2).max() / np.abs(r2).max() < 1e-10
        y1 = _ops.chol_mult(st, B.to(dev()), False).cpu().numpy()
        assert np.abs(y1 - Lr @ B.numpy()).max() / np.abs(Lr @ B.numpy()).max() < 1e-12
        y2 = _ops.chol_mult(st, B.to(dev()), True).cpu().numpy()
        assert np.abs(y2 - Lr.T @ B.numpy()).max() / np.abs(Lr.T @ B.numpy()).max() < 1e-12
    Ki = _ops.chol_inverse(st).cpu().numpy()
    Kir = np.linalg.inv(Lr @ Lr.T)
    assert np.abs(np.tril(Ki) - np.tril(Kir)).max() / np.abs(Kir).max() < 1e-9


def test_chol_unequal_scales_and_addmat():
    # diagonal spanning many powers of two: s differs per row; Kxx + ycov fused in the equilibration pass
    n = 200
    rng = np.random.default_rng(0)
    A = rng.standard_normal((n, n))
    K = A @ A.T / n + np.eye(n)
    d = 2.0 ** rng.integers(-20, 20, n)
    K = K * d[:, None] * d[None, :]
    ycov = np.diag(rng.uniform(0.1, 1, n)) * d[:, None] * d[None, :]
    st = _ops.chol_factor(torch.tensor(K).to(dev()), addmat=torch.tensor(ycov).to(dev()))
    do = odecomp.Chol(K + ycov)
    Lg = _ops.chol_get_factor(st).cpu().numpy()
    assert np.abs(Lg / do._L.clip(1e-300) - 1)[np.tril_indices(n)].max() < 1e-9 or \
        np.abs(Lg - do._L).max() / np.abs(do._L).max() < 1e-12
    sc = st.scalars().cpu().numpy()
    assert abs(sc[1] * sc[3] - do.eps) / do.eps < 1e-14


@pytest.mark.parametrize('n', [1, 100, 128, 129, 333, 400, 1000, 2500])
def test_vector_solves_match_matrix_solves(n):
    """ m = 1 goes through the single-kernel look-back TRSV sweeps, m > 1 through the GEMM recursion: same results, with
    unequal equilibration scales, for both sweeps, and against the oracle's factor """
    rng = np.random.default_rng(n)
    A = rng.standard_normal((n, n))
    K = A @ A.T / n + np.eye(n)
    d = 2.0 ** rng.integers(-6, 6, n)
    K = K * d[:, None] * d[None, :]
    st = _ops.chol_factor(torch.tensor(K).to(dev()))
    L = odecomp.Chol(K)._L
    B = rng.standard_normal((n, 3))
    Bd = torch.tensor(B).to(dev())
    for trans in (False, True):
        ref = sl.solve_triangular(L, B, lower=True, trans='T' if trans else 'N')
        Xm = _ops.chol_solve(st, Bd, trans).cpu().numpy()[:, :3]
        X1 = _ops.chol_solve(st, Bd[:, :1].contiguous(), trans).cpu().numpy()[:, 0]
        scale = np.abs(ref).max()
        assert np.abs(Xm - ref).max() / scale < 1e-10
        assert np.abs(X1 - ref[:, 0]).max() / scale < 1e-10
    # both sweeps in place on a strided vector (a column of a wider matrix), twice in a row on the same stream
    wide = _ops.aligned_empty(n, 4, dev())
    for rep in range(2):
        wide.copy_(torch.tensor(np.concatenate([B, B[:, :1]], axis=1)).to(dev()))
        col = wide[:, 2:3]  # (16-byte aligned: the C ABI requires it)
        lib = _lib.load()
        for trans in (0, 1):
            _ops.check(lib.lgp_chol_solve(_lib.stream_ptr(), _lib.ptr(st.W), st.W.stride(0), _lib.ptr(st.aux), st.n,
                                          col.data_ptr(), wide.stride(0), 1, trans), 'lgp_chol_solve')
        ref = sl.cho_solve((L, True), B[:, 2])
        got = wide.cpu().numpy()
        assert np.abs(got[:, 2] - ref).max() / np.abs(ref).max() < 1e-9
        assert np.array_equal(got[:, 1], B[:, 1]) and np.array_equal(got[:, 3], B[:, 0])  # neighbours untouched


def test_vector_solves_on_fresh_streams():
    """ first use of a caller stream allocates and clears the flag workspace of the TRSV sweeps IN STREAM ORDER (a
    cudaMemset on the NULL stream raced with the first sweep on a non-blocking stream): several new streams, solved
    right after their creation, from several host threads """
    import threading
    n = 1500
    K = spd(n, 3).to(dev())
    st = _ops.chol_factor(K)
    y = torch.randn(n, 1, dtype=torch.float64, device=dev())
    ref = _ops.chol_solve(st, _ops.chol_solve(st, y, False), True)
    torch.cuda.synchronize()
    outs, errs = {}, []

    def work(k):
        try:
            s = torch.cuda.Stream(dev())
            s.wait_stream(torch.cuda.default_stream(dev()))
            with torch.cuda.stream(s):
                for rep in range(3):
                    outs[k, rep] = _ops.chol_solve(st, _ops.chol_solve(st, y, False), True)
            s.synchronize()
        except Exception as e:  # noqa: BLE001
            errs.append(e)
    threads = [threading.Thread(target=work, args=(k,)) for k in range(6)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errs
    for v in outs.values():
        assert torch.equal(v, ref)  # the sweeps are deterministic


@pytest.mark.parametrize('n', [1, 64, 130, 333, 1000, 2111])
@pytest.mark.parametrize('kind', ['expquad', 'matern12', 'matern52', 'matern72', 'cauchy', 'matern52_nowhite', 'const'])
def test_gram_fused_with_equilibration_matches_two_pass(n, kind):
    """ lgp_gram_iso_prepare + lgp_chol_factor[_inverse]_prepared (Gram build writing the equilibrated lower triangle and
    the Gershgorin partial sums straight into the factor's storage) against lgp_gram_iso + lgp_chol_factor[_inverse]: same
    scales (bit for bit), same eps up to the order of the row sums, same factor / logdet / inverse """
    rng = np.random.default_rng(n)
    x = torch.tensor(rng.uniform(0, 6, (2, n))).to(dev())
    white = dict(kind=_lib.K_WHITE, term=1, dimmask=3, amp=0.3)
    main = {'expquad': dict(kind=_lib.K_EXPQUAD, term=0, dimmask=3, scale_x=1.3, scale_y=1.3, amp=37.0),
            'matern12': dict(kind=_lib.K_MATERNP, term=0, dimmask=3, ipar=0, par0=0.0, scale_x=2.0, scale_y=2.0, amp=1.0),
            'matern52': dict(kind=_lib.K_MATERNP, term=0, dimmask=3, ipar=2, par0=0.0, scale_x=1.5, scale_y=1.5, amp=0.02),
            'matern72': dict(kind=_lib.K_MATERNP, term=0, dimmask=3, ipar=3, par0=0.0, scale_x=0.7, scale_y=0.7, loc_x=0.5,
                             loc_y=0.5, amp=5.0),
            'cauchy': dict(kind=_lib.K_CAUCHY, term=0, dimmask=3, par0=2.0, par1=3.0, scale_x=1.1, scale_y=1.1, amp=1.0),
            'matern52_nowhite': dict(kind=_lib.K_MATERNP, term=0, dimmask=3, ipar=2, par0=0.0, scale_x=0.4, scale_y=0.4,
                                     amp=1.0),
            'const': dict(kind=_lib.K_EXPQUAD, term=0, dimmask=3, scale_x=1.0, scale_y=1.0, amp=2.0)}[kind]
    descs = [main] if kind == 'matern52_nowhite' else [main, white]
    if kind == 'const':
        descs = descs + [dict(kind=_lib.K_CONSTANT, term=2, dimmask=0, amp=0.7)]
    K = _ops.gram_iso(descs, x, x, symmetric=True)
    ref = _ops.chol_factor(K)
    got = _ops.gram_chol_factor(descs, x)
    assert got is not None
    npad = ref.npad
    assert torch.equal(got.aux[:2 * npad], ref.aux[:2 * npad])                      # s and 1/s
    sr, sg = ref.scalars().cpu().numpy(), got.scalars().cpu().numpy()
    assert abs(sg[0] - sr[0]) <= 1e-14 * sr[0] and abs(sg[1] - sr[1]) <= 1e-14 * sr[1]   # Gershgorin bound, eps
    assert int(got.info.item()) == int(ref.info.item()) == 0
    assert abs(sg[4] - sr[4]) <= 1e-12 * max(1.0, abs(sr[4]))                       # logdet
    Lr, Lg = _ops.chol_get_factor(ref), _ops.chol_get_factor(got)
    assert relerr(Lg, Lr) < 1e-10
    # factorisation + inverse in one call
    side = torch.cuda.Stream(dev())
    st2, Kinv2 = _ops.gram_chol_factor(descs, x, side=side)
    torch.cuda.current_stream().wait_stream(side)
    st1, Kinv1 = _ops.chol_factor_inverse(K, side)
    torch.cuda.current_stream().wait_stream(side)
    assert relerr(torch.tril(Kinv2), torch.tril(Kinv1)) < 1e-9
    assert relerr(_ops.chol_get_factor(st2), Lr) < 1e-10


def test_gram_fused_unsupported_kernels_fall_back():
    x = torch.rand(3, 200, dtype=torch.float64, device=dev())
    # Maternp proper (offset 1e-30) without a White term: its diagonal does not take the library path
    assert _ops.gram_chol_factor([dict(kind=_lib.K_MATERNP, term=0, dimmask=7, ipar=2, par0=1e-30, amp=1.0)], x) is None
    # Matern of real order: general kernel
    assert _ops.gram_chol_factor([dict(kind=_lib.K_MATERN, term=0, dimmask=7, par0=1.3, amp=1.0),
                                  dict(kind=_lib.K_WHITE, term=1, dimmask=7, amp=0.1)], x) is None


def test_chol_failure_reporting():
    K = torch.eye(200, dtype=torch.float64, device=dev())
    K[150, 150] = 1e-30
    K[150, 10] = K[10, 150] = 1.0   # not positive definite; diagonal stays positive so equilibration is finite
    st = _ops.chol_factor(K, epsrel=0.0)
    assert int(st.info.item()) == 151
    st = _ops.chol_factor(-torch.eye(5, dtype=torch.float64, device=dev()))
    assert int(st.info.item()) != 0


def np_r2(x, y, scale, loc=0.0):
    u = (x - loc) / scale
    v = (y - loc) / scale
    r2 = None
    for f in range(u.shape[0]):
        t = (u[f][:, None] - v[f][None, :]) ** 2
        r2 = t if r2 is None else r2 + t
    return r2


def test_gram_iso_vs_oracle():
    rng = np.random.default_rng(11)
    n, m, d = 333, 257, 3
    x = rng.uniform(0, 10, (d, n))
    y = rng.uniform(0, 10, (d, m))
    xd, yd = torch.tensor(x).to(dev()), torch.tensor(y).to(dev())
    full = (1 << d) - 1

    def check(descs, terms, xx, yy, xxd, yyd):
        Kg = _ops.gram_iso(descs, xxd, yyd).cpu().numpy()
        Kr = ogp.gram(terms, xx, yy)
        err = np.max(np.abs(Kg - Kr) / np.abs(Kr).clip(1e-300))
        assert err < 1e-13, err

    check([dict(kind=_lib.K_EXPQUAD, term=0, dimmask=full, scale_x=1.5, scale_y=1.5)],
          [(1.0, [dict(kind='expquad', scale=1.5)])], x, y, xd, yd)
    check([dict(kind=_lib.K_EXPQUAD, term=0, dimmask=full, scale_x=0.3, scale_y=0.3, loc_x=1.0, loc_y=1.0, amp=3.0)],
          [(3.0, [dict(kind='expquad', scale=0.3, loc=1.0)])], x, y, xd, yd)
    for p in range(5):
        check([dict(kind=_lib.K_MATERNP, term=0, dimmask=full, ipar=p, par0=1e-30, scale_x=2.0, scale_y=2.0, amp=1.3),
               dict(kind=_lib.K_WHITE, term=1, dimmask=full, amp=0.01)],
              [(1.3, [dict(kind='maternp', p=p, scale=2.0)]), (0.01, [dict(kind='white')])], x, x, xd, xd)
        # Matern(nu = p + 1/2) closed form against scipy.special.kv, as the reference evaluates it
        check([dict(kind=_lib.K_MATERNP, term=0, dimmask=full, ipar=p, par0=0.0, scale_x=2.0, scale_y=2.0)],
              [(1.0, [dict(kind='matern', nu=p + 0.5, scale=2.0)])], x, y, xd, yd)
    check([dict(kind=_lib.K_CAUCHY, term=0, dimmask=0b101, par0=2.0, par1=3.0),
           dict(kind=_lib.K_EXPQUAD, term=0, dimmask=0b010, scale_x=0.7, scale_y=0.7, amp=2.0)],
          [(2.0, [dict(kind='cauchy', alpha=2, beta=3.0, dims=[0, 2]), dict(kind='expquad', scale=0.7, dims=[1])])],
          x, y, xd, yd)
    check([dict(kind=_lib.K_CAUCHY, term=0, dimmask=full, par0=1.3, par1=0.7, scale_x=4.0, scale_y=4.0),
           dict(kind=_lib.K_CONSTANT, term=1, dimmask=0, amp=0.25)],
          [(1.0, [dict(kind='cauchy', alpha=1.3, beta=0.7, scale=4.0)]), (0.25, [dict(kind='constant')])], x, y, xd, yd)


def test_gram_second_factor_amp():
    rng = np.random.default_rng(12)
    x = rng.uniform(0, 10, (2, 100))
    xd = torch.tensor(x).to(dev())
    Kg = _ops.gram_iso([dict(kind=_lib.K_EXPQUAD, term=0, dimmask=1), dict(kind=_lib.K_EXPQUAD, term=0, dimmask=2, amp=2.0)],
                       xd, xd).cpu().numpy()
    Kr = ogp.gram([(1.0, [dict(kind='expquad', dims=[0])])], x, x) * (2.0 * ogp.gram([(1.0, [dict(kind='expquad', dims=[1])])], x, x))
    assert np.max(np.abs(Kg - Kr) / Kr) < 1e-13


def test_gram_edge_shapes():
    xd = torch.rand(1, 1, dtype=torch.float64, device=dev())
    d1 = [dict(kind=_lib.K_EXPQUAD, term=0, dimmask=1)]
    assert _ops.gram_iso(d1, xd, xd).item() == 1.0
    yd = torch.rand(1, 65, dtype=torch.float64, device=dev())
    K = _ops.gram_iso(d1, xd, yd)
    assert K.shape == (1, 65)
    np.testing.assert_allclose(K.cpu().numpy(), np.exp(-0.5 * (xd.cpu().numpy().T - yd.cpu().numpy()) ** 2), rtol=1e-14)
    # tiny entries: exp(-r2/2) down to the denormal range keeps 1e-13 relative on normal numbers
    far = torch.tensor([[0.0, 30.0, 37.0]], dtype=torch.float64, device=dev())
    K = _ops.gram_iso(d1, far, far).cpu().numpy()
    ref = np.exp(-0.5 * (far.cpu().numpy().T - far.cpu().numpy()) ** 2)
    assert np.max(np.abs(K - ref) / ref) < 1e-13


def test_gram_vjp_matches_finite_differences():
    rng = np.random.default_rng(13)
    n, d = 150, 2
    x = rng.uniform(0, 5, (d, n))
    xd = torch.tensor(x).to(dev())
    G = rng.standard_normal((n, n))
    Gd = _ops.as_aligned(torch.tensor(G).to(dev()))

    def descs(amp, scale, beta):
        return [dict(kind=_lib.K_CAUCHY, term=0, dimmask=3, par0=2.0, par1=beta, scale_x=scale, scale_y=scale, amp=amp),
                dict(kind=_lib.K_MATERNP, term=0, dimmask=1, ipar=2, par0=1e-30, scale_x=2 * scale, scale_y=2 * scale),
                dict(kind=_lib.K_EXPQUAD, term=1, dimmask=2, scale_x=scale, scale_y=scale, amp=0.5 * amp)]
    p0 = np.array([1.3, 0.8, 2.5])
    f = lambda p: float((torch.tensor(G).to(dev()) * _ops.gram_iso(descs(*p), xd, xd)).sum())
    out = _ops.gram_iso_vjp_general(descs(*p0), xd, xd, Gd).cpu().numpy()
    h = 1e-6
    fd = [(f(p0 + h * e) - f(p0 - h * e)) / (2 * h) for e in np.eye(3)]
    # amp enters factor 0 (x1) and factor 2 (x0.5); scale enters all three factors
    g_amp = out[0, 0] + 0.5 * out[2, 0]
    g_scale = (out[0, 1] + out[1, 1] + out[2, 1]) / p0[1]
    g_beta = out[0, 2]
    np.testing.assert_allclose([g_amp, g_scale, g_beta], fd, rtol=1e-6)
    # symmetric fused form == general form on the symmetrised input
    Gs = G + G.T
    b = rng.standard_normal(n)
    full = _ops.gram_iso_vjp_general(descs(*p0), xd, xd, _ops.as_aligned(torch.tensor(Gs - np.outer(b, b)).to(dev())))
    low = _ops.gram_iso_vjp(descs(*p0), xd, _ops.as_aligned(torch.tensor(Gs).to(dev())), torch.tensor(b).to(dev()))
    np.testing.assert_allclose(low.cpu().numpy(), full.cpu().numpy(), rtol=1e-10, atol=1e-10)


@pytest.mark.parametrize('kind,p', [('expquad', 0), ('maternp', 0), ('maternp', 1), ('maternp', 2), ('maternp', 3),
                                    ('maternp', 4)])
def test_gram_fast_vjp_vs_general(kind, p):
    """the fused symmetric VJP (short in-kernel exp/sqrt where in range, library path elsewhere: diagonal, duplicated
    points, far tails) against the general descriptor kernel on the same symmetric weights"""
    rng = np.random.default_rng(14 + p)
    n, d = 333, 3
    x = rng.uniform(0, 10, (d, n))
    x[:, 7] = x[:, 3]           # duplicated point: r2 == 0 off the diagonal
    x[:, 11] = x[:, 12] + 400   # far point: exp underflows for ExpQuad
    xd = torch.tensor(x).to(dev())
    G = rng.standard_normal((n, n))
    G = G + G.T
    b = rng.standard_normal(n)
    main = dict(kind=_lib.K_EXPQUAD if kind == 'expquad' else _lib.K_MATERNP, term=0, dimmask=7, ipar=p, par0=1e-30 if p % 2 else 0.0,
                scale_x=1.7, scale_y=1.7, amp=1.3)
    descs = [main, dict(kind=_lib.K_WHITE, term=1, dimmask=7, amp=0.01)]
    low = _ops.gram_iso_vjp(descs, xd, _ops.as_aligned(torch.tensor(G).to(dev())), torch.tensor(b).to(dev())).cpu().numpy()
    full = _ops.gram_iso_vjp_general(descs, xd, xd, _ops.as_aligned(torch.tensor(G - np.outer(b, b)).to(dev()))).cpu().numpy()
    np.testing.assert_allclose(low, full, rtol=1e-11, atol=1e-11 * np.abs(full).max())


def test_gram_jvp_matches_finite_differences_and_vjp():
    """ lgp_gram_iso_jvp: dK along a tangent of (amp, log scale, par1) per factor; checked against central differences of
    the Gram build and against the reverse-mode kernel through <G, JVP(t)> == <VJP(G), t> """
    rng = np.random.default_rng(21)
    n, m, d = 130, 97, 2
    xd = torch.tensor(rng.uniform(0, 5, (d, n))).to(dev())
    yd = torch.tensor(rng.uniform(0, 5, (d, m))).to(dev())

    def descs(amp0, ls0, beta, amp2, ls2):
        return [dict(kind=_lib.K_CAUCHY, term=0, dimmask=3, par0=2.0, par1=beta, scale_x=np.exp(ls0), scale_y=np.exp(ls0), amp=amp0),
                dict(kind=_lib.K_MATERN, term=0, dimmask=1, par0=1.3, scale_x=2 * np.exp(ls0), scale_y=2 * np.exp(ls0)),
                dict(kind=_lib.K_MATERNP, term=1, dimmask=2, ipar=2, par0=1e-30, scale_x=np.exp(ls2), scale_y=np.exp(ls2), amp=amp2),
                dict(kind=_lib.K_WHITE, term=2, dimmask=3, amp=0.1)]
    p0 = np.array([1.3, np.log(0.8), 2.5, 0.7, np.log(1.9)])
    t = rng.standard_normal(5)
    # tangent in the (nfactors, 3) layout: log scale of factors 0 and 1 move together
    tan = np.zeros((4, 3))
    tan[0] = [t[0], t[1], t[2]]
    tan[1, 1] = t[1]
    tan[2] = [t[3], t[4], 0.0]
    D = _ops.gram_iso_jvp(descs(*p0), xd, yd, tan).cpu().numpy()
    h = 1e-6
    Kp = _ops.gram_iso(descs(*(p0 + h * t)), xd, yd).cpu().numpy()
    Km = _ops.gram_iso(descs(*(p0 - h * t)), xd, yd).cpu().numpy()
    fd = (Kp - Km) / (2 * h)
    assert np.max(np.abs(D - fd)) < 1e-7 * np.max(np.abs(fd))
    G = rng.standard_normal((n, m))
    vjp = _ops.gram_iso_vjp_general(descs(*p0), xd, yd, _ops.as_aligned(torch.tensor(G).to(dev()))).cpu().numpy()
    np.testing.assert_allclose((G * D).sum(), (vjp * tan).sum(), rtol=1e-11)
    # Frobenius inner product kernel (Fisher contraction)
    A = _ops.as_aligned(torch.tensor(G).to(dev()))
    B = _ops.as_aligned(torch.tensor(D).to(dev()))
    np.testing.assert_allclose(float(_ops.frob_dot(A, B)[0]), (G * D).sum(), rtol=1e-12)
    np.testing.assert_allclose(float(_ops.frob_dot(A[:50, :33], B[:50, :33])[0]), (G[:50, :33] * D[:50, :33]).sum(), rtol=1e-12)


@pytest.mark.parametrize('beta', [0.4, 3.0, 25.0])
def test_gram_rational_quadratic_fast_path(beta):
    """ Cauchy(alpha=2) = rational quadratic through the short log/exp fast path (symmetric v3 and rectangular v2 kernels),
    with White and Constant terms, duplicated and far points, against the oracle (numpy pow), 1e-13 """
    rng = np.random.default_rng(31)
    n, m, d = 333, 257, 3
    x = rng.uniform(0, 10, (d, n))
    x[:, 7] = x[:, 3]
    x[:, 11] = x[:, 12] + 1e6      # far point: tiny but nonzero covariance
    y = rng.uniform(0, 10, (d, m))
    xd, yd = torch.tensor(x).to(dev()), torch.tensor(y).to(dev())
    descs = [dict(kind=_lib.K_CAUCHY, term=0, dimmask=7, par0=2.0, par1=beta, scale_x=1.7, scale_y=1.7, amp=1.3),
             dict(kind=_lib.K_WHITE, term=1, dimmask=7, amp=0.01),
             dict(kind=_lib.K_CONSTANT, term=2, dimmask=0, amp=0.25)]
    terms = [(1.3, [dict(kind='cauchy', alpha=2, beta=beta, scale=1.7)]), (0.01, [dict(kind='white')]),
             (0.25, [dict(kind='constant')])]
    for (a, ad, b, bd, sym) in [(x, xd, x, xd, True), (x, xd, y, yd, False)]:
        Kg = _ops.gram_iso(descs, ad, bd, symmetric=sym).cpu().numpy()
        Kr = ogp.gram(terms, a, b)
        assert np.max(np.abs(Kg - Kr) / np.abs(Kr)) < 1e-13
        if sym:
            assert np.array_equal(Kg, Kg.T)
    # the library-path kernel (LGP_GRAM_LIBM) agrees to rounding
    K1 = _ops.gram_iso(descs[:1], xd, xd, symmetric=True)
    K2 = _ops.gram_iso(descs[:1], xd, xd, symmetric=True, flags=_lib.GRAM_LIBM) if hasattr(_lib, 'GRAM_LIBM') else K1
    assert float(((K1 - K2).abs() / K2).max()) < 1e-13


def test_device_resident_descriptor_entry_points():
    """ lgp_gram_iso_dev / _vjp_dev / _jvp_dev (the entry points an XLA-FFI handler binds: hyperparameters in device
    memory, structure as host attributes) give the results of the host-descriptor entry points for the same numbers """
    rng = np.random.default_rng(31)
    n, m = 300, 170
    x = torch.tensor(rng.uniform(0, 5, (3, n)), device='cuda')
    y = torch.tensor(rng.uniform(0, 5, (3, m)), device='cuda')
    descs = [dict(kind=_lib.K_MATERNP, term=0, dimmask=7, ipar=2, par0=0.0, scale_x=1.3, scale_y=1.3, amp=1.7),
             dict(kind=_lib.K_EXPQUAD, term=0, dimmask=3, scale_x=2.1, scale_y=2.1, loc_x=0.3, loc_y=0.3, amp=1.0),
             dict(kind=_lib.K_CAUCHY, term=1, dimmask=4, par0=2.0, par1=1.5, scale_x=0.8, scale_y=0.8, amp=0.6),
             dict(kind=_lib.K_WHITE, term=2, dimmask=7, amp=0.01)]
    devpar = _ops.devpar_of(descs, 'cuda')
    K_host = _ops.gram_iso(descs, x, y, flags=_lib.GRAM_GENERAL)
    K_dev = _ops.gram_iso_dev(descs, devpar, x, y)
    assert torch.equal(K_dev, K_host)
    # changing the device parameters changes the result without touching the host descriptor
    descs2 = [dict(d) for d in descs]
    descs2[0]['scale_x'] = descs2[0]['scale_y'] = 0.9
    descs2[3]['amp'] = 0.05
    K_dev2 = _ops.gram_iso_dev(descs, _ops.devpar_of(descs2, 'cuda'), x, y)
    assert torch.equal(K_dev2, _ops.gram_iso(descs2, x, y, flags=_lib.GRAM_GENERAL))
    G = torch.tensor(rng.standard_normal((n, m)), device='cuda')
    v_host = _ops.gram_iso_vjp_general(descs, x, y, G)
    v_dev = _ops.gram_iso_vjp_dev(descs, devpar, x, y, G)
    np.testing.assert_allclose(v_dev.cpu().numpy(), v_host.cpu().numpy(), rtol=1e-12, atol=1e-12)
    tan = rng.standard_normal((len(descs), 3))
    D_host = _ops.gram_iso_jvp(descs, x, y, tan)
    D_dev = _ops.gram_iso_jvp_dev(descs, devpar, x, y, torch.tensor(tan, device='cuda'))
    np.testing.assert_allclose(D_dev.cpu().numpy(), D_host.cpu().numpy(), rtol=1e-13, atol=1e-14)
    # symmetric lower-triangle form with the rank-one term
    A = torch.tensor(rng.standard_normal((n, n)), device='cuda')
    Gs = _ops.as_aligned(A + A.T)
    b = torch.tensor(rng.standard_normal(n), device='cuda')
    sym_descs = [descs[0], descs[3]]
    sp = _ops.devpar_of(sym_descs, 'cuda')
    vs = _ops.gram_iso_vjp_dev(sym_descs, sp, x, x, Gs, b=b, symlower=True).cpu().numpy()
    vh = _ops.gram_iso_vjp(sym_descs, x, Gs, b).cpu().numpy()
    np.testing.assert_allclose(vs, vh, rtol=1e-10, atol=1e-10 * np.abs(vh).max())


@pytest.mark.parametrize('n', [300, 1500, 5000])
def test_fused_factor_inverse_matches_separate_calls(n):
    """ lgp_chol_factor_inverse (factorisation on the main stream, inverse-from-factor on a second stream behind the
    complete factor) gives the factor and inverse of the two separate calls """
    rng = np.random.default_rng(n)
    x = torch.tensor(rng.uniform(0, 10, (3, n)), device='cuda')
    descs = [dict(kind=_lib.K_MATERNP, term=0, dimmask=7, ipar=2, par0=0.0, scale_x=1.5, scale_y=1.5, amp=1.0),
             dict(kind=_lib.K_WHITE, term=1, dimmask=7, amp=0.01)]
    K = _ops.gram_iso(descs, x, x, symmetric=True)
    st0 = _ops.chol_factor(K)
    inv0 = _ops.chol_inverse(st0)
    side = torch.cuda.Stream('cuda')
    for _ in range(2):
        st1, inv1 = _ops.chol_factor_inverse(K, side)
        torch.cuda.current_stream().wait_stream(side)
        assert int(st1.info.item()) == 0
        assert torch.equal(torch.tril(st1.W[:n, :n]), torch.tril(st0.W[:n, :n]))
        assert torch.equal(st1.aux[:3 * st1.npad + 8], st0.aux[:3 * st0.npad + 8])
        assert torch.equal(torch.tril(inv1), torch.tril(inv0))
    # same stream for both: plain sequential composition
    st2, inv2 = _ops.chol_factor_inverse(K, torch.cuda.current_stream())
    assert torch.equal(torch.tril(inv2), torch.tril(inv0))
    # an independent check of the inverse itself
    Kr = K.clone()
    eps = float(st0.scalars()[1].item())
    s = st0.aux[:n]
    Kr.diagonal().add_(eps * s * s)
    full = torch.tril(inv0) + torch.tril(inv0, -1).T
    resid = (full @ Kr - torch.eye(n, dtype=torch.float64, device='cuda')).abs().max().item()
    assert resid < 1e-7
