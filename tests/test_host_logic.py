"""Host-side logic that needs no GPU: kernel algebra -> descriptors, StructuredArray, BART bracket folding,
error semantics of the API shell."""
import numpy as np
import pytest

import lsqfitgp_b200 as lgp
from lsqfitgp_b200 import _lib, _array
from lsqfitgp_b200._kernels import _BartSpec
from oracle import bart as obart


def test_kernel_algebra_descriptor():
    k = 2.0 * lgp.ExpQuad(scale=3.0) + lgp.Matern(nu=2.5, scale=(1.5, 1.5)) * lgp.Cauchy(beta=3, dim='b') * 0.5 + 0.1
    descs, index = k._descriptor(['a', 'b'])
    assert [d['kind'] for d in descs] == [_lib.K_EXPQUAD, _lib.K_MATERNP, _lib.K_CAUCHY, _lib.K_CONSTANT]
    assert [d['term'] for d in descs] == [0, 1, 1, 2]
    assert [d['amp'] for d in descs] == [2.0, 0.5, 1.0, 0.1]
    assert descs[0]['scale_x'] == 3.0 and descs[1]['ipar'] == 2 and descs[1]['par0'] == 0.0
    assert descs[2]['dimmask'] == 0b10 and descs[0]['dimmask'] == 0b11
    assert descs[2]['par0'] == 2 and descs[2]['par1'] == 3
    assert isinstance(k, lgp.IsotropicKernel)
    kp = lgp.Maternp(p=1)
    assert kp._descriptor([None])[0][0]['par0'] == 1e-30
    k2 = (lgp.ExpQuad() + lgp.White()) * (lgp.ExpQuad(scale=2) + 1)
    assert len(k2._terms) == 4 and all(len(t.factors) == 2 for t in k2._terms)
    k3 = lgp.ExpQuad() ** 3
    assert len(k3._terms) == 1 and len(k3._terms[0].factors) == 3


def test_kernel_errors():
    with pytest.raises(NotImplementedError):
        lgp.Matern(nu=130.0)
    assert lgp.Matern(nu=1.3)._terms[0].factors[0].kind == 5 and lgp.Matern(nu=1.5)._terms[0].factors[0].kind == 1
    with pytest.raises(AssertionError):
        lgp.ExpQuad(scale=-1)
    with pytest.raises(AssertionError):
        lgp.Cauchy(alpha=3)
    with pytest.raises(NotImplementedError):
        lgp.kernel(lambda x, y: x * y)
    with pytest.raises(TypeError):
        lgp.ExpQuad(dim=3)
    with pytest.raises(TypeError):
        lgp.GP(lambda x, y: 1)
    big = lgp.ExpQuad()
    for _ in range(9):
        big = big * lgp.ExpQuad()
    with pytest.raises(NotImplementedError):
        big._descriptor([None])
    with pytest.raises(ValueError):
        lgp.ExpQuad(dim='a')._descriptor([None])


def test_structured_array():
    x = np.zeros(5, dtype=[('a', float), ('b', float, 2)])
    x['a'] = np.arange(5)
    x['b'] = np.arange(10).reshape(5, 2)
    s = lgp.StructuredArray(x)
    assert s.shape == (5,) and s.dtype.names == ('a', 'b')
    labels, data, shape = _array.columns_of(s)
    assert labels == ['a', ('b', 0), ('b', 1)] and data.shape == (3, 5) and shape == (5,)
    np.testing.assert_array_equal(data[2], x['b'][:, 1])
    t = s[1:3]
    assert t.shape == (2,) and np.array_equal(t['a'], [1, 2])
    r = s.reshape(5, 1)
    assert r.shape == (5, 1) and r['b'].shape == (5, 1, 2)
    u = lgp.unstructured_to_structured(np.arange(6.).reshape(3, 2), names=['p', 'q'])
    assert u.dtype.names == ('p', 'q') and np.array_equal(u['q'], [1, 3, 5])
    labels, data, shape = _array.columns_of(np.arange(4.).reshape(2, 2))
    assert labels == [None] and data.shape == (1, 4) and shape == (2, 2)
    with pytest.raises(TypeError):
        _array.columns_of(np.array(['a', 'b']))


@pytest.mark.parametrize('maxd,reset', [(2, None), (4, 2), (10, [2, 4, 6, 8]), (1, None), (0, None), (6, [2, 4]),
                                        (3, [1]), (6, [1, 2, 4]), (7, [2, 3, 5])])
def test_bart_bracket_folding_matches_oracle(maxd, reset):
    """ stages (including reset patterns that do not fold into one `repeat` sequence: chained stages) against the
    oracle's restatement of the reference's bracket folding, and the derivative rows against the complex step of the
    folding (exact to rounding; the same check as tests/test_bart_core_cpu.py::test_stage_drows_match_complex_step on
    these reset patterns) """
    spec = _BartSpec(1.0, (np.array([3]), None), True, 0.95, 2, maxd, 1, None, True, None, reset)
    widths, nrows, rows, drows, gamma = spec.stages()
    ref = obart.fold_brackets(obart.make_pnt(0.95, 2, maxd), reset)
    assert len(widths) == len(ref) and gamma == 1.0
    r = 0
    for w, nr, (probs, repeat) in zip(widths, nrows, ref):
        assert nr == (repeat or 1) and w * nr == probs.size
        np.testing.assert_array_equal(rows[r:r + nr, :w].ravel(), probs)
        r += nr
    assert r == len(rows) and drows.shape == (2,) + rows.shape
    h = 1e-200
    for q, (a, b) in enumerate([(0.95 + 1j * h, 2), (0.95, 2 + 1j * h)]):
        r = 0
        for w, nr, (probs, repeat) in zip(widths, nrows, obart.fold_brackets(obart.make_pnt(a, b, maxd), reset)):
            np.testing.assert_allclose(drows[q, r:r + nr, :w], probs.imag.reshape(nr, w) / h, rtol=1e-15, atol=0)
            assert np.all(drows[q, r:r + nr, w:] == 0)
            r += nr


def test_bart_unsupported_depth():
    spec = _BartSpec(1.0, (np.array([3]), None), True, 0.95, 2, 4, 1, None, True, None, None)
    with pytest.raises(NotImplementedError):
        spec.stages()


def test_bart_preprocessing_matches_oracle(rng):
    X = np.concatenate([rng.standard_normal((40, 3)), rng.integers(0, 2, (40, 1)).astype(float)], axis=1)
    l1, s1 = lgp.BART.splits_from_coord(X)
    l2, s2 = obart.splits_from_coord(X)
    np.testing.assert_array_equal(l1, l2)
    np.testing.assert_array_equal(s1, s2)
    np.testing.assert_array_equal(lgp.BART.indices_from_coord(X, (l1, s1)), obart.indices_from_coord(X, (l2, s2)))
    xs = lgp.unstructured_to_structured(X)
    l3, s3 = lgp.BART.splits_from_coord(xs)
    np.testing.assert_array_equal(l1, l3)


def test_peer_buffer_addressing():
    """ address arithmetic of the symmetric allocation used by the fused TRSM -> broadcast path (no GPU needed) """
    import types
    import torch
    from lsqfitgp_b200 import _dist
    t = torch.zeros(64 + 100, dtype=torch.float64)
    h = types.SimpleNamespace(buffer_ptrs=[0x1000, 0x9000], multicast_ptr=0x20000)
    pb = _dist._PeerBuffer(t, h, 64)
    assert pb.flag_addr(1, 0) == 0x9000 and pb.flag_addr(0, 17) == 0x1000 + 8 * 17
    assert pb.data_addr(0, 0) == 0x1000 + 8 * 64 and pb.data_addr(1, 10) == 0x9000 + 8 * 74
    assert pb.data_addr('mc', 3) == 0x20000 + 8 * 67
    assert pb.data.numel() == 100 and pb.multicast == 0x20000
    h2 = types.SimpleNamespace(buffer_ptrs=[0x1000], multicast_ptr=0)
    assert _dist._PeerBuffer(t, h2, 64).multicast == 0
    with pytest.raises(AssertionError):
        pb.flag_addr(0, 64)
    # without a process group the reservation is a no-op
    assert _dist.peer_reserve(5000, 512, 'cpu') is False


@pytest.mark.parametrize('tiles', [1, 2, 15, 16, 17, 31, 32, 33, 100, 314])
def test_lower_triangular_tile_enumeration_is_a_bijection(tiles):
    """ the grouped rasterisation of the lower-triangular GEMM launches (csrc/gemm_dmma.cuh: bands of 16 tile rows, column
    by column): every tile on or below the diagonal exactly once, and consecutive CTAs stay inside one band (the locality
    the grouping exists for).  Host-side twin of the kernel's index arithmetic, no GPU needed. """
    import ctypes
    lib = _lib.load()
    lib.lgp_debug_lower_tile.restype = ctypes.c_int
    lib.lgp_debug_lower_tile.argtypes = [ctypes.c_longlong, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
    out = (ctypes.c_int * 2)()
    seen = []
    for b in range(tiles * (tiles + 1) // 2):
        assert lib.lgp_debug_lower_tile(b, tiles, out) == 0
        seen.append((out[0], out[1]))
    assert len(set(seen)) == len(seen) and all(0 <= tn <= tm < tiles for tm, tn in seen)
    bands = [tm // 16 for tm, _ in seen]
    assert bands == sorted(bands)
    assert lib.lgp_debug_lower_tile(tiles * (tiles + 1) // 2, tiles, out) != 0


def test_fused_gram_support_query():
    """ lgp_gram_iso_prepare_supported (host-side, nothing launched): which kernel descriptors the Gram build fused with the
    equilibration pass accepts: the fast family whose diagonal takes the library path of the Gram kernel """
    from lsqfitgp_b200 import _ops
    lib = _lib.load()

    def sup(descs, nd=3):
        return bool(lib.lgp_gram_iso_prepare_supported(_ops.make_factors(descs), len(descs), nd))
    white = dict(kind=_lib.K_WHITE, term=1, dimmask=7, amp=0.1)
    const = dict(kind=_lib.K_CONSTANT, term=2, dimmask=0, amp=0.3)
    m52 = dict(kind=_lib.K_MATERNP, term=0, dimmask=7, ipar=2, par0=0.0, amp=1.0)
    assert sup([m52, white]) and sup([m52]) and sup([m52, white, const])
    assert sup([dict(kind=_lib.K_EXPQUAD, term=0, dimmask=7, amp=2.0)])
    assert sup([dict(kind=_lib.K_CAUCHY, term=0, dimmask=7, par0=2.0, par1=3.0, amp=1.0), white])
    assert not sup([dict(m52, par0=1e-30)])                      # Maternp proper without White: fast-path diagonal
    assert sup([dict(m52, par0=1e-30), white])
    assert not sup([dict(kind=_lib.K_MATERN, term=0, dimmask=7, par0=1.3, amp=1.0), white])   # real order: general kernel
    assert not sup([dict(kind=_lib.K_CAUCHY, term=0, dimmask=7, par0=1.5, par1=3.0, amp=1.0)])
    assert not sup([dict(m52, ipar=5), white])
    assert not sup([m52, dict(kind=_lib.K_EXPQUAD, term=0, dimmask=7, amp=1.0)])              # product of two cores
    assert not sup([dict(m52, scale_y=2.0), white])                                           # asymmetric scales
