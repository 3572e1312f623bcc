"""Thin torch-tensor wrappers over the C ABI (one function per entry point of include/lgp_b200.h).

torch is used for device memory and streams only; all arithmetic happens in liblgpb200.so.
"""

import ctypes

import numpy
import torch

from . import _lib
from ._lib import ptr, stream_ptr, check

f64 = torch.float64


def _even(m):
    return m + (m & 1)


def aligned_empty(rows, cols, device, zero=False):
    """ (rows, cols) float64 view with an even leading dimension and 16-byte aligned base """
    ld = _even(max(cols, 1))
    buf = (torch.zeros if zero else torch.empty)((max(rows, 1), ld), dtype=f64, device=device)
    return buf[:rows, :cols]


def as_aligned(t):
    """ return a 2-d float64 tensor on the device with unit column stride, even row stride, aligned base """
    assert t.ndim == 2 and t.dtype == f64
    if (t.stride(1) == 1 and t.stride(0) % 2 == 0 and t.stride(0) >= t.shape[1] and t.data_ptr() % 16 == 0):
        return t
    out = aligned_empty(t.shape[0], t.shape[1], t.device)
    out.copy_(t)
    return out


def dgemm(A, B, C, *, a_kmajor, b_kmajor, M, N, K, alpha=1.0, flags=0):
    lib = _lib.load()
    check(lib.lgp_dgemm(stream_ptr(), int(a_kmajor), int(b_kmajor), M, N, K, float(alpha), ptr(A), A.stride(0),
                        ptr(B), B.stride(0), ptr(C), C.stride(0), flags), 'lgp_dgemm')
    return C


def axpby(alpha, X, beta, Y, gamma=0.0):
    """ Y = alpha*X + beta*Y + gamma*I in place (X may be None) """
    lib = _lib.load()
    n, m = Y.shape
    assert Y.stride(1) == 1 and (X is None or (X.shape == Y.shape and X.stride(1) == 1))
    check(lib.lgp_axpby(stream_ptr(), n, m, float(alpha), ptr(X), X.stride(0) if X is not None else 0, float(beta),
                        ptr(Y), Y.stride(0), float(gamma)), 'lgp_axpby')
    return Y


# ---------------------------------------------------------------------------------------------
# Gram
# ---------------------------------------------------------------------------------------------

def make_factors(descs):
    """ descs: list of dicts with the fields of struct lgp_factor -> ctypes array """
    arr = (_lib.Factor * len(descs))()
    for a, d in zip(arr, descs):
        a.kind = d['kind']
        a.term = d['term']
        a.dimmask = d['dimmask']
        a.ipar = d.get('ipar', 0)
        a.scale_x = d.get('scale_x', 1.0)
        a.scale_y = d.get('scale_y', 1.0)
        a.loc_x = d.get('loc_x', 0.0)
        a.loc_y = d.get('loc_y', 0.0)
        a.par0 = d.get('par0', 0.0)
        a.par1 = d.get('par1', 0.0)
        a.amp = d.get('amp', 1.0)
    return arr


def gram_iso(descs, x, y, out=None, symmetric=False, flags=0):
    """ x: (ndim, n) float64 device tensor (one row per field), y: (ndim, m). Returns (n, m).
    `flags`: extra LGP_GRAM_* bits (_lib.GRAM_GENERAL, _lib.GRAM_LIBM: A/B checks of the fast paths). """
    lib = _lib.load()
    ndim, n = x.shape
    m = y.shape[1]
    assert y.shape[0] == ndim
    x = x.contiguous() if x.stride(1) != 1 else x
    y = y.contiguous() if y.stride(1) != 1 else y
    if out is None:
        out = aligned_empty(n, m, x.device)
    facs = make_factors(descs)
    check(lib.lgp_gram_iso(stream_ptr(), facs, len(descs), ndim, ptr(x), x.stride(0) if ndim else 0, n, ptr(y),
                           y.stride(0) if ndim else 0, m, ptr(out), out.stride(0), (1 if symmetric else 0) | int(flags)),
          'lgp_gram_iso')
    return out


def gram_iso_vjp(descs, x, Ginv, b):
    """ symmetric fused form: (nfactors, 3) device tensor of sum_ij w_ij (Ginv_ij - b_i b_j) dK_ij/d(amp, log scale,
    par1), reading the lower triangle of Ginv (see lgp_b200.h) """
    lib = _lib.load()
    ndim, n = x.shape
    x = x.contiguous() if x.stride(1) != 1 else x
    buf = torch.empty(3 * len(descs) + 8, dtype=f64, device=x.device)
    facs = make_factors(descs)
    check(lib.lgp_gram_iso_vjp(stream_ptr(), facs, len(descs), ndim, ptr(x), x.stride(0) if ndim else 0, n,
                               ptr(x), x.stride(0) if ndim else 0, n, ptr(Ginv), Ginv.stride(0), ptr(b), 1, ptr(buf)),
          'lgp_gram_iso_vjp')
    return buf[:3 * len(descs)].reshape(len(descs), 3)


def gram_iso_vjp_general(descs, x, y, G):
    """ general form: G dense (n, m); returns (nfactors, 3) """
    lib = _lib.load()
    ndim, n = x.shape
    m = y.shape[1]
    x = x.contiguous() if x.stride(1) != 1 else x
    y = y.contiguous() if y.stride(1) != 1 else y
    assert G.shape == (n, m) and G.stride(1) == 1
    buf = torch.empty(3 * len(descs) + 8, dtype=f64, device=x.device)
    facs = make_factors(descs)
    check(lib.lgp_gram_iso_vjp(stream_ptr(), facs, len(descs), ndim, ptr(x), x.stride(0) if ndim else 0, n,
                               ptr(y), y.stride(0) if ndim else 0, m, ptr(G), G.stride(0), None, 0, ptr(buf)),
          'lgp_gram_iso_vjp')
    return buf[:3 * len(descs)].reshape(len(descs), 3)


def gram_iso_jvp(descs, x, y, tangent, out=None):
    """ forward-mode derivative of the Gram build along `tangent` ((nfactors, 3) host array: d amp, d log scale,
    d par1 per factor, the layout of gram_iso_vjp); returns the dense (n, m) matrix (see lgp_b200.h) """
    lib = _lib.load()
    ndim, n = x.shape
    m = y.shape[1]
    x = x.contiguous() if x.stride(1) != 1 else x
    y = y.contiguous() if y.stride(1) != 1 else y
    if out is None:
        out = aligned_empty(n, m, x.device)
    tan = numpy.ascontiguousarray(numpy.asarray(tangent, dtype=numpy.float64).reshape(-1))
    assert tan.size == 3 * len(descs)
    facs = make_factors(descs)
    check(lib.lgp_gram_iso_jvp(stream_ptr(), facs, len(descs), ndim, ptr(x), x.stride(0) if ndim else 0, n,
                               ptr(y), y.stride(0) if ndim else 0, m, tan.ctypes.data_as(_lib.c_double_p),
                               ptr(out), out.stride(0)), 'lgp_gram_iso_jvp')
    return out


def gram_iso_hvp(descs, x, y, G, tangent, b=None, symlower=False):
    """ second-order contraction (lgp_gram_iso_hvp): (nfactors, 3) device tensor of
    sum_ij G_ij d/d(amp, log scale, par1)_f of sum_g tangent_g dK_ij/dtheta_g; `tangent` as in gram_iso_jvp, G dense
    (n, m), or with symlower=True the lower triangle of a symmetric G less b b' (the G of gram_iso_vjp) """
    lib = _lib.load()
    ndim, n = x.shape
    x = x.contiguous() if x.stride(1) != 1 else x
    y = x if symlower else (y.contiguous() if y.stride(1) != 1 else y)
    m = y.shape[1]
    assert G.shape == (n, m) and G.stride(1) == 1
    tan = numpy.ascontiguousarray(numpy.asarray(tangent, dtype=numpy.float64).reshape(-1))
    assert tan.size == 3 * len(descs)
    buf = torch.empty(3 * len(descs), dtype=f64, device=x.device)
    facs = make_factors(descs)
    if b is not None:
        b = b.contiguous()
    check(lib.lgp_gram_iso_hvp(stream_ptr(), facs, len(descs), ndim, ptr(x), x.stride(0) if ndim else 0, n,
                               ptr(y), y.stride(0) if ndim else 0, m, ptr(G), G.stride(0), ptr(b), 1 if symlower else 0,
                               tan.ctypes.data_as(_lib.c_double_p), ptr(buf)), 'lgp_gram_iso_hvp')
    return buf.reshape(len(descs), 3)


def _ld(p):
    """ leading dimension of a contiguous (ndim, n) point array (a one-row array may carry any stride) """
    return p.stride(0) if p.shape[0] > 1 else p.shape[1]


def gram_iso_xvjp(descs, x, y, G, b=None, symlower=False, need_x=True, need_y=True):
    """ reverse-mode contraction with respect to the points (lgp_gram_iso_xvjp): (gx, gy), gx (ndim, n) =
    sum_j G_ij dK_ij/dx_i, gy (ndim, m) = sum_i G_ij dK_ij/dy_j, G dense (n, m); with symlower=True (y is x) the lower
    triangle of a symmetric G less b b' (the G of gram_iso_vjp), gx the total derivative and gy None.  A side not
    `need`ed is None and not computed. """
    lib = _lib.load()
    ndim, n = x.shape
    x = x.contiguous()
    y = x if symlower else y.contiguous()
    m = y.shape[1]
    assert G.shape == (n, m) and G.stride(1) == 1
    gx = torch.empty((ndim, n), dtype=f64, device=x.device) if (need_x or symlower) else None
    gy = torch.empty((ndim, m), dtype=f64, device=x.device) if (need_y and not symlower) else None
    facs = make_factors(descs)
    if b is not None:
        b = b.contiguous()
    check(lib.lgp_gram_iso_xvjp(stream_ptr(), facs, len(descs), ndim, ptr(x), _ld(x), n, ptr(y), _ld(y), m,
                                ptr(G), G.stride(0), ptr(b), 1 if symlower else 0, ptr(gx), n, ptr(gy), m),
          'lgp_gram_iso_xvjp')
    return gx, gy


def gram_iso_xjvp(descs, x, y, tx, ty, out, accumulate=True):
    """ forward-mode derivative with respect to the points (lgp_gram_iso_xjvp): out (n, m) (+)= sum_d tx[d, i]
    dK_ij/dx_{d,i} + ty[d, j] dK_ij/dy_{d,j}; tx (ndim, n), ty (ndim, m) device tensors or None """
    lib = _lib.load()
    ndim, n = x.shape
    m = y.shape[1]
    x = x.contiguous()
    y = y.contiguous()
    tx = None if tx is None else tx.to(x.device, f64).contiguous()
    ty = None if ty is None else ty.to(x.device, f64).contiguous()
    assert out.shape == (n, m) and out.stride(1) == 1
    facs = make_factors(descs)
    check(lib.lgp_gram_iso_xjvp(stream_ptr(), facs, len(descs), ndim, ptr(x), _ld(x), n, ptr(y), _ld(y), m,
                                ptr(tx), n, ptr(ty), m, ptr(out), out.stride(0), 1 if accumulate else 0),
          'lgp_gram_iso_xjvp')
    return out


def dgemv(P, x, y, alpha=1.0):
    """ y += alpha P x in place (P: 2-D, unit column stride; x, y contiguous device vectors) """
    lib = _lib.load()
    assert P.stride(1) == 1 and x.is_contiguous() and y.is_contiguous()
    check(lib.lgp_dgemv(stream_ptr(), 0, ptr(P), P.stride(0), P.shape[0], P.shape[1], ptr(x), ptr(y), float(alpha)),
          'lgp_dgemv')
    return y


def gram_iso_deriv(descs, x, y, dx_field, dy_field, out=None, symmetric=False):
    """ derivative block d/dx_a d/dy_b k(x, y) (lgp_gram_iso_deriv): a = dx_field, b = dy_field field indices, -1 for
    no derivative on that argument; otherwise as gram_iso """
    lib = _lib.load()
    ndim, n = x.shape
    m = y.shape[1]
    x = x.contiguous() if x.stride(1) != 1 else x
    y = y.contiguous() if y.stride(1) != 1 else y
    if out is None:
        out = aligned_empty(n, m, x.device)
    facs = make_factors(descs)
    check(lib.lgp_gram_iso_deriv(stream_ptr(), facs, len(descs), ndim, ptr(x), x.stride(0), n, ptr(y), y.stride(0), m,
                                 int(dx_field), int(dy_field), ptr(out), out.stride(0), 1 if symmetric else 0),
          'lgp_gram_iso_deriv')
    return out


def gram_iso_deriv_vjp(descs, x, y, dx_field, dy_field, G):
    """ (nfactors, 3) device tensor: sum_ij G_ij d block_ij / d(amp, log scale, par1), G dense (n, m) """
    lib = _lib.load()
    ndim, n = x.shape
    m = y.shape[1]
    x = x.contiguous() if x.stride(1) != 1 else x
    y = y.contiguous() if y.stride(1) != 1 else y
    assert G.shape == (n, m) and G.stride(1) == 1
    buf = torch.empty(3 * len(descs), dtype=f64, device=x.device)
    facs = make_factors(descs)
    check(lib.lgp_gram_iso_deriv_vjp(stream_ptr(), facs, len(descs), ndim, ptr(x), x.stride(0), n, ptr(y), y.stride(0),
                                     m, int(dx_field), int(dy_field), ptr(G), G.stride(0), ptr(buf)),
          'lgp_gram_iso_deriv_vjp')
    return buf.reshape(len(descs), 3)


def gram_iso_deriv_jvp(descs, x, y, dx_field, dy_field, tangent, out=None):
    """ forward-mode derivative of the derivative block along `tangent` (layout of gram_iso_jvp) """
    lib = _lib.load()
    ndim, n = x.shape
    m = y.shape[1]
    x = x.contiguous() if x.stride(1) != 1 else x
    y = y.contiguous() if y.stride(1) != 1 else y
    if out is None:
        out = aligned_empty(n, m, x.device)
    tan = numpy.ascontiguousarray(numpy.asarray(tangent, dtype=numpy.float64).reshape(-1))
    assert tan.size == 3 * len(descs)
    facs = make_factors(descs)
    check(lib.lgp_gram_iso_deriv_jvp(stream_ptr(), facs, len(descs), ndim, ptr(x), x.stride(0), n, ptr(y), y.stride(0),
                                     m, int(dx_field), int(dy_field), tan.ctypes.data_as(_lib.c_double_p), ptr(out),
                                     out.stride(0)), 'lgp_gram_iso_deriv_jvp')
    return out


def devpar_of(descs, device):
    """ (nfactors, 6) device tensor of the numeric descriptor fields in the LGP_DEVPAR_STRIDE order
    (scale_x, scale_y, loc_x, loc_y, par1, amp): what a traced caller keeps on the device """
    rows = [[d.get('scale_x', 1.0), d.get('scale_y', 1.0), d.get('loc_x', 0.0), d.get('loc_y', 0.0), d.get('par1', 0.0),
             d.get('amp', 1.0)] for d in descs]
    return torch.tensor(rows, dtype=f64, device=device)


def _structure_only(descs):
    """ descriptor list with the numeric (device-resident) fields blanked: only kind, term, dimmask, ipar, par0 are kept """
    return [dict(kind=d['kind'], term=d['term'], dimmask=d['dimmask'], ipar=d.get('ipar', 0), par0=d.get('par0', 0.0),
                 scale_x=float('nan'), scale_y=float('nan'), loc_x=float('nan'), loc_y=float('nan'), par1=float('nan'),
                 amp=float('nan')) for d in descs]


def gram_iso_dev(descs, devpar, x, y, out=None):
    """ lgp_gram_iso_dev: Gram matrix with the hyperparameters read from the device tensor `devpar` """
    lib = _lib.load()
    ndim, n = x.shape
    m = y.shape[1]
    x = x.contiguous() if x.stride(1) != 1 else x
    y = y.contiguous() if y.stride(1) != 1 else y
    if out is None:
        out = aligned_empty(n, m, x.device)
    facs = make_factors(_structure_only(descs))
    devpar = devpar.contiguous()
    check(lib.lgp_gram_iso_dev(stream_ptr(), facs, len(descs), ndim, ptr(devpar), ptr(x), x.stride(0) if ndim else 0, n,
                               ptr(y), y.stride(0) if ndim else 0, m, ptr(out), out.stride(0), 0), 'lgp_gram_iso_dev')
    return out


def gram_iso_vjp_dev(descs, devpar, x, y, G, b=None, symlower=False):
    lib = _lib.load()
    ndim, n = x.shape
    m = y.shape[1]
    x = x.contiguous() if x.stride(1) != 1 else x
    y = x if symlower else (y.contiguous() if y.stride(1) != 1 else y)
    buf = torch.empty(3 * len(descs) + 8, dtype=f64, device=x.device)
    facs = make_factors(_structure_only(descs))
    devpar = devpar.contiguous()
    check(lib.lgp_gram_iso_vjp_dev(stream_ptr(), facs, len(descs), ndim, ptr(devpar), ptr(x), x.stride(0) if ndim else 0,
                                   n, ptr(y), y.stride(0) if ndim else 0, m, ptr(G), G.stride(0), ptr(b),
                                   1 if symlower else 0, ptr(buf)), 'lgp_gram_iso_vjp_dev')
    return buf[:3 * len(descs)].reshape(len(descs), 3)


def gram_iso_jvp_dev(descs, devpar, x, y, tangent_dev, out=None):
    lib = _lib.load()
    ndim, n = x.shape
    m = y.shape[1]
    x = x.contiguous() if x.stride(1) != 1 else x
    y = y.contiguous() if y.stride(1) != 1 else y
    if out is None:
        out = aligned_empty(n, m, x.device)
    facs = make_factors(_structure_only(descs))
    devpar = devpar.contiguous()
    tangent_dev = tangent_dev.contiguous().reshape(-1)
    assert tangent_dev.numel() == 3 * len(descs)
    check(lib.lgp_gram_iso_jvp_dev(stream_ptr(), facs, len(descs), ndim, ptr(devpar), ptr(x), x.stride(0) if ndim else 0,
                                   n, ptr(y), y.stride(0) if ndim else 0, m, ptr(tangent_dev), ptr(out), out.stride(0)),
          'lgp_gram_iso_jvp_dev')
    return out


def frob_dot(A, B):
    """ sum_ij A_ij B_ij as a 1-element device tensor (A, B: 2-D, unit column stride) """
    lib = _lib.load()
    assert A.shape == B.shape and A.ndim == 2 and A.stride(1) == 1 and B.stride(1) == 1
    out = torch.empty(1, dtype=f64, device=A.device)
    check(lib.lgp_frob_dot(stream_ptr(), ptr(A), A.stride(0), ptr(B), B.stride(0), A.shape[0], A.shape[1], ptr(out)),
          'lgp_frob_dot')
    return out


def add_scalar(Y, c):
    """ Y += c in place (Y: 2-D, unit column stride) """
    lib = _lib.load()
    assert Y.ndim == 2 and Y.stride(1) == 1
    check(lib.lgp_add_scalar(stream_ptr(), Y.shape[0], Y.shape[1], ptr(Y), Y.stride(0), float(c)), 'lgp_add_scalar')
    return Y


def sym_expand_sub(low, b=None, scale=1.0):
    """ full symmetric (n, n) matrix scale * (sym(lower triangle of low) - b b') """
    lib = _lib.load()
    n = low.shape[0]
    assert low.shape == (n, n) and low.stride(1) == 1
    out = aligned_empty(n, n, low.device)
    if b is not None:
        b = b.contiguous()
    check(lib.lgp_sym_expand_sub(stream_ptr(), ptr(low), low.stride(0), ptr(b), n, float(scale), ptr(out), out.stride(0)),
          'lgp_sym_expand_sub')
    return out


def symlower_dot(low, b, D):
    """ 1-element device tensor sum_ij (G_ij - b_i b_j) D_ij, G symmetric given by the lower triangle of `low` """
    lib = _lib.load()
    n = low.shape[0]
    assert low.shape == (n, n) and D.shape == (n, n) and low.stride(1) == 1
    if D.stride(1) != 1:
        D = D.contiguous()
    if b is not None:
        b = b.contiguous()
    out = torch.empty(1, dtype=f64, device=low.device)
    check(lib.lgp_symlower_dot(stream_ptr(), ptr(low), low.stride(0), ptr(b), ptr(D), D.stride(0), n, ptr(out)),
          'lgp_symlower_dot')
    return out


def colsumsq(A):
    """ device vector of the column sums of squares of A (2-D, unit column stride) """
    lib = _lib.load()
    if A.stride(1) != 1:
        A = A.contiguous()
    out = torch.empty(A.shape[1], dtype=f64, device=A.device)
    check(lib.lgp_colsumsq(stream_ptr(), ptr(A), A.stride(0), A.shape[0], A.shape[1], ptr(out)), 'lgp_colsumsq')
    return out


def searchsorted(splits, x):
    """ splits: (maxlen, p) float64 device (row-major), x: (p, n) float64 device -> (p, n) int32 bin indices (side='left') """
    lib = _lib.load()
    splits = splits.contiguous()
    x = x.contiguous()
    p, n = x.shape
    assert splits.ndim == 2 and splits.shape[1] == p
    out = torch.empty((p, n), dtype=torch.int32, device=x.device)
    check(lib.lgp_searchsorted(stream_ptr(), ptr(splits), splits.shape[0], p, ptr(x), x.stride(0) if p else 0, n,
                               ptr(out), out.stride(0) if p else 0), 'lgp_searchsorted')
    return out


_psi_cache = {}


def digamma_table(length, device):
    """ device table psi[k] = digamma(k), at least `length` entries (one growing table per device) """
    key = str(device)
    t = _psi_cache.get(key)
    if t is None or t.numel() < length:
        lib = _lib.load()
        host = numpy.empty(length, dtype=numpy.float64)
        check(lib.lgp_bart_digamma_table(host.ctypes.data_as(_lib.c_double_p), length), 'lgp_bart_digamma_table')
        t = _psi_cache[key] = torch.from_numpy(host).to(device)
    return t


def _bart_cargs(nsplits, w, widths, nrows, rows, drows):
    """ host-side ctypes views of a BART stage description (see lgp_gram_bart_stages) """
    nsplits = numpy.ascontiguousarray(nsplits, dtype=numpy.int32)
    w = numpy.ascontiguousarray(w, dtype=numpy.float64)
    widths = numpy.ascontiguousarray(widths, dtype=numpy.int32)
    nrows = numpy.ascontiguousarray(nrows, dtype=numpy.int32)
    rows = numpy.ascontiguousarray(rows, dtype=numpy.float64)
    assert rows.ndim == 2 and rows.shape == (int(nrows.sum()), 3) and len(widths) == len(nrows)
    keep = [nsplits, w, widths, nrows, rows]
    dptr = None
    if drows is not None:
        drows = numpy.ascontiguousarray(drows, dtype=numpy.float64)
        assert drows.shape == (2,) + rows.shape
        keep.append(drows)
        dptr = drows.ctypes.data_as(_lib.c_double_p)
    args = (len(nsplits), nsplits.ctypes.data_as(_lib.c_int32_p), w.ctypes.data_as(_lib.c_double_p), len(widths),
            widths.ctypes.data_as(_lib.c_int32_p), nrows.ctypes.data_as(_lib.c_int32_p),
            rows.ctypes.data_as(_lib.c_double_p), dptr)
    return args, keep, nsplits


def gram_bart_stages(nsplits, w, widths, nrows, rows, drows, gamma, amp, ix, iy, out=None, deriv=False, symmetric=False):
    """ BART Gram through lgp_gram_bart_stages.  ix: (p, n) int32 device, iy: (p, m) int32 device (the same tensor for
    symmetric=True).  Returns K, or (K, dKa, dKb) = amp * (corr, d corr / d alpha, d corr / d beta) when deriv. """
    lib = _lib.load()
    p, n = ix.shape
    m = iy.shape[1]
    args, keep, nsplits = _bart_cargs(nsplits, w, widths, nrows, rows, drows)
    if out is None:
        out = aligned_empty(n, m, ix.device)
    dKa = dKb = None
    if deriv:
        dKa = aligned_empty(n, m, ix.device)
        dKb = aligned_empty(n, m, ix.device)
    psi = digamma_table(int(nsplits.max(initial=0)) + 2, ix.device) if p else None
    ix = ix.contiguous()
    iy = ix if symmetric else iy.contiguous()
    check(lib.lgp_gram_bart_stages(stream_ptr(), *args, float(gamma), float(amp), ptr(psi), ptr(ix),
                                   ix.stride(0) if p else 0, n, ptr(iy), iy.stride(0) if p else 0, m, ptr(out),
                                   out.stride(0), ptr(dKa), ptr(dKb), dKa.stride(0) if deriv else 0,
                                   _lib.BART_SYMMETRIC if (symmetric and p) else 0), 'lgp_gram_bart_stages')
    del keep
    return (out, dKa, dKb) if deriv else out


def gram_bart_vjp(nsplits, w, widths, nrows, rows, drows, gamma, amp, ix, iy, G, b=None, symlower=False):
    """ device tensor [sum G corr, sum G amp dcorr/dalpha, sum G amp dcorr/dbeta] (lgp_gram_bart_vjp); symlower: G read
    from its lower triangle as w_ij (G_ij - b_i b_j) """
    lib = _lib.load()
    p, n = ix.shape
    m = iy.shape[1]
    args, keep, nsplits = _bart_cargs(nsplits, w, widths, nrows, rows, drows)
    assert G.shape == (n, m) and G.stride(1) == 1
    psi = digamma_table(int(nsplits.max(initial=0)) + 2, ix.device) if p else None
    ix = ix.contiguous()
    iy = ix if symlower else iy.contiguous()
    out = torch.empty(3, dtype=f64, device=ix.device)
    if b is not None:
        b = b.contiguous()
    check(lib.lgp_gram_bart_vjp(stream_ptr(), *args, float(gamma), float(amp), ptr(psi), ptr(ix),
                                ix.stride(0) if p else 0, n, ptr(iy), iy.stride(0) if p else 0, m, ptr(G), G.stride(0),
                                ptr(b), 1 if symlower else 0, ptr(out)), 'lgp_gram_bart_vjp')
    del keep
    return out


def gram_bart(nsplits, w, rows, gamma, amp, ix, iy, out=None):
    """ single-bracket form (lgp_gram_bart). ix: (p, n) int32 device, iy: (p, m) int32 device; rows: (nrows, width) host """
    lib = _lib.load()
    p, n = ix.shape
    m = iy.shape[1]
    nsplits = numpy.ascontiguousarray(nsplits, dtype=numpy.int32)
    w = numpy.ascontiguousarray(w, dtype=numpy.float64)
    rows = numpy.ascontiguousarray(rows, dtype=numpy.float64)
    nrows, width = rows.shape
    if out is None:
        out = aligned_empty(n, m, ix.device)
    psi = digamma_table(int(nsplits.max(initial=0)) + 2, ix.device) if p else None
    ix = ix.contiguous()
    iy = iy.contiguous()
    check(lib.lgp_gram_bart(stream_ptr(), p, nsplits.ctypes.data_as(_lib.c_int32_p),
                            w.ctypes.data_as(_lib.c_double_p), rows.ctypes.data_as(_lib.c_double_p), nrows, width,
                            float(gamma), float(amp), ptr(psi), ptr(ix), ix.stride(0) if p else 0, n, ptr(iy),
                            iy.stride(0) if p else 0, m, ptr(out), out.stride(0), 0), 'lgp_gram_bart')
    return out


# ---------------------------------------------------------------------------------------------
# Cholesky
# ---------------------------------------------------------------------------------------------

class FactorState:
    """ device-resident factor: W (npad x npad, lower = Lt), aux (s, 1/s, diag, scalars, inverted blocks) """

    __slots__ = ('n', 'npad', 'W', 'aux', 'info', 'device')

    def scalars(self):
        """ device view: [maxrowsum, eps, -, min s^2, sum log L_ii, -] """
        return self.aux[3 * self.npad: 3 * self.npad + 16]


def chol_factor(K, addmat=None, adddiag=None, epsrel='auto', epsabs=0.0):
    lib = _lib.load()
    assert K.ndim == 2 and K.shape[0] == K.shape[1] and K.dtype == f64
    n = K.shape[0]
    if K.stride(1) != 1:
        K = K.contiguous()
    if addmat is not None and addmat.stride(1) != 1:
        addmat = addmat.contiguous()
    if adddiag is not None:
        adddiag = adddiag.contiguous()
    st = FactorState()
    st.n = n
    st.npad = int(lib.lgp_chol_npad(n))
    st.device = K.device
    st.W = torch.empty((st.npad, st.npad), dtype=f64, device=K.device)
    st.aux = torch.empty(int(lib.lgp_chol_aux_doubles(n)), dtype=f64, device=K.device)
    st.info = torch.empty(1, dtype=torch.int32, device=K.device)
    er = -1.0 if (isinstance(epsrel, str) and epsrel == 'auto') else float(epsrel)
    ea = 2.220446049250313e-16 if (isinstance(epsabs, str) and epsabs == 'auto') else float(epsabs)
    check(lib.lgp_chol_factor(stream_ptr(), ptr(K), K.stride(0), ptr(addmat),
                              addmat.stride(0) if addmat is not None else 0, ptr(adddiag), n, er, ea, ptr(st.W),
                              st.W.stride(0), ptr(st.aux), ptr(st.info)), 'lgp_chol_factor')
    return st


def chol_factor_inverse(K, side, addmat=None, adddiag=None, epsrel='auto', epsabs=0.0):
    """ factorisation on the current stream and inverse-from-factor on the torch stream `side`, overlapped inside the
    library (lgp_chol_factor_inverse).  Returns (FactorState, Kinv view (n, n), lower triangle valid): the factor is
    ready in current-stream order, Kinv in `side` order (wait for `side` before reading it). """
    lib = _lib.load()
    assert K.ndim == 2 and K.shape[0] == K.shape[1] and K.dtype == f64
    n = K.shape[0]
    if K.stride(1) != 1:
        K = K.contiguous()
    if addmat is not None and addmat.stride(1) != 1:
        addmat = addmat.contiguous()
    if adddiag is not None:
        adddiag = adddiag.contiguous()
    st = FactorState()
    st.n = n
    st.npad = int(lib.lgp_chol_npad(n))
    st.device = K.device
    st.W = torch.empty((st.npad, st.npad), dtype=f64, device=K.device)
    st.aux = torch.empty(int(lib.lgp_chol_aux_doubles(n)), dtype=f64, device=K.device)
    st.info = torch.empty(1, dtype=torch.int32, device=K.device)
    main = torch.cuda.current_stream()
    with torch.cuda.stream(side):   # the inverse buffers come from the side stream's allocator pool (kept warm there)
        scratch = torch.empty((st.npad, st.npad), dtype=f64, device=K.device)
        Kinv = torch.empty((st.npad, st.npad), dtype=f64, device=K.device)
    er = -1.0 if (isinstance(epsrel, str) and epsrel == 'auto') else float(epsrel)
    ea = 2.220446049250313e-16 if (isinstance(epsabs, str) and epsabs == 'auto') else float(epsabs)
    check(lib.lgp_chol_factor_inverse(ctypes.c_void_p(main.cuda_stream), ctypes.c_void_p(side.cuda_stream), ptr(K),
                                      K.stride(0), ptr(addmat), addmat.stride(0) if addmat is not None else 0,
                                      ptr(adddiag), n, er, ea, ptr(st.W), st.W.stride(0), ptr(st.aux), ptr(st.info),
                                      ptr(scratch), ptr(Kinv), Kinv.stride(0)), 'lgp_chol_factor_inverse')
    # buffers of one stream's pool used by the other stream: keep the allocator from recycling them too early
    for t in (st.W, st.aux, K):
        t.record_stream(side)
    scratch.record_stream(side)
    del scratch
    return st, Kinv[:n, :n]



def gram_chol_factor(descs, x, side=None, epsrel='auto', epsabs=0.0):
    """ Gram build fused with the equilibration pass of the factorisation (lgp_gram_iso_prepare), then the factorisation
    (lgp_chol_factor_prepared) or, with a torch stream `side`, factorisation + inverse-from-factor
    (lgp_chol_factor_inverse_prepared).  x: (ndim, n) float64 device tensor; the matrix K itself is never written.
    Returns FactorState (side is None) or (FactorState, Kinv view) like chol_factor / chol_factor_inverse, or None when the
    kernel is outside the fused family (the caller then builds the Gram matrix and factors it). """
    lib = _lib.load()
    ndim, n = x.shape
    if ndim < 1 or n < 1:
        return None
    facs = make_factors(descs)
    if not lib.lgp_gram_iso_prepare_supported(facs, len(descs), ndim):
        return None   # (asked before any buffer is allocated)
    x = x.contiguous() if x.stride(1) != 1 else x
    st = FactorState()
    st.n = n
    st.npad = int(lib.lgp_chol_npad(n))
    st.device = x.device
    st.W = torch.empty((st.npad, st.npad), dtype=f64, device=x.device)
    st.aux = torch.empty(int(lib.lgp_chol_aux_doubles(n)), dtype=f64, device=x.device)
    st.info = torch.empty(1, dtype=torch.int32, device=x.device)
    main = torch.cuda.current_stream()
    nwork = int(lib.lgp_gram_prepare_work_doubles(n))
    if side is not None:
        with torch.cuda.stream(side):   # the inverse buffers come from the side stream's allocator pool (kept warm there)
            scratch = torch.empty((st.npad, st.npad), dtype=f64, device=x.device)
            Kinv = torch.empty((st.npad, st.npad), dtype=f64, device=x.device)
        # the partial row sums of the Gram build live in the inverse's scratch (unused until the factor is complete); it
        # was allocated on the side stream: order the main stream behind whatever used that block there before
        main.wait_stream(side)
        work = scratch
    else:
        work = torch.empty(nwork, dtype=f64, device=x.device)
    rc = lib.lgp_gram_iso_prepare(ctypes.c_void_p(main.cuda_stream), facs, len(descs), ndim, ptr(x), x.stride(0), n,
                                  ptr(st.W), st.W.stride(0), ptr(st.aux), ptr(work))
    if rc == -4:
        return None
    check(rc, 'lgp_gram_iso_prepare')
    er = -1.0 if (isinstance(epsrel, str) and epsrel == 'auto') else float(epsrel)
    ea = 2.220446049250313e-16 if (isinstance(epsabs, str) and epsabs == 'auto') else float(epsabs)
    if side is None:
        check(lib.lgp_chol_factor_prepared(ctypes.c_void_p(main.cuda_stream), n, er, ea, ptr(st.W), st.W.stride(0),
                                           ptr(st.aux), ptr(st.info)), 'lgp_chol_factor_prepared')
        return st
    check(lib.lgp_chol_factor_inverse_prepared(ctypes.c_void_p(main.cuda_stream), ctypes.c_void_p(side.cuda_stream), n, er,
                                               ea, ptr(st.W), st.W.stride(0), ptr(st.aux), ptr(st.info), ptr(scratch),
                                               ptr(Kinv), Kinv.stride(0)), 'lgp_chol_factor_inverse_prepared')
    for t in (st.W, st.aux):
        t.record_stream(side)
    scratch.record_stream(main)
    del scratch
    return st, Kinv[:n, :n]


def chol_solve(st, B, trans, inplace=False):
    """ B: (n, m) device tensor -> L^-1 B (trans=False) or L^-T B (trans=True) """
    lib = _lib.load()
    Bw = as_aligned(B)
    if Bw is B and not inplace:
        Bw = aligned_empty(B.shape[0], B.shape[1], B.device)
        Bw.copy_(B)
    check(lib.lgp_chol_solve(stream_ptr(), ptr(st.W), st.W.stride(0), ptr(st.aux), st.n, ptr(Bw), Bw.stride(0),
                             Bw.shape[1], int(bool(trans))), 'lgp_chol_solve')
    return Bw


def chol_mult(st, X, trans):
    lib = _lib.load()
    Xa = as_aligned(X)
    Y = aligned_empty(X.shape[0], X.shape[1], X.device)
    tmp = aligned_empty(X.shape[0], X.shape[1], X.device) if trans else None
    check(lib.lgp_chol_mult(stream_ptr(), ptr(st.W), st.W.stride(0), ptr(st.aux), st.n, ptr(Xa), Xa.stride(0),
                            Xa.shape[1], ptr(Y), Y.stride(0), ptr(tmp), tmp.stride(0) if trans else 0,
                            int(bool(trans))), 'lgp_chol_mult')
    return Y


def chol_get_factor(st):
    lib = _lib.load()
    L = torch.empty((st.n, st.n), dtype=f64, device=st.device)
    check(lib.lgp_chol_get_factor(stream_ptr(), ptr(st.W), st.W.stride(0), ptr(st.aux), st.n, ptr(L), L.stride(0)),
          'lgp_chol_get_factor')
    return L


def chol_inverse(st):
    """ lower triangle of (L L^T)^-1 in an (npad, npad) buffer; returns the (n, n) view (upper part undefined) """
    lib = _lib.load()
    scratch = torch.empty((st.npad, st.npad), dtype=f64, device=st.device)
    Kinv = torch.empty((st.npad, st.npad), dtype=f64, device=st.device)
    check(lib.lgp_chol_inverse(stream_ptr(), ptr(st.W), st.W.stride(0), ptr(st.aux), st.n, ptr(scratch), ptr(Kinv),
                               Kinv.stride(0)), 'lgp_chol_inverse')
    del scratch
    return Kinv[:st.n, :st.n]


def chol_logdet_quad(st, a=None):
    """ device tensor [sum_i log L_ii, sum_i a_i^2] """
    lib = _lib.load()
    out = torch.empty(2, dtype=f64, device=st.device)
    if a is not None:
        a = a.contiguous()
    check(lib.lgp_chol_logdet_quad(stream_ptr(), ptr(st.aux), st.n, ptr(a), ptr(out)), 'lgp_chol_logdet_quad')
    return out
