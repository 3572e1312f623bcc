"""Concrete kernels on the GP-fitting hot path.

Reference definitions: src/lsqfitgp/_kernels/_basic.py:34-75,315-343 (Constant, White, ExpQuad, Cauchy),
src/lsqfitgp/_kernels/_matern.py:29-76 (Maternp, Matern), src/lsqfitgp/_kernels/_bart.py (BART).
The arithmetic is in csrc/gram_iso.cu and csrc/gram_bart.cu.
"""

import numpy
import torch

from . import _array
from . import _lib
from . import _ops
from ._Kernel import IsotropicKernel, Kernel, _f

__all__ = ['Constant', 'White', 'ExpQuad', 'Cauchy', 'Maternp', 'Matern', 'BART']


class Constant(IsotropicKernel):
    """ k(x, y) = 1 (reference _kernels/_basic.py:34-46) """
    _kind = _lib.K_CONSTANT

    def __new__(cls, **kw):
        return cls._make(cls._kind, derivable=numpy.inf, **kw)


class White(IsotropicKernel):
    """ k(x, y) = 1 if x == y else 0 (reference _kernels/_basic.py:48-59) """
    _kind = _lib.K_WHITE

    def __new__(cls, **kw):
        return cls._make(cls._kind, **kw)


class ExpQuad(IsotropicKernel):
    """ k(r) = exp(-r^2/2) (reference _kernels/_basic.py:61-75) """
    _kind = _lib.K_EXPQUAD

    def __new__(cls, **kw):
        return cls._make(cls._kind, derivable=numpy.inf, **kw)


class Cauchy(IsotropicKernel):
    """ k(r) = (1 + r^alpha/beta)^(-beta/alpha); alpha=2 is the rational quadratic (reference _basic.py:315-343) """
    _kind = _lib.K_CAUCHY

    def __new__(cls, alpha=2, beta=2, **kw):
        assert 0 < _f(alpha) <= 2, alpha
        assert 0 < _f(beta), beta
        return cls._make(cls._kind, par0=alpha, par1=beta, derivable=numpy.inf if _f(alpha) == 2 else 0, **kw)


class Maternp(IsotropicKernel):
    """ Matern kernel of half-integer order nu = p + 1/2 (reference _kernels/_matern.py:29-49) """
    _kind = _lib.K_MATERNP

    def __new__(cls, p=None, **kw):
        assert p is not None and int(p) == p and p >= 0, p
        return cls._make(cls._kind, ipar=int(p), par0=1e-30, derivable=int(p), **kw)


class Matern(IsotropicKernel):
    """ Matern kernel of real order nu (reference _kernels/_matern.py:55-76).

    Half-integer orders are evaluated in closed form (same polynomial as Maternp without the 1e-30 offset,
    equal to 2/Gamma(nu) (x/2)^nu K_nu(x) to ~1e-15, SURVEY.md section 6).  Other orders, 0 <= nu <= 100, evaluate
    the modified Bessel function K_nu inside the Gram kernel (csrc/bessel_k.cuh: Temme series / Steed continued
    fraction), where the reference calls scipy.special.kv on the host through jax.pure_callback
    (_special/_bessel.py:35,70-82).  As in the reference, nu itself is not differentiable. """
    _kind = _lib.K_MATERNP

    def __new__(cls, nu=None, **kw):
        assert nu is not None and 0 <= _f(nu) < numpy.inf, nu
        if isinstance(nu, torch.Tensor) and nu.requires_grad:
            raise NotImplementedError('Matern: derivatives with respect to nu are not implemented (nor in the reference)')
        p = _f(nu) - 0.5
        if p >= 0 and p == int(p) and p <= 8:
            return cls._make(_lib.K_MATERNP, ipar=int(p), par0=0.0, derivable=int(p), **kw)
        if _f(nu) > 100:
            raise NotImplementedError(f'Matern(nu={nu!r}): orders above 100 are not implemented on the device')
        return cls._make(_lib.K_MATERN, par0=_f(nu), derivable=max(0, int(numpy.ceil(_f(nu))) - 1), **kw)


# -------------------------------------------------------------------------------------------------
# BART
# -------------------------------------------------------------------------------------------------

class _BartSpec:
    """ parameters of one BART term (amplitude * BART correlation) """

    def __init__(self, amp, splits, indices, alpha, beta, maxd, gamma, pnt, intercept, weights, reset, swapped=False):
        self.amp = amp
        self.splits = splits
        self.indices = indices
        self.alpha = alpha
        self.beta = beta
        self.maxd = maxd
        self.gamma = gamma
        self.pnt = pnt
        self.intercept = intercept
        self.weights = weights
        self.reset = reset

    def scaled(self, c):
        new = _BartSpec.__new__(_BartSpec)
        new.__dict__.update(self.__dict__)
        if isinstance(c, torch.Tensor) or isinstance(self.amp, torch.Tensor):
            new.amp = torch.as_tensor(self.amp, dtype=torch.float64) * torch.as_tensor(c, dtype=torch.float64)
        else:
            new.amp = float(self.amp) * float(c)
        return new

    def swapped(self):
        return self

    def hyperparams(self):
        """ (kind, spec, 0, tensor) for the torch scalars that require grad: amplitude, alpha, beta """
        out = []
        if isinstance(self.amp, torch.Tensor) and self.amp.requires_grad:
            out.append(('bart_amp', self, 0, self.amp))
        for name in ('alpha', 'beta'):
            v = getattr(self, name)
            if isinstance(v, torch.Tensor) and v.requires_grad:
                if self.pnt is not None:
                    raise NotImplementedError(f'gradient w.r.t. BART {name} with explicit pnt')
                out.append(('bart_' + name, self, 0, v))
        for name in ('gamma', 'weights', 'pnt'):
            v = getattr(self, name)
            if isinstance(v, torch.Tensor) and v.requires_grad:
                raise NotImplementedError(f'gradient w.r.t. BART {name}')
        return out

    def stages(self):
        """ bracket folding of BART.correlation (reference _bart.py:372-447) -> (stage_width, stage_nrows, rows, drows,
        gamma): the stages in evaluation order (deepest bracket first), each `nrows` rows of `width` probabilities stored
        3 per row; drows[0] / drows[1] = derivative of every entry w.r.t. alpha / beta (pnt_d = alpha / (1 + d)^beta:
        pnt_d / alpha and -pnt_d log(1 + d); 0 for the entries the folding fixes to 1), None for a user-given `pnt`. """
        if self.pnt is None:
            assert self.maxd == int(self.maxd) and self.maxd >= 0, self.maxd
            alpha, beta = _f(self.alpha), _f(self.beta)
            assert 0 <= alpha <= 1, 'alpha must be in [0, 1]'
            assert beta >= 0, 'beta must be in [0, inf)'
            d = numpy.arange(int(self.maxd) + 1)
            pnt = alpha / (1 + d) ** beta
            dpa = 1 / (1 + d) ** beta
            dpb = -pnt * numpy.log1p(d)
        else:
            pnt = numpy.asarray(self.pnt, dtype=float)
            dpa = dpb = None
        assert numpy.all((0 <= pnt) & (pnt <= 1)), 'pnt must be in [0, 1]'
        gamma = self.gamma
        if isinstance(gamma, str):
            raise NotImplementedError("gamma='auto'")
        gamma = _f(gamma)
        assert 0 <= gamma <= 1, 'gamma must be in [0, 1]'
        depth = numpy.arange(len(pnt))  # which pnt_d an entry is; -1: fixed to 1
        if not self.intercept:
            pnt = pnt.copy()
            pnt[0] = 1
            depth[0] = -1
        reset = self.reset
        if reset is None:
            reset = []
        if not hasattr(reset, '__len__'):
            reset = [reset]
        reset = [0] + list(reset) + [len(pnt) - 1]
        for i, j in zip(reset, reset[1:]):
            assert int(j) == j and i <= j, (i, j)
        brackets_norep = list(zip(reset, reset[1:]))
        brackets = [brackets_norep[0] + (1,)]
        for t, b in brackets_norep[1:]:
            lt, lb, lr = brackets[-1]
            if lr * (b - t) == lb - lt and b - t <= 2:
                brackets[-1] = lt, b, lr + 1
            else:
                brackets.append((t, b, 1))
        widths, nrows, rows, idxs = [], [], [], []
        for t, b, repeat in reversed(brackets):
            idx = depth[t:b + 1].copy()
            if t > 0:
                idx[0] = -1
            if repeat > 1:
                head = idx[0:1]
                one = numpy.full_like(head, -1)
                pieces = [[head if i == 0 else one, p] for i, p in enumerate(numpy.split(idx[1:], repeat))]
                idx = numpy.concatenate(sum(reversed(pieces), start=[]))
            else:
                repeat = 1
            width = len(idx) // repeat
            if width > 3:
                raise NotImplementedError(
                    f'BART bracket of depth {width - 1} > 2: the exponential-cost generic recursion '
                    '(reference _bart.py:759-806) is not implemented on the device; use reset= to keep brackets <= 2')
            widths.append(width)
            nrows.append(repeat)
            idx3 = numpy.full((repeat, 3), -1)
            idx3[:, :width] = idx.reshape(repeat, width)
            idxs.append(idx3)
        idx = numpy.concatenate(idxs, axis=0)
        if len(idx) > _lib.BART_MAX_ROWS or len(widths) > _lib.BART_MAX_STAGES:
            raise NotImplementedError(f'BART: more than {_lib.BART_MAX_ROWS} rows / {_lib.BART_MAX_STAGES} stages')
        fixed = idx < 0
        safe = numpy.where(fixed, 0, idx)
        rows = numpy.where(fixed, 1.0, pnt[safe])
        drows = None
        if dpa is not None:
            drows = numpy.stack([numpy.where(fixed, 0.0, dpa[safe]), numpy.where(fixed, 0.0, dpb[safe])])
        return numpy.array(widths, numpy.int32), numpy.array(nrows, numpy.int32), rows, drows, gamma

    def _indices(self, xd, yd):
        length, splits = self.splits
        length = numpy.asarray(length)
        p = xd.shape[0]
        if p != length.size:
            raise ValueError(f'splitting grid is for {length.size} dimensions, found {p}')
        if self.indices:
            ix = xd.to(torch.int32)
            iy = yd.to(torch.int32) if yd is not xd else ix
        else:
            ix = _bart_indices_device(xd, splits)
            iy = _bart_indices_device(yd, splits) if yd is not xd else ix
        w = numpy.ones(p) if self.weights is None else numpy.asarray(self.weights, dtype=float)
        assert numpy.all(w >= 0), 'weights must be in [0, inf)'
        return length, w, ix, iy

    def gram_device(self, xd, yd, labels, out=None, deriv=False):
        """ amp * BART correlation on the device; deriv: also amp * d corr / d alpha, d beta (forward mode) """
        length, w, ix, iy = self._indices(xd, yd)
        widths, nrows, rows, drows, gamma = self.stages()
        if deriv and drows is None:
            raise NotImplementedError('derivatives w.r.t. alpha / beta with explicit pnt')
        return _ops.gram_bart_stages(length, w, widths, nrows, rows, drows, gamma, _f(self.amp), ix, iy, out=out,
                                     deriv=deriv, symmetric=iy is ix)

    def vjp_device(self, xd, yd, G, b=None, symlower=False):
        """ device tensor [dL/d amp, dL/d alpha, dL/d beta] for the cotangent G of the Gram block (reverse mode, one pass,
        nothing materialised); symlower: G_ij = w_ij (G[i][j] - b_i b_j) from the lower triangle """
        length, w, ix, iy = self._indices(xd, xd if symlower else yd)
        widths, nrows, rows, drows, gamma = self.stages()
        if drows is None:
            drows = numpy.zeros((2,) + rows.shape)
        return _ops.gram_bart_vjp(length, w, widths, nrows, rows, drows, gamma, _f(self.amp), ix, iy, G, b=b,
                                  symlower=symlower)


def _bart_indices_device(xd, splits):
    """ searchsorted(side='left') per dimension (reference _bart.py:503-514) on the device: lgp_searchsorted """
    s = torch.as_tensor(numpy.asarray(splits), dtype=torch.float64, device=xd.device)
    if s.ndim == 1:
        s = s[:, None]
    return _ops.searchsorted(s, xd)


class BART(Kernel):
    """BART prior covariance (reference _kernels/_bart.py:32-202). See `splits_from_coord`,
    `indices_from_coord`, `correlation`."""

    _kind = 'bart'

    def __new__(cls, alpha=0.95, beta=2, maxd=2, gamma=1, splits=None, pnt=None, intercept=True, weights=None,
                reset=None, indices=False, **kw):
        if kw.get('scale') is not None or kw.get('loc') is not None or kw.get('dim') is not None:
            raise NotImplementedError('scale/loc/dim on the BART kernel')
        self = object.__new__(cls)
        splits = cls._check_splits(splits, indices)
        self._terms = ()
        self._bart = (_BartSpec(1.0, splits, bool(indices), alpha, beta, maxd, gamma, pnt, intercept, weights, reset),)
        return self

    @staticmethod
    def _check_splits(splits, indices):
        if splits is None:
            raise ValueError('splits not specified')
        l, s = splits
        l = numpy.asarray(l)
        assert l.ndim == 1
        if not indices:
            s = numpy.asarray(s)
            assert 1 <= s.ndim <= 2
            if s.ndim == 1:
                s = s[:, None]
            assert l.size == s.shape[1]
            assert numpy.all((0 <= l) & (l <= s.shape[0])), 'length out of bounds'
            assert numpy.all(numpy.sort(s, axis=0) == s), 'unsorted splitting points'
        return l, s

    @staticmethod
    def _check_x(x):
        x = _array.asarray(x)
        if isinstance(x, _array.StructuredArray):
            cols = x.leaf_columns()
            return numpy.stack([numpy.asarray(c[1]).reshape(x.shape) for c in cols], axis=-1)
        return numpy.asarray(x)

    @classmethod
    def splits_from_coord(cls, x):
        """ (length (p,), splits (n-1, p)): midpoints of consecutive unique values per column
        (reference _bart.py:209-259).  One-off host preprocessing ("next" row f3 of SURVEY section 8). """
        x = cls._check_x(x)
        x = x.reshape(-1, x.shape[-1]) if x.size else x.reshape(1, x.shape[-1])
        fill = numpy.finfo(x.dtype).max if numpy.issubdtype(x.dtype, numpy.inexact) else numpy.iinfo(x.dtype).max
        lengths, mids = [], []
        for xi in x.T:
            u = numpy.unique(xi)
            u = numpy.concatenate([u, numpy.full(xi.size - u.size, fill, dtype=u.dtype)])
            with numpy.errstate(over='ignore'):
                m = numpy.where(u[1:] < fill, (u[1:] + u[:-1]) / 2, fill)
            lengths.append(numpy.searchsorted(m, fill))
            mids.append(m)
        return numpy.array(lengths), numpy.stack(mids, axis=1)

    @classmethod
    def indices_from_coord(cls, x, splits):
        """ bin index of every coordinate w.r.t. the splitting points (reference _bart.py:261-299) """
        splits = cls._check_splits(splits, False)
        x = cls._check_x(x)
        if x.shape[-1] != splits[0].size:
            raise ValueError(f'splitting grid is for {splits[0].size} dimensions, found {x.shape[-1]}')
        out = numpy.empty(x.shape, dtype=numpy.int64)
        for i in range(x.shape[-1]):
            out[..., i] = numpy.searchsorted(splits[1][:, i], x[..., i])
        return out

    @classmethod
    def correlation(cls, splitsbefore_or_totalsplits, splitsbetween_or_index1, splitsafter_or_index2, *, alpha=0.95,
                    beta=2, gamma=1, maxd=2, debug=False, pnt=None, intercept=True, weights=None, reset=None,
                    altinput=False):
        """ BART prior correlation between points given as split counts or (altinput) bin indices
        (reference _bart.py:301-455), evaluated on the device pair by pair. """
        if debug:
            raise NotImplementedError('debug=True (shortcut-free recursion)')
        a = numpy.asarray(splitsbefore_or_totalsplits)
        b = numpy.asarray(splitsbetween_or_index1)
        c = numpy.asarray(splitsafter_or_index2)
        for v in (a, b, c):
            assert numpy.issubdtype(v.dtype, numpy.integer)
        assert numpy.all(a >= 0), 'splitting counts must be nonnegative'
        if altinput:
            assert numpy.all((0 <= b) & (b <= a)), 'splitting index must be in [0, n]'
            assert numpy.all((0 <= c) & (c <= a)), 'splitting index must be in [0, n]'
            n, ix, iy = a, b, c
        else:
            assert numpy.all(b >= 0) and numpy.all(c >= 0), 'splitting counts must be nonnegative'
            # counts (before, between, after) -> equivalent indices: ix = nminus, iy = nminus + n0, n = total
            n, ix, iy = a + b + c, a, a + b
        n, ix, iy = numpy.broadcast_arrays(n, ix, iy)
        shape = ix.shape[:-1]
        p = ix.shape[-1]
        if p == 0:
            return numpy.ones(shape)  # no covariates: correlation 1 (reference _bart.py:659-661)
        flatn = n.reshape(-1, p)
        out = numpy.empty(flatn.shape[0])
        _lib.require_cuda()
        dev = torch.device('cuda', torch.cuda.current_device())
        # group pairs by their split-count vector (the kernel takes one `n` per launch)
        uniq, inv = numpy.unique(flatn, axis=0, return_inverse=True)
        inv = inv.reshape(-1)
        fx = ix.reshape(-1, p)
        fy = iy.reshape(-1, p)
        for u, nu in enumerate(uniq):
            sel = numpy.nonzero(inv == u)[0]
            spec = _BartSpec(1.0, (nu, None), True, alpha, beta, maxd, gamma, pnt, intercept, weights, reset)
            # pair-wise evaluation: 64 x 64 blocks of pairs, of which only the diagonal is wanted (never an m x m Gram)
            xa = torch.from_numpy(numpy.ascontiguousarray(fx[sel].T.astype(numpy.float64))).to(dev)
            ya = torch.from_numpy(numpy.ascontiguousarray(fy[sel].T.astype(numpy.float64))).to(dev)
            res = torch.empty(len(sel), dtype=torch.float64, device=dev)
            for s0 in range(0, len(sel), 64):
                G = spec.gram_device(xa[:, s0:s0 + 64].contiguous(), ya[:, s0:s0 + 64].contiguous(), None)
                res[s0:s0 + 64] = torch.diagonal(G)
            out[sel] = res.cpu().numpy()
        return out.reshape(shape)
