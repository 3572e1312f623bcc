"""Kernel objects: lsqfitgp's CrossKernel / Kernel / IsotropicKernel API on top of descriptor-driven
CUDA Gram kernels.

In the reference a kernel wraps an arbitrary Python/JAX `core(x, y)` callable and every transformation
wraps the previous closure (src/lsqfitgp/_Kernel/_crosskernel.py:152-249, _Kernel/_ops.py, _alg.py).
Here a kernel is a *value*: a sum of terms, each a scalar amplitude times a product of isotropic factors
(kind, parameters, scale, loc, selected fields).  The value is flattened into `lgp_factor_t` records and
evaluated by one fused CUDA kernel (lgp_gram_iso), so the call signature `k(x, y)`, the constructor
keywords `scale=, loc=, dim=` and the algebra `c*k`, `k+k`, `k*k`, `k**n` are those of the reference,
but kernels that cannot be expressed as such a descriptor raise NotImplementedError (no CPU fallback).

Hyperparameters (amplitudes, scales, Cauchy beta) may be torch float64 scalars that require grad: the
log marginal likelihood is differentiable w.r.t. them through torch.autograd (see _linalg.py /
_GP.py), which replaces the reference's JAX tracing of the same scalars.
"""

import numbers

import numpy
import torch

from . import _array
from ._Deriv import Deriv
from . import _lib
from . import _ops

__all__ = ['CrossKernel', 'Kernel', 'CrossStationaryKernel', 'StationaryKernel', 'CrossIsotropicKernel',
           'IsotropicKernel', 'kernel', 'stationarykernel', 'isotropickernel', 'crosskernel',
           'crossstationarykernel', 'crossisotropickernel']


def _isscalar(x):
    if isinstance(x, numbers.Number):
        return True
    if isinstance(x, numpy.ndarray) and x.ndim == 0 and numpy.issubdtype(x.dtype, numpy.number):
        return True
    if isinstance(x, torch.Tensor) and x.ndim == 0:
        return True
    return False


def _f(x):
    """ python float value of a hyperparameter """
    if isinstance(x, torch.Tensor):
        return float(x.detach())
    return float(x)


def _pair(arg):
    """ linop argument: value or (left, right) tuple -> (left, right) """
    if isinstance(arg, tuple):
        if len(arg) != 2:
            raise ValueError('transformation argument tuple must have length 2')
        return arg
    return (arg, arg)


class _Factor:
    """ one isotropic factor: core(kind, params) applied to r2 over selected fields after loc/scale """

    __slots__ = ('kind', 'ipar', 'par0', 'par1', 'scale', 'loc', 'dim', 'derivable')

    def __init__(self, kind, ipar=0, par0=0.0, par1=0.0, scale=(None, None), loc=(None, None), dim=(None, None),
                 derivable=0):
        self.kind = kind
        self.derivable = derivable   # how many times the factor may be differentiated w.r.t. each of its fields
        self.ipar = ipar
        self.par0 = par0
        self.par1 = par1
        self.scale = scale
        self.loc = loc
        self.dim = dim

    def replace(self, **kw):
        new = _Factor(self.kind, self.ipar, self.par0, self.par1, self.scale, self.loc, self.dim, self.derivable)
        for k, v in kw.items():
            setattr(new, k, v)
        return new

    def swapped(self):
        return self.replace(scale=self.scale[::-1], loc=self.loc[::-1], dim=self.dim[::-1])


class _Term:
    __slots__ = ('amp', 'factors')

    def __init__(self, amp, factors):
        self.amp = amp
        self.factors = tuple(factors)


class CrossKernel:
    """Base class of kernels (covariance functions of two possibly different processes)."""

    _kind = None          # set by concrete kernels (_kernels.py)
    _derivable = None
    _diff = None          # (Deriv of x, Deriv of y) of a kernel made by linop('diff')

    def __new__(cls, *args, **kw):
        if cls._kind is None and (args or kw):
            raise NotImplementedError(
                'lsqfitgp_b200 evaluates kernels with fused CUDA code: arbitrary Python `core` callables '
                '(reference: CrossKernel(core, ...), @kernel decorators) are not supported; combine the built-in '
                'kernels with +, * and scalar factors instead')
        self = object.__new__(cls)
        self._terms = ()
        self._bart = ()
        self._diff = None
        return self

    # ---- construction helpers used by _kernels.py
    @classmethod
    def _make(cls, kind, *, ipar=0, par0=0.0, par1=0.0, scale=None, loc=None, dim=None, derivable=None, maxdim=None,
              forcekron=False, batchbytes=None):
        if forcekron:
            raise NotImplementedError('forcekron')
        self = object.__new__(cls)
        sx, sy = _pair(scale)
        lx, ly = _pair(loc)
        dx, dy = _pair(dim)
        for s in (sx, sy):
            if s is not None and not (0 < _f(s) < numpy.inf):
                raise AssertionError(s)  # the reference asserts 0 < scale < inf (_ops.py:324-325)
        for l in (lx, ly):
            if l is not None and not (-numpy.inf < _f(l) < numpy.inf):
                raise AssertionError(l)
        for d in (dx, dy):
            if d is not None and not isinstance(d, (str, list)):
                raise TypeError(f'dim must be a (list of) string, found {d!r}')
        fac = _Factor(kind, ipar, par0, par1, (sx, sy), (lx, ly), (dx, dy), 0 if derivable is None else derivable)
        self._terms = (_Term(1.0, (fac,)),)
        self._bart = ()
        self._diff = None
        self._maxdim = maxdim
        return self

    def _clone(self, cls=None, terms=None, bart=None):
        new = object.__new__(cls or type(self))
        new._terms = self._terms if terms is None else tuple(terms)
        new._bart = self._bart if bart is None else tuple(bart)
        new._diff = None
        return new

    # ---- algebra (reference: _Kernel/_alg.py:32-143, _crosskernel.py:235-249)
    def __add__(self, other):
        _no_algebra_on_diff(self, other)
        if _isscalar(other):
            const = _Term(other, (_Factor(_lib.K_CONSTANT, derivable=numpy.inf),))
            return self._clone(_common_class(type(self), IsotropicKernel), terms=self._terms + (const,))
        if isinstance(other, CrossKernel):
            return self._clone(_common_class(type(self), type(other)), terms=self._terms + other._terms,
                               bart=self._bart + other._bart)
        return NotImplemented

    __radd__ = __add__

    def __mul__(self, other):
        _no_algebra_on_diff(self, other)
        if _isscalar(other):
            terms = [_Term(_mulamp(t.amp, other), t.factors) for t in self._terms]
            bart = [b.scaled(other) for b in self._bart]
            return self._clone(terms=terms, bart=bart)
        if isinstance(other, CrossKernel):
            if self._bart or other._bart:
                raise NotImplementedError('products involving the BART kernel are not supported by the fused kernels')
            terms = []
            for a in self._terms:
                for b in other._terms:
                    terms.append(_Term(_mulamp(a.amp, b.amp), a.factors + b.factors))
            return self._clone(_common_class(type(self), type(other)), terms=terms)
        return NotImplemented

    __rmul__ = __mul__

    def __pow__(self, exponent):
        if not (isinstance(exponent, numbers.Integral) and exponent >= 0):
            raise NotImplementedError('kernel ** non-integer')
        if exponent == 0:
            return self * 0 + 1
        out = self
        for _ in range(int(exponent) - 1):
            out = out * self
        return out

    def _swap(self):
        terms = [_Term(t.amp, [f.swapped() for f in t.factors]) for t in self._terms]
        return self._clone(CrossKernel, terms=terms, bart=[b.swapped() for b in self._bart])

    def linop(self, transfname, *args):
        """ subset of CrossKernel.linop: 'scale', 'loc', 'dim' applied to every factor (reference _ops.py) """
        if len(args) == 1:
            args = args * 2
        if all(a is None for a in args):
            return self
        if transfname == 'diff':
            return self._linop_diff(*args)
        if transfname not in ('scale', 'loc', 'dim'):
            raise NotImplementedError(f'linop {transfname!r}')
        if self._diff is not None:
            raise NotImplementedError(f'linop {transfname!r} after linop(\'diff\')')
        if self._bart:
            raise NotImplementedError(f'linop {transfname!r} on the BART kernel')
        terms = []
        for t in self._terms:
            facs = []
            for f in t.factors:
                old = getattr(f, transfname)
                if any(o is not None for o in old) and transfname != 'dim':
                    raise NotImplementedError(f'composition of two {transfname!r} transformations')
                facs.append(f.replace(**{transfname: tuple(args)}))
            terms.append(_Term(t.amp, facs))
        return self._clone(terms=terms)

    def _linop_diff(self, dx, dy):
        """ k(x, y) -> d/dx_a d/dy_b k(x, y) for derivatives of order <= 1 on each argument (reference
        _Kernel/_crosskernel.py linop('diff') and _Kernel/_ops.py, Diff) """
        dx, dy = Deriv(dx), Deriv(dy)
        if not dx and not dy:
            return self
        if self._diff is not None:
            raise NotImplementedError("composition of two 'diff' transformations")
        self._check_derivable(dx, 0)
        self._check_derivable(dy, 1)
        new = self._clone(CrossKernel)
        new._diff = (dx, dy)
        return new

    def _check_derivable(self, deriv, side):
        """ ValueError if the derivative `deriv` of argument `side` (0 = x, 1 = y) exceeds the derivability of a factor
        that depends on its field (factors that do not depend on it impose no limit); NotImplementedError for what the
        kernels cannot compute (order > 1 on one argument, Matern of non-half-integer order) """
        if not deriv:
            return
        for field, order in deriv:
            for t in self._terms:
                for f in t.factors:
                    if not _factor_depends_on(f, field, side):
                        continue
                    if order > f.derivable:
                        raise ValueError(f'derivative of order {order} w.r.t. {field!r} exceeds the derivability '
                                         f'{f.derivable} of the kernel')
            if self._bart:
                raise ValueError(f'derivative of order {order} w.r.t. {field!r} exceeds the derivability 0 of the '
                                 'BART kernel')
        if deriv.order > 1:
            raise NotImplementedError(f'derivative of order {deriv.order} > 1 on one argument')
        for field, order in deriv:
            for t in self._terms:
                for f in t.factors:
                    if f.kind == _lib.K_MATERN and _factor_depends_on(f, field, side):
                        raise NotImplementedError('derivatives of Matern of non-half-integer order')

    def batch(self, maxnbytes):
        """ the reference chunks the evaluation to bound temporaries (_jaxext/_batcher.py); the fused kernel has none """
        return self

    # ---- evaluation
    def __call__(self, x, y):
        """ k(x, y) with numpy broadcasting of x and y; returns a numpy array """
        _lib.require_cuda()
        lx, cx, sx = _array.columns_of(x)
        ly, cy, sy = _array.columns_of(y)
        if lx != ly:
            raise ValueError(f'x and y have different fields: {lx} vs {ly}')
        shape = numpy.broadcast_shapes(sx, sy)
        dfields = None
        if self._diff is not None:
            dfields = (deriv_field(self._diff[0], lx), deriv_field(self._diff[1], ly))
        dev = torch.device('cuda', torch.cuda.current_device())
        xd, yd = (c.detach().to(dev).contiguous() if isinstance(c, torch.Tensor) else
                  torch.from_numpy(numpy.ascontiguousarray(c)).to(dev) for c in (cx, cy))
        G = self._gram_device(xd, yd, lx, dfields=dfields).cpu().numpy()
        ix = numpy.broadcast_to(numpy.arange(cx.shape[1]).reshape(sx), shape)
        iy = numpy.broadcast_to(numpy.arange(cy.shape[1]).reshape(sy), shape)
        return G[ix, iy]

    def _descriptor(self, labels):
        """ flatten to (list of lgp_factor dicts, list of (term index, factor index)) for the given field labels """
        ndim = len(labels)
        if ndim > _lib.MAX_DIMS:
            raise NotImplementedError(f'more than {_lib.MAX_DIMS} covariate dimensions')
        descs, index = [], []
        for ti, t in enumerate(self._terms):
            for fi, f in enumerate(t.factors):
                mx = _dimmask(labels, f.dim[0])
                my = _dimmask(labels, f.dim[1])
                if mx != my:
                    raise NotImplementedError('different `dim` for the two arguments')
                sx, sy = f.scale
                lx, ly = f.loc
                descs.append(dict(
                    kind=f.kind, term=ti, dimmask=mx, ipar=int(f.ipar), par0=_f(f.par0), par1=_f(f.par1),
                    scale_x=1.0 if sx is None else _f(sx), scale_y=1.0 if sy is None else _f(sy),
                    loc_x=0.0 if lx is None else _f(lx), loc_y=0.0 if ly is None else _f(ly),
                    amp=_f(t.amp) if fi == 0 else 1.0))
                index.append((ti, fi))
        if len(descs) > _lib.MAX_FACTORS:
            raise NotImplementedError(f'kernel expression has {len(descs)} factors > {_lib.MAX_FACTORS}')
        return descs, index

    def _gram_device(self, xd, yd, labels, out=None, symmetric=False, dfields=None):
        """ Gram matrix on the device. xd: (ndim, n), yd: (ndim, m) float64 cuda tensors; dfields: (a, b) field
        indices of a derivative block d/dx_a d/dy_b (-1: none on that argument), see deriv_field """
        n, m = xd.shape[1], yd.shape[1]
        if out is None:
            out = _ops.aligned_empty(n, m, xd.device)
        if dfields is not None and dfields != (-1, -1):
            assert not self._bart   # rejected by _check_derivable
            if self._terms:
                descs, _ = self._descriptor(labels)
                _ops.gram_iso_deriv(descs, xd, yd, dfields[0], dfields[1], out=out, symmetric=symmetric)
            else:
                out.zero_()
            return out
        have = False
        if self._terms:
            descs, _ = self._descriptor(labels)
            _ops.gram_iso(descs, xd, yd, out=out, symmetric=symmetric)
            have = True
        for b in self._bart:
            if have:
                tmp = b.gram_device(xd, yd, labels)
                _ops.axpby(1.0, tmp, 1.0, out)
            else:
                b.gram_device(xd, yd, labels, out=out)
                have = True
        if not have:
            out.zero_()
        return out

    # ---- hyperparameter gradient plumbing (used by _linalg.logml autograd function)
    def _hyperparams(self):
        """ list of (kind, term index, factor index, tensor) for torch tensors that require grad """
        out = []
        for ti, t in enumerate(self._terms):
            if isinstance(t.amp, torch.Tensor) and t.amp.requires_grad:
                out.append(('amp', ti, 0, t.amp))
            for fi, f in enumerate(t.factors):
                sx, sy = f.scale
                if isinstance(sx, torch.Tensor) and sx.requires_grad:
                    if sy is not sx:
                        raise NotImplementedError('gradient w.r.t. a scale applied to one argument only')
                    out.append(('scale', ti, fi, sx))
                if isinstance(f.par1, torch.Tensor) and f.par1.requires_grad:
                    out.append(('par1', ti, fi, f.par1))
                for l in f.loc:
                    if isinstance(l, torch.Tensor) and l.requires_grad:
                        raise NotImplementedError('gradient w.r.t. loc')
                if isinstance(f.par0, torch.Tensor) and f.par0.requires_grad:
                    raise NotImplementedError('gradient w.r.t. this kernel parameter')
        for b in self._bart:
            out += b.hyperparams()
        return out


def _no_algebra_on_diff(a, b):
    if getattr(a, '_diff', None) is not None or getattr(b, '_diff', None) is not None:
        raise NotImplementedError("algebra on a kernel transformed by linop('diff')")


def _factor_depends_on(f, field, side):
    """ whether factor f depends on `field` (None: the coordinate of unstructured points) of argument `side` """
    if f.kind == _lib.K_CONSTANT:
        return False
    dim = f.dim[side]
    if dim is None or field is None:
        return True
    return field in ([dim] if isinstance(dim, str) else dim)


def deriv_field(deriv, labels):
    """ index into `labels` of the field of a first-order derivative, -1 for no derivative """
    deriv = Deriv(deriv)
    if not deriv:
        return -1
    if labels == [None]:
        if not deriv.implicit:
            raise ValueError(f'derivative {deriv!r} w.r.t. named fields of non-structured points')
        return 0
    if deriv.implicit:
        raise ValueError(f'implicit derivative {deriv!r} of structured points: name the field')
    out = []
    for field, _ in deriv:
        idx = [i for i, lab in enumerate(labels) if (lab[0] if isinstance(lab, tuple) else lab) == field]
        if not idx:
            raise ValueError(f'derivative field {field!r} not in x')
        if len(idx) != 1 or isinstance(labels[idx[0]], tuple):
            raise NotImplementedError(f'derivative w.r.t. {field!r}, which is not a single scalar field')
        out.append(idx[0])
    if len(out) != 1 or deriv.order != 1:
        raise NotImplementedError(f'derivative {deriv!r} of order > 1 on one argument')
    return out[0]


def _mulamp(a, b):
    if isinstance(a, torch.Tensor) or isinstance(b, torch.Tensor):
        return torch.as_tensor(a, dtype=torch.float64) * torch.as_tensor(b, dtype=torch.float64)
    return float(a) * float(b)


def _dimmask(labels, dim):
    full = (1 << len(labels)) - 1
    if dim is None:
        return full
    if labels == [None]:
        raise ValueError(f'cannot get dim={dim!r} from non-structured input')
    want = [dim] if isinstance(dim, str) else list(dim)
    mask = 0
    for i, lab in enumerate(labels):
        name = lab[0] if isinstance(lab, tuple) else lab
        if name in want:
            mask |= 1 << i
    for w in want:
        if not any((lab[0] if isinstance(lab, tuple) else lab) == w for lab in labels):
            raise KeyError(w)
    return mask


class Kernel(CrossKernel):
    """ symmetric positive semidefinite kernel """
    pass


class CrossStationaryKernel(CrossKernel):
    pass


class StationaryKernel(CrossStationaryKernel, Kernel):
    pass


class CrossIsotropicKernel(CrossStationaryKernel):
    pass


class IsotropicKernel(CrossIsotropicKernel, StationaryKernel):
    pass


_ORDER = [IsotropicKernel, StationaryKernel, Kernel, CrossIsotropicKernel, CrossStationaryKernel, CrossKernel]


def _common_class(a, b):
    """ most specific class of the hierarchy that both operands are instances of """
    for cls in _ORDER:
        if issubclass(a, cls) and issubclass(b, cls):
            return cls
    return CrossKernel


def _unsupported_decorator(name):
    def deco(*args, **kw):
        raise NotImplementedError(
            f'@{name}: user-defined Python kernel cores cannot be compiled into the fused CUDA Gram kernel; '
            'there is deliberately no CPU fallback (see DESIGN.md, boundary B2)')
    deco.__name__ = name
    return deco


kernel = _unsupported_decorator('kernel')
stationarykernel = _unsupported_decorator('stationarykernel')
isotropickernel = _unsupported_decorator('isotropickernel')
crosskernel = _unsupported_decorator('crosskernel')
crossstationarykernel = _unsupported_decorator('crossstationarykernel')
crossisotropickernel = _unsupported_decorator('crossisotropickernel')
