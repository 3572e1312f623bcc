"""The GP object: elements (points, user covariances, linear transformations), covariance block assembly,
decomposition cache, posterior and marginal likelihood.

Mirror of the parts of src/lsqfitgp/_GP/ on the fitting hot path:
  _gp.py:114-129        GP.__init__ keywords
  _elements.py:158-242  addx            :408-552 addcov         :248-406 addtransf / addlintransf
  _elements.py:554-649  _makecovblock_points / _lintransf_any / _covblock / _assemblecovblocks
  _elements.py:758-817  prior(raw=True)
  _compute.py:45-94     _solver         :96-136 _flatgiven      :138-334 pred / predfromdata / predfromfit
  _compute.py:336-422   _prior_decomp / marginal_likelihood     :430-516 decompose
Everything numeric runs on the device: Gram blocks are written by the CUDA Gram kernels directly into the
slices of the assembled matrix, `Kxx + ycov` is folded into the equilibration pass of the factorisation.

gvar is not available, so only the "raw" (arrays in, arrays out) interfaces exist.  Hyperparameters given as
torch tensors that require grad make `marginal_likelihood` return a differentiable torch scalar
(torch.autograd replaces the JAX tracing used by the reference, src/lsqfitgp/_fit.py:679-702).
"""

import math
import threading

import numpy
import torch

from . import _array
from . import _Kernel
from ._Deriv import Deriv
from . import _lib
from . import _linalg
from . import _ops
from . import _timing

__all__ = ['GP']

f64 = torch.float64


def _device():
    _lib.require_cuda()
    return torch.device('cuda', torch.cuda.current_device())


def _newself(meth):
    """ methods that modify the GP return a modified shallow clone (reference _GP/_base.py:86-104) """
    def newmeth(self, *args, **kw):
        new = self._clone()
        meth(new, *args, **kw)
        return new
    newmeth.__name__ = meth.__name__
    newmeth.__doc__ = meth.__doc__
    return newmeth


class _Element:
    shape = None

    @property
    def size(self):
        return math.prod(self.shape)


class _Points(_Element):
    def __init__(self, labels, xd, shape, deriv=None, dfield=-1):
        self.labels = labels
        self.xd = xd          # (ndim, n) float64 device tensor
        self.shape = shape
        self.deriv = Deriv(deriv)
        self.dfield = dfield  # index of the differentiated field in labels, -1: the process itself


def _plain_points(elem):
    """ points of the process itself (no derivative): what the fused single-key fast paths handle """
    return isinstance(elem, _Points) and elem.dfield < 0


class _LinTransf(_Element):
    def __init__(self, transf, keys, shape, tensors=None):
        self.transf = transf
        self.keys = keys
        self.shape = shape
        self.tensors = tensors  # dict key -> scalar/tensor when built by addtransf


class _Cov(_Element):
    def __init__(self, blocks, shape):
        self.blocks = blocks
        self.shape = shape


# ---------------------------------------------------------------------------------------------------------
# autograd nodes
# ---------------------------------------------------------------------------------------------------------

class _GramFn(torch.autograd.Function):
    """ K = kernel(x, y) as a differentiable function of the kernel hyperparameters and of the points xd, yd.
    backward = lgp_gram_iso_vjp: sum_ij G_ij dK_ij/dtheta without materialising dK, and lgp_gram_iso_xvjp for the points
    (reference: jax.vjp of the Gram build, src/lsqfitgp/_fit.py:687-702).  BART terms depend on the points only through
    integer bin indices: their contribution to the point gradient is 0, as under jax. """

    @staticmethod
    def forward(ctx, kern, xd, yd, labels, dfields, *params):
        ctx.kern, ctx.xd, ctx.yd, ctx.labels, ctx.dfields = kern, xd, yd, labels, dfields
        return kern._gram_device(xd, yd, labels, symmetric=xd is yd, dfields=dfields)

    @staticmethod
    def backward(ctx, G):
        kern, xd, yd, labels, dfields = ctx.kern, ctx.xd, ctx.yd, ctx.labels, ctx.dfields
        hyper = kern._hyperparams()
        need_x, need_y = ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        if (need_x or need_y) and dfields != (-1, -1):
            raise NotImplementedError(_NO_POINT_GRAD_DERIV)
        if torch.is_grad_enabled():   # create_graph: the gradient itself must be differentiable
            why = _no_second_order(hyper, dfields)
            if why is None and (need_x or need_y):
                why = _NO_POINT_SECOND_ORDER
            if why is None:
                return (None, None, None, None, None, *_gram_vjp_graph(kern, xd, yd, labels, G, hyper))
            with torch.no_grad():
                first = _GramFn.backward(ctx, G.detach())
            gpts = [gp for gp in first[1:3] if gp is not None]
            outs = _NoSecondOrder.apply(why, gpts + list(first[5:]), *[h[3] for h in hyper],
                                        *((xd, yd) if gpts else ()))
            it = iter(outs[:len(gpts)])
            gx = next(it) if first[1] is not None else None
            gy = next(it) if first[2] is not None else None
            return (None, gx, gy, None, None, *outs[len(gpts):])
        gx = gy = None
        if need_x or need_y:
            if kern._terms:
                descs, _ = kern._descriptor(labels)
                gx, gy = _ops.gram_iso_xvjp(descs, xd.detach(), yd.detach(), _ops.as_aligned(G.contiguous()),
                                            need_x=need_x, need_y=need_y)
            else:
                gx = torch.zeros_like(xd) if need_x else None
                gy = torch.zeros_like(yd) if need_y else None
        grads = []
        vjp = None
        if kern._terms:
            descs, index = kern._descriptor(labels)
            Ga = _ops.as_aligned(G.contiguous())
            if dfields != (-1, -1):
                vjp = _ops.gram_iso_deriv_vjp(descs, xd, yd, dfields[0], dfields[1], Ga).cpu()
            else:
                vjp = _ops.gram_iso_vjp_general(descs, xd, yd, Ga).cpu()
            pos = {tf: i for i, tf in enumerate(index)}
        bart_vjp = {}  # one fused pass per BART term: [d/d amp, d/d alpha, d/d beta]
        for kind, ti, fi, tensor in hyper:
            if kind == 'amp':
                g = vjp[pos[(ti, 0)], 0]
            elif kind == 'scale':
                g = vjp[pos[(ti, fi)], 1] / tensor.detach().cpu()
            elif kind == 'par1':
                g = vjp[pos[(ti, fi)], 2]
            elif kind in ('bart_amp', 'bart_alpha', 'bart_beta'):
                spec = ti
                if id(spec) not in bart_vjp:
                    bart_vjp[id(spec)] = spec.vjp_device(xd, yd, _ops.as_aligned(G.contiguous())).cpu()
                g = bart_vjp[id(spec)][('bart_amp', 'bart_alpha', 'bart_beta').index(kind)]
            else:  # pragma: no cover
                raise NotImplementedError(kind)
            grads.append(g.to(tensor.device, tensor.dtype).reshape(tensor.shape))
        return (None, gx, gy, None, None, *grads)

    @staticmethod
    def jvp(ctx, _kern, tx, ty, _labels, _dfields, *tangents):
        """ forward mode (torch.autograd.forward_ad): dK along the tangent of the hyperparameters, one pass of
        lgp_gram_iso_jvp, plus that of the points tx, ty (lgp_gram_iso_xjvp, accumulated); what jax.jacfwd of the Gram
        build gives the reference's Fisher path (_fit.py:676-683) """
        kern, xd, yd, labels, dfields = ctx.kern, ctx.xd, ctx.yd, ctx.labels, ctx.dfields
        hyper = kern._hyperparams()
        assert len(hyper) == len(tangents)
        # points that are not on the dual level arrive with a materialised zero tangent: it contributes nothing
        tx, ty = (None if t is None or not bool(torch.any(t != 0)) else t for t in (tx, ty))
        if (tx is not None or ty is not None) and dfields != (-1, -1):
            raise NotImplementedError(_NO_POINT_GRAD_DERIV)
        D = None
        if kern._terms:
            descs, index = kern._descriptor(labels)
            pos = {tf: i for i, tf in enumerate(index)}
            tan = numpy.zeros((len(descs), 3))
            for (kind, ti, fi, tensor), t in zip(hyper, tangents):
                if t is None or kind.startswith('bart_'):
                    continue
                tv = float(t.detach())
                if kind == 'amp':
                    tan[pos[(ti, 0)], 0] += tv
                elif kind == 'scale':
                    tan[pos[(ti, fi)], 1] += tv / float(tensor.detach())
                elif kind == 'par1':
                    tan[pos[(ti, fi)], 2] += tv
                else:  # pragma: no cover
                    raise NotImplementedError(kind)
            if dfields != (-1, -1):
                D = _ops.gram_iso_deriv_jvp(descs, xd, yd, dfields[0], dfields[1], tan)
            else:
                D = _ops.gram_iso_jvp(descs, xd, yd, tan)
            if tx is not None or ty is not None:
                _ops.gram_iso_xjvp(descs, xd.detach(), yd.detach(), tx, ty, D, accumulate=True)
        # BART terms: D += t_amp corr + t_alpha amp dcorr/dalpha + t_beta amp dcorr/dbeta, one kernel pass per term
        bart_tan = {}
        for (kind, ti, fi, tensor), t in zip(hyper, tangents):
            if kind.startswith('bart_') and t is not None:
                bart_tan.setdefault(id(ti), [ti, 0.0, 0.0, 0.0])[1 + ('bart_amp', 'bart_alpha', 'bart_beta').index(kind)] \
                    += float(t.detach())
        for spec, ta, tal, tbe in bart_tan.values():
            amp = float(spec.amp.detach() if isinstance(spec.amp, torch.Tensor) else spec.amp)
            need_d = tal != 0.0 or tbe != 0.0
            res = spec.gram_device(xd, yd, labels, deriv=need_d)
            Kb, dKa, dKb = res if need_d else (res, None, None)
            if D is None:
                D = torch.zeros(xd.shape[1], yd.shape[1], dtype=f64, device=xd.device)
                D = _ops.as_aligned(D)
            if ta != 0.0:
                _ops.axpby(ta / amp, Kb, 1.0, D)
            if tal != 0.0:
                _ops.axpby(tal, dKa, 1.0, D)
            if tbe != 0.0:
                _ops.axpby(tbe, dKb, 1.0, D)
        if D is None:
            D = torch.zeros(xd.shape[1], yd.shape[1], dtype=f64, device=xd.device)
        return D


_NO_POINT_GRAD_DERIV = ('gradients with respect to the points through a derivative-observation block are not '
                        'implemented: they need one more derivative order of the kernel')
_NO_POINT_SECOND_ORDER = ('second derivatives with respect to the points are not implemented: the point derivatives '
                          'of the Gram build are first-order only')


def _no_second_order(hyper, dfields):
    """ why the gradient of a Gram block with respect to `hyper` can not be differentiated again, or None """
    if any(kind.startswith('bart_') for kind, _, _, _ in hyper):
        return ('second derivatives through the BART kernel are not implemented: its alpha/beta derivatives are '
                'first-order only')
    if dfields != (-1, -1):
        return ('second derivatives of the marginal likelihood with derivative observations are not implemented: they '
                'would need the fourth derivative of the kernel core')
    return None


class _NoSecondOrder(torch.autograd.Function):
    """ passes first-order gradients through; differentiating them raises NotImplementedError(why) (the inputs
    `params` only attach the outputs to the graph, so that a second differentiation reaches this node) """

    @staticmethod
    def forward(ctx, why, values, *params):
        ctx.why = why
        return tuple(v.clone() for v in values)

    @staticmethod
    def backward(ctx, *grads):
        raise NotImplementedError(ctx.why)


def _gram_vjp_graph(kern, xd, yd, labels, G, hyper):
    """ gradients with respect to the tensors of `hyper` of sum_ij G_ij K_ij, as differentiable functions of G and of
    the hyperparameters: the per-factor contractions come from _GramVJPFn, their map to the user's tensors (the
    1/scale of d/d log scale) stays in the torch graph """
    params = [h[3] for h in hyper]
    _, index = kern._descriptor(labels)
    pos = {tf: i for i, tf in enumerate(index)}
    vjp = _GramVJPFn.apply(kern, xd, yd, labels, G, *params).cpu()
    grads = []
    for kind, ti, fi, tensor in hyper:
        if kind == 'amp':
            g = vjp[pos[(ti, 0)], 0]
        elif kind == 'scale':
            g = vjp[pos[(ti, fi)], 1] / tensor.cpu()
        elif kind == 'par1':
            g = vjp[pos[(ti, fi)], 2]
        else:  # pragma: no cover
            raise NotImplementedError(kind)
        grads.append(g.to(tensor.device, tensor.dtype).reshape(tensor.shape))
    return grads


class _GramVJPFn(torch.autograd.Function):
    """ (G, theta) -> (nfactors, 3) per-factor contractions sum_ij G_ij dK_ij/d(amp, log scale, par1): the backward of
    _GramFn as a differentiable function, for second derivatives.  Its backward, for a cotangent V on the contractions,
    gives G the matrix sum_f V_f dK/dtheta_f (lgp_gram_iso_jvp) and the hyperparameters the second-order contraction
    sum_ij G_ij d/dtheta (sum_f V_f dK_ij/dtheta_f) (lgp_gram_iso_hvp). """

    @staticmethod
    def forward(ctx, kern, xd, yd, labels, G, *params):
        ctx.kern, ctx.xd, ctx.yd, ctx.labels = kern, xd, yd, labels
        ctx.save_for_backward(G)
        descs, _ = kern._descriptor(labels)
        return _ops.gram_iso_vjp_general(descs, xd, yd, _ops.as_aligned(G.contiguous())).clone()

    @staticmethod
    def backward(ctx, V):
        kern, xd, yd, labels = ctx.kern, ctx.xd, ctx.yd, ctx.labels
        G, = ctx.saved_tensors
        descs, index = kern._descriptor(labels)
        tan = V.detach().cpu().numpy()
        gG = _ops.gram_iso_jvp(descs, xd, yd, tan) if ctx.needs_input_grad[4] else None
        hvp = _ops.gram_iso_hvp(descs, xd, yd, _ops.as_aligned(G.detach().contiguous()), tan).cpu()
        pos = {tf: i for i, tf in enumerate(index)}
        grads = []
        for kind, ti, fi, tensor in kern._hyperparams():
            if kind == 'amp':
                g = hvp[pos[(ti, 0)], 0]
            elif kind == 'scale':
                g = hvp[pos[(ti, fi)], 1] / tensor.detach().cpu()
            else:
                g = hvp[pos[(ti, fi)], 2]
            grads.append(g.to(tensor.device, tensor.dtype).reshape(tensor.shape))
        return (None, None, None, None, gG, *grads)


class _NegLogDensityGradFn(torch.autograd.Function):
    """ (K, r, g) -> (g/2 (K^-1 - b b'), g b), b = K^-1 r: the backward of _NegLogDensityFn as a differentiable function,
    for second derivatives.  K^-1 is the inverse of the jittered matrix that `dec` factors, as in the first-order
    backward; K itself only routes the cotangent to the graph that built it.  For cotangents (W, w), W symmetrised:
      K: g [-1/2 K^-1 W K^-1 + 1/2 (K^-1 W b b' + b b' W K^-1) - 1/2 (K^-1 w b' + b w' K^-1)]
      r: g (K^-1 w - K^-1 W b)          g: 1/2 <W, K^-1 - b b'> + <w, b>
    with K^-1 W K^-1 as two DMMA GEMMs, the second one on its lower triangle only. """

    @staticmethod
    def forward(ctx, dec, a, K, r, g):
        b = dec._solve(a[:, None], True)[:, 0].contiguous()
        low = dec.inverse_lower()
        ctx.dec, ctx.low, ctx.b, ctx.g = dec, low, b, float(g)
        return _ops.sym_expand_sub(low, b, scale=0.5 * float(g)), g * b

    @staticmethod
    def backward(ctx, W, w):
        low, b, g = ctx.low, ctx.b, ctx.g
        n = b.shape[0]
        dev = b.device
        Kinv = _ops.sym_expand_sub(low, None)
        d = torch.zeros(n, dtype=f64, device=dev)    # K^-1 W b - K^-1 w
        cot_g = torch.zeros((), dtype=f64, device=dev)
        cotK = None
        if W is not None:
            W = _ops.as_aligned(0.5 * (W + W.T))
            M1 = _ops.aligned_empty(n, n, dev)
            _ops.dgemm(Kinv, W, M1, a_kmajor=True, b_kmajor=True, M=n, N=n, K=n, flags=_lib.GEMM_BETA0)
            M2 = _ops.aligned_empty(n, n, dev)
            _ops.dgemm(M1, Kinv, M2, a_kmajor=True, b_kmajor=True, M=n, N=n, K=n,
                       flags=_lib.GEMM_BETA0 | _lib.GEMM_LOWER)
            del M1
            Wb = _ops.dgemv(W, b, torch.zeros(n, dtype=f64, device=dev))
            _ops.dgemv(Kinv, Wb, d)
            cot_g = cot_g + 0.5 * (_ops.symlower_dot(low, b, W)[0])
            cotK = _ops.sym_expand_sub(M2, None, scale=-0.5 * g)
            del M2
        if w is not None:
            w = w.contiguous()
            _ops.dgemv(Kinv, w, d, alpha=-1.0)
            cot_g = cot_g + torch.dot(w, b)
        if cotK is None:
            cotK = torch.zeros((n, n), dtype=f64, device=dev)
        cotK += (0.5 * g) * (torch.outer(d, b) + torch.outer(b, d))
        return None, None, cotK, -g * d, cot_g


class _NegLogDensityFn(torch.autograd.Function):
    """ value = 1/2 (n log 2pi + log det K + r' K^-1 r)  (reference _decomp.py:484-488);
    backward: dvalue/dK = 1/2 (K^-1 - b b'), dvalue/dr = b, b = K^-1 r (reference _decomp.py:505-512). """

    @staticmethod
    def forward(ctx, K, r, kw):
        _timing.mark('gp&cov')
        dec = _linalg.Chol(K, **kw)
        _timing.mark('decomp')
        ldq, a = dec.logdet_quad(r)
        ctx.dec, ctx.a = dec, a
        ctx.save_for_backward(K, r)
        n = dec.n
        half = torch.tensor(0.5, dtype=f64, device=K.device)
        return half * (n * math.log(2 * math.pi) + 2 * ldq[0] + ldq[1])

    @staticmethod
    def backward(ctx, g):
        dec, a = ctx.dec, ctx.a
        if torch.is_grad_enabled():   # create_graph: the gradient itself must be differentiable
            K, r = ctx.saved_tensors
            gK, gr = _NegLogDensityGradFn.apply(dec, a, K, r, g)
            return gK if ctx.needs_input_grad[0] else None, gr if ctx.needs_input_grad[1] else None, None
        b = dec._solve(a[:, None], True)[:, 0]
        gK = gr = None
        if ctx.needs_input_grad[0]:
            # g/2 (K^-1 - b b') as a full matrix, one kernel pass over the lower triangle of the inverse
            gK = _ops.sym_expand_sub(dec.inverse_lower(), b.contiguous(), scale=0.5 * float(g))
        if ctx.needs_input_grad[1]:
            gr = g * b
        return gK, gr, None


_SIDE_STREAMS = {}
_SIDE_LOCK = threading.Lock()


def _side_stream_for(main):
    """ one persistent side stream per caller stream: its allocator pool keeps the inverse buffers warm from one
    evaluation to the next (a fresh stream per call would allocate 2 n^2 doubles in a new pool every time) """
    key = (main.device_index, main.cuda_stream)
    with _SIDE_LOCK:
        side = _SIDE_STREAMS.get(key)
        if side is None:
            side = _SIDE_STREAMS[key] = torch.cuda.Stream(torch.device('cuda', main.device_index))
        return side


def _fusable(kw):
    """ solver keywords the fused Gram -> factor path understands """
    return set(kw) <= {'epsrel', 'epsabs'}


class _FusedNegLogMLFn(torch.autograd.Function):
    """ Gram -> Chol -> value in one node for the common case (one set of points, kernel-only covariance):
    the backward pass feeds the lower triangle of K^-1 and b = K^-1 r straight into the symmetric Gram-VJP
    kernel, so no dense n x n gradient matrix is ever formed (the two dK_vjp calls of the reference,
    _decomp.py:505-509, collapse into one pass over the lower triangle).  The points xd are differentiable too: their
    gradient is one more pass over the same triangle (lgp_gram_iso_xvjp). """

    @staticmethod
    def forward(ctx, kern, xd, labels, r, kw, *params):
        # the gradient will need K^-1: factorisation and inverse-from-factor in ONE library call, the inverse on a
        # persistent side stream (the latency-bound triangular solves below overlap its GEMMs)
        need_inverse = any(ctx.needs_input_grad[5:]) or ctx.needs_input_grad[1]
        side = _side_stream_for(torch.cuda.current_stream()) if need_inverse else None
        # kernels of the fast family: the Gram build writes the equilibrated lower triangle and the Gershgorin partial
        # sums straight into the factor's storage (K itself is never materialised)
        descs, _ = kern._descriptor(labels)
        dec = _linalg.Chol._from_kernel(descs, xd, _inverse_stream=side, **kw) if _fusable(kw) else None
        if dec is None:
            K = kern._gram_device(xd, xd, labels, symmetric=True)
            _timing.mark('gp&cov')
            dec = _linalg.Chol(K, _inverse_stream=side, **kw) if side is not None else _linalg.Chol(K, **kw)
            del K
        else:
            _timing.mark('gp&cov')
        _timing.mark('decomp')
        ldq, a = dec.logdet_quad(r)
        ctx.kern, ctx.xd, ctx.labels, ctx.dec, ctx.a = kern, xd, labels, dec, a
        ctx.save_for_backward(r)
        half = torch.tensor(0.5, dtype=f64, device=xd.device)
        return half * (dec.n * math.log(2 * math.pi) + 2 * ldq[0] + ldq[1])

    @staticmethod
    def backward(ctx, g):
        kern, xd, labels, dec, a = ctx.kern, ctx.xd, ctx.labels, ctx.dec, ctx.a
        if torch.is_grad_enabled() and ctx.needs_input_grad[1]:
            # create_graph with differentiable points: first order only
            r, = ctx.saved_tensors
            with torch.no_grad():
                first = _FusedNegLogMLFn.backward(ctx, g.detach())
            keep = [i for i in (1, 3) if first[i] is not None] + list(range(5, len(first)))
            outs = _NoSecondOrder.apply(_NO_POINT_SECOND_ORDER, [first[i] for i in keep],
                                        *[h[3] for h in kern._hyperparams()], xd, r)
            res = [None] * len(first)
            for i, o in zip(keep, outs):
                res[i] = o
            return tuple(res)
        if torch.is_grad_enabled():
            # create_graph: the same second order as the assembled route, through K built here (never on the
            # first-order path) and the lower triangle of K^-1 kept by `dec`
            r, = ctx.saved_tensors
            hyper = kern._hyperparams()
            K = _GramFn.apply(kern, xd, xd, labels, (-1, -1), *[h[3] for h in hyper])
            gK, gr = _NegLogDensityGradFn.apply(dec, a, K, r, g)
            grads = _gram_vjp_graph(kern, xd, xd, labels, gK, hyper) if hyper else []
            return (None, None, None, gr if ctx.needs_input_grad[3] else None, None, *grads)
        b = dec._solve(a[:, None], True)[:, 0].contiguous()
        gr = g * b if ctx.needs_input_grad[3] else None
        hyper = kern._hyperparams()
        grads = []
        gx = None
        if hyper or ctx.needs_input_grad[1]:
            low = dec.inverse_lower()   # joins the side stream if the inverse was started in forward
            descs, index = kern._descriptor(labels)
            if ctx.needs_input_grad[1]:
                # the G of the hyperparameters' contraction: g/2 w_ij (K^-1 - b b')_ij on the lower triangle
                gx = (0.5 * g) * _ops.gram_iso_xvjp(descs, xd.detach(), None, low, b, symlower=True)[0]
            if hyper:
                vjp = (0.5 * _ops.gram_iso_vjp(descs, xd, low, b)).cpu()
            del low
            dec._low = None   # 8 n^2 bytes: not needed again
        if hyper:
            pos = {tf: i for i, tf in enumerate(index)}
            gc = g.cpu()
            for kind, ti, fi, tensor in hyper:
                if kind == 'amp':
                    v = vjp[pos[(ti, 0)], 0]
                elif kind == 'scale':
                    v = vjp[pos[(ti, fi)], 1] / tensor.detach().cpu()
                elif kind == 'par1':
                    v = vjp[pos[(ti, fi)], 2]
                else:  # pragma: no cover
                    raise NotImplementedError(kind)
                grads.append((gc * v).to(tensor.device, tensor.dtype).reshape(tensor.shape))
        return (None, gx, None, gr, None, *grads)


class GP:
    """Object that represents a Gaussian process over arbitrary input.

    Parameters follow lsqfitgp.GP (reference _GP/_gp.py:114-129).  `checkpos` is accepted but the LOBPCG
    positivity check is not run (the reference skips it too whenever the code is traced).
    """

    def __init__(self, covfun=None, *, solver='chol', checkpos=True, checksym=True, checkfinite=True, checklin=True,
                 posepsfac=1, halfmatrix=False, **kw):
        if covfun is not None and not isinstance(covfun, _Kernel.Kernel):
            raise TypeError('covariance function must be of class Kernel')
        self._covfun = covfun
        self._elements = {}       # key -> _Element
        self._covblocks = {}      # (key, key) -> device matrix
        self._decompcache = {}    # tuple of keys -> Decomposition
        self._dtype_names = None
        self._checkpos = bool(checkpos)
        self._posepsfac = float(posepsfac)
        self._checksym = bool(checksym)
        self._checkfinite = bool(checkfinite)
        self._checklin = bool(checklin)
        self._halfmatrix = bool(halfmatrix)
        if self._halfmatrix:
            assert not self._checksym, 'halfmatrix=True requires checksym=False'
        decomp = self._getdecomp(solver)
        self._solver_name = solver
        self._solverkw = dict(kw)
        self._decompclass = lambda K, **kwargs: decomp(K, **kwargs, **self._solverkw)
        self._decompbase = decomp

    def _clone(self):
        new = object.__new__(type(self))
        new.__dict__.update(self.__dict__)
        new._elements = dict(self._elements)
        new._covblocks = dict(self._covblocks)
        new._decompcache = dict(self._decompcache)
        return new

    # ------------------------------------------------------------------------------------------------
    # elements
    # ------------------------------------------------------------------------------------------------
    @_newself
    def addx(self, x, key=None, *, deriv=0, proc=None):
        """ Add points where the Gaussian process is evaluated (reference _elements.py:158-242).
        `deriv` (see `Deriv`): the points are of the first derivative of the process w.r.t. that field (order <= 1). """
        deriv = Deriv(deriv)
        if proc is not None:
            raise NotImplementedError('multiple processes')
        if self._covfun is None:
            raise KeyError('process named DefaultProcess not found')
        if hasattr(x, 'keys') and not isinstance(x, _array.StructuredArray):
            if key is not None:
                raise ValueError('can not specify key if x is a dictionary')
            if None in x:
                raise ValueError('None key in x not allowed')
        else:
            if key is None:
                raise ValueError('x is not dictionary but key is None')
            x = {key: x}
        dev = _device()
        for key in x:
            if key in self._elements:
                raise KeyError('key {!r} already in GP'.format(key))
            labels, data, shape = _array.columns_of(x[key])
            names = tuple(labels)
            if self._dtype_names is not None and self._dtype_names != names:
                raise TypeError(f'x[{key!r}] has fields {names!r} not compatible with {self._dtype_names!r}')
            dfield = _Kernel.deriv_field(deriv, labels) if deriv.order <= 1 else None
            self._covfun._check_derivable(deriv, 0)
            self._dtype_names = names
            if isinstance(data, torch.Tensor):
                # points given as torch tensors stay on their autograd graph (and on a forward-mode dual level): the
                # marginal likelihood is then differentiable with respect to them
                xd = data.to(dev).contiguous()
            else:
                xd = torch.from_numpy(numpy.ascontiguousarray(data)).to(dev)
            self._elements[key] = _Points(labels, xd, tuple(shape), deriv, dfield)

    @_newself
    def addcov(self, covblocks, key=None, *, decomps=None):
        """ Add user-defined covariance blocks (reference _elements.py:408-552) """
        if hasattr(covblocks, 'keys'):
            if key is not None:
                raise ValueError('can not specify key if covblocks is a dictionary')
            if None in covblocks:
                raise ValueError('None key in covblocks not allowed')
            if decomps is not None and not hasattr(decomps, 'keys'):
                raise TypeError('covblocks is dictionary but decomps is not')
        else:
            if key is None:
                raise ValueError('covblocks is not dictionary but key is None')
            covblocks = {(key, key): covblocks}
            if decomps is not None:
                decomps = {key: decomps}
        if decomps is None:
            decomps = {}
        dev = _device()
        shapes, preblocks = {}, {}
        for keys, block in covblocks.items():
            for k in keys:
                if k in self._elements:
                    raise KeyError(f'key {k!r} already in GP')
            xkey, ykey = keys
            if block is None:
                raise TypeError(f'block {keys!r} is None')
            if isinstance(block, torch.Tensor):
                block = block.to(dev, f64)
            else:
                block = torch.as_tensor(numpy.asarray(block, dtype=numpy.float64)).to(dev)
            if xkey == ykey:
                if block.ndim % 2 == 1:
                    raise ValueError(f'diagonal block {xkey!r} has odd number of axes')
                half = block.ndim // 2
                head, tail = tuple(block.shape[:half]), tuple(block.shape[half:])
                if head != tail:
                    raise ValueError(f'shape {tuple(block.shape)!r} of diagonal block {xkey!r} is not symmetric')
                shapes[xkey] = head
            preblocks[keys] = block
        for k, dec in decomps.items():
            if k not in shapes:
                raise KeyError(f'key {k!r} in decomps not found in diagonal blocks')
            if not isinstance(dec, _linalg.Decomposition):
                raise TypeError(f'decomps[{k!r}] = {dec!r} is not a decomposition')
            if dec.n != math.prod(shapes[k]):
                raise ValueError(f'decomposition matrix size {dec.n} != diagonal block size for key {k!r}')
        blocks = {}
        for keys, block in preblocks.items():
            if self._checkfinite and not bool(torch.all(torch.isfinite(block))):
                raise ValueError(f'block {keys!r} not finite')
            xkey, ykey = keys
            if xkey == ykey:
                size = math.prod(shapes[xkey])
                block = block.reshape(size, size)
                if self._checksym and not bool(torch.allclose(block, block.T)):
                    raise ValueError(f'diagonal block {xkey!r} is not symmetric')
                blocks[keys] = block
            else:
                for k in keys:
                    if k not in shapes:
                        raise KeyError(f'key {k!r} from off-diagonal block {keys!r} not found in diagonal blocks')
                eshape = shapes[xkey] + shapes[ykey]
                if tuple(block.shape) != eshape:
                    raise ValueError(f'shape {tuple(block.shape)!r} of block {keys!r} is not {eshape!r} as expected '
                                     'from diagonal blocks')
                block = block.reshape(math.prod(shapes[xkey]), math.prod(shapes[ykey]))
                blocks[keys] = block
                if keys[::-1] not in preblocks:
                    blocks[keys[::-1]] = block.T
        if self._checksym:
            for keys, block in blocks.items():
                if keys[0] != keys[1] and not bool(torch.allclose(block.T, blocks[keys[::-1]])):
                    raise ValueError(f'block {keys!r} is not the transpose of block {keys[::-1]!r}')
        for k, shape in shapes.items():
            self._elements[k] = _Cov(blocks, shape)
            dec = decomps.get(k)
            if dec is not None:
                self._decompcache[k,] = dec

    @_newself
    def addtransf(self, tensors, key, *, axes=1):
        """ Linear transformation sum_k tensordot(tensors[k], process[k], axes) (reference _elements.py:248-330) """
        assert isinstance(axes, int) and axes >= 0, axes
        if key is None:
            raise ValueError('key can not be None')
        if key in self._elements:
            raise KeyError(f'key {key!r} already in GP')
        for k in tensors:
            if k not in self._elements:
                raise KeyError(k)
        if len(tensors) == 0:
            raise ValueError('empty tensors, undetermined output shape')
        dev = _device()
        tens = {}
        shapes = []
        for k, t in tensors.items():
            if isinstance(t, torch.Tensor):
                t = t.to(dev, f64)
            else:
                t = torch.as_tensor(numpy.asarray(t, dtype=numpy.float64)).to(dev)
            if self._checkfinite and not bool(torch.all(torch.isfinite(t))):
                raise ValueError(f'tensors[{k!r}] contains infs/nans')
            rshape = self._elements[k].shape
            if t.ndim and tuple(t.shape[t.ndim - axes:]) != tuple(rshape[:axes]):
                raise ValueError(f'tensors[{k!r}].shape = {tuple(t.shape)!r} can not be multiplied with shape '
                                 f'{rshape!r} with {axes}-axes contraction')
            tens[k] = t
            shapes.append(tuple(t.shape[:t.ndim - axes]) + tuple(rshape[axes:]) if t.ndim else tuple(rshape))
        try:
            shape = tuple(numpy.broadcast_shapes(*shapes))
        except ValueError:
            raise ValueError('can not broadcast tensors with shapes [' + ', '.join(repr(tuple(t.shape)) for t in
                             tens.values()) + '] contracted with arrays with shapes [' +
                             ', '.join(repr(self._elements[k].shape) for k in tens) + ']')

        def equiv_lintransf(*args):
            out = None
            for a, t in zip(args, tens.values()):
                b = torch.tensordot(t, a, axes) if t.ndim else t * a
                out = b if out is None else out + b
            return out
        self._elements[key] = _LinTransf(equiv_lintransf, list(tens.keys()), shape, tensors=tens)

    @_newself
    def addlintransf(self, transf, keys, key, *, checklin=None):
        """ Finite linear transformation given as a function of torch tensors; the function receives each
        element with one extra trailing (batch) axis (reference _elements.py:332-406 uses jax.vmap(-1, -1)). """
        if key is None:
            raise ValueError('key can not be None')
        if key in self._elements:
            raise KeyError(f'key {key!r} already in GP')
        for k in keys:
            if k not in self._elements:
                raise KeyError(k)
        dev = _device()
        probe = [torch.zeros(self._elements[k].shape + (1,), dtype=f64, device=dev) for k in keys]
        out = transf(*probe)
        shape = tuple(out.shape[:-1])
        if checklin is None:
            checklin = self._checklin
        if checklin:
            g = torch.Generator(device='cpu').manual_seed(202310)
            a = [torch.randn(p.shape, generator=g, dtype=f64).to(dev) for p in probe]
            b = [torch.randn(p.shape, generator=g, dtype=f64).to(dev) for p in probe]
            lhs = transf(*[2.5 * u - 1.5 * v for u, v in zip(a, b)])
            rhs = 2.5 * transf(*a) - 1.5 * transf(*b)
            if not bool(torch.allclose(lhs, rhs, rtol=1e-9, atol=1e-12)):
                raise RuntimeError('the transformation is not linear')
        self._elements[key] = _LinTransf(transf, list(keys), shape)

    # ------------------------------------------------------------------------------------------------
    # covariance blocks
    # ------------------------------------------------------------------------------------------------
    def _grad_mode(self):
        return self._covfun is not None and torch.is_grad_enabled() and (
            bool(self._covfun._hyperparams()) or any(isinstance(e, _Points) and e.xd.requires_grad
                                                     for e in self._elements.values()))

    def _makecovblock_points(self, xkey, ykey, out=None):
        x = self._elements[xkey]
        y = self._elements[ykey]
        kern = self._covfun
        yd = x.xd if y is x else y.xd
        dfields = (x.dfield, y.dfield)
        if self._grad_mode():
            params = [h[3] for h in kern._hyperparams()]
            cov = _GramFn.apply(kern, x.xd, yd, x.labels, dfields, *params)
            if out is not None:
                raise RuntimeError('internal: out= in grad mode')
            return cov
        return kern._gram_device(x.xd, yd, x.labels, out=out, symmetric=y is x, dfields=dfields)

    def _makecovblock_lintransf_any(self, xkey, ykey):
        x = self._elements[xkey]
        y = self._elements[ykey]
        covs = []
        for k in x.keys:
            elem = self._elements[k]
            cov = self._covblock(k, ykey)
            covs.append(cov.reshape(elem.shape + (y.size,)))
        cov = x.transf(*covs)
        assert tuple(cov.shape) == tuple(x.shape) + (y.size,), (cov.shape, x.shape, y.size)
        return cov.reshape(x.size, y.size)

    # ---- scalar linear combinations (addtransf with scalar tensors, e.g. the bayestree.bart recipe
    # train = trainmean + trainnoise + mean): cov(x, y) = sum_ab c_a c_b cov(a, b) accumulated block by block straight
    # into one matrix, structurally zero blocks skipped (the generic path materialises every block, zeros included, and
    # sums them with one pass each: reference _elements.py:581-601)
    def _expand_scalar(self, key):
        """ [(coefficient, base key), ...] if `key` is a scalar linear combination of non-transformed elements with
        plain-number coefficients, else None """
        e = self._elements[key]
        if not isinstance(e, _LinTransf):
            return [(1.0, key)]
        if e.tensors is None:
            return None
        out = []
        for k, t in e.tensors.items():
            if t.ndim != 0 or t.requires_grad:
                return None
            sub = self._expand_scalar(k)
            if sub is None:
                return None
            c = float(t)
            out += [(c * cs, ks) for cs, ks in sub]
        return out

    def _scalar_shapes_ok(self, key, parts):
        """ every base element of the combination has the size of the result or size 1 (broadcast scalar) """
        size = self._elements[key].size
        return all(self._elements[k].size in (size, 1) for _, k in parts)

    def _structurally_zero(self, a, b):
        ea, eb = self._elements[a], self._elements[b]
        if isinstance(ea, _Points) and isinstance(eb, _Points):
            return False
        if isinstance(ea, _Cov) and isinstance(eb, _Cov):
            return not (ea.blocks is eb.blocks and (a, b) in ea.blocks)
        return True   # points and user covariances are independent

    def _makecovblock_scalar_combination(self, xkey, ykey, xs, ys):
        x, y = self._elements[xkey], self._elements[ykey]
        n, m = x.size, y.size
        grad = self._grad_mode() or any(getattr(b, 'requires_grad', False) for e in self._elements.values()
                                        if isinstance(e, _Cov) for b in e.blocks.values())
        acc = None
        for ca, a in xs:
            for cb, b in ys:
                if self._structurally_zero(a, b) or ca * cb == 0.0:
                    continue
                blk = self._covblock(a, b)
                c = ca * cb
                if grad or blk.requires_grad:
                    term = blk * c if c != 1.0 else blk
                    if tuple(term.shape) != (n, m):
                        term = term.expand(n, m)
                    acc = term if acc is None else acc + term
                    continue
                if acc is None:
                    acc = _ops.aligned_empty(n, m, _device(), zero=True)
                if tuple(blk.shape) == (n, m):
                    _ops.axpby(c, blk if blk.stride(1) == 1 else blk.contiguous(), 1.0, acc)
                elif blk.numel() == 1:
                    _ops.add_scalar(acc, c * float(blk.reshape(())))
                else:
                    acc.add_(blk.expand(n, m), alpha=c)   # other broadcast patterns: rare, generic
        if acc is None:
            acc = torch.zeros((n, m), dtype=f64, device=_device())
        return acc

    def _makecovblock(self, xkey, ykey, out=None):
        x = self._elements[xkey]
        y = self._elements[ykey]
        xs = ys = None
        if isinstance(x, _LinTransf) or isinstance(y, _LinTransf):
            xs, ys = self._expand_scalar(xkey), self._expand_scalar(ykey)
        if isinstance(x, _Points) and isinstance(y, _Points):
            cov = self._makecovblock_points(xkey, ykey, out=out)
        elif xs is not None and ys is not None and self._scalar_shapes_ok(xkey, xs) and self._scalar_shapes_ok(ykey, ys):
            cov = self._makecovblock_scalar_combination(xkey, ykey, xs, ys)
        elif isinstance(x, _LinTransf):
            cov = self._makecovblock_lintransf_any(xkey, ykey)
        elif isinstance(y, _LinTransf):
            cov = self._makecovblock_lintransf_any(ykey, xkey).T
        elif isinstance(x, _Cov) and isinstance(y, _Cov) and x.blocks is y.blocks and (xkey, ykey) in x.blocks:
            cov = x.blocks[xkey, ykey]
        else:
            cov = torch.zeros((x.size, y.size), dtype=f64, device=_device())
        if self._checkfinite and not cov.requires_grad and not bool(torch.all(torch.isfinite(cov))):
            raise RuntimeError(f'covariance block {(xkey, ykey)!r} is not finite')
        if self._checksym and xkey == ykey and not cov.requires_grad and not bool(torch.allclose(cov, cov.T)):
            raise RuntimeError(f'covariance block {(xkey, ykey)!r} is not symmetric')
        return cov

    def _covblock(self, row, col, out=None):
        if self._grad_mode():
            return self._makecovblock(row, col)  # no caching of graph-attached blocks
        if (row, col) not in self._covblocks:
            block = self._makecovblock(row, col, out=out)
            if row != col:
                self._covblocks[col, row] = block.T
            self._covblocks[row, col] = block
        return self._covblocks[row, col]

    def _assemblecovblocks(self, rowkeys, colkeys=None):
        """ block matrix of the covariances between rowkeys and colkeys (reference _elements.py:642-649);
        Gram blocks of points are written by the CUDA kernel directly into their slice """
        if colkeys is None:
            colkeys = rowkeys
        rowkeys, colkeys = list(rowkeys), list(colkeys)
        if len(rowkeys) == 1 and len(colkeys) == 1:
            return self._covblock(rowkeys[0], colkeys[0])
        if self._grad_mode():
            return torch.cat([torch.cat([self._covblock(r, c) for c in colkeys], 1) for r in rowkeys], 0)
        rs = [self._elements[k].size for k in rowkeys]
        cs = [self._elements[k].size for k in colkeys]
        out = _ops.aligned_empty(sum(rs), sum(cs), _device())
        r0 = 0
        for r, nr in zip(rowkeys, rs):
            c0 = 0
            for c, nc in zip(colkeys, cs):
                view = out[r0:r0 + nr, c0:c0 + nc]
                if (r, c) in self._covblocks:
                    view.copy_(self._covblocks[r, c])
                elif (isinstance(self._elements[r], _Points) and isinstance(self._elements[c], _Points)
                      and c0 % 2 == 0):
                    self._covblock(r, c, out=view)
                else:
                    view.copy_(self._covblock(r, c))
                c0 += nc
            r0 += nr
        return out

    # ------------------------------------------------------------------------------------------------
    # prior
    # ------------------------------------------------------------------------------------------------
    def prior(self, key=None, *, raw=False):
        """ Prior covariance (raw=True only: there is no gvar here; reference _elements.py:758-817) """
        if not raw:
            raise NotImplementedError('prior(raw=False) needs gvar; use raw=True to get the covariance matrix')
        if key is None:
            outkeys = list(self._elements)
        elif isinstance(key, list):
            outkeys = key
        else:
            elem = self._elements[key]
            cov = self._covblock(key, key)
            return cov.detach().cpu().numpy().reshape(elem.shape + elem.shape)
        return {
            (row, col): self._covblock(row, col).detach().cpu().numpy().reshape(
                self._elements[row].shape + self._elements[col].shape)
            for row in outkeys for col in outkeys
        }

    # ------------------------------------------------------------------------------------------------
    # compute
    # ------------------------------------------------------------------------------------------------
    def _solver(self, keys, ycov=None, *, covtransf=None, **kw):
        """ decomposition of the covariance of `keys` plus ycov (reference _compute.py:45-94) """
        keys = tuple(keys)
        if ycov is None:
            cache = self._decompcache.get(keys)
            if cache is not None:
                return cache
        if (hasattr(self._decompbase, 'from_kernel') and len(keys) == 1 and ycov is None and not covtransf
                and _plain_points(self._elements[keys[0]]) and self._covfun._terms and not self._covfun._bart
                and (keys[0], keys[0]) not in self._covblocks):
            # distributed solver on one set of points with a kernel-only covariance: every rank generates its own tiles
            # from the replicated points; the n x n matrix is never assembled (the case that outgrows one GPU)
            elem = self._elements[keys[0]]
            descs, _ = self._covfun._descriptor(elem.labels)
            _timing.mark('gp&cov')
            skw = dict(self._solverkw)
            skw.update(kw)
            decomp = self._decompbase.from_kernel(descs, elem.xd, **skw)
            _timing.mark('decomp')
            self._decompcache[keys] = decomp
            return decomp
        if (self._solver_name == 'chol' and len(keys) == 1 and ycov is None and not covtransf
                and _plain_points(self._elements[keys[0]]) and self._covfun is not None and self._covfun._terms
                and not self._covfun._bart and (keys[0], keys[0]) not in self._covblocks and not self._grad_mode()):
            # one set of points, kernel-only covariance, matrix not built yet: Gram build fused with the equilibration pass
            # of the factorisation (lgp_gram_iso_prepare), for the kernels of the fast family.  The finiteness check of the
            # block moves to the points (a finite kernel of finite points is finite); anything else takes the usual path,
            # which builds the block, checks it and reports the error
            elem = self._elements[keys[0]]
            skw = dict(self._solverkw)
            skw.update(kw)
            if _fusable(skw) and (not self._checkfinite or bool(torch.all(torch.isfinite(elem.xd)))):
                descs, _ = self._covfun._descriptor(elem.labels)
                if all(math.isfinite(float(v)) for d in descs for v in d.values()):
                    decomp = _linalg.Chol._from_kernel(descs, elem.xd, **skw)
                    if decomp is not None:
                        _timing.mark('gp&cov')
                        _timing.mark('decomp')
                        self._decompcache[keys] = decomp
                        return decomp
        Kxx = self._assemblecovblocks(keys)
        if covtransf:
            if ycov is not None:
                Kxx = Kxx + ycov
                ycov = None
            Kxx = covtransf(Kxx)
        _timing.mark('gp&cov')
        if ycov is not None:
            decomp = self._decompclass(Kxx, _addmat=ycov, **kw)  # Kxx + ycov fused into the equilibration pass
        else:
            decomp = self._decompclass(Kxx, **kw)
        _timing.mark('decomp')
        if ycov is None and not covtransf:
            self._decompcache[keys] = decomp
        return decomp

    def _flatgiven(self, given, givencov):
        if not hasattr(given, 'keys'):
            raise TypeError('`given` must be dict')
        gcblack = givencov is None or isinstance(givencov, _linalg.Decomposition)
        if not gcblack and not hasattr(givencov, 'keys'):
            raise TypeError('`givenconv` must be None, dict or Decomposition')
        dev = _device()
        ylist, keylist = [], []
        for key, l in given.items():
            if key not in self._elements:
                raise KeyError(key)
            if isinstance(l, torch.Tensor):
                l = l.to(dev, f64)
            else:
                l = numpy.asarray(l)
                if l.dtype == object:
                    raise NotImplementedError('given contains objects (gvars): pass means and `givencov` instead')
                if not numpy.issubdtype(l.dtype, numpy.number):
                    raise TypeError('given[{!r}] has non-numerical dtype {!r}'.format(key, l.dtype))
                l = torch.as_tensor(l.astype(numpy.float64)).to(dev)
            shape = self._elements[key].shape
            if tuple(l.shape) != tuple(shape):
                raise ValueError('given[{!r}] has shape {!r} different from shape {!r}'.format(
                    key, tuple(l.shape), shape))
            ylist.append(l.reshape(-1))
            keylist.append(key)
        if gcblack:
            covblocks = givencov
        else:
            def get(i, j):
                b = givencov[keylist[i], keylist[j]]
                if isinstance(b, torch.Tensor):
                    b = b.to(dev, f64)
                else:
                    b = torch.as_tensor(numpy.asarray(b, dtype=numpy.float64)).to(dev)
                return b.reshape(ylist[i].shape + ylist[j].shape)
            covblocks = [[get(i, j) for j in range(len(keylist))] for i in range(len(keylist))]
        return ylist, keylist, covblocks

    @staticmethod
    def _block(blocks):
        if len(blocks) == 1 and len(blocks[0]) == 1:
            return blocks[0][0]
        return torch.cat([torch.cat(row, 1) for row in blocks], 0)

    def _check_ymean(self, ymean):
        if self._checkfinite and not ymean.requires_grad and not bool(torch.all(torch.isfinite(ymean))):
            raise ValueError('mean of `given` is not finite')

    def _check_ycov(self, ycov):
        if ycov is None or isinstance(ycov, _linalg.Decomposition) or ycov.requires_grad:
            return
        if self._checkfinite and not bool(torch.all(torch.isfinite(ycov))):
            raise ValueError('covariance matrix of `given` is not finite')
        if self._checksym and not bool(torch.allclose(ycov, ycov.T)):
            raise ValueError('covariance matrix of `given` is not symmetric')

    def _slices(self, keys):
        sizes = [self._elements[k].size for k in keys]
        stops = numpy.pad(numpy.cumsum(sizes), (1, 0))
        return [slice(stops[i - 1], stops[i]) for i in range(1, len(stops))]

    def pred(self, given, key=None, givencov=None, *, fromdata=None, raw=False, keepcorr=None):
        """ Posterior mean and covariance (raw=True only; reference _compute.py:138-322).
        Returns numpy arrays. """
        if fromdata is None:
            raise ValueError('you must specify if `given` is data or fit result')
        fromdata = bool(fromdata)
        raw = bool(raw)
        if keepcorr is None:
            keepcorr = not raw
        if keepcorr and raw:
            raise ValueError('both keepcorr=True and raw=True')
        if not raw:
            raise NotImplementedError('pred(raw=False) needs gvar; use raw=True')
        strip = False
        if key is None:
            outkeys = list(self._elements)
        elif isinstance(key, list):
            outkeys = key
        else:
            outkeys = [key]
            strip = True
        outslices = self._slices(outkeys)
        ylist, inkeys, ycovblocks = self._flatgiven(given, givencov)
        y = torch.cat(ylist)
        with torch.no_grad():
            Kxxs = self._assemblecovblocks(inkeys, outkeys)
            ycov = self._block(ycovblocks) if ycovblocks is not None else None
            self._check_ycov(ycov)
            ymean = y
            self._check_ymean(ymean)
            Kxsxs = self._assemblecovblocks(outkeys)
            if fromdata:
                solver = self._solver(inkeys, ycov)
            else:
                solver = self._solver(inkeys)
            if not hasattr(solver, '_solve'):
                # generic Decomposition (e.g. the distributed solver): the two interface calls of the reference
                # (_compute.py:259-260)
                mean = solver.pinv_bilinear(Kxxs, ymean)
                cov = Kxsxs - solver.ginv_quad(Kxxs)
                if not fromdata and ycov is not None:
                    A = solver.ginv_linear(Kxxs)
                    cov = cov + A.T @ ycov @ A
                return self._pred_out(mean, cov, outkeys, outslices, strip)
            # mean = (L⁻¹Kxxs)'(L⁻¹y), cov = Kxsxs - (L⁻¹Kxxs)'(L⁻¹Kxxs): one TRSM shared by both
            invLA = solver._solve(_ops.as_aligned(Kxxs), False)
            invLy = solver._solve(ymean[:, None], False)
            mean = solver._matmul_tn(invLA, invLy)[:, 0]
            cov = _ops.aligned_empty(Kxsxs.shape[0], Kxsxs.shape[1], Kxsxs.device)
            cov.copy_(Kxsxs)
            A = _ops.as_aligned(invLA)
            _ops.dgemm(A, A, cov, a_kmajor=False, b_kmajor=False, M=cov.shape[0], N=cov.shape[1], K=A.shape[0],
                       alpha=-1.0)
            if not fromdata and ycov is not None:
                Ainv = solver._solve(invLA, True)  # K⁻¹ Kxxs
                T = solver._matmul_tn(_ops.as_aligned(ycov.contiguous()), Ainv)  # ycov' A (ycov symmetric)
                cov = cov + solver._matmul_tn(Ainv, T)
        return self._pred_out(mean, cov, outkeys, outslices, strip)

    def _pred_out(self, mean, cov, outkeys, outslices, strip):
        mean = mean.cpu().numpy()
        cov = cov.cpu().numpy()
        if not strip:
            meandict = {k: mean[s].reshape(self._elements[k].shape) for k, s in zip(outkeys, outslices)}
            covdict = {
                (row, col): cov[rs, cs].reshape(self._elements[row].shape + self._elements[col].shape)
                for row, rs in zip(outkeys, outslices) for col, cs in zip(outkeys, outslices)
            }
            return meandict, covdict
        outkey, = outkeys
        return mean.reshape(self._elements[outkey].shape), cov.reshape(2 * self._elements[outkey].shape)

    def predfromfit(self, *args, **kw):
        """ Like `pred` with ``fromdata=False`` """
        return self.pred(*args, fromdata=False, **kw)

    def predfromdata(self, *args, **kw):
        """ Like `pred` with ``fromdata=True`` """
        return self.pred(*args, fromdata=True, **kw)

    def _prior_decomp(self, given, givencov=None, **kw):
        """ (decomposition of Kxx + ycov, flattened data) (reference _compute.py:336-367) """
        ylist, inkeys, ycovblocks = self._flatgiven(given, givencov)
        ymean = torch.cat(ylist)
        self._check_ymean(ymean)
        ycov = self._block(ycovblocks) if ycovblocks is not None else None
        self._check_ycov(ycov)
        decomp = self._solver(inkeys, ycov, **kw)
        return decomp, ymean

    def _prior_matrix(self, given, givencov=None):
        """ (Kxx + ycov, flattened data) as torch tensors attached to the autograd graph of the hyperparameters: the
        argument of the decomposition in `_prior_decomp`, before decomposing (reference _compute.py:45-94,336-367).
        Used by the Fisher path of empbayes_fit, which needs its forward-mode derivative. """
        ylist, inkeys, ycovblocks = self._flatgiven(given, givencov)
        ymean = torch.cat(ylist)
        self._check_ymean(ymean)
        ycov = self._block(ycovblocks) if ycovblocks is not None else None
        self._check_ycov(ycov)
        Kxx = self._assemblecovblocks(inkeys)
        if ycov is not None:
            Kxx = Kxx + ycov
        return Kxx, ymean

    def marginal_likelihood(self, given, givencov=None, **kw):
        """ Logarithm of the probability of the data (reference _compute.py:383-422).

        Returns a float, or a differentiable torch scalar (on the device) when kernel hyperparameters, data or
        given covariance are torch tensors that require grad. """
        ylist, inkeys, ycovblocks = self._flatgiven(given, givencov)
        ymean = torch.cat(ylist)
        self._check_ymean(ymean)
        ycov = self._block(ycovblocks) if ycovblocks is not None else None
        self._check_ycov(ycov)
        grad = torch.is_grad_enabled() and (self._grad_mode() or ymean.requires_grad
                                            or (ycov is not None and ycov.requires_grad)
                                            or any(getattr(b, 'requires_grad', False) for e in
                                                   self._elements.values() if isinstance(e, _Cov)
                                                   for b in e.blocks.values()))
        if not grad:
            with torch.no_grad():
                decomp = self._solver(inkeys, ycov, **kw)
                mll, _, _, _, _ = decomp.minus_log_normal_density(ymean, value=True)
            return -float(mll)
        if self._solver_name != 'chol':
            raise NotImplementedError(f"derivatives of marginal_likelihood with solver={self._solver_name!r}: the "
                                      "distributed decomposition is value-only, use solver='chol' for gradients")
        solverkw = dict(self._solverkw)
        solverkw.update(kw)
        if (len(inkeys) == 1 and ycov is None and _plain_points(self._elements[inkeys[0]])
                and self._covfun._terms and not self._covfun._bart):
            elem = self._elements[inkeys[0]]
            params = [h[3] for h in self._covfun._hyperparams()]
            return -_FusedNegLogMLFn.apply(self._covfun, elem.xd, elem.labels, ymean, solverkw, *params)
        Kxx = self._assemblecovblocks(inkeys)
        if ycov is not None:
            Kxx = Kxx + ycov
        return -_NegLogDensityFn.apply(Kxx, ymean, solverkw)

    @staticmethod
    def _getdecomp(solver):
        """ solver registry (reference _compute.py:424-428: {'chol': Chol}); 'chol-dist' is the same decomposition
        sharded 2-D block-cyclic over the GPUs of the default process group (lsqfitgp_b200._dist) """
        if solver == 'chol-dist':
            from . import _dist
            return _dist.DistCholDecomposition
        return {'chol': _linalg.Chol}[solver]

    @classmethod
    def decompose(cls, posdefmatrix, solver='chol', **kw):
        """ Decompose a nonnegative definite matrix (reference _compute.py:430-516) """
        m = posdefmatrix if isinstance(posdefmatrix, torch.Tensor) else numpy.asarray(posdefmatrix)
        assert m.size > 0 if not isinstance(m, torch.Tensor) else m.numel() > 0
        assert m.ndim % 2 == 0
        half = m.ndim // 2
        head, tail = tuple(m.shape[:half]), tuple(m.shape[half:])
        assert head == tail
        n = math.prod(head)
        m = m.reshape(n, n)
        return cls._getdecomp(solver)(m, **kw)
