"""empbayes_fit: maximum a posteriori fit of the hyperparameters of a GP.

Mirror of src/lsqfitgp/_fit.py (empbayes_fit :145-371, _parse_hyperprior :444-489,
_prepare_functions :598-754, _prepare_minargs :756-772, _posterior_covariance :808-845) without gvar and
without JAX:

  * the hyperprior is a dictionary key -> (mean, sdev) of independent Normal priors (scalars or arrays), or a
    pair (mean vector, covariance matrix); keys spelled 'log(x)' / 'sqrt(x)' are exposed to `gpfactory`
    as hp['x'] = exp(.) / square(.) like gvar.BufferDict does (reference _patch_gvar.py:58-63);
  * `gpfactory(hp, **gpfactorykw)` receives torch float64 scalars/arrays that require grad and must build the
    kernel from them with torch operations; the objective
        -logML(hp(p)) + 1/2 (k log 2pi + p.p) + additional_loss(hp)          (reference _fit.py:659-668,718-721)
    is differentiated by torch.autograd, whose backward runs the CUDA inverse-from-factor and Gram-VJP kernels;
  * the same scipy.optimize.minimize drivers are used: 'nograd' -> Nelder-Mead, 'gradient' -> BFGS,
    'fisher' -> dogleg with the Fisher information plus the prior precision as hessian (reference _fit.py:732-743,
    756-772): dK/dp comes from torch forward-mode AD through the Gram JVP kernel (lgp_gram_iso_jvp), the matrix
    itself from Chol.minus_log_normal_density(fisher=True) (two blocked TRSMs per parameter on the DMMA path);
    'hessian' -> trust-exact with the exact Hessian of the objective (torch.autograd.functional.hessian through the
    twice-differentiable marginal likelihood).  trust-exact, not dogleg, because it accepts the indefinite Hessians
    met away from the optimum, where dogleg requires positive definiteness;
  * covariance: 'fisher', 'minhess', 'none', 'auto' as the reference, and 'hessian': the inverse of the exact Hessian
    at the optimum (a RuntimeError if it is not positive definite).  'hessmod' is not implemented.
"""

import math
import re
import time
import warnings

import numpy
import torch
from scipy import linalg, optimize

from . import _linalg
from . import _timing

__all__ = ['empbayes_fit']

f64 = torch.float64

_EXT = re.compile(r'^([\w{}., ]+)\((.+)\)$')


def _copula_beta21(z):
    """ Normal -> Beta(2, 1): ppf(Phi(z)) with ppf(u) = sqrt(u) (reference copula.beta(2, 1), copula/_copulas.py:43-50) """
    return torch.exp(0.5 * torch.special.log_ndtr(z))


def _copula_invgamma11(z):
    """ Normal -> InvGamma(1, 1): ppf(u) = -1/log(u), evaluated through the upper tail for z >= 0 as the reference does
    (copula/_copulas.py:141-163) """
    lo = -1.0 / torch.special.log_ndtr(torch.clamp(z, max=0.0))
    hi = -1.0 / torch.log1p(-torch.exp(torch.special.log_ndtr(-torch.clamp(z, min=0.0))))
    return torch.where(z < 0, lo, hi)


# key 'f(x)' in the hyperprior is exposed to gpfactory as hp['x'] = f^-1(value), like gvar.BufferDict does
# (reference _patch_gvar.py:58-63); the two copula names are the ones copula.makedict produces for the priors of
# bayestree.bart (bayestree/_bart.py:175-184), the only closed-form members of that family needed on this path
_INV = {'log': torch.exp, 'sqrt': torch.square,
        '__copula_beta{2, 1}': _copula_beta21, '__copula_invgamma{1, 1}': _copula_invgamma11}


class _HyperDict(dict):
    """ dictionary of hyperparameters; hp['x'] falls back to the inverse transform of a stored 'f(x)' key """

    def __missing__(self, key):
        for name, inv in _INV.items():
            k = f'{name}({key})'
            if dict.__contains__(self, k):
                return inv(dict.__getitem__(self, k))
        raise KeyError(key)

    def __contains__(self, key):
        return dict.__contains__(self, key) or any(dict.__contains__(self, f'{n}({key})') for n in _INV)

    def get(self, key, default=None):
        try:
            return self[key]
        except KeyError:
            return default


class Logger:
    """ indented logging with a verbosity level (reference _fit.py:79-143) """

    def __init__(self, verbosity=0):
        self._verbosity = verbosity
        self._loglevel = 0

    def log(self, message, verbosity=1, level=None):
        if verbosity > self._verbosity:
            return
        indent = '    ' * (self._loglevel if level is None else level)
        for line in str(message).split('\n'):
            print(indent + line)


class empbayes_fit(Logger):

    SEPARATE_JAC = False

    def __init__(self, hyperprior, gpfactory, data, *, raises=True, minkw={}, gpfactorykw={}, jit=True,
                 method='gradient', initial='priormean', verbosity=0, covariance='auto', fix=None, mlkw={},
                 forward=False, additional_loss=None, multistart=0, multistart_seed=0, in_flight=1):
        Logger.__init__(self, verbosity)
        self.log('**** call lsqfitgp_b200.empbayes_fit ****')
        assert callable(gpfactory)
        if method not in ('nograd', 'gradient', 'fisher', 'hessian'):
            raise KeyError(method)
        if covariance not in ('auto', 'fisher', 'minhess', 'hessian', 'none'):
            raise KeyError(covariance)
        # `jit`: there is no tracing compiler here.  `forward`: the reference's forward mode materialises dK (n, n, k) with
        # jax.jacfwd and contracts it (_fit.py:679-685, _decomp.py:524-531); the same gradient is obtained here in ONE
        # reverse sweep by the fused VJP kernels (lgp_gram_iso_vjp / lgp_gram_bart_vjp), whatever the flag says: the
        # values are identical (tests/test_gpu_api.py::test_gradfwd_equals_gradrev), only the work differs.
        self._forward = bool(forward)
        del jit

        hpinitial, hpunflat = self._parse_hyperprior(hyperprior, initial, fix)
        self.data = data
        if isinstance(data, tuple) and len(data) == 1:
            data, = data
        if callable(data):
            cachedargs = None
        elif isinstance(data, tuple):
            assert len(data) == 2
            cachedargs = data
        else:
            cachedargs = (data,)

        self.gpfactory = gpfactory
        self.gpfactorykw = gpfactorykw
        self._ncalls = {'fun': 0, 'fun&jac': 0}
        self._timer = _timing.PhaseTimer()   # device time of the three phases of the reference's timer (_fit.py:410-442)
        self._hpunflat = hpunflat

        def total_of(pt):
            """ the objective as a torch function of the whitened parameters; starts the phase timer """
            hp = hpunflat(pt)
            gp = gpfactory(hp, **gpfactorykw)
            args = data(hp, **gpfactorykw) if cachedargs is None else cachedargs
            if not isinstance(args, tuple):
                args = (args,)
            self._timer.start()
            try:
                ml = gp.marginal_likelihood(*args, **mlkw)
            except BaseException:
                self._timer.stop()
                raise
            loss = -ml
            prior = 1 / 2 * (len(pt) * math.log(2 * math.pi) + pt @ pt)
            if isinstance(loss, torch.Tensor):
                total = loss.cpu() + prior
            else:
                total = prior + loss
            if additional_loss is not None:
                extra = additional_loss(hp)
                total = total + (extra.cpu() if isinstance(extra, torch.Tensor) else extra)
            return total

        def objective(p, need_grad):
            pt = torch.tensor(numpy.asarray(p, dtype=float), dtype=f64, requires_grad=need_grad)
            with torch.set_grad_enabled(need_grad):
                total = total_of(pt)
            if not need_grad:
                self._timer.stop()
                return float(total)
            try:
                grad, = torch.autograd.grad(total, pt, allow_unused=True)
            finally:
                self._timer.stop()
            if grad is None:
                grad = torch.zeros_like(pt)
            return float(total.detach()), grad.numpy().astype(float)

        def fisher(p):
            """ Fisher information of the hyperparameters plus prior precision (reference _fit.py:732-743) """
            import torch.autograd.forward_ad as fwAD
            if additional_loss is not None:
                raise NotImplementedError('Fisher matrix not implemented with additional_loss')
            self._ncalls['fisher'] = self._ncalls.get('fisher', 0) + 1
            p = numpy.asarray(p, dtype=float)
            k = len(p)
            K0 = r0 = None
            dKs, drs = [], []
            for q in range(k):
                pt = torch.tensor(p, dtype=f64, requires_grad=True)
                e = torch.zeros(k, dtype=f64)
                e[q] = 1.0
                with fwAD.dual_level():
                    hp = hpunflat(fwAD.make_dual(pt, e))
                    gp = gpfactory(hp, **gpfactorykw)
                    args = data(hp, **gpfactorykw) if cachedargs is None else cachedargs
                    if not isinstance(args, tuple):
                        args = (args,)
                    K, r = gp._prior_matrix(*args)
                    Kp, Kt = fwAD.unpack_dual(K)
                    rp, rt = fwAD.unpack_dual(r)
                    if K0 is None:
                        K0, r0 = Kp.detach(), rp.detach()
                    dKs.append(torch.zeros_like(K0) if Kt is None else Kt.detach())
                    drs.append(torch.zeros_like(r0) if rt is None else rt.detach().to(r0.device))
                del K, Kp, Kt
            solverkw = dict(getattr(gp, '_solverkw', {}))
            solverkw.update(mlkw)
            dec = _linalg.Chol(K0, **solverkw)
            del K0
            lkw = dict(dK=dKs)
            if any(bool(torch.any(d != 0)) for d in drs):
                lkw.update(dr=torch.stack(drs, dim=1))
            _, _, _, fm, _ = dec.minus_log_normal_density(r0, fisher=True, **lkw)
            fm = fm.cpu().numpy() if isinstance(fm, torch.Tensor) else numpy.asarray(fm)
            return fm + numpy.eye(k)

        def hessian(p):
            """ exact Hessian of the objective in p: torch.autograd.functional.hessian through the twice-differentiable
            marginal likelihood (the GP term's second order runs lgp_gram_iso_hvp, lgp_gram_iso_jvp and DMMA GEMMs) """
            self._ncalls['hess'] = self._ncalls.get('hess', 0) + 1
            pt = torch.tensor(numpy.asarray(p, dtype=float), dtype=f64)
            try:
                H = torch.autograd.functional.hessian(total_of, pt)
            finally:
                self._timer.stop()
            return H.numpy().astype(float)

        def fun(p):
            self._ncalls['fun'] += 1
            return objective(p, False)

        def fun_and_jac(p):
            self._ncalls['fun&jac'] += 1
            return objective(p, True)

        def jac(p):
            return objective(p, True)[1]

        minargs = dict(fun=fun_and_jac, jac=True, x0=hpinitial)
        if self.SEPARATE_JAC:
            minargs.update(fun=fun, jac=jac)
        if method == 'nograd':
            minargs.update(fun=fun, jac=None, method='nelder-mead')
        elif method == 'gradient':
            minargs.update(method='bfgs')
        elif method == 'fisher':
            # dogleg requires positive definiteness; the Fisher matrix is p.s.d. and the prior precision is the identity
            minargs.update(hess=fisher, method='dogleg')
        elif method == 'hessian':
            # trust-exact accepts the indefinite Hessians met away from the optimum, which dogleg does not
            minargs.update(hess=hessian, method='trust-exact')
        self.log(f'method {method!r}', 2)

        def callback(intermediate_result=None, *a):
            if self._verbosity >= 3:
                try:
                    self.log(f'iteration: fun = {intermediate_result.fun:.15g}', 3)
                except AttributeError:
                    self.log('iteration', 3)
        minargs.update(callback=callback)
        minargs.update(minkw)

        # multi-start (not in the reference, whose optimiser evaluates one point at a time, _fit.py:338): the objective
        # at `multistart` draws of the whitened parameters from their prior N(0, I), plus the requested starting point,
        # is evaluated as ONE batch sharded over the GPUs of the process group (lsqfitgp_b200.eval_batch_sharded, with
        # `in_flight` evaluations kept in flight per GPU); the best point starts the minimiser.  Every rank gets the
        # same batch results, hence runs the same (replicated) minimisation afterwards.
        self.multistart = None
        if multistart and len(hpinitial):
            from . import _dist
            rng = numpy.random.default_rng(multistart_seed)
            starts = numpy.vstack([hpinitial, rng.standard_normal((int(multistart), len(hpinitial)))])

            def safe(p):
                try:
                    return numpy.array([objective(p, False)])
                except (numpy.linalg.LinAlgError, RuntimeError):
                    return numpy.array([numpy.inf])
            dev = torch.device('cuda', torch.cuda.current_device()) if torch.cuda.is_available() else None
            vals = _dist.eval_batch_sharded(safe, starts, device=dev, in_flight=in_flight)[:, 0]
            vals = numpy.where(numpy.isfinite(vals), vals, numpy.inf)
            best = int(numpy.argmin(vals))
            self.multistart = dict(starts=starts, values=vals, best=best)
            self.log(f'multistart: best of {len(starts)} starting points has objective {vals[best]:.6g}', 2)
            minargs.update(x0=starts[best])
        self.log(f'minimizer method {minargs["method"]!r}', 2)
        total = time.perf_counter()
        result = optimize.minimize(**minargs)
        total = time.perf_counter() - total

        if result.success:
            self.log(f'minimization succeeded: {result.message}')
        else:
            msg = f'minimization failed: {result.message}'
            if raises:
                raise RuntimeError(msg)
            elif self._verbosity == 0:
                warnings.warn(msg)
            else:
                self.log(msg)

        cov = self._posterior_covariance(method, covariance, result, fisher, hessian)
        self._pcov_p = cov
        # the reference's totals line (_fit.py:775-794): device time per phase, the rest of the wall clock as 'other'
        times = dict(self._timer.totals)
        times['other'] = max(total - sum(times.values()), 0.0)
        self.times = times
        self.log(f'calls: {self._ncalls}')
        self.log(f'total time: {total:.3g} s')
        self.log('partials: ' + ', '.join(f'{k} {v:.3g} s' for k, v in times.items()), 2)

        # posterior of the hyperparameters in the original parametrisation: hp = mean + L p (linear map)
        xt = torch.tensor(result.x, dtype=f64)
        self.pmean = self._tonumpy(hpunflat(xt, raw=True))
        flatmean, J = self._flat_and_jac(result.x)
        if numpy.ndim(cov) == 1:
            fullcov = numpy.full((len(flatmean), len(flatmean)), numpy.nan)
        else:
            fullcov = J @ numpy.asarray(cov) @ J.T
        self._flatpcov = fullcov
        self.pcov = self._unflat_cov(fullcov)
        sdev = numpy.sqrt(numpy.clip(numpy.diag(fullcov), 0, None)) if numpy.all(numpy.isfinite(fullcov)) else \
            numpy.full(len(flatmean), numpy.nan)
        self.p = self._unflat_pairs(flatmean, sdev)
        self.minresult = result
        self.minargs = minargs
        self.log('**** exit lsqfitgp_b200.empbayes_fit ****')

    # ------------------------------------------------------------------------------------------------
    def hp_at(self, p):
        """ hyperparameters (as `gpfactory` receives them: a dictionary that also resolves transformed keys such as
        hp['x'] for a stored 'log(x)') at the whitened parameter vector p, detached """
        with torch.no_grad():
            return self._hpunflat(torch.tensor(numpy.asarray(p, dtype=float), dtype=f64))

    def hp_sdev(self, p, names):
        """ first-order standard deviation of the (transformed) hyperparameters `names` at p from the posterior
        covariance of p: what gvar's error propagation gives fit.p['x'] in the reference """
        cov = numpy.asarray(self._pcov_p)
        out = {}
        for name in names:
            pt = torch.tensor(numpy.asarray(p, dtype=float), dtype=f64, requires_grad=True)
            v = self._hpunflat(pt)[name]
            g, = torch.autograd.grad(v.sum(), pt, allow_unused=True)
            g = numpy.zeros(len(cov)) if g is None else g.numpy()
            out[name] = float(numpy.sqrt(max(g @ cov @ g, 0.0))) if cov.ndim == 2 and numpy.all(numpy.isfinite(cov)) \
                else float('nan')
        return out

    def hp_sample(self, rng=None):
        """ hyperparameters at a sample of p from its Gaussian posterior approximation (the reference samples
        fit.pmean / fit.pcov with _fastraniter.sample, bayestree/_bart.py:229-238) """
        from . import _fastraniter
        x = _fastraniter.sample(numpy.asarray(self.minresult.x), numpy.asarray(self._pcov_p), rng=rng)
        return self.hp_at(x)

    def _parse_hyperprior(self, hyperprior, initial, fix):
        """ -> (x0, hpunflat); whitening with Chol of the prior covariance (reference _fit.py:444-489) """
        self._isdict = hasattr(hyperprior, 'keys')
        if self._isdict:
            self._keys = list(hyperprior.keys())
            for k in self._keys:
                m = _EXT.match(k) if isinstance(k, str) else None
                if m and m.group(1) in _INV and m.group(2) in hyperprior:
                    raise ValueError(f'duplicate keys {m.group(2)!r} and {k!r} in hyperprior')
            means, sdevs, self._shapes = [], [], []
            for k in self._keys:
                mu, sd = hyperprior[k]
                mu = numpy.asarray(mu, dtype=float)
                sd = numpy.broadcast_to(numpy.asarray(sd, dtype=float), mu.shape)
                self._shapes.append(mu.shape)
                means.append(mu.reshape(-1))
                sdevs.append(sd.reshape(-1))
            mean = numpy.concatenate(means)
            cov = numpy.diag(numpy.concatenate(sdevs) ** 2)
        else:
            mu, c = hyperprior
            mean = numpy.atleast_1d(numpy.asarray(mu, dtype=float)).reshape(-1)
            c = numpy.asarray(c, dtype=float)
            self._shapes = [numpy.shape(mu)]
            self._keys = [None]
            cov = numpy.diag(numpy.broadcast_to(c, mean.shape) ** 2) if c.ndim < 2 else c.reshape(mean.size, mean.size)
        self.prior = hyperprior
        nflat = mean.size

        # fixed parameters
        flatfix = numpy.zeros(nflat, bool)
        if fix is not None:
            if self._isdict:
                assert hasattr(fix, 'keys'), 'hyperprior is dictionary but fix is array'
                off = 0
                for k, shape in zip(self._keys, self._shapes):
                    size = int(numpy.prod(shape, dtype=int))
                    key = k
                    m = _EXT.match(k) if isinstance(k, str) else None
                    if m and m.group(1) in _INV and m.group(2) in fix:
                        assert k not in fix, f'duplicate keys {k!r} and {m.group(2)!r} in fix'
                        key = m.group(2)
                    if key in fix:
                        flatfix[off:off + size] = numpy.broadcast_to(fix[key], shape).reshape(-1)
                    off += size
            else:
                assert not hasattr(fix, 'keys'), 'fix is dictionary but hyperprior is array'
                flatfix[:] = numpy.broadcast_to(fix, self._shapes[0]).reshape(-1)
        self.fix = fix
        free = ~flatfix
        fmean = mean[free]
        fcov = cov[numpy.ix_(free, free)]
        nfree = int(free.sum())
        self.log(f'{nfree}/{nflat} free hyperparameters', 2)
        # whitening: hp_free = mean + L p  with L the Cholesky factor of the prior covariance, computed with
        # the same Chol class (device) as the reference does (_fit.py:457)
        if nfree:
            dec = _linalg.Chol(fcov)
            L = dec.factor().cpu().numpy()
        else:
            L = numpy.zeros((0, 0))

        # starting point
        if isinstance(initial, str):
            if initial == 'priormean':
                flatinitial = mean.copy()
            elif initial == 'priorsample':
                fulldec = _linalg.Chol(cov)
                flatinitial = mean + fulldec.correlate(numpy.random.randn(nflat))
            else:
                raise KeyError(initial)
        else:
            if self._isdict:
                assert hasattr(initial, 'keys'), 'hyperprior is dictionary but initial is array'
                assert set(initial.keys()) == set(self._keys)
                flatinitial = numpy.concatenate([numpy.asarray(initial[k], dtype=float).reshape(-1) for k in self._keys])
            else:
                flatinitial = numpy.asarray(initial, dtype=float).reshape(-1)
        self.initial = self._unflat_numpy(flatinitial)
        x0 = numpy.linalg.solve(L, flatinitial[free] - fmean) if nfree else numpy.zeros(0)

        Lt = torch.tensor(L, dtype=f64)
        mt = torch.tensor(fmean, dtype=f64)
        fixed_values = torch.tensor(flatinitial[flatfix], dtype=f64)
        free_idx = torch.tensor(numpy.nonzero(free)[0])
        fixed_idx = torch.tensor(numpy.nonzero(flatfix)[0])
        self._L, self._free = L, free

        def unflat(x, raw=False):
            assert x.ndim == 1
            xf = mt + Lt @ x
            y = torch.zeros(nflat, dtype=f64)
            y = y.index_put((free_idx,), xf)
            y = y.index_put((fixed_idx,), fixed_values)
            return self._unflat_torch(y, raw)
        return x0, unflat

    def _unflat_torch(self, y, raw=False):
        if not self._isdict:
            return y.reshape(self._shapes[0])
        out = {} if raw else _HyperDict()
        off = 0
        for k, shape in zip(self._keys, self._shapes):
            size = int(numpy.prod(shape, dtype=int))
            out[k] = y[off:off + size].reshape(shape)
            off += size
        return out

    def _unflat_numpy(self, y):
        t = self._unflat_torch(torch.tensor(y, dtype=f64), raw=True)
        return self._tonumpy(t)

    @staticmethod
    def _tonumpy(t):
        if isinstance(t, dict):
            return {k: v.detach().numpy() for k, v in t.items()}
        return t.detach().numpy()

    def _flat_and_jac(self, x):
        """ flat posterior mean of the hyperparameters and jacobian d hp_flat / d p """
        nflat = len(self._free)
        J = numpy.zeros((nflat, len(x)))
        J[self._free] = self._L
        xt = torch.tensor(x, dtype=f64)
        y = self._unflat_torch_flat(xt)
        return y, J

    def _unflat_torch_flat(self, xt):
        t = self._unflat_torch_raw(xt)
        return t

    def _unflat_torch_raw(self, xt):
        # recompute the flat vector (mean + L p with fixed values) as numpy
        d = self.pmean
        if isinstance(d, dict):
            return numpy.concatenate([numpy.asarray(d[k]).reshape(-1) for k in self._keys])
        return numpy.asarray(d).reshape(-1)

    def _unflat_cov(self, fullcov):
        if not self._isdict:
            return fullcov.reshape(self._shapes[0] + self._shapes[0])
        out = {}
        offs = numpy.cumsum([0] + [int(numpy.prod(s, dtype=int)) for s in self._shapes])
        for i, ki in enumerate(self._keys):
            for j, kj in enumerate(self._keys):
                out[ki, kj] = fullcov[offs[i]:offs[i + 1], offs[j]:offs[j + 1]].reshape(self._shapes[i] + self._shapes[j])
        return out

    def _unflat_pairs(self, mean, sdev):
        if not self._isdict:
            return (mean.reshape(self._shapes[0]), sdev.reshape(self._shapes[0]))
        out = {}
        off = 0
        for k, shape in zip(self._keys, self._shapes):
            size = int(numpy.prod(shape, dtype=int))
            out[k] = (mean[off:off + size].reshape(shape), sdev[off:off + size].reshape(shape))
            off += size
        return out

    def _posterior_covariance(self, method, covariance, result, fisher_func, hessian_func):
        """ reference _fit.py:808-845 """
        if covariance == 'auto':
            covariance = 'minhess' if (hasattr(result, 'hess_inv') or hasattr(result, 'hess')) else 'none'
        if covariance == 'fisher':
            self.log('use fisher plus prior precision as precision', 2)
            prec = result.hess if method == 'fisher' else fisher_func(result.x)
            return _linalg.Chol(prec).ginv()
        if covariance == 'hessian':
            self.log('use the hessian at the optimum as precision', 2)
            try:
                cho = linalg.cho_factor(hessian_func(result.x), lower=True)
            except numpy.linalg.LinAlgError:
                raise RuntimeError('the hessian of the objective at the optimum is not positive definite') from None
            return linalg.cho_solve(cho, numpy.eye(result.x.size))
        if covariance == 'minhess':
            if hasattr(result, 'hess_inv'):
                hessinv = result.hess_inv
                if isinstance(hessinv, optimize.LbfgsInvHessProduct):
                    bfgs = optimize.BFGS()
                    bfgs.initialize(hessinv.shape[0], 'inv_hess')
                    for i in range(hessinv.n_corrs):
                        bfgs.update(hessinv.sk[i], hessinv.yk[i])
                    return bfgs.get_matrix()
                return numpy.asarray(hessinv)
            if hasattr(result, 'hess'):
                return _linalg.Chol(result.hess).ginv()
            raise RuntimeError('the minimizer did not return an estimate of the hessian')
        return numpy.full(result.x.size, numpy.nan)
