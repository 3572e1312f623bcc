"""Oracle: BART kernel (NumPy restatement of src/lsqfitgp/_kernels/_bart.py).

  splits_from_coord    :240-259
  indices_from_coord   :294-299, 503-514
  correlation          :301-455  (probabilities, weights, bracket folding with `repeat`)
  _correlation         :628-806  (fast closed forms for width 1/2/3, generic recursion otherwise)
  _correlation_old     :516-610  (independent older implementation, used by the reference's tests as cross-check)

The pair-level functions here take `ix`, `iy` of shape (..., p) and broadcast like the reference's
jnp.vectorize wrapper (:808-815).
"""

import numpy as np
from scipy import special

from . import fasthash


def splits_from_coord(x):
    """ x: (n, p) array -> (length (p,), splits (n-1, p)) ; _bart.py:240-259 """
    x = np.asarray(x)
    x = x.reshape(-1, x.shape[-1]) if x.size else x.reshape(1, x.shape[-1])
    if np.issubdtype(x.dtype, np.inexact):
        fill = np.finfo(x.dtype).max
    else:
        fill = np.iinfo(x.dtype).max
    lengths, mids = [], []
    for xi in x.T:
        u = np.unique(xi)
        u = np.concatenate([u, np.full(xi.size - u.size, fill, dtype=u.dtype)])  # jnp.unique(size=, fill_value=)
        with np.errstate(over='ignore'):
            m = np.where(u[1:] < fill, (u[1:] + u[:-1]) / 2, fill)
        l = np.searchsorted(m, fill)
        lengths.append(l)
        mids.append(m)
    return np.array(lengths), np.stack(mids, axis=1) if mids else np.empty((max(len(x) - 1, 0), 0))


def indices_from_coord(x, splits):
    """ _bart.py:294-299,503-514: searchsorted (side='left') per column """
    length, s = splits
    x = np.asarray(x)
    out = np.empty(x.shape, dtype=np.int64)
    for i in range(x.shape[-1]):
        out[..., i] = np.searchsorted(s[:, i], x[..., i])
    return out


def make_pnt(alpha, beta, maxd):
    d = np.arange(maxd + 1)
    return alpha / (1 + d) ** beta  # _bart.py:379-382


def _inexact(x):
    """ x as a float64 array, or complex128 when it is complex (the complex-step derivatives of gram_derivs) """
    x = np.asarray(x)
    return x.astype(np.result_type(x, float), copy=False)


def fold_brackets(pnt, reset, altinput=True, debug=False):
    """ _bart.py:415-447 -> list of (probs, repeat) in evaluation order (deepest first) """
    pnt = _inexact(pnt)
    if reset is None:
        reset = []
    if not hasattr(reset, '__len__'):
        reset = [reset]
    reset = [0] + list(reset) + [pnt.shape[-1] - 1]
    for i, j in zip(reset, reset[1:]):
        assert int(j) == j and i <= j, (i, j)
    brackets_norep = list(zip(reset, reset[1:]))
    brackets = [brackets_norep[0] + (1,)]
    for t, b in brackets_norep[1:]:
        lt, lb, lr = brackets[-1]
        if altinput and not debug and lr * (b - t) == lb - lt and b - t <= 2:
            brackets[-1] = lt, b, lr + 1
        else:
            brackets.append((t, b, 1))
    out = []
    for t, b, repeat in reversed(brackets):
        probs = pnt[..., t:b + 1].copy()
        if t > 0:
            probs[..., 0] = 1
        if repeat > 1:
            head = probs[..., 0:1]
            one = np.ones_like(head)
            pieces = [[head if i == 0 else one, p] for i, p in enumerate(np.split(probs[..., 1:], repeat, axis=-1))]
            probs = np.concatenate(sum(reversed(pieces), start=[]), axis=-1)
        else:
            repeat = None
        out.append((probs, repeat))
    return out


def correlation(n, ix, iy, *, alpha=0.95, beta=2, gamma=1, maxd=2, debug=False, pnt=None, intercept=True,
                weights=None, reset=None, altinput=True, use_hash=False):
    """ BART.correlation (_bart.py:301-455), altinput (index) form.
    n (p,), ix/iy (..., p) integer arrays. """
    n = np.asarray(n)
    ix = np.asarray(ix)
    iy = np.asarray(iy)
    if pnt is None:
        pnt = make_pnt(alpha, beta, maxd)
    else:
        pnt = _inexact(pnt)
    if weights is None:
        weights = np.ones(n.shape[-1])
    else:
        weights = np.asarray(weights, dtype=float)
    gamma = _inexact(gamma)
    if not intercept:
        pnt = pnt.copy()
        pnt[..., 0] = 1
    corr = gamma
    for probs, repeat in fold_brackets(pnt, reset, altinput, debug):
        if altinput:
            corr = _correlation(n, ix, iy, probs, corr, weights, debug, repeat, use_hash=use_hash)
        else:
            assert repeat is None
            corr = _correlation_old_vec(n, ix, iy, probs, corr, weights, debug)
    return corr


def _correlation(n, ix, iy, pnt, gamma, w, debug=False, repeat=None, use_hash=False):
    """ vectorised over leading axes of ix, iy and gamma; _bart.py:628-806 """
    n = np.asarray(n)
    ix, iy = np.broadcast_arrays(np.asarray(ix), np.asarray(iy))
    pnt = _inexact(pnt)
    w = np.asarray(w, dtype=float)
    gamma = _inexact(gamma)
    if repeat is not None:
        assert not debug and repeat > 0 and pnt.size % repeat == 0 and pnt.size // repeat <= 3
    else:
        repeat = 1
    batch = ix.shape[:-1]
    if n.size == 0:
        return np.ones(batch)
    # ignore zero-weight axes (:669-672)
    n = np.where(w, n, 0)
    ix = np.where(w, ix, 0)
    iy = np.where(w, iy, 0)
    # equality of the points (:675-678); the reference compares 64-bit hashes
    if use_hash:
        hx = fasthash.fasthash64_rows(ix.reshape(-1, ix.shape[-1]).astype(ix.dtype)).reshape(batch)
        hy = fasthash.fasthash64_rows(iy.reshape(-1, iy.shape[-1]).astype(iy.dtype)).reshape(batch)
        anyn0 = hx != hy
    else:
        anyn0 = np.any(ix != iy, axis=-1)
    rows = pnt.reshape(repeat, -1)
    width = pnt.size // repeat

    if width == 1:
        for row in rows:
            gamma = np.where(anyn0, 1 - (1 - gamma) * row[0], 1)
        return gamma + np.zeros(batch, gamma.dtype)

    Wn = np.sum(np.where(n, w, 0))  # :694

    if width == 2 and not debug:
        n0 = np.abs(ix - iy)
        with np.errstate(divide='ignore', invalid='ignore'):
            wn = np.where(n, w / n, 0)
        sum_term = _dot(wn, n0)
        for row in rows:
            Q = 1 - row[1] + gamma * row[1]
            P0 = row[0]
            result = 1 - P0 + Q * (P0 - P0 / Wn * sum_term)
            gamma = np.where(anyn0, result, 1)
        return gamma

    xlty = ix < iy
    minxy = np.where(xlty, ix, iy)
    maxxy = np.where(xlty, iy, ix)
    n0 = maxxy - minxy

    if width == 3 and not debug:
        nminus0 = maxxy
        nplus0 = n - minxy
        nout = n - n0
        with np.errstate(divide='ignore', invalid='ignore'):
            inv_Wn = 1 / Wn
            inv_Wnmod = 1 / (Wn - np.where(n, w, 0))
            inv_Wnminus = np.where(nplus0, inv_Wn, inv_Wnmod)
            inv_Wnplus = np.where(nminus0, inv_Wn, inv_Wnmod)
            wn = np.where(n, w / n, 0)
            S = _dot(wn, nout)
            t = wn * n0
            terms1 = (S[..., None] + t) * (inv_Wnminus + inv_Wnplus + inv_Wn * (nout - 2))
            terms2 = np.where(nplus0, w * inv_Wn * n0 / nplus0, w * inv_Wnmod)
            terms2 = terms2 + np.where(nminus0, w * inv_Wn * n0 / nminus0, w * inv_Wnmod)
            psin = special.digamma(np.where(n, n, 1).astype(float))
            psiminus = np.where(xlty, special.digamma((1 + iy).astype(float)), special.digamma((1 + ix).astype(float)))
            psiplus = np.where(xlty, special.digamma((1 + n - ix).astype(float)),
                               special.digamma((1 + n - iy).astype(float)))
            terms3 = w * inv_Wn * n0 * (2 * psin - psiminus - psiplus)
            terms = terms1 - terms2 - terms3
            sumi = _dot(wn, terms)
        for row in rows:
            Q = 1 + row[2] * (gamma - 1)
            sump = S + row[1] * (Q * sumi - S)
            result = 1 + row[0] * (inv_Wn * sump - 1)
            gamma = np.where(anyn0, result, 1)
        return gamma

    # generic recursion (:759-806), scalar python loops: small cases only
    assert repeat == 1
    flat_ix = ix.reshape(-1, ix.shape[-1])
    flat_iy = iy.reshape(-1, iy.shape[-1])
    g = np.broadcast_to(gamma, batch).reshape(-1)
    out = np.empty(flat_ix.shape[0])
    for q in range(flat_ix.shape[0]):
        out[q] = _correlation_rec(n, flat_ix[q], flat_iy[q], pnt, float(g[q]), w, debug)
    return out.reshape(batch)


def _dot(a, b):
    """ wn @ v over the last axis, sequential accumulation in field order """
    a, b = np.broadcast_arrays(a, b)
    acc = np.zeros(a.shape[:-1])
    for i in range(a.shape[-1]):
        acc = acc + a[..., i] * b[..., i]
    return acc


def _correlation_rec(n, ix, iy, pnt, gamma, w, debug):
    """ scalar generic recursion, _bart.py:759-806 (dispatching to the closed forms like the reference) """
    if not debug and pnt.size <= 3:
        return float(_correlation(n, ix, iy, pnt, gamma, w, debug, None))
    if pnt.size == 1:
        return float(_correlation(n, ix, iy, pnt, gamma, w, debug, None))
    n = np.where(w, n, 0)
    ix = np.where(w, ix, 0)
    iy = np.where(w, iy, 0)
    anyn0 = bool(np.any(ix != iy))
    if not anyn0:
        return 1.0
    Wn = np.sum(np.where(n, w, 0))
    minxy = np.minimum(ix, iy)
    maxxy = np.maximum(ix, iy)
    n0 = maxxy - minxy
    nminus = minxy
    nplus = n - maxxy
    p = len(nminus)
    sump = 0.0
    for i in range(p):
        ni = nminus[i] + n0[i] + nplus[i]
        if ni == 0:
            continue
        sumn = 0.0
        for k in range(nminus[i] + nplus[i]):
            nm = nminus.copy()
            npl = nplus.copy()
            if k < nminus[i]:
                nm[i] = k
            else:
                npl[i] = k - nminus[i]
            nn = nm + n0 + npl
            sumn += _correlation_rec(nn, nm, nm + n0, pnt[1:], gamma, w, debug)
        sump += w[i] * sumn / ni
    return 1 - pnt[0] * (1 - sump / Wn)


def _correlation_old(nminus, n0, nplus, pnt, gamma, w, debug=False):
    """ scalar; _bart.py:516-610 """
    nminus = np.where(w, nminus, 0)
    n0 = np.where(w, n0, 0)
    nplus = np.where(w, nplus, 0)
    if nminus.size == 0:
        return 1.0
    anyn0 = bool(np.any(np.logical_and(n0, w)))
    if pnt.size == 1:
        return 1 - (1 - gamma) * pnt[0] if anyn0 else 1.0
    nout = nminus + nplus
    n = nout + n0
    Wn = np.sum(np.where(n, w, 0))
    with np.errstate(divide='ignore', invalid='ignore'):
        if pnt.size == 2 and not debug:
            Q = 1 - (1 - gamma) * pnt[1]
            sump = Q * np.sum(np.where(n, w * nout / n, 0))
            return 1 - pnt[0] * (1 - sump / Wn) if anyn0 else 1.0
        if pnt.size == 3 and not debug:
            Q = 1 - (1 - gamma) * pnt[2]
            s = w * nout / n
            S = np.sum(np.where(n, s, 0))
            t = w * n0 / n
            psin = special.digamma(n.astype(float))

            def terms(nminus, nplus):
                nminus0 = nminus + n0
                Wnmod = Wn - np.where(nminus0, 0, w)
                frac = np.where(nminus0, w * nminus / nminus0, 0)
                terms1 = (S - s + frac) / Wnmod
                psi1nminus0 = special.digamma((1 + nminus0).astype(float))
                terms2 = ((nplus - 1) * (S + t) - w * n0 * (psin - psi1nminus0)) / Wn
                return np.where(nplus, terms1 + terms2, 0)
            tplus = terms(nminus, nplus)
            tminus = terms(nplus, nminus)
            tall = np.where(n, w * (tplus + tminus) / n, 0)
            sump = (1 - pnt[1]) * S + pnt[1] * Q * np.sum(tall)
            return 1 - pnt[0] * (1 - sump / Wn) if anyn0 else 1.0
    if not anyn0:
        return 1.0
    p = len(nminus)
    sump = 0.0
    for i in range(p):
        ni = nminus[i] + n0[i] + nplus[i]
        if ni == 0:
            continue
        sumn = 0.0
        for k in range(nminus[i] + nplus[i]):
            nm = nminus.copy()
            npl = nplus.copy()
            if k < nminus[i]:
                nm[i] = k
            else:
                npl[i] = k - nminus[i]
            sumn += _correlation_old(nm, n0, npl, pnt[1:], gamma, w, debug)
        sump += w[i] * sumn / ni
    return 1 - pnt[0] * (1 - sump / Wn)


def _correlation_old_vec(nminus, n0, nplus, pnt, gamma, w, debug):
    nminus, n0, nplus = np.broadcast_arrays(nminus, n0, nplus)
    batch = nminus.shape[:-1]
    g = np.broadcast_to(gamma, batch).reshape(-1)
    a = nminus.reshape(-1, nminus.shape[-1])
    b = n0.reshape(-1, n0.shape[-1])
    c = nplus.reshape(-1, nplus.shape[-1])
    out = np.array([_correlation_old(a[q], b[q], c[q], _inexact(pnt), g[q], np.asarray(w, float), debug)
                    for q in range(a.shape[0])])
    return out.reshape(batch)


def gram(n, ix, iy, *, chunk=256, **kw):
    """ full (len(ix), len(iy)) BART Gram matrix, row-chunked like batchufunc (_jaxext/_batcher.py:81-120) """
    ix = np.asarray(ix)
    iy = np.asarray(iy)
    cplx = any(np.iscomplexobj(kw.get(k)) for k in ('alpha', 'beta', 'gamma', 'pnt'))
    out = np.empty((ix.shape[0], iy.shape[0]), complex if cplx else float)
    for s in range(0, ix.shape[0], chunk):
        out[s:s + chunk] = correlation(n, ix[s:s + chunk, None, :], iy[None, :, :], **kw)
    return out


def _complex_step(f, n, ix, iy, alpha, beta, h, kw):
    """ (f, df/dalpha, df/dbeta) with the derivatives Im f(alpha + ih) / h: alpha and beta enter only through
    pnt_d = alpha / (1 + d)^beta, and everything after is +, -, *, / and index-selected branches, so there is no
    subtractive cancellation and the result is exact to rounding """
    return (f(n, ix, iy, alpha=alpha, beta=beta, **kw), f(n, ix, iy, alpha=alpha + 1j * h, beta=beta, **kw).imag / h,
            f(n, ix, iy, alpha=alpha, beta=beta + 1j * h, **kw).imag / h)


def correlation_derivs(n, ix, iy, *, alpha=0.95, beta=2, h=1e-200, **kw):
    """ (correlation, d/dalpha, d/dbeta) per pair, by complex step """
    return _complex_step(correlation, n, ix, iy, alpha, beta, h, kw)


def gram_derivs(n, ix, iy, *, alpha=0.95, beta=2, h=1e-200, **kw):
    """ (K, dK/dalpha, dK/dbeta) of `gram` (K without amplitude), by complex step """
    return _complex_step(gram, n, ix, iy, alpha, beta, h, kw)
