#!/usr/bin/env python
"""bench.py -- headline benchmark of the GP-fitting hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--n 20000] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[1] -- Matern(nu=2.5), 3-D covariates, n = 20000, float64,
one step = one evaluation of log marginal likelihood AND its gradient w.r.t. (log scale, log sigma_f, log sigma_n):
Gram build -> equilibrated/jittered Cholesky -> triangular solves + log-determinant -> inverse from the factor ->
Gram-VJP contraction.  Metric: logML(+gradient) evaluations per second, whole job.

  value : device-timed (CUDA events), inputs (x, y) already resident in HBM, kernels through the C ABI.  The batch of
          N*K hyperparameter points goes through the product's sharding function `lsqfitgp_b200.eval_batch_sharded`
          (round-robin over the ranks, one all_gather of (1 + k) doubles per point) at every N, N = 1 included.
  e2e   : the same metric through the public API (lgp.GP(...).marginal_likelihood + torch.autograd.grad) from HOST
          arrays, host->device copies of x, y and the device->host read of (logML, gradient) inside the timed region.
  N > 1 : one process per GPU (torchrun); independent units, no data-path collective -> weak scaling; time = max over
          ranks.  Extra keys: c3_batch (BASELINE configs[2]), dist_chol (configs[4]: block-cyclic Cholesky n = 150000
          with its parity block at n = 30000 against the single-GPU factorisation and the CPU oracle).
  --impl reference : the CPU restatement of the reference path (oracle/, NumPy/SciPy/OpenBLAS on all host cores;
          jax/gvar are not installable here so the reference itself cannot run) on a bounded sample of the same
          workload, every phase extrapolated with its own exponent, plus one measured full-size value-only evaluation.
"""

import os
import sys

if any(a == 'reference' or a == '--impl=reference' for a in sys.argv):
    # torchrun exports OMP_NUM_THREADS=1: the CPU arm uses every host core whatever launched it (set before numpy loads)
    for _v in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
        os.environ[_v] = str(os.cpu_count() or 1)

import argparse
import json
import math
import subprocess
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'logML+gradient evaluations/s at n=20000 fp64 (Gram+Chol+solve+inverse+VJP)'
UNIT = 'evals/s'
FP64_DMMA_PEAK_FALLBACK = 37.0   # round-1 measurement (profiles/peaks_fp64_r1.log); the line reports the live probe

# DRAM traffic of one lgp_chol_factor call at n=20000 comes from an ncu capture (it cannot be measured in this process)
CHOL_TRAFFIC_BYTES_N20000 = 47.37e9   # profiles/traffic_chol20k_r2c.txt (33.5 GB read + 13.8 GB written)


def make_data(n, seed=2002):
    """ SURVEY.md section 8(d), config C2 """
    rng = np.random.default_rng(seed)
    X = rng.uniform(0, 10, (n, 3))
    y = np.sin(X[:, 0]) + np.cos(X[:, 1]) * X[:, 2] / 10 + 0.1 * rng.standard_normal(n)
    return X, y


def make_data_c3(n=10000, seed=3003):
    """ SURVEY.md section 8(d), config C3 """
    rng = np.random.default_rng(seed)
    X = rng.uniform(0, 100, (n, 2))
    y = np.sin(X[:, 0] / 5) + np.cos(X[:, 1] / 7) + 0.1 * rng.standard_normal(n)
    return X, y


def theta_for(i):
    """ hyperparameter point i of the batch: (log ell, log sigma_f, log sigma_n) """
    rng = np.random.default_rng(3004 + i)
    return np.array([np.log(1.5), 0.0, np.log(0.1)]) + 0.05 * rng.standard_normal(3)


# --------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores
# --------------------------------------------------------------------------------------------------------------

PHASE_EXPONENT = dict(gram=2, chol=3, solve=2, inverse=3, dgram=2)   # cost of each oracle phase as a power of n


def c2_terms(theta):
    ell, sf, sn = np.exp(theta)
    return [(sf ** 2, [dict(kind='matern', nu=2.5, scale=ell)]), (sn ** 2, [dict(kind='white')])]


def cpu_eval(X, y, theta, timers=None):
    from oracle import gp as ogp
    ell, sf, sn = np.exp(theta)
    val, g = ogp.logml_and_grad(c2_terms(theta), X.T.copy(), y, [('logscale', 0, 0), ('amp', 0), ('amp', 1)],
                                timers=timers)
    return val, np.array([g[0], g[1] * 2 * sf ** 2, g[2] * 2 * sn ** 2])


def use_all_cores():
    """ pin the BLAS pool to every host core (torchrun sets OMP_NUM_THREADS=1); returns (limiter, threads in use) """
    cores = os.cpu_count() or 1
    lim = None
    try:
        import threadpoolctl
        lim = threadpoolctl.threadpool_limits(limits=cores)
        infos = threadpoolctl.threadpool_info()
        if infos:
            cores = max(i.get('num_threads', 1) for i in infos)
    except Exception:
        pass
    return lim, cores


def cpu_phase_model(n_full, sizes, reps=1):
    """ time the oracle's phases at the sizes in `sizes` (largest last) and extrapolate EACH phase to n_full with its
    own exponent (Gram / derivative Gram / solves ~ n^2, Cholesky / inverse ~ n^3); the measured exponents between
    the two largest sizes are reported next to the nominal ones. """
    meas = {}
    for n in sizes:
        X, y = make_data(n)
        best = None
        for r in range(reps):
            t = {}
            t0 = time.perf_counter()
            cpu_eval(X, y, theta_for(r), timers=t)
            t['total'] = time.perf_counter() - t0
            if best is None or t['total'] < best['total']:
                best = t
        meas[n] = best
    n1 = sizes[-1]
    ext = {p: meas[n1][p] * (n_full / n1) ** e for p, e in PHASE_EXPONENT.items()}
    fitted = None
    if len(sizes) > 1:
        n0 = sizes[-2]
        fitted = {p: round(math.log(max(meas[n1][p], 1e-9) / max(meas[n0][p], 1e-9)) / math.log(n1 / n0), 2)
                  for p in PHASE_EXPONENT}
    return dict(n_measured=n1, seconds_measured=meas[n1]['total'],
                phases_seconds_measured={p: meas[n1][p] for p in PHASE_EXPONENT},
                phases_seconds_extrapolated=ext, seconds_extrapolated=sum(ext.values()),
                exponents_nominal=PHASE_EXPONENT, exponents_fitted=fitted,
                sizes={str(n): meas[n]['total'] for n in sizes})


def cpu_baseline(n_full, n_sample):
    """ cpu_baseline key of the GPU arm (N = 1 only): bounded sample, per-phase extrapolation """
    lim, cores = use_all_cores()
    X, y = make_data(500)
    cpu_eval(X, y, theta_for(0))  # warm up the BLAS threads
    sizes = [n_sample // 2, n_sample] if n_sample >= 1000 else [n_sample]
    m = cpu_phase_model(n_full, sizes)
    return dict(value=1.0 / m['seconds_extrapolated'], unit=UNIT, cores=cores, kind='port', extrapolated=True,
                n_measured=m['n_measured'],
                sample=f"oracle (NumPy/SciPy OpenBLAS restatement of the reference path, {cores} threads) logML+gradient "
                       f"measured at n={m['n_measured']} in {m['seconds_measured']:.2f} s; each phase extrapolated to "
                       f"n={n_full} with its own exponent (gram/solve/dgram n^2, chol/inverse n^3) -> "
                       f"{m['seconds_extrapolated']:.1f} s per evaluation",
                model=m)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    lim, cores = use_all_cores()
    n_sample = args.ref_n
    if n_sample <= 0:
        # bounded sample: about 100 s for the K + W steps (a step costs ~15 s at n=5000, mostly the n^2 scipy.special.kv Gram)
        n_sample = int(min(5000, max(2000, 5000 * math.sqrt(100.0 / (15.0 * max(args.steps + args.warmup, 1))))))
        n_sample -= n_sample % 100
    X, y = make_data(n_sample)
    cpu_eval(X[:500], y[:500], theta_for(0))
    for w in range(args.warmup):
        cpu_eval(X, y, theta_for(w))
    per = []
    t0 = time.perf_counter()
    for s in range(args.steps):
        t = {}
        cpu_eval(X, y, theta_for(s), timers=t)
        per.append(t)
    t_sample = (time.perf_counter() - t0) / args.steps
    phases = {p: float(np.mean([t[p] for t in per])) for p in PHASE_EXPONENT}
    ext = {p: phases[p] * (args.n / n_sample) ** e for p, e in PHASE_EXPONENT.items()}
    fitted = None
    if n_sample >= 1000:
        Xh, yh = make_data(n_sample // 2)
        th = {}
        cpu_eval(Xh, yh, theta_for(0), timers=th)
        fitted = {p: round(math.log(max(phases[p], 1e-9) / max(th[p], 1e-9)) / math.log(2.0), 2) for p in PHASE_EXPONENT}
    # one MEASURED full-size evaluation (value only: Gram + Cholesky + forward solve); its phases replace the
    # extrapolated ones, so that only the gradient part (inverse, derivative Gram) of the figure is extrapolated
    full = None
    used = dict(ext)
    if args.ref_full and args.n >= 2 * n_sample:
        try:
            import psutil
            if psutil.virtual_memory().available > 2.5 * 8 * args.n ** 2:
                from oracle import gp as ogp
                Xf, yf = make_data(args.n)
                tm = {}
                t1 = time.perf_counter()
                v, L, eps = ogp.logml_value_lean(c2_terms(theta_for(0)), Xf.T.copy(), yf, timers=tm)
                full = dict(n=args.n, seconds=time.perf_counter() - t1, phases_seconds=tm, neg_logml=float(v),
                            extrapolated_same_phases_seconds=dict(gram=ext['gram'], chol=ext['chol']),
                            note='value-only evaluation (Gram + Cholesky + forward solve), measured at full size')
                del L
                used['gram'], used['chol'] = tm['gram'], tm['chol']
            else:
                full = dict(skipped='host RAM')
        except Exception as e:  # never lose the line to the optional full-size run
            full = dict(error=repr(e)[:200])
    t_full = sum(used.values())
    value = 1.0 / t_full
    measured = 'gram and chol measured at full size, ' if full and 'seconds' in full else ''
    sample = (f'each step = oracle logML+gradient at n={n_sample} ({t_sample:.2f} s measured, {cores} threads); {measured}'
              f'the other phases extrapolated to n={args.n} with their own exponents (solve/dgram n^2, inverse n^3) -> '
              f'{t_full:.1f} s per evaluation; the reference itself needs jax+gvar, not installable here')
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=t_full * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f64',
                data='synthetic', impl='reference', extrapolated=True, n_measured=n_sample,
                ms_per_step_measured_sample=t_sample * 1e3,
                scale=dict(exponents_nominal=PHASE_EXPONENT, exponents_fitted=fitted, phases_seconds_measured=phases,
                           phases_seconds_extrapolated=ext, phases_seconds_used=used),
                full_size_value_only=full,
                config=dict(workload=f'Matern(nu=2.5) 3-D n={args.n} fp64 logML+gradient (BASELINE configs[1])',
                            n=args.n, d=3, kernel='sf^2*Matern(nu=2.5, scale=ell) + sn^2*White'),
                cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind='port', sample=sample, extrapolated=True,
                                  n_measured=n_sample),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------------------

def c5_problem(n):
    """ BASELINE.json configs[4] / SURVEY.md 8(d) C5: X = U(0,1000)^2 (density kept for other n), ExpQuad(scale=5) + 0.01 I """
    from lsqfitgp_b200 import _lib
    box = 1000.0 * math.sqrt(n / 150000.0)
    rng = np.random.default_rng(5005)
    X = rng.uniform(0, box, (n, 2))
    b = rng.standard_normal(n)
    descs = [dict(kind=_lib.K_EXPQUAD, term=0, dimmask=3, scale_x=5.0, scale_y=5.0, amp=1.0),
             dict(kind=_lib.K_WHITE, term=1, dimmask=3, amp=0.01)]
    terms = [(1.0, [dict(kind='expquad', scale=5.0)]), (0.01, [dict(kind='white')])]
    return X, b, descs, terms


def llt_check(dc, n, dev, nvec=4):
    """ max over `nvec` random v of |L(L^T v) - (K + eps S^2) v| / |(K + eps S^2) v| (K regenerated strip-wise) """
    import torch
    worst = 0.0
    g = torch.Generator(device='cpu').manual_seed(77)
    for _ in range(nvec):
        v = torch.randn(n, generator=g, dtype=torch.float64).to(dev)
        kv = dc.matvec(v)
        llv = dc.correlate(dc.back_correlate(v))
        worst = max(worst, float((llv - kv).norm().item() / kv.norm().item()))
    return worst


def dist_chol_parity(n, tile, dev, rank, world, oracle=True):
    """ SURVEY.md 8(d) C5 parity items on the ranks of this run: DistChol at n (default 30000) against (i) the single-GPU
    lgp_chol_factor path on every rank, (ii) the CPU oracle value on rank 0, (iii) L(L^T v) = K v for 4 random v. """
    import torch
    import torch.distributed as dist
    from lsqfitgp_b200 import _dist, _ops, _linalg
    X, b, descs, terms = c5_problem(n)
    x = torch.tensor(np.ascontiguousarray(X.T)).to(dev)
    bd = torch.tensor(b).to(dev)
    dc = _dist.DistChol(descs, x, tile=tile)
    ld_d, sol_d, eps_d = dc.logdet(), dc.solve(bd), dc.eps
    quad_d = float((bd * sol_d).sum().item())
    out = dict(n=n, tile=tile, grid=[dc.lay.Pr, dc.lay.Pc], panel_broadcast=getattr(dc, 'peer_mode', 'nccl'))
    out['llt_v_relerr_max4'] = llt_check(dc, n, dev)
    del dc
    torch.cuda.empty_cache()
    # (i) single-GPU factorisation of the same matrix (every rank has a GPU of its own)
    K = _ops.gram_iso(descs, x, x, symmetric=True)
    ch = _linalg.Chol(K)
    del K
    ldq, _ = ch.logdet_quad(None)
    ld_s = 2.0 * float(ldq[0].item())
    sol_s = ch.ginv_linear(bd)
    eps_s = ch.eps
    out['vs_single_gpu'] = dict(
        logdet_relerr=abs(ld_d - ld_s) / abs(ld_s),
        solve_relerr=float((sol_d - sol_s).norm().item() / sol_s.norm().item()),
        eps_relerr=abs(eps_d - eps_s) / abs(eps_s))
    del ch
    torch.cuda.empty_cache()
    # (ii) CPU oracle on rank 0 (one n x n host buffer; skipped when the host lacks the RAM)
    if oracle and rank == 0:
        try:
            import psutil
            if psutil.virtual_memory().available > 2.5 * 8 * n * n:
                from oracle import gp as ogp
                from scipy import linalg
                use_all_cores()
                t0 = time.perf_counter()
                v, L, eps_o = ogp.logml_value_lean(terms, np.ascontiguousarray(X.T), b)
                ld_o = 2.0 * float(np.sum(np.log(np.diagonal(L))))
                y1 = linalg.solve_triangular(L, b, lower=True, check_finite=False)
                quad_o = float(y1 @ y1)
                val_o = 0.5 * (n * math.log(2 * math.pi) + ld_o + quad_o)
                val_d = 0.5 * (n * math.log(2 * math.pi) + ld_d + quad_d)
                out['vs_cpu_oracle'] = dict(logdet_relerr=abs(ld_d - ld_o) / abs(ld_o),
                                            quad_relerr=abs(quad_d - quad_o) / abs(quad_o),
                                            neg_logml_relerr=abs(val_d - val_o) / abs(val_o),
                                            eps_relerr=abs(eps_d - eps_o) / abs(eps_o),
                                            oracle_seconds=time.perf_counter() - t0)
                del L
            else:
                out['vs_cpu_oracle'] = dict(skipped='host RAM')
        except Exception as e:
            out['vs_cpu_oracle'] = dict(error=repr(e)[:200])
    if world > 1:
        dist.barrier()
    bars = dict(logdet=1e-12, solve=1e-10, eps=1e-12, llt=1e-12, oracle=1e-9)
    s = out['vs_single_gpu']
    ok = (s['logdet_relerr'] <= bars['logdet'] and s['solve_relerr'] <= bars['solve'] and s['eps_relerr'] <= bars['eps']
          and out['llt_v_relerr_max4'] <= bars['llt'])
    o = out.get('vs_cpu_oracle')
    if o and 'logdet_relerr' in o:
        ok = ok and o['logdet_relerr'] <= bars['oracle'] and o['neg_logml_relerr'] <= bars['oracle']
    out['bars'] = bars
    out['pass'] = bool(ok)
    return out


def dist_chol_measure(n, tile, dev, rank, world, dmma_peak, reps=1):
    """ Block-cyclic multi-GPU Cholesky (BASELINE.json configs[4] / SURVEY.md 8(d) C5): K generated tile-wise in place,
    factor, solve K x = b, logdet.  Device-timed (CUDA events on each rank's main stream), max over ranks. """
    import torch
    import torch.distributed as dist
    from lsqfitgp_b200 import _dist, _ops
    X, b, descs, _ = c5_problem(n)
    Xh = torch.tensor(np.ascontiguousarray(X.T)).pin_memory()
    bh = torch.tensor(b).pin_memory()

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up at a small size: NCCL broadcast channels, kernel attributes, allocator
    w = _dist.DistChol(descs, Xh[:, :4096].to(dev), tile=min(tile, 512))
    w.solve(bh[:4096].to(dev))
    del w
    _dist.peer_reserve(n, tile, dev)  # pooled peer-mapped slab buffers of the fused TRSM -> broadcast path (allocation)
    best = None
    for _ in range(reps):
        sync()
        t0 = time.perf_counter()
        x = Xh.to(dev, non_blocking=True)                       # e2e: host -> device copy of the points
        dc = _dist.DistChol(descs, x, tile=tile)
        ld = dc.logdet()                                        # device -> host read of the result
        torch.cuda.synchronize()
        t_e2e = time.perf_counter() - t0
        fms = dc.factor_ms()
        sync()
        t0 = time.perf_counter()
        sol = dc.solve(bh.to(dev))
        torch.cuda.synchronize()
        t_solve = time.perf_counter() - t0
        tt = torch.tensor([fms, t_e2e * 1e3, t_solve * 1e3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        fms, e2e_ms, solve_ms = (float(v) for v in tt.cpu())
        if best is None or fms < best['factor_ms']:
            best = dict(factor_ms=fms, e2e_ms=e2e_ms, solve_ms=solve_ms, logdet=ld)
        # size-independent checks: residual of the jittered system on 512 sampled rows, and L (L^T v) = K v
        idx = torch.as_tensor(np.random.default_rng(1).choice(n, 512, replace=False), device=dev)
        Ks = _ops.gram_iso(descs, x.index_select(1, idx).contiguous(), x)
        r = Ks @ sol + float(dc._epsout[1].item()) * (dc.s[idx] ** 2) * sol[idx] - bh.to(dev)[idx]
        best['resid_sampled'] = float(r.norm().item() / bh[idx.cpu()].norm().item())
        del Ks
        best['llt_v_relerr_max4'] = llt_check(dc, n, dev)
        grid = [dc.lay.Pr, dc.lay.Pc]
        peer_mode = getattr(dc, 'peer_mode', 'nccl')
        del dc, sol
        torch.cuda.empty_cache()
    flops = n ** 3 / 3
    tf = flops / (best['factor_ms'] * 1e-3) / 1e12
    return dict(n=n, tile=tile, grid=grid, n_gpus=world, panel_broadcast=peer_mode, storage='lower-packed tiles',
                factor_ms=best['factor_ms'],
                factor_TFLOPs=tf,
                per_gpu_TFLOPs=tf / world, frac_of_dmma_peak=tf / world / dmma_peak, dmma_peak_TFLOPs=dmma_peak,
                e2e_ms=best['e2e_ms'], e2e_TFLOPs=flops / (best['e2e_ms'] * 1e-3) / 1e12,
                solve_ms=best['solve_ms'], logdet=best['logdet'], resid_sampled=best['resid_sampled'],
                llt_v_relerr_max4=best['llt_v_relerr_max4'],
                h2d_bytes=n * 2 * 8, d2h_bytes=8,
                note='n^3/3 flop; Gram generated in place by tile owners; e2e = H2D of points + Gram + equilibration + '
                     'factor + logdet readback; panel_broadcast: multimem = TRSM epilogue stores through the NVSwitch '
                     'multicast mapping, p2p = one NVLink store per peer, nccl = copy + ncclBroadcast; llt_v = '
                     '|L(L^T v) - (K + eps S^2) v| / |.| with K regenerated strip-wise, 4 random v')


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.stop_flag = threading.Event()
        self.maxmhz = None

    def run(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(['nvidia-smi', f'--id={self.index}', f'--query-gpu={q}',
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(',')]
                self.samples.append(float(parts[0]))
                self.maxmhz = float(parts[1])
                for nm, v in zip(names, parts[2:]):
                    if v.lower().startswith('active'):
                        self.reasons.add(nm)
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.samples:
            return dict(sm_mhz=None, sm_max_mhz=self.maxmhz, reasons=sorted(self.reasons))
        return dict(sm_mhz=float(np.median(self.samples)), sm_max_mhz=self.maxmhz, reasons=sorted(self.reasons),
                    samples=len(self.samples))


def measure_fp64_peaks(dev):
    """ live roofline denominators: the library's register-resident DMMA.8x8x4 / DFMA loops (lgp_peak_probe), timed with
    CUDA events: burst = best of 5 short launches, sustained = back-to-back launches for about a second """
    import ctypes
    import torch
    from lsqfitgp_b200 import _lib
    lib = _lib.load()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    scratch = torch.empty(512 * sms, dtype=torch.float64, device=dev)
    fl = ctypes.c_double(0.0)
    out = {}
    for kind, name in ((0, 'dmma'), (1, 'dfma')):
        def launch(iters):
            _lib.check(lib.lgp_peak_probe(_lib.stream_ptr(), kind, iters, _lib.ptr(scratch), scratch.numel(),
                                          ctypes.byref(fl)), 'lgp_peak_probe')
            return fl.value
        launch(1000)
        torch.cuda.synchronize()
        best = 0.0
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f = launch(20000)
            e1.record()
            e1.synchronize()
            best = max(best, f / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        out[name + '_burst_TFLOPs'] = best
        if kind == 0:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            tot = 0.0
            for _ in range(20):
                tot += launch(100000)
            e1.record()
            e1.synchronize()
            out['dmma_sustained_TFLOPs'] = tot / (e0.elapsed_time(e1) * 1e-3) / 1e12
            out['dmma_sustained_seconds'] = e0.elapsed_time(e1) * 1e-3
    return out


DUMP_FACTOR_SAMPLES = 1 << 20


def dump_outputs(path, last):
    """ --dump-outputs: what the last timed evaluation computed, as float64 .npy files (8.5 MB at n = 20000): the
    negative log marginal likelihood, its gradient w.r.t. (log ell, log sigma_f, log sigma_n), the diagonal of the
    Cholesky factor L and a fixed seeded sample of 2^20 entries of its lower triangle (the whole of L is 3.2 GB) """
    import torch
    from lsqfitgp_b200 import _ops
    st = last['st']
    n = st.n
    L = _ops.chol_get_factor(st)
    rng = np.random.default_rng(6006)
    i, j = rng.integers(0, n, (2, DUMP_FACTOR_SAMPLES))
    flat = torch.as_tensor(np.maximum(i, j) * n + np.minimum(i, j), device=L.device)
    arrays = dict(neg_logml=np.array([last['val']]), neg_logml_grad=last['grad'],
                  chol_factor_diag=torch.diagonal(L).cpu().numpy(),
                  chol_factor_sample=L.reshape(-1).index_select(0, flat).cpu().numpy())
    del L
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), np.asarray(a, dtype=np.float64))


def run_gpu(args):
    import torch
    import torch.distributed as dist
    import lsqfitgp_b200 as lgp
    from lsqfitgp_b200 import _lib, _ops

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    lib = _lib.load()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxrank(*vals):
        if world == 1:
            return [float(v) for v in vals]
        tt = torch.tensor(vals, dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return [float(v) for v in tt.cpu()]

    peaks = measure_fp64_peaks(dev)
    dmma_peak = peaks['dmma_sustained_TFLOPs']   # the factorisation is timed inside a long step: sustained figure

    n = args.n
    X, y = make_data(n)
    xd = torch.tensor(np.ascontiguousarray(X.T)).to(dev)          # (3, n) field-major, resident in HBM
    yd = torch.tensor(y).to(dev)
    names = ['f0', 'f1', 'f2']

    def descs_for(theta):
        ell, sf, sn = np.exp(theta)
        return [dict(kind=_lib.K_MATERNP, term=0, dimmask=7, ipar=2, par0=0.0, scale_x=ell, scale_y=ell, amp=sf ** 2),
                dict(kind=_lib.K_WHITE, term=1, dimmask=7, amp=sn ** 2)]

    # events: 0 gram 1 [factorisation on the main stream; the library starts the inverse of the leading half on the side
    # stream behind the half-way panel] 2 [solves on the main stream | rest of the inverse on the side stream] 3 [join] 4 vjp 5
    phases = ['gram_fused_into_next_phase', 'gram_chol_overlapped_with_early_inverse', 'solves_overlapped_with_inverse', 'inverse_tail_after_solves',
              'vjp']
    K = _ops.aligned_empty(n, n, dev)
    side = torch.cuda.Stream(dev)
    ev_log = []

    def step_device(theta, Kbuf=None, record=False, side_stream=None):
        """ one logML+gradient evaluation with device-resident inputs, straight through the C ABI """
        descs = descs_for(theta)
        Kb = K if Kbuf is None else Kbuf
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)] if record else None

        def mark(i):
            if ev is not None:
                ev[i].record()
        mark(0)
        # Gram build fused with the equilibration pass (lgp_gram_iso_prepare: K itself is never written), then
        # factorisation + inverse-from-factor in one library call (lgp_chol_factor_inverse_prepared): the inverse runs on a
        # side stream, the latency-bound triangular solves on the main stream overlap it (the public API does the same in
        # _GP._FusedNegLogMLFn.forward)
        main = torch.cuda.current_stream()
        sd = side if side_stream is None else side_stream
        mark(1)
        fused = _ops.gram_chol_factor(descs, xd, side=sd)
        if fused is None:   # (kernel outside the fused family: not the case for the headline config)
            _ops.gram_iso(descs, xd, xd, out=Kb, symmetric=True)
            fused = _ops.chol_factor_inverse(Kb, sd)
        st, Kinv = fused
        mark(2)
        a = _ops.chol_solve(st, yd[:, None], False)
        ldq = _ops.chol_logdet_quad(st, a[:, 0].contiguous())
        b = _ops.chol_solve(st, a, True, inplace=True)
        mark(3)
        main.wait_stream(sd)
        Kinv.record_stream(main)
        mark(4)
        vjp = _ops.gram_iso_vjp(descs, xd, Kinv, b[:, 0].contiguous())
        mark(5)
        if record:
            ev_log.append(ev)
        return ldq, vjp, st

    def finish(theta, ldq, vjp):
        ld, q = ldq.cpu().numpy()
        v = vjp.cpu().numpy()
        ell, sf, sn = np.exp(theta)
        val = 0.5 * (n * math.log(2 * math.pi) + 2 * ld + q)
        grad = 0.5 * np.array([v[0, 1], v[0, 0] * 2 * sf ** 2, v[1, 0] * 2 * sn ** 2])
        return val, grad

    record_flag = [False]
    last = {}   # --dump-outputs: the latest evaluation of the device arm (its factor stays alive until the next one)

    def fun_device(theta):
        """ unit of the sharded batch: (neg logML, gradient) of one hyperparameter point, device-resident inputs """
        ldq, vjp, st = step_device(theta, record=record_flag[0])
        assert int(st.info.item()) == 0
        val, grad = finish(theta, ldq, vjp)
        if args.dump_outputs:
            last.update(val=val, grad=grad, st=st)
        return np.r_[val, grad]

    # pinned host staging for the end-to-end arm
    Xh = torch.empty((n, 3), dtype=torch.float64).pin_memory()
    Xh.copy_(torch.tensor(X))
    yh = torch.empty(n, dtype=torch.float64).pin_memory()
    yh.copy_(torch.tensor(y))
    Xnp, ynp = Xh.numpy(), yh.numpy()

    def fun_e2e(theta):
        """ public API from host buffers: H2D of x and y, D2H of (logML, gradient) """
        th = torch.tensor(theta, dtype=torch.float64, requires_grad=True)
        ell, sf, sn = torch.exp(th[0]), torch.exp(th[1]), torch.exp(th[2])
        kern = sf ** 2 * lgp.Matern(nu=2.5, scale=ell) + sn ** 2 * lgp.White()
        xs = lgp.unstructured_to_structured(Xnp, names=names)
        gp = lgp.GP(kern, checkpos=False, checksym=False, checkfinite=False).addx(xs, 'data')
        ml = gp.marginal_likelihood({'data': ynp})
        g, = torch.autograd.grad(ml, th)
        return np.r_[-float(ml.detach()), -g.numpy()]

    def batch(first, count):
        """ `count` hyperparameter points per rank, numbered from `first` """
        return np.stack([theta_for(first + i) for i in range(count * world)])

    def timed_batch(fun, thetas, in_flight=1):
        """ the product's sharding function on the whole batch; device-timed on this rank's current stream """
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        out = lgp.eval_batch_sharded(fun, thetas, device=dev, in_flight=in_flight)
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        t_dev = e0.elapsed_time(e1) / 1e3
        barrier()
        t_dev, wall = maxrank(t_dev, wall)
        return out, t_dev, wall

    # ---- correctness guard: the two arms agree (the oracle comparison lives in tests/ and smoke())
    th0 = theta_for(0)
    r_dev = fun_device(th0)
    r_api = fun_e2e(th0)
    assert abs(r_dev[0] - r_api[0]) <= 1e-9 * abs(r_dev[0]), (r_dev, r_api)
    assert np.max(np.abs(r_dev[1:] - r_api[1:])) <= 1e-9 * np.max(np.abs(r_dev[1:])), (r_dev, r_api)

    # ---- device-resident arm
    if args.warmup:
        timed_batch(fun_device, batch(1000, args.warmup))
    launches0 = lib.lgp_launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    record_flag[0] = True
    out_dev, t_dev, wall_dev = timed_batch(fun_device, batch(0, args.steps))
    record_flag[0] = False
    sampler.stop_flag.set()
    launches = lib.lgp_launch_count() - launches0
    assert out_dev.shape == (args.steps * world, 4) and np.all(np.isfinite(out_dev))
    phase_ms = {p: float(np.mean([ev[i].elapsed_time(ev[i + 1]) for ev in ev_log])) for i, p in enumerate(phases)}
    chol_inverse_span_ms = float(np.mean([ev[1].elapsed_time(ev[4]) for ev in ev_log]))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    last.clear()

    # ---- the Gram kernel alone (inside the step it is fused with the equilibration pass of the factorisation)
    gram_alone = []
    for _ in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _ops.gram_iso(descs_for(theta_for(0)), xd, xd, out=K, symmetric=True)
        e1.record()
        e1.synchronize()
        gram_alone.append(e0.elapsed_time(e1))
    gram_alone_ms = float(np.mean(gram_alone[1:]))

    # ---- the factorisation alone (lgp_chol_factor, nothing overlapped): the kernel-level roofline figure
    _ops.gram_iso(descs_for(theta_for(0)), xd, xd, out=K, symmetric=True)
    chol_alone = []
    for _ in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        st_ = _ops.chol_factor(K)
        e1.record()
        e1.synchronize()
        chol_alone.append(e0.elapsed_time(e1))
        del st_
    chol_alone_ms = float(np.mean(chol_alone[1:]))

    # ---- end-to-end arm
    if args.warmup:
        timed_batch(fun_e2e, batch(1000, min(args.warmup, 2)))
    out_e2e, _, t_e2e = timed_batch(fun_e2e, batch(0, args.steps))
    assert np.max(np.abs(out_e2e - out_dev)) <= 1e-8 * np.max(np.abs(out_dev))

    # ---- batch arm (extra key, not the headline): the same evaluations with `in_flight` of them in flight per GPU (one
    # host thread + stream per slot): the panel chains of one factorisation overlap the GEMMs of another
    batch_tp = None
    if args.in_flight > 1:
        nb = max(args.steps, 2 * args.in_flight)
        Ks = [K] + [_ops.aligned_empty(n, n, dev) for _ in range(args.in_flight - 1)]
        sides = [torch.cuda.Stream(dev) for _ in range(args.in_flight)]   # persistent: allocator pools stay warm
        slot_of = {}
        lock = threading.Lock()

        def fun_slot(theta):
            with lock:
                slot = slot_of.setdefault(threading.get_ident(), len(slot_of))
            ldq, vjp, st = step_device(theta, Kbuf=Ks[slot % args.in_flight], side_stream=sides[slot % args.in_flight])
            val, grad = finish(theta, ldq, vjp)
            return np.r_[val, grad]
        timed_batch(fun_slot, batch(2000, args.in_flight), in_flight=args.in_flight)   # warm-up: per-stream setup
        slot_of.clear()
        out_b, _, t_batch = timed_batch(fun_slot, batch(0, nb), in_flight=args.in_flight)
        assert abs(out_b[0, 0] - out_dev[0, 0]) <= 1e-12 * abs(out_dev[0, 0]), (out_b[0], out_dev[0])
        del Ks
        batch_tp = dict(value=nb * world / t_batch, unit=UNIT, in_flight=args.in_flight, evaluations_per_gpu=nb,
                        timing='host wall clock between device synchronisations (several streams)')
    del K
    torch.cuda.empty_cache()

    # ---- c3_batch (extra key): BASELINE configs[2], ExpQuad + noise, n = 10000, a batch of hyperparameter points theta_b
    # ~ prior (seed 3004), 8 per GPU (B = 64 on 8 GPUs), through the public API from host arrays, sharded by
    # eval_batch_sharded with `in_flight` swept
    c3 = None
    if args.c3_per_gpu > 0:
        X3, y3 = make_data_c3()
        x3 = lgp.unstructured_to_structured(X3, names=['a', 'b'])
        B3 = args.c3_per_gpu * world
        th3 = np.array([np.log(3), 0.0, np.log(0.1)]) + 0.5 * np.random.default_rng(3004).standard_normal((B3, 3))

        def fun_c3(theta):
            th = torch.tensor(theta, dtype=torch.float64, requires_grad=True)
            k = torch.exp(th[1]) ** 2 * lgp.ExpQuad(scale=torch.exp(th[0])) + torch.exp(th[2]) ** 2 * lgp.White()
            gp = lgp.GP(k, checkpos=False, checksym=False, checkfinite=False).addx(x3, 'data')
            ml = gp.marginal_likelihood({'data': y3})
            g, = torch.autograd.grad(ml, th)
            return np.r_[float(ml.detach()), g.numpy()]
        sweep = {}
        ref_out = None
        for c in (1, 2, 4):
            timed_batch(fun_c3, th3[:c * world], in_flight=c)
            o3, _, t3 = timed_batch(fun_c3, th3, in_flight=c)
            if ref_out is None:
                ref_out = o3
            else:
                assert np.max(np.abs(o3 - ref_out)) <= 1e-9 * np.max(np.abs(ref_out))
            sweep[str(c)] = B3 / t3
        bestc = max(sweep, key=sweep.get)
        c3 = dict(value=sweep[bestc], unit=UNIT, in_flight_best=int(bestc), evals_per_s_by_in_flight=sweep, batch=B3,
                  per_gpu=args.c3_per_gpu, n=10000,
                  workload='BASELINE configs[2]: sf^2*ExpQuad(scale=ell)+sn^2*White, n=10000 2-D, logML+gradient of a '
                           'batch theta_b ~ N((log 3, 0, log 0.1), 0.5^2) (seed 3004) via lgp.eval_batch_sharded + public API',
                  timing='host wall clock incl. H2D of x, y and D2H of results, max over ranks')
        torch.cuda.empty_cache()

    # ---- c1 latency (extra key, N = 1): BASELINE configs[0] through the public API
    c1 = None
    if world == 1 and args.c1:
        rng = np.random.default_rng(1001)
        x1 = np.sort(rng.uniform(0, 100, 1000))
        y1 = np.sin(x1 / 3) + 0.1 * rng.standard_normal(1000)
        xp = np.linspace(-5, 105, 500)
        ycov1 = {('d', 'd'): 0.01 * np.eye(1000)}

        def c1_fun():
            gp = lgp.GP(lgp.ExpQuad(scale=3), checkpos=False, checksym=False).addx(x1, 'd').addx(xp, 'p')
            ml = gp.marginal_likelihood({'d': y1}, ycov1)
            m, c = gp.predfromdata({'d': y1}, 'p', ycov1, raw=True)
            return ml
        for _ in range(3):
            c1_fun()
        torch.cuda.synchronize()
        ts = []
        for _ in range(10):
            t0 = time.perf_counter()
            c1_fun()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        c1 = dict(ms=min(ts) * 1e3, ms_median=float(np.median(ts)) * 1e3,
                  workload='BASELINE configs[0]: GP(ExpQuad(scale=3)) n=1000, marginal_likelihood + predfromdata on 500 '
                           'points, host arrays in / out (reference docs: 4.8 ms jitted on a laptop CPU)')

    # ---- c4_bart (extra key, N = 1): BASELINE configs[3], lgp.BART kernel at n = 5000, p = 10 (8 continuous + 2 binary
    # covariates): Gram build, Cholesky, and one objective + gradient evaluation of the bayestree.bart recipe
    # (lambda^2 BART(alpha, beta) + sigma^2 I + k^2 11', epsrel = 0; derivatives w.r.t. alpha, beta, lambda, sigma^2)
    c4 = None
    if world == 1 and args.c4:
        rng = np.random.default_rng(4004)
        n4 = 5000
        X4 = np.concatenate([rng.standard_normal((n4, 8)), rng.integers(0, 2, (n4, 2)).astype(float)], axis=1)
        y4 = rng.standard_normal(n4)
        splits = lgp.BART.splits_from_coord(X4)
        idx = lgp.BART.indices_from_coord(X4, splits)
        xi = lgp.unstructured_to_structured(idx.astype(np.int32), names=[f'c{i}' for i in range(10)])
        kb = lgp.BART(splits=splits, indices=True, alpha=0.95, beta=2, maxd=10, reset=[2, 4, 6, 8], gamma=1)
        ixd = torch.tensor(np.ascontiguousarray(idx.T.astype(np.float64)), device=dev)

        def dev_ms(fn, reps=5):
            fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            e1.synchronize()
            return e0.elapsed_time(e1) / reps
        gram_ms = dev_ms(lambda: kb._gram_device(ixd, ixd, None, symmetric=True))
        Kb = kb._gram_device(ixd, ixd, None, symmetric=True)
        Kb.diagonal().add_(0.1)
        chol_ms = dev_ms(lambda: _ops.chol_factor(Kb))
        del Kb

        def fit_step():
            th = torch.tensor([0.95, 2.0, 1.1, 0.5], dtype=torch.float64, requires_grad=True)
            k4 = th[2] ** 2 * lgp.BART(splits=splits, indices=True, alpha=th[0], beta=th[1], maxd=10, reset=[2, 4, 6, 8])
            gp4 = (lgp.GP(k4, checkpos=False, checksym=False, checkfinite=False, epsrel=0).addx(xi, 'trainmean')
                   .addcov(torch.diag((th[3] * torch.ones(n4, dtype=torch.float64)).to(dev)), 'trainnoise')
                   .addcov(0.49, 'mean').addtransf({'trainmean': 1, 'trainnoise': 1, 'mean': 1}, 'train'))
            ml = gp4.marginal_likelihood({'train': y4})
            g, = torch.autograd.grad(ml, th)
            return float(ml.detach()), g.numpy()
        fit_step()
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            fit_step()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        c4 = dict(n=n4, p=10, gram_ms=gram_ms, gram_Gpairs_per_s=n4 * n4 / (gram_ms * 1e-3) / 1e9, chol_ms=chol_ms,
                  chol_TFLOPs=n4 ** 3 / 3 / (chol_ms * 1e-3) / 1e12, recipe_value_and_gradient_ms=min(ts) * 1e3,
                  workload='BASELINE configs[3]: lgp.BART(maxd=10, reset=[2,4,6,8]) n=5000 p=10: symmetric Gram build, '
                           'Cholesky, and one bayestree.bart objective+gradient evaluation (alpha, beta, lambda, sigma^2) '
                           'through the public API, wall clock')
        torch.cuda.empty_cache()

    sampler.join(timeout=2)

    dist_chol = None
    if args.dist_n > 0 and (world > 1 or args.dist_n1 > 0):
        try:
            if world > 1:
                dist_chol = dist_chol_measure(args.dist_n, args.dist_tile, dev, rank, world, dmma_peak)
            else:
                # 1-GPU point of the curve: the largest n that fits one B200 with the dense local layout
                dist_chol = dist_chol_measure(args.dist_n1, args.dist_tile, dev, rank, world, dmma_peak)
                dist_chol['note_1gpu'] = ('same code path on a 1 x 1 process grid; lower-packed tile storage (84 GiB at '
                                          'n = 150000)')
            if args.dist_parity_n > 0:
                dist_chol['parity'] = {f'n{args.dist_parity_n}': dist_chol_parity(args.dist_parity_n, args.dist_tile, dev,
                                                                                  rank, world)}
        except Exception as e:  # never lose the headline line to the secondary measurement
            dist_chol = dict(error=repr(e)[:300])

    rc = 0
    if rank == 0:
        value = args.steps * world / t_dev
        e2e_value = args.steps * world / t_e2e
        chol_tflops = n ** 3 / 3 / (chol_alone_ms * 1e-3) / 1e12
        line = dict(
            metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
            ms_per_step=t_dev / args.steps * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None,
            dtype='f64', data='synthetic',
            config=dict(workload=f'Matern(nu=2.5) 3-D n={n} fp64 logML+gradient (BASELINE configs[1])', n=n, d=3,
                        kernel='sf^2*Matern(nu=2.5, scale=ell) + sn^2*White',
                        parallelism=f'hyperparameter batch of {args.steps * world} points sharded x{world} by '
                                    'lsqfitgp_b200.eval_batch_sharded (all_gather of results inside the timed region)',
                        l2='working set (3.2 GB matrix) exceeds the 126 MB L2; no flush needed'),
            clocks=sampler.summary(),
            e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=n * 3 * 8 + n * 8, d2h_bytes_per_step=4 * 8,
                     ms_per_step=t_e2e / args.steps * 1e3,
                     api='lgp.eval_batch_sharded(lgp.GP(kernel).addx(x).marginal_likelihood({..}) + torch.autograd.grad)'),
            gpu_launches=int(launches),
            wall_ms_per_step=wall_dev / args.steps * 1e3,
            roofline=dict(bound='tensor', kernel='gemm_dmma_kernel (Cholesky: lgp_chol_factor timed alone in this run, mean of 3 '
                                                 'calls after one warm-up; inside the step it overlaps the inverse)',
                          achieved=chol_tflops, peak=dmma_peak, unit='TFLOP/s',
                          frac=chol_tflops / dmma_peak,
                          traffic=CHOL_TRAFFIC_BYTES_N20000 if n == 20000 else None,
                          traffic_source='ncu dram__bytes_read.sum + dram__bytes_write.sum over the kernels of one '
                                         'lgp_chol_factor call at n=20000 (profiles/traffic_chol20k_r2c.txt; ncu cannot run '
                                         'inside this process): 33.5 GB read + 13.8 GB written (82.9 GB before the grouped '
                                         'rasterisation of the lower-triangular tile enumeration, profiles/traffic_chol20k_r2.txt); '
                                         'the right-looking updates re-read the trailing matrix once per panel; '
                                         'tensor-bound (0.56 TB/s average)',
                          peak_source='measured in THIS run: register-resident DMMA.8x8x4 loop of the library '
                                      '(lgp_peak_probe), sustained over %.1f s; burst %.2f; MEASURED_PEAKS.json has no '
                                      'FP64 entry' % (peaks['dmma_sustained_seconds'], peaks['dmma_burst_TFLOPs']),
                          peaks_measured=peaks,
                          algorithmic_flops_per_launch=n ** 3 / 3),
            phases_ms=phase_ms,
            chol_inverse_span_ms=chol_inverse_span_ms, chol_alone_ms=chol_alone_ms,
            phases_note='the Gram build writes the equilibrated lower triangle straight into the factor storage '
                        '(lgp_gram_iso_prepare; gram_alone_ms = the plain Gram kernel timed alone); one library call '
                        '(lgp_chol_factor_inverse_prepared) does the factorisation (main stream) and the '
                        'inverse-from-factor (side stream, leading half started behind the half-way panel): the phases of '
                        'the main stream are spans, not costs; chol_inverse_span_ms = Gram + factorisation + inverse together '
                        '(n^3 flop); chol_alone_ms = lgp_chol_factor with nothing overlapped',
            gram_alone_ms=gram_alone_ms,
            phase_rates=dict(gram_GBps=8 * n * n / (gram_alone_ms * 1e-3) / 1e9,
                             gram_frac_of_hbm_peak=8 * n * n / (gram_alone_ms * 1e-3) / 1e9 / hbm_peak(),
                             chol_TFLOPs=chol_tflops,
                             chol_plus_inverse_TFLOPs=n ** 3 / (chol_inverse_span_ms * 1e-3) / 1e12,
                             vjp_GBps=4 * n * n / (phase_ms['vjp'] * 1e-3) / 1e9,
                             step_TFLOPs=n ** 3 / (t_dev / args.steps) / 1e12,
                             step_frac_of_dmma_peak=n ** 3 / (t_dev / args.steps) / 1e12 / dmma_peak),
        )
        if batch_tp is not None:
            line['batch_throughput'] = batch_tp
        if c3 is not None:
            line['c3_batch'] = c3
        if c1 is not None:
            line['c1_latency'] = c1
        if c4 is not None:
            line['c4_bart'] = c4
        if dist_chol is not None:
            line['dist_chol'] = dist_chol
            par = dist_chol.get('parity') or {}
            if any(not v.get('pass', True) for v in par.values()):
                rc = 3   # a parity bar was missed: the run fails loudly (the line is still printed for diagnosis)
        if world == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'] = cpu_baseline(n, args.ref_n if args.ref_n > 0 else 5000)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return rc


def hbm_peak():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs'])
    except Exception:
        return 6530.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--n', type=int, default=20000)
    ap.add_argument('--ref-n', type=int, default=0,
                    help='sample size of the CPU baseline / reference arm (0: 5000 for the baseline key; for the reference '
                         'arm sized from --steps/--warmup so that the run ends within a few minutes)')
    ap.add_argument('--ref-full', type=int, default=1,
                    help='reference arm: also run ONE measured value-only evaluation at the full size (0: skip)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dist-n', type=int, default=150000,
                    help='size of the block-cyclic multi-GPU Cholesky reported under "dist_chol" at N > 1 (0 = skip)')
    ap.add_argument('--dist-n1', type=int, default=150000,
                    help='N = 1 only: size of the 1-GPU point of the dist_chol curve (lower-packed tiles: 84 GiB at '
                         'n = 150000 on one B200); 0 = skip')
    ap.add_argument('--dist-parity-n', type=int, default=30000,
                    help='size of the DistChol parity block (vs single-GPU factorisation and CPU oracle; 0 = skip)')
    ap.add_argument('--dist-tile', type=int, default=1024)
    ap.add_argument('--in-flight', type=int, default=2,
                    help='extra key batch_throughput: the same evaluations with this many in flight per GPU (0: skip)')
    ap.add_argument('--c3-per-gpu', type=int, default=8, help='extra key c3_batch: points per GPU (0: skip)')
    ap.add_argument('--c1', type=int, default=1, help='extra key c1_latency at N = 1 (0: skip)')
    ap.add_argument('--c4', type=int, default=1, help='extra key c4_bart at N = 1 (0: skip)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one computed as DIR/<name>.npy (float64, about '
                         '8.5 MB): neg_logml, neg_logml_grad, chol_factor_diag, chol_factor_sample; the inputs depend on '
                         'the arguments only, so two builds can be compared output for output')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs applies to the GPU arm (--impl ours)')
    if args.impl == 'reference':
        return run_reference(args)
    return run_gpu(args)


if __name__ == '__main__':
    sys.exit(main())
