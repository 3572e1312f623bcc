/*
 * lgp_b200.h -- C ABI of liblgpb200.so, the B200-native (sm_100a) GP-fitting hot path:
 * Gram-matrix build -> equilibrated, jittered dense Cholesky -> triangular solves, log-determinant,
 * inverse-from-factor and the hyperparameter-gradient contraction.
 *
 * The reference (Gattocrucco/lsqfitgp 0.22.dev0) is pure Python/JAX and has no FFI for this path; each
 * entry point below names the reference code it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every pointer is caller-owned DEVICE memory unless stated otherwise (torch tensors on the Python side)
 *   - matrices are row-major float64 with an explicit leading dimension in elements
 *   - `stream` is a cudaStream_t passed as void*; all calls are asynchronous on it and never synchronise
 *   - return value: 0 = launched ok; <0 = argument/launch error (LGP_ERR_*).  Numerical failure of the
 *     factorisation is reported in the device-side `info` word (LAPACK convention, 1-based pivot index)
 *   - every matrix and vector the library works on is the caller's: nothing is allocated on the data path.  On first use
 *     per device it creates a few CUDA streams and events (one high-priority panel stream per caller stream, side streams
 *     for the inverse recursion) and, per caller stream that issues vector solves (lgp_chol_solve with m = 1,
 *     lgp_tile_trsv), one 256 KiB flag workspace (cudaMalloc once: that first call synchronises the device)
 *   - thread safety: entry points may be called concurrently from several host threads on different streams
 *
 * Environment switches, for kernel experiments only (the product path needs none): LGP_TRACE (per-panel timeline of the
 * factorisation, synchronises), LGP_PANEL_BLOCKS (panel width in 128-blocks, default 4), LGP_TAIL_BLOCKS /
 * LGP_FIRST_BLOCKS / LGP_CHAIN_BLOCKS (panel schedule).
 */
#ifndef LGP_B200_H
#define LGP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LGP_ABI_VERSION 1

#define LGP_OK 0
#define LGP_ERR_BADARG (-1)
#define LGP_ERR_ALIGN (-2) /* pointer not 16-byte aligned or odd leading dimension */
#define LGP_ERR_CUDA (-3)
#define LGP_ERR_UNSUPPORTED (-4)

typedef void *lgp_stream_t;

int lgp_abi_version(void);
/* static string: compiler, arch, build flags */
const char *lgp_build_info(void);
/* number of CUDA kernel launches issued by the library since load (instrumentation for bench.py) */
long long lgp_launch_count(void);

/* Roofline probe: launches ONE register-resident loop kernel on `stream` (2 CTAs of 256 threads per SM, `iters`
 * iterations of 16 independent accumulators per thread) and stores the number of floating-point operations it performs
 * in *flops_out (HOST).  kind = LGP_PEAK_DMMA: mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4, the FP64 tensor pipe the
 * factorisation runs on); LGP_PEAK_DFMA: scalar DFMA.  The caller times the launch with CUDA events: bench.py measures
 * the denominators of roofline.frac in the run that reports them.  scratch: device, >= 512 * (number of SMs) doubles. */
#define LGP_PEAK_DMMA 0
#define LGP_PEAK_DFMA 1
int lgp_peak_probe(lgp_stream_t stream, int kind, int iters, double *scratch, int64_t scratch_doubles,
                   double *flops_out /*host*/);

/* ------------------------------------------------------------------------------------------------
 * Gram matrix of a sum of products of isotropic kernel factors.
 * Replaces GPElements._makecovblock_points -> CrossKernel.__call__ -> IsotropicKernel core
 * (src/lsqfitgp/_GP/_elements.py:554-579, _Kernel/_crosskernel.py:192-200, _Kernel/_ops.py:292-326,
 *  _Kernel/_isotropic.py:61-81, _Kernel/_util.py:74-99, _kernels/_basic.py:34-75,315-343,
 *  _kernels/_matern.py:29-76, _special/_bessel.py:101-110, _Kernel/_alg.py:48-82).
 *
 *   K[i][j] = sum_terms prod_{factors f in term} amp_f * core_f( r2_f(i,j) )
 *   r2_f(i,j) = sum_{fields d in dimmask_f, ascending} ( (x[d][i]-loc_x)/scale_x - (y[d][j]-loc_y)/scale_y )^2
 * with every operation individually rounded (no FMA contraction), as the reference does.
 * ---------------------------------------------------------------------------------------------- */
#define LGP_K_EXPQUAD 0  /* exp(-r2/2)                                   _basic.py:75 */
#define LGP_K_MATERNP 1  /* half-integer Matern, nu = ipar + 1/2; par0 = offset added to (2p+1)*r2
                            (1e-30 for Maternp, 0 for Matern(nu=p+1/2))   _matern.py:48-49,74-76 */
#define LGP_K_CAUCHY 2   /* (1 + r2^(par0/2)/par1)^(-par1/par0)           _basic.py:339-343 */
#define LGP_K_WHITE 3    /* prod_d (x_d == y_d)                           _basic.py:59 */
#define LGP_K_CONSTANT 4 /* 1                                             _basic.py:46 */
#define LGP_K_MATERN 5   /* Matern of real order nu = par0 in [0, 100]: 2/Gamma(nu) (x/2)^nu K_nu(x), x = sqrt(2 nu r2),
                            K_nu evaluated in the kernel (Temme series / Steed CF2); the reference calls
                            scipy.special.kv on the host            _matern.py:55-76, _special/_bessel.py:70-99 */

#define LGP_MAX_FACTORS 8
#define LGP_MAX_DIMS 32

typedef struct lgp_factor {
    int32_t kind;     /* LGP_K_* */
    int32_t term;     /* additive term index; factors with equal term multiply */
    uint32_t dimmask; /* bit d set: field d enters r2 */
    int32_t ipar;     /* MATERNP: p */
    double scale_x, scale_y, loc_x, loc_y;
    double par0, par1;
    double amp;
} lgp_factor_t;

/* x: ndim fields of n points, x[d*ldx + i]; y likewise (m points).  K_out[i*ldk + j], i<n, j<m.
 * `factors` is HOST memory (copied into kernel parameters).
 * flags: LGP_GRAM_SYMMETRIC asserts x==y (same pointer): lower tiles are evaluated once and mirrored. */
#define LGP_GRAM_SYMMETRIC 1
#define LGP_GRAM_GENERAL 2 /* force the general (sum-of-products) kernel even when the fast path applies */
#define LGP_GRAM_LIBM 4    /* fast path with CUDA libm exp/sqrt instead of the short in-kernel versions (A/B checks) */
int lgp_gram_iso(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                 int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, double *K_out, int64_t ldk,
                 int flags);

/* Reverse-mode contraction of the Gram build (what jax.vjp of the Gram function gives the reference,
 * src/lsqfitgp/_fit.py:687-702), without materialising dK:
 *   out[3f+0] = sum_ij G_ij * dK_ij/d amp_f
 *   out[3f+1] = sum_ij G_ij * dK_ij/d log(scale_f)        (scale_x == scale_y == scale_f)
 *   out[3f+2] = sum_ij G_ij * dK_ij/d par1_f              (Cauchy beta; 0 otherwise)
 * symlower = 0: G is a dense n x m matrix (ldg).  symlower = 1: x == y and G_ij = w_ij (G[i][j] - b_i b_j) read from
 * the LOWER triangle only, w = 2 off the diagonal: with G = (K+eps)^-1 and b = K^-1 r this is
 * dK_vjp(invK) - dK_vjp(outer(invKr, invKr)) of Chol.minus_log_normal_density collapsed into one pass
 * (src/lsqfitgp/_linalg/_decomp.py:505-509).  b may be NULL.  out: device memory, 3*nfactors + 8 doubles (the tail is scratch)
 * (accumulated with atomicAdd: summation order, hence the last bits, may vary from run to run). */
int lgp_gram_iso_vjp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                     int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, const double *G, int64_t ldg,
                     const double *b, int symlower, double *out);

/* Forward-mode derivative of the Gram build (what jax.jacfwd of decomp.matrix() gives the reference for the Fisher
 * matrix, src/lsqfitgp/_fit.py:676-683, _linalg/_decomp.py:535-558), one tangent direction at a time:
 *   D[i][j] = sum_f tangent[3f+0] dK_ij/d amp_f + tangent[3f+1] dK_ij/d log(scale_f) + tangent[3f+2] dK_ij/d par1_f
 * `tangent` is HOST memory (3*nfactors doubles, same layout as the output of lgp_gram_iso_vjp). */
int lgp_gram_iso_jvp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                     int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, const double *tangent,
                     double *D_out, int64_t ldd);

/* Second-order contraction of the Gram build, the derivative of lgp_gram_iso_vjp along `tangent` (what a second
 * jax.vjp through the Gram build gives the reference's Hessian, src/lsqfitgp/_fit.py empbayes_fit(method='hessian'),
 * without materialising the k^2 matrices d2K/dtheta_a dtheta_b):
 *   out[3f+k] = sum_ij G_ij d/dtheta_{f,k} ( sum_{g,l} tangent[3g+l] dK_ij/dtheta_{g,l} ),
 *   theta_{f,.} = (amp_f, log(scale_f), par1_f)      (scale_x == scale_y == scale_f)
 * G, b and symlower as in lgp_gram_iso_vjp; `tangent` is HOST memory (3*nfactors doubles, the layout of
 * lgp_gram_iso_jvp).  Every kind of the general kernel.  out: device memory, 3*nfactors doubles (zeroed by the call;
 * accumulated with atomicAdd). */
int lgp_gram_iso_hvp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                     int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, const double *G, int64_t ldg,
                     const double *b, int symlower, const double *tangent, double *out);

/* Derivatives of the Gram build with respect to the points (what jax differentiating through the points of `gpfactory`
 * gives the reference, src/lsqfitgp/_fit.py:687-702).  For a factor with field d in its dimmask,
 *   dK/dx_{d,i} = amp c'(r2) 2 (u_{d,i} - v_{d,j}) / scale_x,   dK/dy_{d,j} = -amp c'(r2) 2 (u_{d,i} - v_{d,j}) / scale_y,
 * u = (x - loc_x)/scale_x, v = (y - loc_y)/scale_y, with the product rule across the factors of a term; White and
 * Constant contribute 0.  c' (u - v) is taken as 0 where u - v = 0, also where c' diverges at r = 0 (Maternp p = 0,
 * Matern of low order, Cauchy alpha < 2): the exact value on the diagonal, where K(x_i, x_i) is constant.
 *
 * Reverse mode: gx[d*ldgx + i] = sum_j G_ij dK_ij/dx_{d,i}, gy[d*ldgy + j] = sum_i G_ij dK_ij/dy_{d,j}.  symlower = 0:
 * G dense n x m (ldg), b_i b_j subtracted if b is not NULL; gx or gy may be NULL (not both).  symlower = 1: x == y,
 * G_ij = w_ij (G[i][j] - b_i b_j) read from the LOWER triangle only, w = 2 off the diagonal, as in lgp_gram_iso_vjp;
 * gx then receives the total derivative (both arguments) and gy must be NULL.  Outputs are device memory, zeroed by the
 * call (fields outside every dimmask stay 0), accumulated with atomicAdd: the last bits may vary from run to run. */
int lgp_gram_iso_xvjp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                      int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, const double *G, int64_t ldg,
                      const double *b, int symlower, double *gx, int64_t ldgx, double *gy, int64_t ldgy);

/* Forward mode: D[i][j] (+)= sum_d tx[d*ldtx + i] dK_ij/dx_{d,i} + ty[d*ldty + j] dK_ij/dy_{d,j}, tx and ty device
 * (ndim, n) / (ndim, m) arrays, either may be NULL (a zero tangent).  accumulate = 1 adds to D, 0 overwrites it. */
int lgp_gram_iso_xjvp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                      int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, const double *tx, int64_t ldtx,
                      const double *ty, int64_t ldty, double *D_out, int64_t ldd, int accumulate);

/* Derivative blocks: the covariance between first derivatives of the process, cov(d f(x)/d x_a, d f(y)/d y_b), with
 * a = dx_field, b = dy_field (field indices; -1 = no derivative on that argument, both -1 is LGP_ERR_BADARG).
 * Replaces the reference's jax derivatives of the kernel core behind addx(deriv=) and CrossKernel.linop('diff')
 * (src/lsqfitgp/_GP/_elements.py:190-242, _Kernel/_crosskernel.py:281-347, _Kernel/_ops.py:200-290):
 *   K[i][j] = d/dx_a d/dy_b k(x_i, y_j)   (only the derivatives requested),
 * the derivatives taken with respect to the raw coordinates (1/scale chain factors included).  Only first derivatives;
 * a factor that depends on a differentiated field must be ExpQuad, Maternp with p >= 1 or Cauchy with alpha = 2
 * (otherwise LGP_ERR_UNSUPPORTED); the other factors may be of any kind.  Same layouts as lgp_gram_iso;
 * flags: LGP_GRAM_SYMMETRIC with x == y and dx_field == dy_field evaluates the lower tiles once and mirrors them. */
int lgp_gram_iso_deriv(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                       int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, int dx_field, int dy_field,
                       double *K_out, int64_t ldk, int flags);

/* Reverse-mode contraction of a derivative block (dense G, n x m, ldg), the out layout of lgp_gram_iso_vjp:
 * out[3f+k] = sum_ij G_ij d K_ij / d(amp_f, log scale_f, par1_f).  out: device, 3*nfactors doubles (zeroed by the call;
 * atomicAdd accumulation). */
int lgp_gram_iso_deriv_vjp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                           int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, int dx_field, int dy_field,
                           const double *G, int64_t ldg, double *out);

/* Forward-mode derivative of a derivative block along `tangent` (HOST, 3*nfactors doubles, layout of lgp_gram_iso_jvp). */
int lgp_gram_iso_deriv_jvp(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                           int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, int dx_field, int dy_field,
                           const double *tangent, double *D_out, int64_t ldd);

/* Variants with DEVICE-RESIDENT hyperparameters: what an XLA-FFI custom call needs, where traced scalars arrive as device
 * buffers and must not be read on the host (the boundary B3 of SURVEY.md section 8b: jax.ffi handlers wrapping these are in
 * lsqfitgp_b200/csrc/xla_ffi_shim.cc, INTEGRATION.md section 3).  `factors` (HOST) carries only the structure: kind, term,
 * dimmask, ipar and par0 (Matern order / Maternp offset / Cauchy alpha: static, not differentiable, as in the reference);
 * its other fields are ignored.  `devpar` (DEVICE): LGP_DEVPAR_STRIDE doubles per factor, in the order scale_x, scale_y,
 * loc_x, loc_y, par1, amp.  `tangent_dev` (DEVICE): 3*nfactors doubles.  Same results as the host-descriptor entry points
 * for the same numbers; they run the general (sum-of-products) kernels, not the single-term fast paths. */
#define LGP_DEVPAR_STRIDE 6
int lgp_gram_iso_dev(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *devpar,
                     const double *x, int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m, double *K_out,
                     int64_t ldk, int flags);
int lgp_gram_iso_vjp_dev(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *devpar,
                         const double *x, int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m,
                         const double *G, int64_t ldg, const double *b, int symlower, double *out);
int lgp_gram_iso_jvp_dev(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *devpar,
                         const double *x, int64_t ldx, int64_t n, const double *y, int64_t ldy, int64_t m,
                         const double *tangent_dev, double *D_out, int64_t ldd);

/* out[0] = sum_{i<rows, j<cols} A[i*lda+j] * B[i*ldb+j]: the contraction einsum('kij,qij->kq') of the Fisher matrix
 * (src/lsqfitgp/_linalg/_decomp.py:553), one (k, q) pair per call.  out: device memory, 1 double. */
int lgp_frob_dot(lgp_stream_t stream, const double *A, int64_t lda, const double *B, int64_t ldb, int64_t rows,
                 int64_t cols, double *out);

/* ------------------------------------------------------------------------------------------------
 * BART Gram (fast path of BART._correlation: src/lsqfitgp/_kernels/_bart.py:628-757, with the
 * bracket folding of BART.correlation :415-455 done by the caller).
 * ix[d*ldx + i], iy[d*ldy + j]: int32 bin indices in [0, nsplits[d]]; w[p] weights; rows: `nrows` rows of width
 * `width` (1..3) of non-termination probabilities, deepest bracket first (row-major, host memory); gamma scalar.
 * ---------------------------------------------------------------------------------------------- */
int lgp_gram_bart(lgp_stream_t stream, int p, const int32_t *nsplits /*host*/, const double *w /*host*/,
                  const double *rows /*host*/, int nrows, int width, double gamma, double amp,
                  const double *psi /*device: psi[k] = digamma(k), k <= max(nsplits)+1; needed for width 3*/,
                  const int32_t *ix, int64_t ldx, int64_t n, const int32_t *iy, int64_t ldy, int64_t m,
                  double *K_out, int64_t ldk, int flags);

/* General form: a chain of `nstages` bracket stages (the brackets of BART.correlation that do not fold into one
 * `repeat` sequence, _bart.py:447-455: the per-pair result of one stage is the gamma of the next), optional derivative
 * outputs, optional symmetric evaluation.
 *   stage_width[s] in 1..3, stage_nrows[s] >= 1 (HOST); rows: sum(stage_nrows) rows of THREE doubles each (entries beyond
 *   the stage's width ignored), in evaluation order (deepest bracket first); at most LGP_BART_MAX_ROWS rows in total.
 *   drows (HOST, may be NULL when no derivative is requested): 2 x (total rows) x 3: d rows / d alpha, then d rows / d beta
 *   (for pnt_d = alpha / (1 + d)^beta: pnt_d / alpha and -pnt_d log(1 + d); 0 for entries fixed to 1).
 *   K_out = amp * corr (may be NULL if only derivatives are wanted); dKa_out = amp * d corr / d alpha, dKb_out likewise
 *   for beta (each may be NULL; ld = ldd): what jax.jacfwd of the BART kernel gives `bayestree.bart`
 *   (src/lsqfitgp/bayestree/_bart.py:175-227 with forward=True, _fit.py:679-685).
 *   flags: LGP_BART_SYMMETRIC asserts ix == iy (same pointer) and n == m: only tiles on or below the diagonal are
 *   evaluated and mirrored.
 *   More than LGP_BART_MAX_STAGES stages, LGP_BART_MAX_ROWS rows or 64 covariates of non-zero weight: LGP_ERR_UNSUPPORTED
 *   (here and in lgp_gram_bart_vjp). */
#define LGP_BART_MAX_ROWS 16
#define LGP_BART_MAX_STAGES 8
#define LGP_BART_SYMMETRIC 1
int lgp_gram_bart_stages(lgp_stream_t stream, int p, const int32_t *nsplits /*host*/, const double *w /*host*/,
                         int nstages, const int32_t *stage_width /*host*/, const int32_t *stage_nrows /*host*/,
                         const double *rows /*host*/, const double *drows /*host*/, double gamma, double amp,
                         const double *psi /*device*/, const int32_t *ix, int64_t ldx, int64_t n, const int32_t *iy,
                         int64_t ldy, int64_t m, double *K_out, int64_t ldk, double *dKa_out, double *dKb_out,
                         int64_t ldd, int flags);

/* Reverse-mode contraction of the BART Gram build without materialising the derivatives (what jax.vjp of the kernel
 * gives empbayes_fit in reverse mode, src/lsqfitgp/_fit.py:687-702 with _linalg/_decomp.py:505-509):
 *   out[0] = sum_ij G_ij corr_ij            (= d/d amp)
 *   out[1] = sum_ij G_ij amp d corr_ij / d alpha,   out[2] likewise for beta
 * symlower = 0: G dense n x m.  symlower = 1: ix == iy and G_ij = w_ij (G[i][j] - b_i b_j) read from the LOWER triangle
 * only, w = 2 off the diagonal (b may be NULL), as in lgp_gram_iso_vjp.  out: device, 3 doubles (zeroed by the call;
 * accumulated with atomicAdd). */
int lgp_gram_bart_vjp(lgp_stream_t stream, int p, const int32_t *nsplits /*host*/, const double *w /*host*/, int nstages,
                      const int32_t *stage_width /*host*/, const int32_t *stage_nrows /*host*/,
                      const double *rows /*host*/, const double *drows /*host*/, double gamma, double amp,
                      const double *psi /*device*/, const int32_t *ix, int64_t ldx, int64_t n, const int32_t *iy,
                      int64_t ldy, int64_t m, const double *G, int64_t ldg, const double *b, int symlower, double *out);
/* fills HOST buffer psi_out[k] = digamma(k), k = 1..len-1 (psi_out[0] = -inf): jspecial.digamma of integers
 * (_bart.py:735-743) by an extended-precision recurrence */
int lgp_bart_digamma_table(double *psi_out, int64_t len);

/* ------------------------------------------------------------------------------------------------
 * FP64 GEMM on the DMMA tensor pipe:  C[i][j] (+)= alpha * sum_k Aop[i][k]*Bop[j][k]
 *   a_kmajor: Aop[i][k] = A[i*lda+k], else A[k*lda+i];  b_kmajor: Bop[j][k] = B[j*ldb+k], else B[k*ldb+j]
 * flags: LGP_GEMM_*.  Replaces the dgemm/dsyrk custom calls under `@`/einsum in _decomp.py:409,420,472.
 * ---------------------------------------------------------------------------------------------- */
#define LGP_GEMM_LOWER 1
#define LGP_GEMM_BETA0 2
#define LGP_GEMM_A_LOWER_K 4
#define LGP_GEMM_B_LOWER_K 8
#define LGP_GEMM_A_UPPER_K 16
#define LGP_GEMM_B_UPPER_K 32
int lgp_dgemm(lgp_stream_t stream, int a_kmajor, int b_kmajor, int64_t M, int64_t N, int64_t K, double alpha,
              const double *A, int64_t lda, const double *B, int64_t ldb, double *C, int64_t ldc, int flags);

/* Y = alpha*X + beta*Y + gamma*I over an n x m block (X may be NULL).  The elementwise block sums of
 * _assemblecovblocks / addtransf with scalar tensors (src/lsqfitgp/_GP/_elements.py:581-601,642-649) and
 * `Kxx + ycov` (src/lsqfitgp/_GP/_compute.py:84-85). */
int lgp_axpby(lgp_stream_t stream, int64_t n, int64_t m, double alpha, const double *X, int64_t ldx, double beta,
              double *Y, int64_t ldy, double gamma);

/* Y += c over an n x m block: blocks of scalar covariances broadcast through addtransf (the `k^2 11^T` term of
 * bayestree.bart, src/lsqfitgp/bayestree/_bart.py:199-204, _GP/_elements.py:581-601). */
int lgp_add_scalar(lgp_stream_t stream, int64_t n, int64_t m, double *Y, int64_t ldy, double c);

/* out (n x n, ldo) = scale * (sym(low) - b b^T) as a FULL symmetric matrix, `low` given by its LOWER triangle (ldl; the
 * upper triangle is not read), b optional n-vector: dvalue/dK = 1/2 (K^-1 - K^-1 r r^T K^-1) of the normal density for
 * consumers that need the full matrix (generic dK_vjp callbacks, reverse mode through assembled blocks),
 * src/lsqfitgp/_linalg/_decomp.py:505-509.  One pass: reads n^2/2, writes n^2. */
int lgp_sym_expand_sub(lgp_stream_t stream, const double *low, int64_t ldl, const double *b, int64_t n, double scale,
                       double *out, int64_t ldo);

/* out[0] = sum_ij (G_ij - b_i b_j) D_ij with symmetric G given by its LOWER triangle (`low`, ldl) and D any n x n matrix
 * (ldd): tr(K^-1 dK) - r^T K^-1 dK K^-1 r of the forward-mode gradient, einsum('ij,ijk->k') and einsum('i,ijk,j->k') of
 * src/lsqfitgp/_linalg/_decomp.py:524-531, one k per call.  out: device, 1 double (zeroed by the call; atomicAdd). */
int lgp_symlower_dot(lgp_stream_t stream, const double *low, int64_t ldl, const double *b, const double *D, int64_t ldd,
                     int64_t n, double *out);

/* out[j] = sum_i A[i*lda + j]^2, j < cols: diag(A^T K^-1 A) from L^-1 A, Chol.ginv_diagquad,
 * src/lsqfitgp/_linalg/_decomp.py:422-427.  out: device, cols doubles (zeroed by the call; atomicAdd). */
int lgp_colsumsq(lgp_stream_t stream, const double *A, int64_t lda, int64_t rows, int64_t cols, double *out);

/* BART bin indices on the device: out[d*ldo + i] = searchsorted(splits[:, d], x[d*ldx + i], side='left') over the whole
 * padded column, d < p, i < n (BART.indices_from_coord, src/lsqfitgp/_kernels/_bart.py:294-299,503-514).
 * splits: maxlen x p row-major (as BART.splits_from_coord returns it, padded with the dtype maximum), DEVICE memory. */
int lgp_searchsorted(lgp_stream_t stream, const double *splits, int64_t maxlen, int p, const double *x, int64_t ldx,
                     int64_t n, int32_t *out, int64_t ldo);

/* ------------------------------------------------------------------------------------------------
 * Cholesky with lsqfitgp's equilibration + Gershgorin jitter (Chol.__init__,
 * src/lsqfitgp/_linalg/_decomp.py:245-255,349-361,380-393):
 *   s_i = 2^rint(log2(K_ii)/2) (1 if K_ii == 0);  Kt = K/s/s^T;  eps = epsrel*max_i sum_j |Kt_ij| + epsabs;
 *   Kt_ii += eps;  Lt = chol(Kt);  L = diag(s) Lt.
 * The factor is kept as (Lt, s): W holds Lt in the lower triangle of an npad x npad matrix
 * (npad = n rounded up to 128, identity padding), aux holds s, 1/s, diag(Lt), the scalars and the
 * inverted 128x128 diagonal blocks.
 *   K      : n x n input (ldk); only read.  addmat (optional, may be NULL): n x n matrix added to K
 *            (GPCompute._solver `Kxx + ycov`, src/lsqfitgp/_GP/_compute.py:84-85);
 *            adddiag (optional): n-vector added to the diagonal.
 *   epsrel < 0 means 'auto' = n * 2^-52.
 *   aux scalars (doubles at aux + 3*npad): [0] max row abs-sum of Kt, [1] eps, [2] reserved,
 *            [3] min_i s_i^2  (so Chol.eps = [1]*[3]); [4] = sum_i log(L_ii) again (written by the final reduction),
 *            [5] = 0
 *   info   : device int32; 0 on success, else 1-based index of the first non-positive/NaN pivot.
 * ---------------------------------------------------------------------------------------------- */
int64_t lgp_chol_npad(int64_t n);
int64_t lgp_chol_aux_doubles(int64_t n);
#define LGP_AUX_S(npad) (0)
#define LGP_AUX_SINV(npad) (npad)
#define LGP_AUX_DIAG(npad) (2 * (npad))
#define LGP_AUX_SCALARS(npad) (3 * (npad))
#define LGP_AUX_INVDIAG(npad) (3 * (npad) + 16)
int lgp_chol_factor(lgp_stream_t stream, const double *K, int64_t ldk, const double *addmat, int64_t ldadd,
                    const double *adddiag, int64_t n, double epsrel, double epsabs, double *W, int64_t ldw,
                    double *aux, int32_t *info);

/* B (n x m, ldb even, 16-byte aligned) <- L^-1 B (trans=0) or L^-T B (trans=1), L = diag(s) Lt.
 * Replaces jax.scipy.linalg.solve_triangular in _decomp.py:402-403,407-408,419,426,439,467-469.
 * m = 1: ONE kernel per sweep (block rows chained by device flags in ticket order; up to 128 distinct caller streams per
 * device, LGP_ERR_UNSUPPORTED beyond); m > 1: recursion over DMMA GEMMs with the inverted diagonal blocks. */
int lgp_chol_solve(lgp_stream_t stream, const double *W, int64_t ldw, const double *aux, int64_t n, double *B,
                   int64_t ldb, int64_t m, int trans);

/* Y (n x m) = L X (trans=0) or L^T X (trans=1).  Chol.correlate / back_correlate (_decomp.py:429-435). */
/* tmp (n x m, ldt even, 16-byte aligned) is scratch, required for trans=1 only. X, tmp: ld even, aligned. */
int lgp_chol_mult(lgp_stream_t stream, const double *W, int64_t ldw, const double *aux, int64_t n, const double *X,
                  int64_t ldx, int64_t m, double *Y, int64_t ldy, double *tmp, int64_t ldt, int trans);

/* Lout (n x n) = L = diag(s) Lt with zeros above the diagonal. */
int lgp_chol_get_factor(lgp_stream_t stream, const double *W, int64_t ldw, const double *aux, int64_t n,
                        double *Lout, int64_t ldl);

/* Kinv (npad x npad, ld = ldk) lower triangle <- (L L^T)^-1 via TRTRI + LAUUM on the DMMA pipe
 * (2n^3/3 flop instead of the reference's L^-1 I and invL^T invL = 3n^3, _decomp.py:471-472).
 * scratch: npad x npad doubles (ld = npad). */
int lgp_chol_inverse(lgp_stream_t stream, const double *W, int64_t ldw, const double *aux, int64_t n,
                     double *scratch, double *Kinv, int64_t ldk);

/* lgp_chol_factor followed by lgp_chol_inverse in ONE call: what a logML + gradient evaluation needs
 * (Chol.__init__ and the invL / invK of minus_log_normal_density, src/lsqfitgp/_linalg/_decomp.py:380-393,466-472).
 * The factorisation runs on `stream` (on return the factor, aux and info are complete in `stream` order, exactly as after
 * lgp_chol_factor); the inverse runs on `inv_stream` (Kinv is complete in `inv_stream` order: make consumers wait for
 * that stream).  The inverse starts behind the complete factor; while it runs on `inv_stream` the caller's latency-bound
 * triangular solves on `stream` overlap its GEMMs.  inv_stream == stream gives the plain sequential composition.
 * Arguments as in the two calls. */
int lgp_chol_factor_inverse(lgp_stream_t stream, lgp_stream_t inv_stream, const double *K, int64_t ldk,
                            const double *addmat, int64_t ldadd, const double *adddiag, int64_t n, double epsrel,
                            double epsabs, double *W, int64_t ldw, double *aux, int32_t *info, double *scratch,
                            double *Kinv, int64_t ldkinv);

/* Gram build FUSED with the equilibration pass of the factorisation (north_star: "Gram epilogue -> equilibration / row
 * sums"): for one set of points and a kernel of the fast family (ExpQuad, Matern nu = p + 1/2 with p <= 3, rational
 * quadratic, each optionally + White + Constant) the entries K_ij / (s_i s_j), j <= i, are written straight into the
 * npad x npad factor storage W (identity padding beyond n), s = 2^rint(log2(K_ii)/2) being uniform because the diagonal
 * of a stationary kernel is constant, and the partial sums of |entry| per tile go to `work` and are reduced in a fixed
 * order to the Gershgorin bound (aux scalar 0).  K itself is never written: it replaces _makecovblock_points
 * (_GP/_elements.py:554-579) + diag_scale_pow2 / eigval_bound (_decomp.py:349-361,384-385) for that case, saving the
 * 8 n^2-byte matrix, its mirror stores and the 12 n^2 bytes of the separate pass.  Returns LGP_ERR_UNSUPPORTED when the
 * kernel is outside that family (the caller then uses lgp_gram_iso + lgp_chol_factor).  Follow it with
 * lgp_chol_factor_prepared / lgp_chol_factor_inverse_prepared on the same stream.
 * work: lgp_gram_prepare_work_doubles(n) doubles (= npad^2 / 64; may alias the `scratch` of the inverse). */
int64_t lgp_gram_prepare_work_doubles(int64_t n);
/* 1 if lgp_gram_iso_prepare accepts this kernel descriptor (host-side query, nothing is launched), else 0 */
int lgp_gram_iso_prepare_supported(const lgp_factor_t *factors, int nfactors, int ndim);
int lgp_gram_iso_prepare(lgp_stream_t stream, const lgp_factor_t *factors, int nfactors, int ndim, const double *x,
                         int64_t ldx, int64_t n, double *W, int64_t ldw, double *aux, double *work);
/* lgp_chol_factor / lgp_chol_factor_inverse on a W / aux pair filled by lgp_gram_iso_prepare: jitter, factorisation (and
 * inverse); same outputs as the plain calls (eps may differ in the last bits: the row sums are added in another order) */
int lgp_chol_factor_prepared(lgp_stream_t stream, int64_t n, double epsrel, double epsabs, double *W, int64_t ldw,
                             double *aux, int32_t *info);
int lgp_chol_factor_inverse_prepared(lgp_stream_t stream, lgp_stream_t inv_stream, int64_t n, double epsrel, double epsabs,
                                     double *W, int64_t ldw, double *aux, int32_t *info, double *scratch, double *Kinv,
                                     int64_t ldkinv);

/* out[0] = sum_i log L_ii ; out[1] = sum_i a_i^2 for a (n-vector, may be NULL -> 0).
 * The reductions of Chol.minus_log_normal_density (value), _decomp.py:484-488. */
int lgp_chol_logdet_quad(lgp_stream_t stream, const double *aux, int64_t n, const double *a, double *out);

/* ------------------------------------------------------------------------------------------------
 * Tile-level building blocks of the 2-D block-cyclic multi-GPU factorisation (one process per GPU; the
 * collectives are issued by the host code in lsqfitgp_b200/_dist.py through torch.distributed/NCCL).  The reference
 * is single-device; these distribute Chol.__init__ (src/lsqfitgp/_linalg/_decomp.py:380-393) and the solves
 * (:398-439) for matrices larger than one GPU's memory.
 *
 * Tile (I, J) of the t x t tiling of the (padded) n x n matrix lives on process (I mod nprow, J mod npcol) at local
 * tile position (I div nprow, J div npcol) of a dense row-major local matrix A (lda).
 * ---------------------------------------------------------------------------------------------- */
typedef struct lgp_grid {
    int64_t n;    /* true matrix size */
    int32_t tile; /* t, multiple of 128 */
    int32_t nprow, npcol, prow, pcol;
} lgp_grid_t;

/* rows/cols of the local matrix of this process */
int lgp_dist_local_shape(const lgp_grid_t *grid, int64_t *rows, int64_t *cols);
/* d[i] = A_ii for the diagonal entries (i < n) stored on this process; other entries of d are left untouched */
int lgp_dist_diag(lgp_stream_t stream, const lgp_grid_t *grid, const double *A, int64_t lda, double *d);
/* s_i = 2^rint(log2(d_i)/2) (1 if d_i == 0 or i >= n), sinv = 1/s: diag_scale_pow2, _decomp.py:356-361 */
int lgp_dist_scale_from_diag(lgp_stream_t stream, const double *d, int64_t n, int64_t npad, double *s, double *sinv);
/* A <- A/s_i/s_j, identity in the padding rows/columns (global index >= n); rowsum[i] = sum over the LOCAL columns of
 * |A_ij| for the rows stored here (other entries untouched): the partial Gershgorin sums of eigval_bound,
 * _decomp.py:349-354, to be summed over processes */
int lgp_dist_prepare(lgp_stream_t stream, const lgp_grid_t *grid, double *A, int64_t lda, const double *sinv,
                     double *rowsum);
/* out[0] = max_i rowsum_i, out[1] = eps = epsrel*out[0] + epsabs (epsrel < 0: 'auto' = n*2^-52), _decomp.py:245-255 */
int lgp_dist_eps(lgp_stream_t stream, const double *rowsum, int64_t n, double epsrel, double epsabs, double *out);
/* A_ii += eps[0] for the diagonal entries (i < n) stored on this process (_decomp.py:386-387) */
int lgp_dist_add_diag(lgp_stream_t stream, const lgp_grid_t *grid, double *A, int64_t lda, const double *eps);

/* Cholesky of one t x t diagonal tile in place (lower triangle), plus the inverted 128x128 diagonal blocks
 * (invd: t/128 blocks), the diagonal of the factor (dvec[j0 + i], i < t) and info (atomicMin of the 1-based GLOBAL
 * index j0 + i + 1 of a failed pivot; initialise to INT_MAX). */
int lgp_tile_potrf(lgp_stream_t stream, double *A, int64_t lda, int64_t t, double *invd, double *dvec, int32_t *info,
                   int64_t j0);
/* B (rows x t, ldb) <- B L^-T for a factored diagonal tile L (t x t, ldl) with its inverted diagonal blocks */
int lgp_tile_trsm_right(lgp_stream_t stream, const double *L, int64_t ldl, const double *invd, int64_t t, double *B,
                        int64_t ldb, int64_t rows);

/* Fused panel solve + broadcast over peer memory (block-cyclic Cholesky, step "TRSM -> broadcast of the panel slab"):
 * same result in B as lgp_tile_trsm_right, and every final entry B[i][j] is also stored by the epilogue of the last
 * product at dst[d] + i*ld_dst + j for d < n_dst (<= 8).  dst[d] are device addresses valid on THIS GPU: local buffers,
 * buffers of peer GPUs mapped over NVLink (one store per peer), or, with multimem != 0, ONE NVSwitch multicast address
 * (n_dst == 1; a single multimem.st reaches the buffer of every GPU of the group, the local one included).
 * `dst` is a HOST array.  Replaces copy + ncclBroadcast of the slab; order readers with lgp_flag_signal/lgp_flag_wait. */
int lgp_tile_trsm_right_bcast(lgp_stream_t stream, const double *L, int64_t ldl, const double *invd, int64_t t, double *B,
                              int64_t ldb, int64_t rows, int n_dst, void *const *dst, int64_t ld_dst, int multimem);

/* Cross-GPU ordering for the peer stores: monotone 64-bit counters living in peer-mapped memory.
 * lgp_flag_signal: after everything enqueued before it on `stream` (system-scope fence), store `value` with release
 *   semantics to each of the n (<= LGP_MAX_FLAGS) addresses flag_ptrs[i] (HOST array of device addresses, local or peer).
 * lgp_flag_wait: block `stream` until flags[i] >= value for all i < n (acquire loads on LOCAL memory); after
 *   timeout_ms without progress it gives up and sets *err = 1 (device int32, caller-initialised to 0) instead of
 *   spinning forever. */
#define LGP_MAX_FLAGS 16
int lgp_flag_signal(lgp_stream_t stream, void *const *flag_ptrs, int n, uint64_t value);
int lgp_flag_wait(lgp_stream_t stream, const uint64_t *flags, int n, uint64_t value, int64_t timeout_ms, int32_t *err);

/* Copy a rows x cols block (src, lds) to n_dst (<= 8) destinations dst[d] + i*ld_dst + j at once: peer-mapped buffers
 * (one NVLink store per destination) or, with multimem != 0, ONE NVSwitch multicast address (n_dst == 1).  Used to
 * hand the factored diagonal tile and its inverted 128x128 blocks to the other GPUs of a process column without
 * ncclBroadcast; order readers with lgp_flag_signal / lgp_flag_wait.  `dst` is a HOST array. */
int lgp_copy2d_bcast(lgp_stream_t stream, const double *src, int64_t lds, int64_t rows, int64_t cols, int n_dst,
                     void *const *dst, int64_t ld_dst, int multimem);
/* b (t contiguous doubles) <- L^-1 b (trans=0) or L^-T b (trans=1) */
int lgp_tile_trsv(lgp_stream_t stream, const double *L, int64_t ldl, const double *invd, int64_t t, double *b,
                  int trans);
/* Trailing update of step k for the local tile columns lj in [lj_begin, lj_end):
 *   A[I, J] -= L[I, k] L[J, k]^T   for the local tiles with I >= J > k,
 * panel[r] (r < nprow; HOST array of device pointers) = the tiles L[I, k], I > k, I mod nprow == r, stacked in
 * increasing I as a contiguous (count*t) x t matrix (what process (r, k mod npcol) broadcasts).  One DMMA GEMM launch
 * per local tile column. */
int lgp_dist_trailing_update(lgp_stream_t stream, const lgp_grid_t *grid, double *A, int64_t lda, int64_t k,
                             const double *const *panel, int64_t lj_begin, int64_t lj_end);
/* Lower-packed local storage (half the memory: n = 150000 fits ONE B200): local tile column lj (global tile column
 * J = pcol + npcol*lj) is one contiguous panel of leading dimension t that holds only the local tile rows
 * li >= first = #{I < J : I mod nprow == prow}, i.e. the tiles I >= J, stacked in increasing I.
 * lgp_dist_panel_rows: first stored local tile row and number of stored tile rows of panel lj (host outputs).
 * lgp_dist_panel_diag / _prepare / _add_diag: the per-panel forms of lgp_dist_diag / lgp_dist_prepare / lgp_dist_add_diag;
 *   _prepare ACCUMULATES (atomicAdd) into rowsum, which the caller zero-initialises: tiles strictly below the diagonal
 *   contribute their column sums as well (the mirrored entries are not stored), so that the sum over processes is again
 *   the full Gershgorin row sum of eigval_bound (_decomp.py:349-354).
 * lgp_dist_trailing_update_packed: as lgp_dist_trailing_update with colpanels[lj] (HOST array of device pointers, one per
 *   local tile column) instead of the dense local matrix. */
int lgp_dist_panel_rows(const lgp_grid_t *grid, int64_t lj, int64_t *first_tile_row, int64_t *tile_rows);
int lgp_dist_panel_diag(lgp_stream_t stream, const lgp_grid_t *grid, int64_t lj, const double *panel, double *d);
int lgp_dist_panel_prepare(lgp_stream_t stream, const lgp_grid_t *grid, int64_t lj, double *panel, const double *sinv,
                           double *rowsum);
int lgp_dist_panel_add_diag(lgp_stream_t stream, const lgp_grid_t *grid, int64_t lj, double *panel, const double *eps);
int lgp_dist_trailing_update_packed(lgp_stream_t stream, const lgp_grid_t *grid, double *const *colpanels, int64_t k,
                                    const double *const *panel, int64_t lj_begin, int64_t lj_end);
/* y += alpha * P x (trans=0; P rows x cols, x cols, y rows) or y += alpha * P^T x (trans=1; x rows, y cols):
 * the HBM-streaming vector updates of the distributed triangular solves */
int lgp_dgemv(lgp_stream_t stream, int trans, const double *P, int64_t ldp, int64_t rows, int64_t cols,
              const double *x, double *y, double alpha);
/* dst (ldd) <- src (lds), rows x cols; ld even, 16-byte aligned bases (panel staging) */
int lgp_copy2d(lgp_stream_t stream, const double *src, int64_t lds, double *dst, int64_t ldd, int64_t rows,
               int64_t cols);

#ifdef __cplusplus
}
#endif
#endif /* LGP_B200_H */
