"""CPU restatement (NumPy/SciPy, float64) of lsqfitgp's GP-fitting hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under `lsqfitgp_b200/` imports this package; only `tests/`,
`__graft_entry__.smoke()` and the `cpu_baseline` / `--impl reference` legs of `bench.py` do, and only
as the checker or as the timed CPU baseline.

Why a restatement: the reference (Gattocrucco/lsqfitgp 0.22.dev0) hard-imports `jax`, `jaxlib` and
`gvar`, none of which exist in this image (no network, not in /opt/wheelhouse), so it cannot be
imported here or on the GPU box.  Every function cites the reference lines it follows (paths
relative to the reference root).  The arithmetic lives in third-party code in the reference too:
  jax/jaxlib >= 0.4.35 (pyproject.toml:42-43): jnp elementwise ops -> here numpy ufuncs;
      jax.scipy.linalg.cholesky / solve_triangular -> LAPACK dpotrf / dtrsm -> here scipy.linalg (same routines);
      jax.scipy.special.digamma -> here scipy.special.digamma
  scipy >= 1.10: scipy.special.kv (called by the reference itself through pure_callback) -> same function.

Pinning status (see tests/test_oracle_*.py, tests/golden/):
  * fasthash64: pinned to the reference's 20 golden vectors (tests/test_jax.py:112-186).
  * Chol: pinned by the reference's own test battery restated (tests/linalg/test_decomp.py:145-261:
    every method against scipy.linalg.solve / eigvalsh / finite differences).
  * Matern/Maternp cores: pinned by tests/test_special.py:68-97 restated (mpmath / scipy kv).
  * BART: the fast path is pinned against a restatement of the reference's independent recursive
    implementation `_correlation_old` (tests/kernels/test_bart.py:332-353) and the property tests.
  * THE REFERENCE'S OWN SOURCE, executed under a numpy stand-in for the jax API (oracle/refshim.py): lgp.GP
    .marginal_likelihood / .predfromdata(raw=True), every supported kernel class, _linalg.Chol (value, forward gradient,
    Fisher matrix, solves) and BART (preprocessing, correlation) produce tests/golden/reference_vectors.npz
    (tests/golden/gen_reference_vectors.py).  The restatement reproduces those vectors to 0-2 ulp on Gram blocks, exactly
    on eps, to 1e-13 on logML (tests/test_reference_vectors.py); logML / posterior values of the BASELINE configs are
    therefore pinned to the reference's code, though not to the JAX runtime (XLA's own rounding is not reproduced; LAPACK
    is scipy's).  A 50-digit mpmath anchor (tests/test_oracle_mpmath_anchor.py) is the implementation-independent check.
"""
