"""ctypes binding of liblgpb200.so (the C ABI declared in include/lgp_b200.h).

The library is the product path: there is no CPU or PyTorch fallback. Importing this module never
needs a GPU (so the CPU test tier can check that every declared symbol is exported); calling a
compute entry point without the library or without a CUDA device raises.
"""

import ctypes
import os
import pathlib

_HERE = pathlib.Path(__file__).resolve().parent
LIB_PATH = _HERE / 'csrc' / 'liblgpb200.so'

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int32_p = ctypes.POINTER(ctypes.c_int32)

LGP_OK = 0
ERRORS = {-1: 'bad argument', -2: 'misaligned pointer or odd leading dimension', -3: 'CUDA launch error',
          -4: 'unsupported configuration'}

# kernel kinds (lgp_b200.h)
K_EXPQUAD, K_MATERNP, K_CAUCHY, K_WHITE, K_CONSTANT, K_MATERN = range(6)
GRAM_SYMMETRIC, GRAM_GENERAL, GRAM_LIBM = 1, 2, 4  # LGP_GRAM_* flags of lgp_gram_iso
MAX_FACTORS = 8
DEVPAR_STRIDE = 6  # scale_x, scale_y, loc_x, loc_y, par1, amp
BART_MAX_ROWS, BART_MAX_STAGES, BART_SYMMETRIC = 16, 8, 1
MAX_DIMS = 32

GEMM_LOWER, GEMM_BETA0, GEMM_A_LOWER_K, GEMM_B_LOWER_K, GEMM_A_UPPER_K, GEMM_B_UPPER_K = 1, 2, 4, 8, 16, 32


class Factor(ctypes.Structure):
    """ struct lgp_factor (include/lgp_b200.h) """
    _fields_ = [
        ('kind', ctypes.c_int32),
        ('term', ctypes.c_int32),
        ('dimmask', ctypes.c_uint32),
        ('ipar', ctypes.c_int32),
        ('scale_x', ctypes.c_double),
        ('scale_y', ctypes.c_double),
        ('loc_x', ctypes.c_double),
        ('loc_y', ctypes.c_double),
        ('par0', ctypes.c_double),
        ('par1', ctypes.c_double),
        ('amp', ctypes.c_double),
    ]


class Grid(ctypes.Structure):
    """ struct lgp_grid (include/lgp_b200.h) """
    _fields_ = [
        ('n', ctypes.c_int64),
        ('tile', ctypes.c_int32),
        ('nprow', ctypes.c_int32),
        ('npcol', ctypes.c_int32),
        ('prow', ctypes.c_int32),
        ('pcol', ctypes.c_int32),
    ]


_vp = ctypes.c_void_p
_i64 = ctypes.c_int64
_int = ctypes.c_int
_dbl = ctypes.c_double

# name -> (restype, argtypes); must list every function declared in include/lgp_b200.h
SIGNATURES = {
    'lgp_abi_version': (_int, []),
    'lgp_build_info': (ctypes.c_char_p, []),
    'lgp_launch_count': (ctypes.c_longlong, []),
    'lgp_peak_probe': (_int, [_vp, _int, _int, _vp, _i64, c_double_p]),
    'lgp_gram_iso': (_int, [_vp, ctypes.POINTER(Factor), _int, _int, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _int]),
    'lgp_gram_iso_vjp': (_int, [_vp, ctypes.POINTER(Factor), _int, _int, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64,
                                _vp, _int, _vp]),
    'lgp_gram_iso_jvp': (_int, [_vp, ctypes.POINTER(Factor), _int, _int, _vp, _i64, _i64, _vp, _i64, _i64, c_double_p,
                                _vp, _i64]),
    'lgp_gram_iso_hvp': (_int, [_vp, ctypes.POINTER(Factor), _int, _int, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64,
                                _vp, _int, c_double_p, _vp]),
    'lgp_gram_iso_xvjp': (_int, [_vp, ctypes.POINTER(Factor), _int, _int, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64,
                                 _vp, _int, _vp, _i64, _vp, _i64]),
    'lgp_gram_iso_xjvp': (_int, [_vp, ctypes.POINTER(Factor), _int, _int, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64,
                                 _vp, _i64, _vp, _i64, _int]),
    'lgp_gram_iso_deriv': (_int, [_vp, ctypes.POINTER(Factor), _int, _int, _vp, _i64, _i64, _vp, _i64, _i64, _int, _int,
                                  _vp, _i64, _int]),
    'lgp_gram_iso_deriv_vjp': (_int, [_vp, ctypes.POINTER(Factor), _int, _int, _vp, _i64, _i64, _vp, _i64, _i64, _int,
                                      _int, _vp, _i64, _vp]),
    'lgp_gram_iso_deriv_jvp': (_int, [_vp, ctypes.POINTER(Factor), _int, _int, _vp, _i64, _i64, _vp, _i64, _i64, _int,
                                      _int, c_double_p, _vp, _i64]),
    'lgp_gram_iso_dev': (_int, [_vp, ctypes.POINTER(Factor), _int, _int, _vp, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64,
                                _int]),
    'lgp_gram_iso_vjp_dev': (_int, [_vp, ctypes.POINTER(Factor), _int, _int, _vp, _vp, _i64, _i64, _vp, _i64, _i64, _vp,
                                    _i64, _vp, _int, _vp]),
    'lgp_gram_iso_jvp_dev': (_int, [_vp, ctypes.POINTER(Factor), _int, _int, _vp, _vp, _i64, _i64, _vp, _i64, _i64, _vp,
                                    _vp, _i64]),
    'lgp_frob_dot': (_int, [_vp, _vp, _i64, _vp, _i64, _i64, _i64, _vp]),
    'lgp_gram_bart': (_int, [_vp, _int, c_int32_p, c_double_p, c_double_p, _int, _int, _dbl, _dbl, _vp,
                             _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _int]),
    'lgp_gram_bart_stages': (_int, [_vp, _int, c_int32_p, c_double_p, _int, c_int32_p, c_int32_p, c_double_p, c_double_p,
                                    _dbl, _dbl, _vp, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _vp, _vp, _i64, _int]),
    'lgp_gram_bart_vjp': (_int, [_vp, _int, c_int32_p, c_double_p, _int, c_int32_p, c_int32_p, c_double_p, c_double_p,
                                 _dbl, _dbl, _vp, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _vp, _int, _vp]),
    'lgp_bart_digamma_table': (_int, [c_double_p, _i64]),
    'lgp_dgemm': (_int, [_vp, _int, _int, _i64, _i64, _i64, _dbl, _vp, _i64, _vp, _i64, _vp, _i64, _int]),
    'lgp_axpby': (_int, [_vp, _i64, _i64, _dbl, _vp, _i64, _dbl, _vp, _i64, _dbl]),
    'lgp_add_scalar': (_int, [_vp, _i64, _i64, _vp, _i64, _dbl]),
    'lgp_sym_expand_sub': (_int, [_vp, _vp, _i64, _vp, _i64, _dbl, _vp, _i64]),
    'lgp_symlower_dot': (_int, [_vp, _vp, _i64, _vp, _vp, _i64, _i64, _vp]),
    'lgp_colsumsq': (_int, [_vp, _vp, _i64, _i64, _i64, _vp]),
    'lgp_searchsorted': (_int, [_vp, _vp, _i64, _int, _vp, _i64, _i64, _vp, _i64]),
    'lgp_chol_npad': (_i64, [_i64]),
    'lgp_chol_aux_doubles': (_i64, [_i64]),
    'lgp_chol_factor': (_int, [_vp, _vp, _i64, _vp, _i64, _vp, _i64, _dbl, _dbl, _vp, _i64, _vp, _vp]),
    'lgp_chol_factor_inverse': (_int, [_vp, _vp, _vp, _i64, _vp, _i64, _vp, _i64, _dbl, _dbl, _vp, _i64, _vp, _vp, _vp, _vp,
                                       _i64]),
    'lgp_gram_prepare_work_doubles': (_i64, [_i64]),
    'lgp_gram_iso_prepare_supported': (_int, [ctypes.POINTER(Factor), _int, _int]),
    'lgp_gram_iso_prepare': (_int, [_vp, ctypes.POINTER(Factor), _int, _int, _vp, _i64, _i64, _vp, _i64, _vp, _vp]),
    'lgp_chol_factor_prepared': (_int, [_vp, _i64, _dbl, _dbl, _vp, _i64, _vp, _vp]),
    'lgp_chol_factor_inverse_prepared': (_int, [_vp, _vp, _i64, _dbl, _dbl, _vp, _i64, _vp, _vp, _vp, _vp, _i64]),
    'lgp_chol_solve': (_int, [_vp, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _int]),
    'lgp_chol_mult': (_int, [_vp, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _vp, _i64, _vp, _i64, _int]),
    'lgp_chol_get_factor': (_int, [_vp, _vp, _i64, _vp, _i64, _vp, _i64]),
    'lgp_chol_inverse': (_int, [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _i64]),
    'lgp_chol_logdet_quad': (_int, [_vp, _vp, _i64, _vp, _vp]),
    'lgp_dist_local_shape': (_int, [ctypes.POINTER(Grid), ctypes.POINTER(_i64), ctypes.POINTER(_i64)]),
    'lgp_dist_diag': (_int, [_vp, ctypes.POINTER(Grid), _vp, _i64, _vp]),
    'lgp_dist_scale_from_diag': (_int, [_vp, _vp, _i64, _i64, _vp, _vp]),
    'lgp_dist_prepare': (_int, [_vp, ctypes.POINTER(Grid), _vp, _i64, _vp, _vp]),
    'lgp_dist_eps': (_int, [_vp, _vp, _i64, _dbl, _dbl, _vp]),
    'lgp_dist_add_diag': (_int, [_vp, ctypes.POINTER(Grid), _vp, _i64, _vp]),
    'lgp_tile_potrf': (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _i64]),
    'lgp_tile_trsm_right': (_int, [_vp, _vp, _i64, _vp, _i64, _vp, _i64, _i64]),
    'lgp_tile_trsm_right_bcast': (_int, [_vp, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _int, ctypes.POINTER(_vp), _i64,
                                         _int]),
    'lgp_copy2d_bcast': (_int, [_vp, _vp, _i64, _i64, _i64, _int, ctypes.POINTER(_vp), _i64, _int]),
    'lgp_flag_signal': (_int, [_vp, ctypes.POINTER(_vp), _int, ctypes.c_uint64]),
    'lgp_flag_wait': (_int, [_vp, _vp, _int, ctypes.c_uint64, _i64, _vp]),
    'lgp_tile_trsv': (_int, [_vp, _vp, _i64, _vp, _i64, _vp, _int]),
    'lgp_dist_trailing_update': (_int, [_vp, ctypes.POINTER(Grid), _vp, _i64, _i64, ctypes.POINTER(_vp), _i64, _i64]),
    'lgp_dist_panel_rows': (_int, [ctypes.POINTER(Grid), _i64, ctypes.POINTER(_i64), ctypes.POINTER(_i64)]),
    'lgp_dist_panel_diag': (_int, [_vp, ctypes.POINTER(Grid), _i64, _vp, _vp]),
    'lgp_dist_panel_prepare': (_int, [_vp, ctypes.POINTER(Grid), _i64, _vp, _vp, _vp]),
    'lgp_dist_panel_add_diag': (_int, [_vp, ctypes.POINTER(Grid), _i64, _vp, _vp]),
    'lgp_dist_trailing_update_packed': (_int, [_vp, ctypes.POINTER(Grid), ctypes.POINTER(_vp), _i64, ctypes.POINTER(_vp),
                                               _i64, _i64]),
    'lgp_dgemv': (_int, [_vp, _int, _vp, _i64, _i64, _i64, _vp, _vp, _dbl]),
    'lgp_copy2d': (_int, [_vp, _vp, _i64, _vp, _i64, _i64, _i64]),
}

_lib = None


class LibraryMissing(RuntimeError):
    pass


def load():
    """Load liblgpb200.so (built in-tree by `__graft_entry__.build()` / `make -C lsqfitgp_b200/csrc`)."""
    global _lib
    if _lib is not None:
        return _lib
    path = pathlib.Path(os.environ.get('LGP_LIB_PATH', LIB_PATH))  # override for kernel experiments only
    if not path.exists():
        raise LibraryMissing(
            f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
            f'or `make -C {LIB_PATH.parent}`. There is no CPU fallback.')
    lib = ctypes.CDLL(os.fspath(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != LGP_OK:
        raise RuntimeError(f'{what} failed: {ERRORS.get(rc, rc)}')


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """ device pointer of a torch tensor (or None) """
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError('lsqfitgp_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback')
    load()
