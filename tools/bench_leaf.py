"""128x128 leaf (Cholesky + inverse of the factor in one CTA, chol_leaf3.cuh): correctness against torch, phase clocks and
time per call."""
import sys, ctypes
import numpy as np
import torch
sys.path.insert(0, '.')
from lsqfitgp_b200 import _lib
lib = _lib.load()
lib.lgp_debug_leaf.restype = ctypes.c_int
lib.lgp_debug_leaf.argtypes = [ctypes.c_void_p] * 2 + [ctypes.c_int64] + [ctypes.c_void_p] * 3 + [ctypes.c_int]
lib.lgp_debug_leaf3_clocks.argtypes = [ctypes.c_void_p]
dev = torch.device('cuda:0')
torch.manual_seed(0)
A = torch.randn(128, 128, dtype=torch.float64, device=dev)
K = A @ A.T + 128 * torch.eye(128, dtype=torch.float64, device=dev)
L = torch.linalg.cholesky(K)
Linv = torch.linalg.inv(L)
clk = (ctypes.c_longlong * 32)()
names3 = ['load'] + sum([[f'panel{J}', f'colupd{J}'] for J in range(4)], [])[:-1] + ['store']
invd = torch.full((128, 128), 7.0, dtype=torch.float64, device=dev)
dvec = torch.empty(128, dtype=torch.float64, device=dev)
info = torch.full((1,), 2**31 - 1, dtype=torch.int32, device=dev)
W = K.clone()
W += torch.triu(torch.full_like(W, 3.0), 1)  # the strict upper triangle of the input is scratch: must be ignored
rc = lib.lgp_debug_leaf(_lib.stream_ptr(), _lib.ptr(W), 128, _lib.ptr(invd), _lib.ptr(dvec), _lib.ptr(info), 1)
torch.cuda.synchronize()
print(f'rc={rc}: L err {float((W - L).abs().max() / L.abs().max()):.2e} (upper zero: {bool((torch.triu(W, 1) == 0).all())}), '
      f'inverse err {float((invd - Linv).abs().max() / Linv.abs().max()):.2e}, diag err {float((dvec - torch.diagonal(L)).abs().max()):.2e}, info {int(info.item())}')
# odd leading dimension / unaligned base: the scalar load and store paths
Wbig = torch.zeros(128, 131, dtype=torch.float64, device=dev)
Wbig[:, 1:129] = K
Wv = Wbig[:, 1:129]
rc = lib.lgp_debug_leaf(_lib.stream_ptr(), Wv.data_ptr(), 131, _lib.ptr(invd), _lib.ptr(dvec), _lib.ptr(info), 1)
torch.cuda.synchronize()
print(f'   ld = 131, base + 8 bytes: L err {float((Wv - L).abs().max() / L.abs().max()):.2e}, inverse err {float((invd - Linv).abs().max() / Linv.abs().max()):.2e}')
# failure reporting: a negative pivot at column 70
Kb = K.clone(); Kb[70, 70] = -1.0
info.fill_(2**31 - 1)
lib.lgp_debug_leaf(_lib.stream_ptr(), _lib.ptr(Kb), 128, _lib.ptr(invd), _lib.ptr(dvec), _lib.ptr(info), 1)
torch.cuda.synchronize()
print(f'   bad pivot reported at {int(info.item())} (expect 71)')
for rep in range(2):
    W = K.clone()
    lib.lgp_debug_leaf(_lib.stream_ptr(), _lib.ptr(W), 128, _lib.ptr(invd), _lib.ptr(dvec), _lib.ptr(info), 1)
    torch.cuda.synchronize()
    lib.lgp_debug_leaf3_clocks(clk)
    c = np.array(list(clk)[:10], dtype=np.int64)
    print('   phases (cycles):', ', '.join(f'{n} {v}' for n, v in zip(names3, np.diff(c))), '| total', c[-1] - c[0])
for trial in range(2):
    Ws = [K.clone() for _ in range(50)]  # a fresh (valid) input for every launch
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for Wi in Ws:
        lib.lgp_debug_leaf(_lib.stream_ptr(), _lib.ptr(Wi), 128, _lib.ptr(invd), _lib.ptr(dvec), _lib.ptr(info), 1)
    e1.record(); torch.cuda.synchronize()
    print(f'   {e0.elapsed_time(e1)*1e3/50:.1f} us per leaf (50 launches, fresh inputs)')
