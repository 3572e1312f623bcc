"""Oracle: fasthash64 (src/lsqfitgp/_jaxext/_fasthash.py:56-97 == tests/fast-hash/fasthash.c:34-66)."""

import numpy as np

M = 0x880355f21e6d1965
MASK = (1 << 64) - 1
BART_SEED = 16132933535611723338  # src/lsqfitgp/_kernels/_bart.py:675


def _mix(h):
    h ^= h >> 23
    h = (h * 0x2127599bf4325c37) & MASK
    h ^= h >> 47
    return h


def fasthash64(buf, seed):
    """ buf: bytes-like; returns python int """
    buf = bytes(buf)
    n = len(buf)
    h = (seed ^ ((n * M) & MASK)) & MASK
    nw = n // 8
    for i in range(nw):
        v = int.from_bytes(buf[8 * i: 8 * i + 8], 'little')
        h ^= _mix(v)
        h = (h * M) & MASK
    tail = buf[8 * nw:]
    if tail:
        v = int.from_bytes(tail, 'little')
        h ^= _mix(v)
        h = (h * M) & MASK
    return _mix(h)


def fasthash32(buf, seed):
    h = fasthash64(buf, seed)
    return (h - (h >> 32)) & 0xffffffff


def fasthash64_rows(a, seed=BART_SEED):
    """ hash each row of a 2-d integer array over its raw bytes (as BART._correlation does on ix, iy) """
    a = np.ascontiguousarray(a)
    return np.array([fasthash64(row.tobytes(), seed) for row in a], dtype=np.uint64)
