"""Pin the fasthash64 oracle to the reference's golden vectors (tests/test_jax.py:112-186 of the reference)
and to the C restatement."""
import ctypes
import pathlib

import numpy as np
import pytest

from oracle import fasthash

INPUTS = [
    [], [234], [194, 116], [160, 237, 166], [72, 56, 46, 113], [152, 22, 163, 7, 234],
    [100, 11, 190, 249, 103, 74], [119, 52, 46, 248, 188, 178, 216], [81, 10, 197, 4, 19, 41, 69, 164],
    [53, 246, 128, 162, 79, 228, 71, 137, 255], [145, 141, 43, 100, 125, 107, 12, 4, 147, 229],
    [117, 92, 35, 144, 76, 140, 59, 36, 42, 13, 94], [91, 207, 0, 152, 226, 159, 190, 164, 136, 176, 194, 59],
    [126, 94, 132, 168, 44, 150, 242, 165, 199, 149, 248, 82, 141],
    [26, 101, 134, 203, 216, 141, 100, 242, 248, 225, 83, 131, 27, 100],
    [153, 2, 211, 91, 131, 54, 101, 233, 213, 71, 216, 126, 60, 48, 157],
    [114, 165, 8, 26, 213, 17, 112, 170, 104, 161, 164, 95, 53, 17, 149, 170],
    [40, 198, 242, 87, 28, 55, 234, 142, 22, 200, 236, 65, 198, 91, 197, 233, 46],
    [208, 21, 5, 101, 61, 240, 41, 134, 164, 25, 109, 253, 108, 140, 229, 255, 39, 199],
    [240, 22, 57, 231, 226, 172, 97, 114, 34, 20, 14, 47, 118, 129, 193, 93, 43, 209, 75],
]
HASHES64 = [
    7502587791032603753, 16941272163545924368, 10988138224395471776, 9507901428091620561, 8215232957141175337,
    18053746358964717198, 12425373722766252877, 2946925277746383721, 12402381367179054957, 755910146092029036,
    3255785893224143811, 12592656301469221220, 428602295608661196, 5824169786726525377, 1508071078291841094,
    11448092356368632731, 6157277036160160880, 9731805725958528408, 3366289320067065534, 17424790981778646777,
]
HASHES32 = [
    1004310665, 2046185678, 3566082500, 2790396102, 2182032100, 2323244336, 1312080940, 2492442272, 1823551547,
    3569298354, 1867203821, 2449676296, 2938746445, 3041190206, 3115372248, 3527005061, 1217622642, 4177513530,
    303099792, 2425579332,
]
SEED32 = 2428169863
SEED64 = 6361217807637034346


def test_golden_vectors():
    for inp, h32, h64 in zip(INPUTS, HASHES32, HASHES64):
        buf = bytes(inp)
        assert fasthash.fasthash64(buf, SEED64) == h64
        assert fasthash.fasthash32(buf, SEED32) == h32


def test_c_restatement(rng):
    p = pathlib.Path(fasthash.__file__).resolve().parent / 'liboracle_c.so'
    if not p.exists():
        pytest.skip('oracle/liboracle_c.so not built')
    lib = ctypes.CDLL(str(p))
    lib.oracle_fasthash64.restype = ctypes.c_uint64
    lib.oracle_fasthash64.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_uint64]
    for inp, h64 in zip(INPUTS, HASHES64):
        assert lib.oracle_fasthash64(bytes(inp), len(inp), SEED64) == h64


def test_rows_equal_iff_hash_equal(rng):
    """ what BART._correlation uses the hash for (reference _bart.py:675-678): equality of index vectors """
    a = rng.integers(0, 5, (50, 4), dtype=np.int32)
    b = a.copy()
    b[::2, 1] += 1
    ha = fasthash.fasthash64_rows(a)
    hb = fasthash.fasthash64_rows(b)
    assert np.array_equal(ha != hb, np.any(a != b, axis=1))
