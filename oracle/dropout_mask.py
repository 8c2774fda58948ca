"""Host restatement of the dropout hash of xfm_b200/csrc/common.cuh (drop_keep_idx), in numpy uint32 arithmetic.

Every dropout in the library (GEMM epilogue, attention probabilities, dropout_apply) keeps element `idx` of a mask stream
exactly when keep(seed, idx, p) is true; the kernels differ only in how they number their elements:
  * dropout_apply and the GEMM epilogue: idx = row * N + col;
  * attention: idx = ((b * H + h) * Lq + q) * ((Lk + 1) & ~1) + key (an even row stride, so keys 2k and 2k+1 share one
    hash pair).
The seed is the one passed to the kernel plus the device seed salt (xfm_seed_salt_*), which tests set to zero.
"""
import numpy as np


def _mix32(x):
    x = x ^ (x >> np.uint32(16))
    x = x * np.uint32(0x7FEB352D)
    x = x ^ (x >> np.uint32(15))
    x = x * np.uint32(0x846CA68B)
    return x ^ (x >> np.uint32(16))


def keep(seed, idx, p):
    """drop_keep_idx(seed, idx, p) for every element index in `idx` (any integer array): a bool array of idx's shape."""
    idx = np.asarray(idx, dtype=np.uint64)
    thr = np.uint32(np.float32(p) * np.float32(65536.0) + np.float32(0.5))
    s = np.uint32((seed & 0xFFFFFFFF) ^ (((seed >> 32) * 0x85EBCA6B) & 0xFFFFFFFF))
    pair = idx >> np.uint64(1)
    lo, hi = (pair & np.uint64(0xFFFFFFFF)).astype(np.uint32), (pair >> np.uint64(32)).astype(np.uint32)
    with np.errstate(over="ignore"):
        x = _mix32((lo + hi * np.uint32(0x9E3779B1)) ^ s)
    bits = np.where((idx & np.uint64(1)) == 1, x >> np.uint32(16), x & np.uint32(0xFFFF))
    return bits >= thr


def attention_index(B, H, Lq, Lk):
    """Element indices of an attention probability mask as a [B, H, Lq, Lk] uint64 array."""
    lke = (Lk + 1) & ~1
    rows = np.arange(B * H * Lq, dtype=np.uint64).reshape(B, H, Lq, 1)
    return rows * np.uint64(lke) + np.arange(Lk, dtype=np.uint64)
