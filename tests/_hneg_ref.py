"""numpy restatement of the hard-negative candidate draws of ngcf_hard_negatives (csrc/evalsample.cu), used by the
hard-negative tests.

Candidate j of batch row b: ``h = ngcf_hash64(seed + seed_dev, b, b >> 32, j, 'HNEG')`` (four murmur3 finalizer rounds
over the counter words, csrc/common.cuh), ``r = (h.x * n_free) >> 32`` with ``n_free`` the number of items outside the
user's exclusion list, and the candidate is the r-th of those items in ascending order.  The device finds it by a
binary search over the list; here it is an index into ``np.setdiff1d``, so the two do not share an algorithm.
The product package never imports this module.
"""
import numpy as np

from tests._dropout_ref import M32, mix, seed_words

STREAM_HNEG = np.uint64(0x484E4547)       # 'HNEG'


def hash64(seed: int, a, b, c, stream=STREAM_HNEG):
    """ngcf_hash64(seed, a, b, c, stream) -> (x, y), uint64 arrays of 32-bit values."""
    lo, hi = seed_words(seed)
    h = mix((np.asarray(a, dtype=np.uint64) & M32) ^ lo ^ stream)
    h = mix(h ^ (((np.asarray(b, dtype=np.uint64) & M32) + np.uint64(0x9E3779B9)) & M32) ^ hi)
    h = mix((h + (np.asarray(c, dtype=np.uint64) * np.uint64(0x632BE5AB) & M32) + np.uint64(0x7F4A7C15)) & M32)
    return h, mix(h ^ np.uint64(0x68E31DA4))


def free_items(excluded, n_items: int):
    """Ascending items of [0, n_items) outside ``excluded``."""
    return np.setdiff1d(np.arange(n_items, dtype=np.int64), np.asarray(excluded, dtype=np.int64))


def candidates(seed: int, u_id, rows, n_items: int, M: int):
    """int64 [B, M]: the candidates ngcf_hard_negatives draws for batch users ``u_id`` under key ``seed`` (seed +
    *seed_dev); ``rows[u]`` = user u's excluded items."""
    u_id = np.asarray(u_id, dtype=np.int64)
    B = u_id.size
    b = np.repeat(np.arange(B, dtype=np.uint64), M)
    j = np.tile(np.arange(M, dtype=np.uint64), B)
    x, _ = hash64(seed, b & M32, b >> np.uint64(32), j)
    out = np.empty(B * M, dtype=np.int64)
    cache = {}
    for i in range(B * M):
        u = int(u_id[i // M])
        if u not in cache:
            cache[u] = free_items(rows[u], n_items)
        free = cache[u]
        r = int((int(x[i]) * free.size) >> 32)
        out[i] = free[r]
    return out.reshape(B, M)
