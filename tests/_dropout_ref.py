"""numpy restatement of the device-RNG dropout decisions (csrc/common.cuh), used by the dropout-RNG tests.

Node dropout: entry (row, col) of L has the static key ``node_key(row, col)``; per step, group g of four layers draws
two murmur3 finalizer rounds of ``key ^ seed_lo ^ g * 0x632BE5AB ^ 'NODE'`` (the second one also mixes in seed_hi),
which give four 16-bit uniforms.  Bit k of the decision byte = the entry survives layers 0..k (cumulative).
The seed's high word enters only the second round, so the decisions of layers 0, 1, 4 and 5 depend on the seed's low
word alone; per-step seeds differ in their low words (NGCF draws them at random, a graph replay adds an odd
constant), so this costs no freshness.
Message dropout: element (row, col) of a layer's [n_rows, d_out] output, with ``row`` global (local row + the shard's
row offset), belongs to quad ``((row * d_out + col) >> 2)``; one hash of (seed, layer, quad) gives the quad's four
uniforms, element ``j = (row * d_out + col) & 3`` takes uniform j.

An element is kept iff its uniform is >= ``thr = uint32(float32(p) * 65536)`` (truncated): the kernels receive p as
a C float, so p is rounded to float32 first, and probabilities are resolved to 2^-16.  The kept value of message
dropout is scaled by ``float32(1) / (float32(1) - float32(p))``, evaluated in float32 as the kernels do; that can
differ from the exactly rounded float32(1 / (1 - p)) by one ulp, far inside every tolerance that uses it.

All arithmetic is on uint64 arrays reduced with ``& 0xffffffff`` after every step that can exceed 32 bits, so numpy
never overflows or promotes.  The product package never imports this module.
"""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)
STREAM_NODE = np.uint64(0x4E4F4445)       # 'NODE'
STREAM_MESS = np.uint64(0x4D455353)       # 'MESS'


def _u32(x):
    return np.asarray(x).astype(np.uint64) & M32


def mix(h):
    """ngcf_mix: the murmur3 32-bit finalizer."""
    h = _u32(h)
    h ^= h >> np.uint64(16)
    h = (h * np.uint64(0x85EBCA6B)) & M32
    h ^= h >> np.uint64(13)
    h = (h * np.uint64(0xC2B2AE35)) & M32
    h ^= h >> np.uint64(16)
    return h


def seed_words(seed: int):
    """(low, high) 32-bit words of a 64-bit seed (taken modulo 2^64, like seed + *seed_dev on the device)."""
    seed = int(seed) % (1 << 64)
    return np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)


def threshold16(p: float) -> int:
    """ngcf_threshold16: keep iff a 16-bit uniform is >= this."""
    return int(np.float32(p) * np.float32(65536.0))


def keep_scale(p: float) -> np.float32:
    """1/(1-p) as the kernels compute it, in float32."""
    return np.float32(1.0) / (np.float32(1.0) - np.float32(p))


def node_key(row, col):
    """ngcf_node_key(row, col): the static 32-bit key of entry (row, col) of L (uint64 array of 32-bit values)."""
    a = mix((_u32(row) + np.uint64(0x9E3779B9)) & M32)
    b = (_u32(col) * np.uint64(0x85EBCA77) + np.uint64(0xC2B2AE3D)) & M32
    return mix(a ^ b)


def node_keep_bits_key(seed: int, p: float, n_layers: int, key):
    """node_keep_bits_key: the cumulative decision bits (bit k = survives layers 0..k) of entries with these keys."""
    lo, hi = seed_words(seed)
    thr = np.uint64(threshold16(p))
    key = _u32(key)
    bits = np.zeros(key.shape, dtype=np.uint64)
    keep = np.ones(key.shape, dtype=bool)
    for g in range((n_layers + 3) // 4):
        h = mix(key ^ lo ^ np.uint64((g * 0x632BE5AB) & 0xFFFFFFFF) ^ STREAM_NODE)
        y = mix(h ^ hi)
        u = (h & np.uint64(0xFFFF), h >> np.uint64(16), y & np.uint64(0xFFFF), y >> np.uint64(16))
        for j in range(4):
            layer = g * 4 + j
            keep &= u[j] >= thr
            if layer < n_layers:
                bits |= keep.astype(np.uint64) << np.uint64(layer)
    return bits


def node_keep_bits(seed: int, p: float, n_layers: int, row, col):
    """node_keep_bits(p, seed, n_layers, row, col) for arrays of global coordinates of L."""
    return node_keep_bits_key(seed, p, n_layers, node_key(row, col))


def edge_keep(seed: int, p: float, n_layers: int, row, col):
    """Per-layer bool keep lists of entries (row, col) of L (COO order in, COO order out): what the CPU oracle takes
    as ``edge_keep``."""
    bits = node_keep_bits(seed, p, n_layers, row, col)
    return [((bits >> np.uint64(k)) & np.uint64(1)).astype(bool) for k in range(n_layers)]


def mess_keep(seed: int, p: float, layer: int, n_rows: int, d_out: int, row_offset: int = 0):
    """bool [n_rows, d_out]: message-dropout decisions of local rows 0..n_rows-1 = global rows row_offset + r."""
    lo, hi = seed_words(seed)
    thr = np.uint64(threshold16(p))
    row = np.arange(n_rows, dtype=np.uint64)[:, None] + np.uint64(row_offset)
    idx = row * np.uint64(d_out) + np.arange(d_out, dtype=np.uint64)[None, :]      # < 2^63 for any real shape
    quad, j = idx >> np.uint64(2), idx & np.uint64(3)
    h = mix((quad & M32) ^ lo ^ STREAM_MESS ^ np.uint64((layer * 0x632BE5AB) & 0xFFFFFFFF))
    h = mix(h ^ (((quad >> np.uint64(32)) + np.uint64(0x9E3779B9)) & M32) ^ hi)
    y = mix(h ^ np.uint64(0x68E31DA4))
    u = np.where(j < 2, h, y)
    u = np.where((j & np.uint64(1)) == 0, u & np.uint64(0xFFFF), u >> np.uint64(16))
    return u >= thr


def mess_mult(seed: int, p: float, layer: int, n_rows: int, d_out: int, row_offset: int = 0):
    """float32 [n_rows, d_out] inverted-dropout multipliers (keep * 1/(1-p)): the oracle's ``mess_mult``."""
    return mess_keep(seed, p, layer, n_rows, d_out, row_offset).astype(np.float32) * keep_scale(p)


def pack_mess_bits(keep):
    """bool [n_rows, d_out] -> the int32 [n_rows, ceil(d_out/32)] word layout of ngcf_mess_dropout_bits
    (bit col & 31 of word col >> 5)."""
    n_rows, d_out = keep.shape
    words = (d_out + 31) // 32
    padded = np.zeros((n_rows, words * 32), dtype=np.uint64)
    padded[:, :d_out] = keep
    weights = np.uint64(1) << np.arange(32, dtype=np.uint64)
    w = (padded.reshape(n_rows, words, 32) * weights).sum(axis=2, dtype=np.uint64)
    return w.astype(np.uint32).view(np.int32)
