"""Properties of the numpy restatement of the device-RNG dropout decisions (tests/_dropout_ref.py): the GPU tests take
it as the reference, so it must itself draw what dropout promises (keep rates, cumulative layers, independent draws)."""
import numpy as np
import pytest

from tests import _dropout_ref as R

SEED = 0x5DEECE66D_2F1A3B7
RNG = np.random.default_rng(0)
ROW = RNG.integers(0, 1 << 27, 200_000)
COL = RNG.integers(0, 1 << 27, 200_000)


@pytest.mark.parametrize("p", [0.05, 0.1, 0.3, 0.5, 0.77, 0.9])
def test_keep_fraction_follows_threshold(p):
    thr = R.threshold16(p)
    assert thr == int(np.float32(p) * 65536)
    keep = 1.0 - thr / 65536
    bits = R.node_keep_bits(SEED, p, 8, ROW, COL)
    sigma = np.sqrt(keep * (1 - keep) / ROW.size)
    for k in range(8):                                         # layer k survives with keep^(k+1)
        f = float(((bits >> np.uint64(k)) & np.uint64(1)).mean())
        want = keep ** (k + 1)
        assert abs(f - want) <= 5 * max(sigma, np.sqrt(want * (1 - want) / ROW.size)) + 1e-6, (k, f, want)
    m = R.mess_keep(SEED, p, 3, 1000, 200, row_offset=12345)
    assert abs(float(m.mean()) - keep) <= 5 * np.sqrt(keep * (1 - keep) / m.size)
    mult = R.mess_mult(SEED, p, 3, 1000, 200, row_offset=12345)
    assert mult.dtype == np.float32 and set(np.unique(mult).tolist()) == {0.0, float(R.keep_scale(p))}
    assert abs(float(R.keep_scale(p)) - 1 / (1 - p)) <= 1e-6 / (1 - p)


def test_node_bits_are_cumulative():
    for p in (0.1, 0.5):
        bits = R.node_keep_bits(SEED, p, 8, ROW, COL)
        assert bits.max() < 256
        for k in range(1, 8):
            on = ((bits >> np.uint64(k)) & np.uint64(1)) == 1
            below = bits & np.uint64((1 << k) - 1)
            assert np.all(below[on] == (1 << k) - 1), k
        # fewer layers = the low bits of the same draws
        for n in (1, 3, 4, 5, 7):
            assert np.array_equal(R.node_keep_bits(SEED, p, n, ROW, COL), bits & np.uint64((1 << n) - 1)), n


def test_layers_4_to_7_are_drawn_from_their_own_group():
    p = 0.5
    bits = R.node_keep_bits(SEED, p, 8, ROW, COL)
    full = bits == 255                                          # survived all 8 layers
    assert 0.5 ** 8 * 0.8 < float(full.mean()) < 0.5 ** 8 * 1.2
    # among the entries that survived layers 0..3, the survival of layers 4..7 is independent of the draws of 0..3
    s3 = (bits & np.uint64(15)) == 15
    f4 = float(((bits[s3] >> np.uint64(4)) & np.uint64(1)).mean())
    assert abs(f4 - 0.5) < 0.03
    # the second group's 16-bit uniforms are not the first group's: compare the raw draws
    key = R.node_key(ROW, COL)
    lo, hi = R.seed_words(SEED)
    h0 = R.mix(key ^ lo ^ np.uint64(0) ^ R.STREAM_NODE)
    h1 = R.mix(key ^ lo ^ np.uint64(0x632BE5AB) ^ R.STREAM_NODE)
    assert float((h0 == h1).mean()) < 1e-4
    assert abs(np.corrcoef((h0 & np.uint64(0xFFFF)).astype(float), (h1 & np.uint64(0xFFFF)).astype(float))[0, 1]) < 0.02


def test_transposed_coordinates_draw_independently():
    a = R.node_keep_bits(SEED, 0.5, 8, ROW, COL) & np.uint64(1)
    b = R.node_keep_bits(SEED, 0.5, 8, COL, ROW) & np.uint64(1)
    assert abs(float((a == b).mean()) - 0.5) < 0.01
    assert not np.array_equal(R.node_key(ROW, COL), R.node_key(COL, ROW))
    assert np.array_equal(R.node_key(ROW[:10], ROW[:10]), R.node_key(ROW[:10], ROW[:10]))


def test_seed_high_word_changes_decisions():
    lo_only = 0x9ABCDEF0
    s1, s2 = (1 << 32) | lo_only, (7 << 32) | lo_only
    for s in (s1, s2):
        assert R.seed_words(s)[0] == R.seed_words(lo_only)[0]
    n0 = R.node_keep_bits(lo_only, 0.5, 8, ROW, COL)
    n1 = R.node_keep_bits(s1, 0.5, 8, ROW, COL)
    n2 = R.node_keep_bits(s2, 0.5, 8, ROW, COL)
    for x, y in ((n0, n1), (n1, n2)):
        # layers 0-1 (and 4-5) of a group come from its first mix, which sees the low word only (see _dropout_ref);
        # layers 2-3 come from the second mix, which folds in the high word
        assert np.array_equal(x & np.uint64(3), y & np.uint64(3))
        both = (x & np.uint64(3)) == 3
        agree = ((x[both] >> np.uint64(2)) & np.uint64(1)) == ((y[both] >> np.uint64(2)) & np.uint64(1))
        assert abs(float(agree.mean()) - 0.5) < 0.02
    m0 = R.mess_keep(lo_only, 0.5, 2, 500, 64, 77)
    m1 = R.mess_keep(s1, 0.5, 2, 500, 64, 77)
    assert abs(float((m0 == m1).mean()) - 0.5) < 0.02
    # the seed is taken modulo 2^64, as seed + *seed_dev wraps on the device
    assert np.array_equal(R.node_keep_bits((1 << 64) + 5, 0.3, 8, ROW[:100], COL[:100]),
                          R.node_keep_bits(5, 0.3, 8, ROW[:100], COL[:100]))


def test_message_decisions_follow_the_global_flat_index():
    """Rows of a shard at row_offset r0 draw what rows r0.. of the whole table draw; the quad index uses its high word."""
    full = R.mess_keep(SEED, 0.4, 5, 300, 65)
    assert np.array_equal(R.mess_keep(SEED, 0.4, 5, 100, 65, row_offset=123), full[123:223])
    assert not np.array_equal(R.mess_keep(SEED, 0.4, 6, 300, 65), full)          # layers draw independently
    big = 1 << 30                                                                  # (2^30 * 128) / 4 > 2^32
    a = R.mess_keep(SEED, 0.5, 1, 4, 128, row_offset=big)
    b = R.mess_keep(SEED, 0.5, 1, 4, 128, row_offset=big - (1 << 32) // 32)       # same low 32 bits of the quad
    assert abs(float((a == b).mean()) - 0.5) < 0.15


def test_pack_mess_bits_layout():
    keep = RNG.random((7, 65)) < 0.5
    w = R.pack_mess_bits(keep).view(np.uint32)
    assert w.shape == (7, 3)
    for r in range(7):
        for c in range(65):
            assert bool((w[r, c >> 5] >> (c & 31)) & 1) == keep[r, c]
    assert np.all(w[:, 2] >> 1 == 0)                                               # columns past d_out stay 0


def test_product_never_imports_dropout_reference():
    import os
    import re
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "seoul_tourism_recommendation_ngcf_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+(tests\b|\S*_dropout_ref\b)", src, flags=re.M), f
                assert "_dropout_ref" not in src, f
