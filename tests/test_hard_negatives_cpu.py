"""CPU checks of dynamic hard-negative sampling: HardNegatives' argument validation, the host restatement of the
candidate draws (support and uniformity), and the refusals of the C entry point before any CUDA call."""
import ctypes

import numpy as np
import pytest
import torch
from scipy import stats

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import _lib
from tests import _hneg_ref as H


def _train(n_user=6, n_items=10):
    return pkg.Interactions.from_pairs([0, 0, 2, 5], [1, 7, 3, 9], n_items, rows=torch.arange(n_user))


def test_hard_negatives_validates_its_arguments():
    hn = pkg.HardNegatives(_train())
    assert hn.n_candidates == 32 and hn.chosen is None and not hn.debug
    assert pkg.HardNegatives(_train(), 1).n_candidates == 1
    assert pkg.HardNegatives(_train(), 64).n_candidates == 64
    with pytest.raises(TypeError, match="Interactions"):
        pkg.HardNegatives((torch.zeros(3, dtype=torch.int64), torch.zeros(0, dtype=torch.int32)))
    for m in (0, 65, -1):
        with pytest.raises(ValueError, match="n_candidates"):
            pkg.HardNegatives(_train(), m)


def test_hard_negatives_refuses_a_user_with_every_item():
    full = pkg.Interactions.from_pairs([0, 1, 1, 1, 1], [2, 0, 1, 2, 3], 4, rows=torch.arange(3))
    with pytest.raises(ValueError, match="row 1 lists all 4 items"):
        pkg.HardNegatives(full)
    one_left = pkg.Interactions.from_pairs([1, 1, 1], [0, 1, 3], 4, rows=torch.arange(3))
    pkg.HardNegatives(one_left)                                          # one free item is enough


def test_restated_hash_words():
    """The restatement's hash of counter (a, b, c) differs in every argument and in the stream constant."""
    x0, y0 = H.hash64(5, 1, 0, 0)
    assert 0 <= int(x0) < 2 ** 32 and 0 <= int(y0) < 2 ** 32
    assert int(H.hash64(5, 2, 0, 0)[0]) != int(x0) and int(H.hash64(5, 1, 1, 0)[0]) != int(x0)
    assert int(H.hash64(5, 1, 0, 1)[0]) != int(x0) and int(H.hash64(5 + (1 << 32), 1, 0, 0)[0]) != int(x0)
    assert int(H.hash64(5, 1, 0, 0, stream=np.uint64(0x53414D50))[0]) != int(x0)


def test_restated_draws_never_hit_an_excluded_item():
    rng = np.random.default_rng(0)
    n_items, n_user = 300, 40
    rows = [np.sort(rng.choice(n_items, rng.integers(0, n_items), replace=False)) for _ in range(n_user)]
    rows[3] = np.delete(np.arange(n_items), 17)                          # exactly one free item
    rows[4] = np.array([], dtype=np.int64)                               # no excluded item
    u_id = np.concatenate([np.arange(n_user), rng.integers(0, n_user, 200)])
    cand = H.candidates(123456789012345, u_id, rows, n_items, 64)
    assert cand.shape == (u_id.size, 64) and cand.min() >= 0 and cand.max() < n_items
    for b, u in enumerate(u_id):
        assert not np.isin(cand[b], rows[u]).any(), b
    assert np.all(cand[u_id == 3] == 17)
    assert len(np.unique(cand[u_id == 4])) > 100                         # spread over the whole item range


def test_restated_draws_are_uniform_over_free_items():
    n_items = 50
    excluded = np.array([0, 1, 2, 10, 11, 30, 48, 49])
    free = H.free_items(excluded, n_items)
    B, M = 400, 64                                                       # 25 600 draws, ~610 per free item
    for seed in (1, 2 ** 40 + 7):
        cand = H.candidates(seed, np.zeros(B, dtype=np.int64), [excluded], n_items, M)
        counts = np.array([(cand == i).sum() for i in free])
        assert counts.sum() == B * M
        assert stats.chisquare(counts).pvalue > 1e-3, seed


def test_c_entry_refuses_bad_arguments():
    lib = _lib.load()
    d = ctypes.c_void_p(16)
    layers, dims = _lib.ptr_array_int([16, 16]), _lib.int_array([64, 64])

    def call(layers=layers, dims=dims, n=2, n_user=10, u_id=d, batch=4, ptr=d, idx=d, n_items=20, M=8, chosen=d):
        return lib.ngcf_hard_negatives(layers, dims, n, n_user, u_id, batch, ptr, idx, n_items, M, 1, None, chosen,
                                       None, None, None)

    for kw, msg in ((dict(n=0), b"blocks"), (dict(n=10), b"blocks"), (dict(dims=_lib.int_array([64, 129])), b"block 1"),
                    (dict(layers=_lib.ptr_array_int([16, 0])), b"block 1"), (dict(n_user=0), b"n_user"),
                    (dict(n_items=0), b"n_items"), (dict(n_items=2 ** 31), b"n_items"), (dict(M=0), b"M 0"),
                    (dict(M=65), b"M 65"), (dict(batch=-1), b"batch"), (dict(u_id=None), b"null"),
                    (dict(ptr=None), b"null"), (dict(chosen=None), b"null")):
        assert call(**kw) != 0, kw
        assert msg in lib.ngcf_last_error(), (kw, lib.ngcf_last_error())
    assert call(batch=0, u_id=None, ptr=None, chosen=None) == 0        # nothing to do, nothing launched


def test_product_never_imports_the_restatement():
    import os
    pkg_dir = os.path.dirname(pkg.__file__)
    for f in os.listdir(pkg_dir):
        if f.endswith(".py"):
            assert "_hneg_ref" not in open(os.path.join(pkg_dir, f)).read(), f
