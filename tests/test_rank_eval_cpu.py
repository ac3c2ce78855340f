"""CPU checks of full-ranking evaluation: the Interactions CSR, the metric definitions on hand-worked lists, and the
argument validation of full_rank_eval / rank_metrics / score_topk(exclude=...) and of the two C entry points."""
import ctypes

import numpy as np
import pytest
import torch

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import _lib
from tests import _rank_ref as R


def test_from_pairs_sorts_and_deduplicates():
    x = pkg.Interactions.from_pairs([3, 0, 3, 3, 1, 0], [5, 2, 1, 5, 0, 2], 10)
    assert (x.n_rows, x.n_items) == (4, 10)
    assert x.ptr.dtype == torch.int64 and x.idx.dtype == torch.int32
    assert x.ptr.tolist() == [0, 1, 2, 2, 4]                       # user 2 has no pairs: an empty row
    assert x.idx.tolist() == [2, 0, 1, 5]
    assert [r.tolist() for r in R.rows_of(x)] == [[2], [0], [], [1, 5]]


def test_from_pairs_rows_remap_and_drop_other_users():
    user = np.array([3, 0, 3, 3, 1, 7, 7])
    item = np.array([5, 2, 1, 5, 0, 9, 4])
    x = pkg.Interactions.from_pairs(user, item, 10, rows=torch.tensor([7, 3, 5]))
    assert x.n_rows == 3
    assert [r.tolist() for r in R.rows_of(x)] == [[4, 9], [1, 5], []]   # row r = user rows[r]; users 0, 1 left out
    e = pkg.Interactions.from_pairs(user, item, 10, rows=[])
    assert e.n_rows == 0 and e.ptr.tolist() == [0] and e.idx.numel() == 0
    z = pkg.Interactions.from_pairs([], [], 10)
    assert z.n_rows == 0 and z.ptr.tolist() == [0]


def test_from_pairs_matches_a_python_restatement():
    rng = np.random.default_rng(0)
    user, item = rng.integers(0, 50, 3000), rng.integers(0, 400, 3000)
    rows = rng.permutation(60)[:40]
    x = pkg.Interactions.from_pairs(torch.from_numpy(user), torch.from_numpy(item), 400, rows=rows)
    want = [sorted(set(item[user == u].tolist())) for u in rows]
    assert [r.tolist() for r in R.rows_of(x)] == want


@pytest.mark.parametrize("user,item,n_items,rows", [
    ([0, 1], [0, 10], 10, None),                 # item id == n_items
    ([0, 1], [-1, 3], 10, None),                 # negative item id
    ([-2, 1], [0, 3], 10, None),                 # negative user id
    ([0, 1, 2], [0, 3], 10, None),               # lengths differ
    ([0, 1], [0, 3], 0, None),                   # no items
    ([0, 1], [0, 3], 10, [1, 1]),                # rows not unique
])
def test_from_pairs_rejects_bad_input(user, item, n_items, rows):
    with pytest.raises(ValueError):
        pkg.Interactions.from_pairs(user, item, n_items, rows=rows)


def test_metric_restatement_on_hand_worked_lists():
    l2 = np.log2
    # one hit at position 1 of 2: recall 1/2, precision 1/2, ndcg = (1/log2 3) / (1 + 1/log2 3)
    got = R.user_metrics([5, 3, 9, 1], {3, 1}, [2, 4])
    np.testing.assert_allclose(got[0], [0.5, 0.5, (1 / l2(3)) / (1 + 1 / l2(3)), 1.0])
    np.testing.assert_allclose(got[1], [1.0, 0.5, (1 / l2(3) + 1 / l2(5)) / (1 + 1 / l2(3)), 1.0])
    # the same hits at other positions: same recall / precision, different ndcg
    a, b = R.user_metrics([3, 1, 5, 9], {3, 1}, [4]), R.user_metrics([5, 9, 3, 1], {3, 1}, [4])
    assert a[0, 0] == b[0, 0] == 1.0 and a[0, 1] == b[0, 1] == 0.5
    assert a[0, 2] == pytest.approx(1.0) and b[0, 2] == pytest.approx((1 / l2(4) + 1 / l2(5)) / (1 + 1 / l2(3)))
    # |T| < K: the ideal list is only |T| long
    np.testing.assert_allclose(R.user_metrics([7, 2, 3], {7}, [3])[0], [1.0, 1 / 3, 1.0, 1.0])
    # |T| > K
    np.testing.assert_allclose(R.user_metrics([1, 9, 2], {1, 2, 3, 4, 5}, [3])[0],
                               [2 / 5, 2 / 3, (1 + 1 / l2(4)) / (1 + 1 / l2(3) + 1 / l2(4)), 1.0])
    # no hit; empty slots (-1) never hit
    np.testing.assert_allclose(R.user_metrics([4, -1, -1], {8}, [3])[0], [0, 0, 0, 0])
    # empty T: zeros, and the user does not count
    means, n, per = R.metrics([[1, 2], [1, 2]], [[], [2]], [2])
    assert n == 1 and np.all(per[0] == 0)
    np.testing.assert_allclose(means[0], [1.0, 0.5, (1 / l2(3)) / 1.0, 1.0])


def _cpu_case():
    u, it = torch.zeros(3, 8), torch.zeros(50, 8)
    tr = pkg.Interactions.from_pairs([0, 1, 2], [1, 2, 3], 50)
    return u, it, tr


@pytest.mark.parametrize("Ks,msg", [((), "cut-offs"), ((20, 10), "ascending"), ((0, 5), "ascending"),
                                    ((10, 10), "ascending"), (tuple(range(1, 10)), "cut-offs"), ((20, 129), "128")])
def test_full_rank_eval_rejects_bad_cutoffs(Ks, msg):
    u, it, tr = _cpu_case()
    with pytest.raises(ValueError, match=msg):
        pkg.full_rank_eval(u, it, train=tr, test=tr, Ks=Ks)


def test_full_rank_eval_rejects_mismatched_interactions_and_cpu_tensors():
    u, it, tr = _cpu_case()
    short = pkg.Interactions.from_pairs([0, 1], [1, 2], 50)
    with pytest.raises(ValueError, match="2 rows"):
        pkg.full_rank_eval(u, it, train=short, test=tr)
    with pytest.raises(ValueError, match="test has"):
        pkg.full_rank_eval(u, it, train=tr, test=pkg.Interactions.from_pairs([0, 1, 2], [1, 2, 3], 60))
    with pytest.raises(TypeError):
        pkg.full_rank_eval(u, it, train=tr, test=None)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.full_rank_eval(u, it, train=tr, test=tr)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.score_topk(u, it, 5, exclude=tr)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.rank_metrics(torch.zeros(3, 20, dtype=torch.int64), tr, Ks=(5, 20))
    with pytest.raises(ValueError, match="list length"):
        pkg.rank_metrics(torch.zeros(3, 20, dtype=torch.int64), tr, Ks=(5, 21))


def test_c_entry_points_validate_before_any_cuda_call():
    lib = _lib.load()
    dummy = ctypes.c_void_p(16)
    ks = _lib.int_array([5, 3])
    assert lib.ngcf_rank_metrics(dummy, 4, 10, dummy, dummy, ks, 2, dummy, dummy, None) != 0
    assert b"ascending" in lib.ngcf_last_error()
    assert lib.ngcf_rank_metrics(dummy, 4, 10, dummy, dummy, _lib.int_array([5, 11]), 2, dummy, dummy, None) != 0
    assert b"rank_metrics" in lib.ngcf_last_error()
    assert lib.ngcf_rank_metrics(dummy, 4, 129, dummy, dummy, _lib.int_array([5]), 1, dummy, dummy, None) != 0
    assert lib.ngcf_rank_metrics(dummy, 4, 10, dummy, dummy, _lib.int_array(range(1, 10)), 9, dummy, dummy, None) != 0
    assert lib.ngcf_score_topk_excluding(dummy, 4, dummy, 100, 64, 10, None, None, dummy, dummy, dummy, 1 << 20,
                                         None) != 0
    assert b"score_topk_excluding" in lib.ngcf_last_error()
    assert lib.ngcf_score_topk_excluding(dummy, 4, dummy, 100, 64, 0, dummy, dummy, dummy, dummy, dummy, 1 << 20,
                                         None) != 0
    assert b"score_topk" in lib.ngcf_last_error()
