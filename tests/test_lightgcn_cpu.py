"""LightGCN without a GPU: constructor checks, the new C entries' refusals (before any CUDA call), the float64
restatement on a hand-worked graph, and that the product never imports the restatement."""
import ctypes
import math
import os

import numpy as np
import pytest
import torch

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import _lib, laplacian, synth
from tests import _lightgcn_ref as R

N_USER, N_ITEM = 6, 4


def _lap(n_user=N_USER, n_item=N_ITEM):
    u = np.arange(n_user) % n_item
    return laplacian.laplacian_coo(np.arange(n_user), u, np.ones(n_user, np.float32), n_user, n_item)


def _model(**kw):
    args = dict(embed_size=8, n_layers=2, lap_list=[_lap()], num_dict=synth.num_dict_for(N_USER, N_ITEM))
    args.update(kw)
    return pkg.LightGCN(args.pop("embed_size"), args.pop("n_layers"), args.pop("lap_list"), args.pop("num_dict"), **args)


def test_constructor_tables_and_init():
    torch.manual_seed(0)
    m = _model(embed_size=65, n_layers=3)
    assert list(m.state_dict()) == ["user_embedding.weight", "item_embedding.weight"]
    assert m.user_embedding.weight.shape == (N_USER, 65) and m.item_embedding.weight.shape == (N_ITEM, 65)
    assert m._node_mode == "bits" and _model(embed_size=64)._node_mode == "compact"
    big = pkg.LightGCN(64, 1, [_lap(3000, 1000)], synth.num_dict_for(3000, 1000))
    assert abs(float(big.user_embedding.weight.std()) - 0.1) < 0.005         # normal_(std=0.1)
    assert abs(float(big.user_embedding.weight.mean())) < 0.005
    mixed = _model(embed_size=65, emb_ratio=1.0)
    assert {"age_emb.weight", "sex_emb.weight", "month_emb.weight", "day_emb.weight", "dow_emb.weight"} <= \
        set(mixed.state_dict())
    assert mixed.feat_widths == [13, 13, 13, 13, 13]
    for bad in (0, 9):
        with pytest.raises(ValueError, match="n_layers"):
            _model(n_layers=bad)
    for bad in (0, 129):
        with pytest.raises(ValueError, match="embed_size"):
            _model(embed_size=bad)
    with pytest.raises(ValueError, match="node_dropout"):
        _model(node_dropout=1.0)
    with pytest.raises(ValueError, match="emb_ratio"):
        _model(emb_ratio=-0.5)
    with pytest.raises(ValueError, match=r"n_user \+ n_item = 10"):
        _model(lap_list=[_lap(), _lap(5, 4)])
    with pytest.raises(NotImplementedError, match="row-sharded"):
        _model().shard()


def test_cpu_device_is_refused():
    m = _model()
    b = {k: torch.from_numpy(v) for k, v in synth.random_batch(N_USER, N_ITEM, 4, seed=1).items()}
    with pytest.raises(RuntimeError, match="CUDA device only"):
        m(b["year"], b["u_id"], b["age"], b["sex"], b["month"], b["day"], b["dow"], b["pos_item"], b["neg_item"], True)


def _rc(fn, *args):
    rc = fn(*args)
    return rc, _lib.load().ngcf_last_error().decode()


def test_c_entries_refuse_bad_arguments():
    """Every refusal returns NGCF_ERR_INVALID (-1) with its own message: nothing reaches the CUDA runtime (which, without
    a device, would fail with NGCF_ERR_CUDA instead).  Pointers are never dereferenced on the host."""
    lib = _lib.load()
    P = 256                                                          # a non-null fake device address
    lay = _lib.ptr_array_int([P] * 3)
    sets = dict(rows=_lib.ptr_array_int([P]), offs=_lib.i64_array([0]), sizes=_lib.i64_array([4]),
                outs=_lib.ptr_array_int([P]))
    cases = [
        (lib.ngcf_layer_mean, (None, 3, 8, None, 0, 4, P, 8, None), "null layer array"),
        (lib.ngcf_layer_mean, (lay, 0, 8, None, 0, 4, P, 8, None), "0 layers"),
        (lib.ngcf_layer_mean, (lay, 10, 8, None, 0, 4, P, 8, None), "10 layers"),
        (lib.ngcf_layer_mean, (lay, 3, 0, None, 0, 4, P, 8, None), "width 0"),
        (lib.ngcf_layer_mean, (lay, 3, 129, None, 0, 4, P, 129, None), "width 129"),
        (lib.ngcf_layer_mean, (lay, 3, 8, None, 0, 4, P, 7, None), "ld_out 7"),
        (lib.ngcf_layer_mean, (_lib.ptr_array_int([P, 0, P]), 3, 8, None, 0, 4, P, 8, None), "null layer 1"),
        (lib.ngcf_layer_mean, (lay, 3, 8, None, 0, -1, P, 8, None), "n_out -1"),
        (lib.ngcf_layer_mean, (lay, 3, 8, None, 0, 4, None, 8, None), "null output"),
        (lib.ngcf_layer_mean_sets, (lay, 3, 8, sets["rows"], sets["offs"], sets["sizes"], sets["outs"], 0, 8, None),
         "n_sets 0"),
        (lib.ngcf_layer_mean_sets, (lay, 3, 8, sets["rows"], sets["offs"], sets["sizes"], sets["outs"], 5, 8, None),
         "n_sets 5"),
        (lib.ngcf_layer_mean_sets, (lay, 3, 8, None, sets["offs"], sets["sizes"], sets["outs"], 1, 8, None),
         "null host array"),
        (lib.ngcf_layer_mean_sets, (lay, 3, 8, _lib.ptr_array_int([0]), sets["offs"], sets["sizes"], sets["outs"], 1, 8,
                                    None), "set 0"),
        (lib.ngcf_layer_mean_sets, (lay, 3, 8, sets["rows"], sets["offs"], _lib.i64_array([-1]), sets["outs"], 1, 8,
                                    None), "set 0"),
        (lib.ngcf_rowgrad_expand, (None, 10, P, 8, 8, 0.5, P, 8, None), "null pointer"),
        (lib.ngcf_rowgrad_expand, (P, 10, None, 8, 8, 0.5, P, 8, None), "null pointer"),
        (lib.ngcf_rowgrad_expand, (P, 10, P, 8, 8, 0.5, None, 8, None), "null pointer"),
        (lib.ngcf_rowgrad_expand, (P, -1, P, 8, 8, 0.5, P, 8, None), "n_rows -1"),
        (lib.ngcf_rowgrad_expand, (P, 1 << 31, P, 8, 8, 0.5, P, 8, None), "n_rows 2147483648"),
        (lib.ngcf_rowgrad_expand, (P, 10, P, 8, 0, 0.5, P, 8, None), "width 0"),
        (lib.ngcf_rowgrad_expand, (P, 10, P, 8, 129, 0.5, P, 129, None), "width 129"),
        (lib.ngcf_rowgrad_expand, (P, 10, P, 7, 8, 0.5, P, 8, None), "row pitches 7 / 8"),
        (lib.ngcf_rowgrad_expand, (P, 10, P, 8, 8, 0.5, P, 4, None), "row pitches 8 / 4"),
    ]
    hn = lambda **kw: tuple({**dict(layers=lay, d=8, n=3, n_user=6, u_id=P, batch=4, ptr=P, idx=P, n_items=4, M=8,
                                    signed=0, seed=1, seed_dev=None, chosen=P, cand=None, score=None, stream=None),
                             **kw}.values())
    cases += [
        (lib.ngcf_hard_negatives_mean, hn(d=0), "bad block 0"),
        (lib.ngcf_hard_negatives_mean, hn(d=129), "bad block 0"),
        (lib.ngcf_hard_negatives_mean, hn(n=10), "10 blocks"),
        (lib.ngcf_hard_negatives_mean, hn(n=0), "0 blocks"),
        (lib.ngcf_hard_negatives_mean, hn(layers=None), "null layer array"),
        (lib.ngcf_hard_negatives_mean, hn(M=0), "M 0 outside"),
        (lib.ngcf_hard_negatives_mean, hn(M=65), "M 65 outside"),
        (lib.ngcf_hard_negatives_mean, hn(n_items=0), "n_items 0"),
        (lib.ngcf_hard_negatives_mean, hn(n_user=0), "n_user 0"),
        (lib.ngcf_hard_negatives_mean, hn(chosen=None), "null pointer"),
    ]
    for fn, args, msg in cases:
        rc, err = _rc(fn, *args)
        assert rc == -1, (fn.__name__, msg, rc, err)
        assert msg in err, (fn.__name__, msg, err)


def test_restatement_by_hand_two_users_two_items():
    """Users u0, u1, items i0, i1; edges u0-i0, u0-i1, u1-i1.  Degrees 2, 1, 1, 2, so L = D^-1/2 A D^-1/2 has
    L[u0,i0] = 1/sqrt(2), L[u0,i1] = 1/2, L[u1,i1] = 1/sqrt(2), and the transposed entries."""
    L = laplacian.laplacian_coo(np.array([0, 0, 1]), np.array([0, 1, 1]), np.ones(3, np.float32), 2, 2)
    r2 = 1 / math.sqrt(2)
    Ld = torch.tensor([[0, 0, r2, 0.5], [0, 0, 0, r2], [r2, 0, 0, 0], [0.5, r2, 0, 0]], dtype=torch.float64)
    assert torch.allclose(L.to_dense().double(), Ld, atol=1e-7)
    user_w = torch.tensor([[1.0], [2.0]], dtype=torch.float64, requires_grad=True)
    item_w = torch.tensor([[3.0], [4.0]], dtype=torch.float64, requires_grad=True)
    # K = 1: E_1 = L E_0 = [3/sqrt2 + 4/2, 4/sqrt2, 1/sqrt2, 1/2 + 2/sqrt2]
    E1 = [3 * r2 + 2, 4 * r2, r2, 0.5 + 2 * r2]
    F = R.final_rows(L, user_w, item_w, 1)
    want = torch.tensor([[(e0 + e1) / 2] for e0, e1 in zip([1, 2, 3, 4], E1)], dtype=torch.float64)
    assert torch.allclose(F, want, rtol=1e-7, atol=0)
    # d F[u0] / d E_0 = (e_u0 + L^T e_u0) / 2 = [1/2, 0, 1/(2 sqrt2), 1/4]
    F[0, 0].backward()
    assert torch.allclose(torch.cat([user_w.grad, item_w.grad]).flatten(),
                          torch.tensor([0.5, 0, r2 / 2, 0.25], dtype=torch.float64), rtol=1e-7, atol=0)
    # K = 2 with u0-i1 (both directions) dropped at layer 1 only: E_2 = L' E_1, L' = L without those entries
    row, col, _ = R.coo_of(L)
    drop = ((row == 0) & (col == 3)) | ((row == 3) & (col == 0))
    keep = [np.ones(row.size, bool), ~drop]
    F2 = R.final_rows(L, user_w.detach(), item_w.detach(), 2, keep)
    E2 = [r2 * E1[2], r2 * E1[3], r2 * E1[0], r2 * E1[1]]
    want2 = torch.tensor([[(a + b + c) / 3] for a, b, c in zip([1, 2, 3, 4], E1, E2)], dtype=torch.float64)
    assert torch.allclose(F2, want2, rtol=1e-7, atol=0)
    u, p, n = R.batch_rows(F2, 2, [1, 0], [1, 1], [0, 0])
    assert torch.equal(u, F2[[1, 0]]) and torch.equal(p, F2[[3, 3]]) and torch.equal(n, F2[[2, 2]])


def test_product_never_imports_the_restatement():
    pkg_dir = os.path.dirname(pkg.__file__)
    for f in os.listdir(pkg_dir):
        if f.endswith(".py"):
            assert "_lightgcn_ref" not in open(os.path.join(pkg_dir, f)).read(), f
