"""Sampled-softmax loss without a GPU: hand-worked values of the float64 restatement, SoftmaxLoss's argument checks,
and the C entry's refusals, all before any CUDA call."""
import ctypes
import math

import pytest
import torch

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import _lib
from tests import _softmax_ref as R


def test_restatement_by_hand_b2():
    u = torch.tensor([[1.0, 0.0], [0.0, 2.0]])
    p = torch.tensor([[1.0, 1.0], [0.0, 1.0]])
    # s = u p^T / 0.5: row 0 = (2, 0), row 1 = (4, 4)
    got = R.loss(u, p, torch.empty(0), temperature=0.5, weight_decay=0.0, batch_size=2)
    want = ((math.log(math.exp(2) + 1) - 2) + (math.log(2 * math.exp(4)) - 4)) / 2
    assert float(got) == pytest.approx(want, rel=1e-12)
    # with wd: |u|^2 + |p|^2 = (1 + 2) + (4 + 1)
    got = R.loss(u, p, torch.empty(0), temperature=0.5, weight_decay=0.1, batch_size=4)
    assert float(got) == pytest.approx((want * 2 + 0.1 * 8) / 4, rel=1e-12)


def test_restatement_by_hand_b3_with_a_masked_column():
    u = torch.eye(3)
    p = torch.tensor([[2.0, 0, 0], [0, 1.0, 0], [1.0, 0, 1.0]])
    n = torch.tensor([[0, 0, 1.0], [1.0, 0, 0], [0, 3.0, 0]])
    pos_ids = torch.tensor([7, 7, 5])                     # rows 0 and 1 share an item: p_1 is not row 0's negative
    neg_ids = torch.tensor([5, 2, 1])                     # n_0 is row 2's positive item: masked for row 2
    keep = R.mask(pos_ids, neg_ids, 3, True)
    assert keep.tolist() == [[True, False, True, True, True, True],
                             [False, True, True, True, True, True],
                             [True, True, True, False, True, True]]
    got = R.loss(u, p, n, temperature=1.0, weight_decay=0.0, batch_size=3, pos_ids=pos_ids, neg_ids=neg_ids)
    # s = u [p; n]^T: row 0 = (2, 0, 1 | 0, 1, 0), row 1 = (0, 1, 0 | 0, 0, 3), row 2 = (0, 0, 1 | 1, 0, 0)
    r0 = math.log(math.exp(2) + math.exp(1) + 1 + math.e + 1) - 2            # p_1 masked
    r1 = math.log(math.e + 1 + 1 + 1 + math.exp(3)) - 1                      # p_0 masked
    r2 = math.log(1 + 1 + math.e + 1 + 1) - 1                                # n_0 masked
    assert float(got) == pytest.approx((r0 + r1 + r2) / 3, rel=1e-12)
    _, gu, gp, gn = R.loss_and_grads(u, p, n, temperature=1.0, weight_decay=0.0, batch_size=3, pos_ids=pos_ids,
                                     neg_ids=neg_ids)
    # row 1's gradient through column 0 (masked for it) is zero: dL/du_1 = sum_j G_1j c_j has no p_0 term
    P1 = torch.tensor([0, math.e, 1, 1, 1, math.exp(3)], dtype=torch.float64) / (math.e + 1 + 1 + 1 + math.exp(3))
    P1[1] -= 1
    cols = torch.cat([p, n]).double()
    assert torch.allclose(gu[1], (P1 @ cols) / 3, rtol=1e-12, atol=1e-15)
    assert gp.shape == (3, 3) and gn.shape == (3, 3)
    # without ids nothing is masked
    full = R.loss(u, p, n, temperature=1.0, weight_decay=0.0, batch_size=3)
    assert float(full) > float(got)


def test_softmax_loss_validates_its_arguments():
    for kw, msg in ((dict(temperature=0.0), "temperature"), (dict(temperature=-1.0), "temperature"),
                    (dict(weight_decay=-0.1), "weight_decay"), (dict(batch_size=0), "batch_size")):
        args = dict(weight_decay=0.025, batch_size=8, temperature=0.2)
        args.update(kw)
        with pytest.raises(ValueError, match=msg):
            pkg.SoftmaxLoss(**args)
    crit = pkg.SoftmaxLoss(0.025, 8, 0.2)
    u = torch.zeros(4, 8)
    with pytest.raises(RuntimeError, match="CUDA"):
        crit(u, u, u)


def test_c_entry_refuses_bad_arguments():
    lib = _lib.load()
    d = ctypes.c_void_p(1024)
    need = ctypes.c_size_t()
    assert lib.ngcf_softmax_loss_workspace(8, 16, 64, ctypes.byref(need)) == 0 and need.value > 0
    one = ctypes.c_size_t()
    assert lib.ngcf_softmax_loss_workspace(8, 8, 64, ctypes.byref(one)) == 0 and one.value < need.value
    for args, msg in (((0, 0, 64), b"batch"), ((4097, 4097, 64), b"batch"), ((8, 16, 0), b"D 0"),
                      ((8, 16, 1153), b"D 1153"), ((8, 12, 64), b"n_cols")):
        assert lib.ngcf_softmax_loss_workspace(*args, ctypes.byref(one)) != 0
        assert msg in lib.ngcf_last_error(), (args, lib.ngcf_last_error())

    def call(u=d, p=d, n=d, B=8, D=64, pos=None, neg=None, tau=0.2, wd=0.0, bs=8.0, loss=d, gu=d, gp=d, gn=d, ws=d,
             ws_bytes=need.value):
        return lib.ngcf_softmax_loss(u, p, n, B, D, pos, neg, tau, wd, bs, loss, gu, gp, gn, ws, ws_bytes, None)

    for kw, msg in ((dict(u=None), b"null"), (dict(p=None), b"null"), (dict(loss=None), b"null"),
                    (dict(B=0), b"batch"), (dict(B=4097), b"batch"), (dict(D=0), b"D 0"), (dict(D=1153), b"D 1153"),
                    (dict(tau=0.0), b"temperature"), (dict(tau=float("nan")), b"temperature"),
                    (dict(tau=float("inf")), b"temperature"), (dict(wd=-1.0), b"weight_decay"),
                    (dict(bs=0.0), b"batch_size"), (dict(gp=None), b"every gradient"),
                    (dict(gn=None), b"every gradient"), (dict(gu=None), b"every gradient"),
                    (dict(n=None), b"gn given without n"), (dict(neg=d), b"neg_ids given without pos_ids"),
                    (dict(pos=d), b"without neg_ids"), (dict(n=None, gn=None, pos=d, neg=d), b"neg_ids given without n")):
        rc = call(**kw)
        assert rc == -1, (kw, rc)
        assert msg in lib.ngcf_last_error(), (kw, lib.ngcf_last_error())
    assert call(ws_bytes=need.value - 1) == -3                           # NGCF_ERR_WORKSPACE
    assert b"workspace" in lib.ngcf_last_error()
    assert call(ws=None) == -3
    assert call(n=None, gn=None, ws_bytes=one.value - 1) == -3           # without n the smaller workspace is checked


def test_product_never_imports_the_restatement():
    import os
    pkg_dir = os.path.dirname(pkg.__file__)
    for f in os.listdir(pkg_dir):
        if f.endswith(".py"):
            assert "_softmax_ref" not in open(os.path.join(pkg_dir, f)).read(), f
