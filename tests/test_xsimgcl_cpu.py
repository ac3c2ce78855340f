"""XSimGCL without a GPU: constructor checks and refusals, the new C entries' refusals (before any CUDA call), the noise
restatement on a hand-worked 2-row example, and that the product never imports the restatement."""
import ctypes
import math
import os

import numpy as np
import pytest
import torch

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import _lib, laplacian, synth
from tests import _xsimgcl_ref as R

N_USER, N_ITEM = 6, 4


def _lap(n_user=N_USER, n_item=N_ITEM):
    u = np.arange(n_user) % n_item
    return laplacian.laplacian_coo(np.arange(n_user), u, np.ones(n_user, np.float32), n_user, n_item)


def _model(**kw):
    args = dict(embed_size=8, n_layers=2, lap_list=[_lap()], num_dict=synth.num_dict_for(N_USER, N_ITEM))
    args.update(kw)
    return pkg.XSimGCL(args.pop("embed_size"), args.pop("n_layers"), args.pop("lap_list"), args.pop("num_dict"), **args)


def test_constructor_defaults_state_dict_and_validation():
    torch.manual_seed(0)
    m = _model(embed_size=65, n_layers=3, cl_layer=3)
    assert isinstance(m, pkg.LightGCN)
    assert list(m.state_dict()) == ["user_embedding.weight", "item_embedding.weight"]
    torch.manual_seed(0)
    lg = pkg.LightGCN(65, 3, [_lap()], synth.num_dict_for(N_USER, N_ITEM))
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), lg.state_dict().values()))
    d = _model()
    assert (d.eps, d.cl_weight, d.cl_layer, d.temperature, d.emb_ratio, d.node_dropout) == (0.2, 0.2, 1, 0.2, 0.0, 0.0)
    assert d.cl_loss is None
    mixed = _model(embed_size=65, emb_ratio=1.0)
    assert {"age_emb.weight", "dow_emb.weight"} <= set(mixed.state_dict())
    for kw, msg in ((dict(eps=-0.1), "eps"), (dict(eps=float("nan")), "eps"), (dict(cl_weight=-1.0), "cl_weight"),
                    (dict(temperature=0.0), "temperature"), (dict(temperature=-1.0), "temperature"),
                    (dict(cl_layer=0), "cl_layer"), (dict(cl_layer=3), "cl_layer"),
                    (dict(n_layers=0), "n_layers"), (dict(n_layers=9), "n_layers"),
                    (dict(embed_size=0), "embed_size"), (dict(embed_size=129), "embed_size"),
                    (dict(emb_ratio=2.0), "emb_ratio")):
        with pytest.raises(ValueError, match=msg):
            _model(**kw)
    with pytest.raises(NotImplementedError, match="row-sharded"):
        _model().shard()


def test_refusals_before_any_device_work():
    m = _model()
    b = {k: torch.from_numpy(v) for k, v in synth.random_batch(N_USER, N_ITEM, 4, seed=1).items()}
    with pytest.raises(RuntimeError, match="CUDA device only"):
        m(b["year"], b["u_id"], b["age"], b["sex"], b["month"], b["day"], b["dow"], b["pos_item"], b["neg_item"], True)
    big = {k: torch.from_numpy(v) for k, v in synth.random_batch(N_USER, N_ITEM, 4097, seed=1).items()}
    with pytest.raises(ValueError, match="4097 rows"):
        m(big["year"], big["u_id"], big["age"], big["sex"], big["month"], big["day"], big["dow"], big["pos_item"],
          big["neg_item"], True)


def test_abi_symbols_present():
    lib = _lib.load()
    for name in ("ngcf_perturb_rows", "ngcf_infonce_workspace", "ngcf_infonce", "ngcf_rowgrad_add"):
        assert hasattr(lib, name) and name in _lib.SIGNATURES
    assert lib.ngcf_abi_version() == 4


def _rc(fn, *args):
    rc = fn(*args)
    return rc, _lib.load().ngcf_last_error().decode()


def test_c_entries_refuse_bad_arguments():
    """Every refusal returns NGCF_ERR_INVALID (-1) with its own message, before any CUDA call.  Pointers are never
    dereferenced on the host."""
    lib = _lib.load()
    P = 256                                                          # a non-null fake device address
    pr = lambda **kw: tuple({**dict(E=P, n=10, d=8, ld=8, eps=0.2, seed=1, seed_dev=None, layer=1, stream=None),
                             **kw}.values())
    nce = lambda **kw: tuple({**dict(x1=P, x2=P, B=16, D=64, ids=P, tau=0.2, loss=P, g1=P, g2=P, ws=P,
                                     bytes=1 << 30, stream=None), **kw}.values())
    one = dict(rows=_lib.ptr_array_int([P, P]), offs=_lib.i64_array([0, 6]), g=_lib.ptr_array_int([P, P]),
               sizes=_lib.i64_array([4, 4]))
    add = lambda **kw: tuple({**dict(rows=one["rows"], offs=one["offs"], g=one["g"], sizes=one["sizes"], n_sets=2, d=8,
                                     slot=P, dst=P, ld=8, stream=None), **kw}.values())
    ws = ctypes.c_size_t()
    cases = [
        (lib.ngcf_perturb_rows, pr(E=None), "null E"),
        (lib.ngcf_perturb_rows, pr(d=0, ld=0), "width 0"),
        (lib.ngcf_perturb_rows, pr(d=129, ld=129), "width 129"),
        (lib.ngcf_perturb_rows, pr(ld=7), "ld 7 < width 8"),
        (lib.ngcf_perturb_rows, pr(n=-1), "n_rows -1"),
        (lib.ngcf_perturb_rows, pr(n=1 << 31), "n_rows 2147483648"),
        (lib.ngcf_perturb_rows, pr(eps=-0.5), "eps -0.5"),
        (lib.ngcf_perturb_rows, pr(eps=float("inf")), "eps inf"),
        (lib.ngcf_perturb_rows, pr(layer=-1), "layer -1"),
        (lib.ngcf_perturb_rows, pr(layer=9), "layer 9"),
        (lib.ngcf_infonce_workspace, (0, 64, ctypes.byref(ws)), "batch 0"),
        (lib.ngcf_infonce_workspace, (4097, 64, ctypes.byref(ws)), "batch 4097"),
        (lib.ngcf_infonce_workspace, (16, 0, ctypes.byref(ws)), "D 0"),
        (lib.ngcf_infonce_workspace, (16, 1153, ctypes.byref(ws)), "D 1153"),
        (lib.ngcf_infonce_workspace, (16, 64, None), "null pointer"),
        (lib.ngcf_infonce, nce(x1=None), "null x1"),
        (lib.ngcf_infonce, nce(x2=None), "null x1, x2"),
        (lib.ngcf_infonce, nce(ids=None), "ids"),
        (lib.ngcf_infonce, nce(loss=None), "loss"),
        (lib.ngcf_infonce, nce(B=0), "batch 0"),
        (lib.ngcf_infonce, nce(B=4097), "batch 4097"),
        (lib.ngcf_infonce, nce(D=0), "D 0"),
        (lib.ngcf_infonce, nce(D=1153), "D 1153"),
        (lib.ngcf_infonce, nce(tau=0.0), "temperature 0"),
        (lib.ngcf_infonce, nce(g2=None), "both gradient buffers"),
        (lib.ngcf_rowgrad_add, add(rows=None), "null pointer"),
        (lib.ngcf_rowgrad_add, add(dst=None), "null pointer"),
        (lib.ngcf_rowgrad_add, add(n_sets=0), "n_sets 0"),
        (lib.ngcf_rowgrad_add, add(n_sets=3), "n_sets 3"),
        (lib.ngcf_rowgrad_add, add(d=0, ld=0), "width 0"),
        (lib.ngcf_rowgrad_add, add(d=129, ld=129), "width 129"),
        (lib.ngcf_rowgrad_add, add(ld=4), "ld_dst 4"),
        (lib.ngcf_rowgrad_add, add(g=_lib.ptr_array_int([P, 0])), "set 1"),
    ]
    for fn, args, msg in cases:
        rc, err = _rc(fn, *args)
        assert rc == -1, (fn.__name__, msg, rc, err)
        assert msg in err, (fn.__name__, msg, err)
    # a short workspace is its own status
    assert lib.ngcf_infonce_workspace(16, 64, ctypes.byref(ws)) == 0 and ws.value > 0
    rc, err = _rc(lib.ngcf_infonce, *nce(bytes=ws.value - 1))
    assert rc == -3 and "workspace" in err, (rc, err)          # NGCF_ERR_WORKSPACE


def _mix(h):
    h ^= h >> 16
    h = (h * 0x85EBCA6B) & 0xFFFFFFFF
    h ^= h >> 13
    h = (h * 0xC2B2AE35) & 0xFFFFFFFF
    return h ^ (h >> 16)


def _uniform_scalar(seed, row, col, layer):
    """ngcf_hash64 written out on Python ints (a second restatement of the numpy one)."""
    lo, hi = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    h = _mix(row ^ lo ^ 0x4E4F4953)
    h = _mix(h ^ ((col + 0x9E3779B9) & 0xFFFFFFFF) ^ hi)
    h = _mix((h + layer * 0x632BE5AB + 0x7F4A7C15) & 0xFFFFFFFF)
    return (h >> 8) / float(1 << 24)


def test_noise_restatement_by_hand_two_rows():
    """Two rows of width 3 at layer 2: row 0 = (1.5, -2, 0), row 1 = (0, 0, 0).  The noise is eps * sign(x) * u / |u|
    with u the row's three uniforms: row 0's third entry and all of row 1 stay zero (sign 0), row 0's second entry
    moves down."""
    seed, eps, layer = 0x1234_5678_9ABC_DEF0, 0.1, 2
    u = R.uniforms(seed, 2, 3, layer)
    for r in range(2):
        for c in range(3):
            want = _uniform_scalar(seed, r, c, layer)
            assert float(u[r, c]) == want and 0.0 <= want < 1.0 and want * (1 << 24) == int(want * (1 << 24))
    x = torch.tensor([[1.5, -2.0, 0.0], [0.0, 0.0, 0.0]], dtype=torch.float64)
    got = x + R.noise(x, seed, layer, eps)
    n0 = math.sqrt(sum(_uniform_scalar(seed, 0, c, layer) ** 2 for c in range(3)))
    want = [[1.5 + eps * _uniform_scalar(seed, 0, 0, layer) / n0, -2.0 - eps * _uniform_scalar(seed, 0, 1, layer) / n0,
             0.0], [0.0, 0.0, 0.0]]
    assert torch.allclose(got, torch.tensor(want, dtype=torch.float64), rtol=1e-15, atol=0)
    # layers and seeds give other uniforms
    assert not torch.equal(u, R.uniforms(seed, 2, 3, layer + 1)) and not torch.equal(u, R.uniforms(seed + 1, 2, 3, layer))


def test_info_nce_restatement_by_hand():
    """Two distinct ids with orthogonal unit rows in both views, tau = 1: each row's logits are (1, 0), so
    InfoNCE = log(e + 1) - 1; a repeated id leaves the loss unchanged."""
    a = torch.tensor([[2.0, 0.0], [0.0, 3.0]], dtype=torch.float64)
    want = math.log(math.e + 1) - 1
    assert float(R.info_nce(a, a, 1.0)) == pytest.approx(want, rel=1e-12)
    Fr = torch.cat([a, a])                                              # 2 users, 2 items with the same rows
    got = R.cl_loss(Fr, Fr, 2, [0, 1, 0, 1], [1, 0, 1, 1], 1.0, 0.5)
    assert float(got) == pytest.approx(0.5 * 2 * want, rel=1e-12)
    assert R.first_occurrences([5, 3, 5, 9, 3]).tolist() == [1, 0, 3]


def test_product_never_imports_the_restatement():
    pkg_dir = os.path.dirname(pkg.__file__)
    for f in os.listdir(pkg_dir):
        if f.endswith(".py"):
            assert "_xsimgcl_ref" not in open(os.path.join(pkg_dir, f)).read(), f
