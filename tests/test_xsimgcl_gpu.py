"""XSimGCL on the GPU against the float64 restatement (tests/_xsimgcl_ref.py): the noise kernel, forward rows and
all_*_emb, the cosine InfoNCE kernel, table gradients of BPR / SoftmaxLoss + cl_loss, the reductions to LightGCN,
GraphedStep + Adam against the eager loop, hard negatives, Experiment, state_dict and a short training run."""
import copy
import ctypes
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import _lib, laplacian, synth
from tests import _hneg_ref as H
from tests import _rank_ref
from tests import _softmax_ref as S
from tests import _xsimgcl_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
N_USER, N_ITEM = 700, 500
GRAPH_STEP = 0x9E3779B97F4A7C15 & (2 ** 62 - 1)          # GraphedStep's per-replay seed_dev increment
FIELDS = ("year", "u_id", "age", "sex", "month", "day", "dow", "pos_item")


@functools.lru_cache(maxsize=None)
def _graph(seed=3):
    u, i, r = synth.powerlaw_bipartite(N_USER, N_ITEM, 20000, seed=seed)
    return u, i, laplacian.laplacian_coo(u, i, r, N_USER, N_ITEM)


def _model(emb, K, seed=0, **kw):
    L = _graph()[2]
    torch.manual_seed(seed)
    return pkg.XSimGCL(emb, K, [L, L], synth.num_dict_for(N_USER, N_ITEM), **kw).to(DEV), L


def _batch(B, seed=4):
    """A batch whose users and items repeat."""
    b = {k: torch.from_numpy(v) for k, v in synth.random_batch(N_USER, N_ITEM, B, seed=seed).items()}
    b["u_id"][:6] = torch.tensor([0, 1, 0, 1, 2, 1])
    b["pos_item"][:4] = torch.tensor([7, 7, 9, 9])
    b["neg_item"][:4] = torch.tensor([9, 7, 8, 8])
    return b


def _call(m, b, neg, node_flag=True):
    d = {k: v.to(DEV) for k, v in b.items()}
    return m(d["year"], d["u_id"], d["age"], d["sex"], d["month"], d["day"], d["dow"], d["pos_item"], neg, node_flag)


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp(min=1e-30))


def _key(m):
    st = m._last
    return (st.seed + (int(st.seed_dev) if st.seed_dev is not None else 0)) % (1 << 64)


def _ref_layers(m, L, uw=None, iw=None, noisy=True):
    """float64 E_0..E_K of m's last forward, signs from the device's own layers."""
    uw = m.user_embedding.weight if uw is None else uw
    iw = m.item_embedding.weight if iw is None else iw
    E0 = torch.cat([uw.double().cpu(), iw.double().cpu()])
    signs = [e.cpu() for e in m._last.E[1:]]
    return R.layers(L, E0, m.n_layer, m.eps if noisy else 0.0, _key(m), signs)


@pytest.mark.parametrize("d", [4, 64, 65, 128])
def test_perturb_rows_equals_the_host_stream(d):
    lib = _lib.load()
    N, eps, seed, layer = 3000, 0.2, 0x0123_4567_89AB_CDEF, 3
    g = torch.Generator().manual_seed(d)
    E = torch.randn(N, d, generator=g)
    E[5] = 0.0                                                          # an all-zero row stays zero
    E[7, : d // 2] = 0.0
    Ed = E.to(DEV)
    seed_dev = torch.tensor([12345], dtype=torch.int64, device=DEV)
    _lib.check(lib.ngcf_perturb_rows(Ed.data_ptr(), N, d, d, eps, seed, seed_dev.data_ptr(), layer,
                                     _lib.current_stream()), "perturb_rows")
    key = (seed + 12345) % (1 << 64)
    want = E.double() + R.noise(E, key, layer, eps)
    got = Ed.double().cpu()
    assert torch.equal(got[5], torch.zeros(d, dtype=torch.float64))
    assert torch.equal(got[7, : d // 2], torch.zeros(d // 2, dtype=torch.float64))
    err = float(((got - want).abs() / want.abs().clamp(min=1e-30))[E != 0].max())
    assert err <= 1e-6, err
    # the uniforms themselves: on a row of ones the added vector is eps * u / |u|, and u / |u| is scale-free
    ones = torch.ones(4, d, device=DEV)
    _lib.check(lib.ngcf_perturb_rows(ones.data_ptr(), 4, d, d, 1.0, seed, None, layer, _lib.current_stream()), "perturb")
    u = R.uniforms(seed, 4, d, layer)
    assert torch.allclose((ones.double().cpu() - 1), u / u.norm(dim=1, keepdim=True), rtol=2e-6, atol=2e-7)
    # a different layer or key draws other noise
    again = torch.ones(4, d, device=DEV)
    _lib.check(lib.ngcf_perturb_rows(again.data_ptr(), 4, d, d, 1.0, seed, None, layer + 1, _lib.current_stream()), "p")
    assert not torch.equal(again, ones)


@pytest.mark.parametrize("cl", ["first", "last"])
@pytest.mark.parametrize("d", [4, 64, 65, 128])
@pytest.mark.parametrize("K", [1, 2, 3, 4])
def test_forward_rows_equal_the_restatement(K, d, cl):
    m, L = _model(d, K, cl_layer=1 if cl == "first" else K)
    b = _batch(203)
    worst = 0.0
    for node_flag in (True, False):
        torch.manual_seed(5)
        with torch.no_grad():
            u, pp, n = _call(m, b, b["neg_item"].to(DEV), node_flag)
        assert (m.cl_loss is not None) == node_flag
        E = _ref_layers(m, L, noisy=node_flag)
        Fr = R.final_rows(E)
        ru, rp, rn = Fr[b["u_id"]], Fr[N_USER + b["pos_item"]], Fr[N_USER + b["neg_item"]]
        errs = [_rel(u, ru), _rel(pp, rp), _rel(n, rn), _rel(m.all_users_emb, Fr[:N_USER]),
                _rel(m.all_items_emb, Fr[N_USER:])]
        if not node_flag:                                               # the clean mean(E_1 .. E_K), no noise at all
            clean = R.final_rows(R.layers(L, E[0], K))
            errs.append(_rel(m.all_users_emb, clean[:N_USER]))
        worst = max(worst, *errs)
    print(f"K={K} d={d} cl={cl}: worst max-relative error {worst:.2e}")
    assert worst <= 1e-5


def _infonce(x1, x2, ids, tau, grad=True):
    lib = _lib.load()
    B, D = x1.shape
    ws_bytes = ctypes.c_size_t()
    _lib.check(lib.ngcf_infonce_workspace(B, D, ctypes.byref(ws_bytes)), "ws")
    ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=DEV)
    loss = torch.empty((), device=DEV)
    g1, g2 = (torch.empty_like(x1), torch.empty_like(x2)) if grad else (None, None)
    _lib.check(lib.ngcf_infonce(x1.data_ptr(), x2.data_ptr(), B, D, ids.data_ptr(), tau, loss.data_ptr(), _lib.ptr(g1),
                                _lib.ptr(g2), ws.data_ptr(), ws_bytes.value, _lib.current_stream()), "infonce")
    return loss, g1, g2


@pytest.mark.parametrize("case", ["repeats", "all_duplicate", "all_distinct", "large_logits", "wide"])
def test_infonce_equals_selfrec_with_unique(case):
    B, D, tau = {"repeats": (1024, 64, 0.2), "all_duplicate": (300, 65, 0.2), "all_distinct": (2048, 64, 0.2),
                 "large_logits": (512, 128, 0.02), "wide": (203, 257, 0.5)}[case]
    g = torch.Generator().manual_seed(B + D)
    if case == "all_duplicate":
        ids = torch.full((B,), 7, dtype=torch.int64)
    elif case == "all_distinct":
        ids = torch.randperm(10 * B, generator=g)[:B]
    else:
        ids = torch.randint(0, B // 3, (B,), generator=g)
    x1 = torch.randn(B, D, generator=g, dtype=torch.float64)
    # large logits: cos / tau up to 50, with views far enough apart that the loss does not vanish
    x2 = x1 + (3.0 if case == "large_logits" else 0.5) * torch.randn(B, D, generator=g, dtype=torch.float64)
    dup = torch.ones(B, dtype=torch.bool)                              # duplicate ids carry the same rows, as gathered
    dup[R.first_occurrences(ids)] = False                               # rows of one table do
    first = {}
    for i, v in enumerate(ids.tolist()):
        first.setdefault(v, i)
    src = torch.tensor([first[v] for v in ids.tolist()])
    x1, x2 = x1[src], x2[src]
    a, b = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)
    fo = R.first_occurrences(ids)
    ref = R.info_nce(a[fo], b[fo], tau)
    ga, gb = torch.autograd.grad(ref, [a, b])
    loss, g1, g2 = _infonce(x1.float().to(DEV), x2.float().to(DEV), ids.to(DEV), tau)
    e_loss = abs(float(loss) - float(ref)) / max(abs(float(ref)), 1e-30)
    e1, e2 = _rel(g1, ga), _rel(g2, gb)
    print(f"{case}: loss {float(loss):.6f} vs {float(ref):.6f}; errors {e_loss:.1e} {e1:.1e} {e2:.1e}")
    assert e_loss <= 1e-5 or (case == "all_duplicate" and abs(float(loss)) <= 1e-6)
    if case != "all_duplicate":
        assert e1 <= 1e-4 and e2 <= 1e-4
    else:
        assert float(g1.abs().max()) <= 1e-6 and float(g2.abs().max()) <= 1e-6
    dd = dup.to(DEV)
    assert float(g1[dd].abs().sum()) == 0.0 and float(g2[dd].abs().sum()) == 0.0     # later occurrences take no part
    again = _infonce(x1.float().to(DEV), x2.float().to(DEV), ids.to(DEV), tau)
    assert torch.equal(loss, again[0]) and torch.equal(g1, again[1]) and torch.equal(g2, again[2])
    fwd_only = _infonce(x1.float().to(DEV), x2.float().to(DEV), ids.to(DEV), tau, grad=False)
    assert torch.equal(loss, fwd_only[0])


def _bpr64(u, p, n, wd, bs):
    x = (u * p).sum(1).abs() - (u * n).sum(1).abs()
    reg = (u * u).sum() + (p * p).sum() + (n * n).sum()
    return (-F.logsigmoid(x).sum() + wd * reg) / bs


@pytest.mark.parametrize("crit", ["bpr", "softmax"])
@pytest.mark.parametrize("emb,K,cl", [(64, 3, 1), (64, 3, 3), (65, 2, 2), (64, 1, 1)])
def test_table_gradients_equal_float64_autograd(emb, K, cl, crit):
    B = 256
    m, L = _model(emb, K, cl_layer=cl, cl_weight=0.5)
    b = _batch(B)
    d = {k: v.to(DEV) for k, v in b.items()}
    torch.manual_seed(21)
    u, p, n = _call(m, b, d["neg_item"])
    rec = pkg.BPR(0.025, B)(u, p, n) if crit == "bpr" else \
        pkg.SoftmaxLoss(0.025, B, 0.2)(u, p, n, d["pos_item"], d["neg_item"])
    loss = rec + m.cl_loss
    loss.backward()
    uw = m.user_embedding.weight.detach().double().cpu().requires_grad_(True)
    iw = m.item_embedding.weight.detach().double().cpu().requires_grad_(True)
    E = _ref_layers(m, L, uw, iw)
    Fr = R.final_rows(E)
    ru, rp, rn = Fr[b["u_id"]], Fr[N_USER + b["pos_item"]], Fr[N_USER + b["neg_item"]]
    ref = _bpr64(ru, rp, rn, 0.025, B) if crit == "bpr" else \
        S.loss(ru, rp, rn, temperature=0.2, weight_decay=0.025, batch_size=B, pos_ids=b["pos_item"], neg_ids=b["neg_item"])
    ref_cl = R.cl_loss(Fr, E[cl], N_USER, b["u_id"], b["pos_item"], 0.2, 0.5)
    gU, gI = torch.autograd.grad(ref + ref_cl, [uw, iw])
    eu, ei = _rel(m.user_embedding.weight.grad, gU), _rel(m.item_embedding.weight.grad, gI)
    print(f"{crit} {emb}x{K} cl={cl}: loss {float(loss):.6f} vs {float(ref + ref_cl):.6f} (cl {float(m.cl_loss):.6f} "
          f"vs {float(ref_cl):.6f}), grad errors {eu:.2e} {ei:.2e}")
    assert abs(float(m.cl_loss) - float(ref_cl)) <= 1e-5 * abs(float(ref_cl))
    assert abs(float(loss) - float(ref + ref_cl)) <= 1e-5 * abs(float(ref + ref_cl))
    assert eu <= 1e-4 and ei <= 1e-4


def test_cl_weight_zero_and_eps_zero_reduce_to_the_expected_models():
    b = _batch(128)
    d = {k: v.to(DEV) for k, v in b.items()}
    # cl_weight = 0: the noise only, no contrastive launches, cl_loss None
    m, L = _model(64, 3, cl_weight=0.0)
    n0 = _lib.load().ngcf_launch_count()
    torch.manual_seed(3)
    u, p, n = _call(m, b, d["neg_item"])
    launches_plain = _lib.load().ngcf_launch_count() - n0
    assert m.cl_loss is None
    Fr = R.final_rows(_ref_layers(m, L))
    assert _rel(u, Fr[b["u_id"]]) <= 1e-5
    m2, _ = _model(64, 3, cl_weight=0.2)
    n0 = _lib.load().ngcf_launch_count()
    torch.manual_seed(3)
    u2, _, _ = _call(m2, b, d["neg_item"])
    assert torch.equal(u, u2)                                           # same key, same noise
    assert _lib.load().ngcf_launch_count() - n0 > launches_plain        # the contrastive term's launches
    # eps = 0: no key is drawn, and the rows are the clean mean(E_1 .. E_K); gradients are LightGCN's chain without E_0
    m3, _ = _model(64, 3, eps=0.0, cl_weight=0.0)
    state = torch.get_rng_state()
    u3, p3, n3 = _call(m3, b, d["neg_item"])
    assert torch.equal(state, torch.get_rng_state()) and m3._last.seed == 0
    clean = R.final_rows(R.layers(L, torch.cat([m3.user_embedding.weight.double().cpu(),
                                                m3.item_embedding.weight.double().cpu()]), 3))
    assert _rel(u3, clean[b["u_id"]]) <= 1e-5
    # eval forward of a trained-mode model equals the LightGCN layers' mean without E_0
    lg = pkg.LightGCN(64, 3, [L, L], synth.num_dict_for(N_USER, N_ITEM)).to(DEV)
    lg.load_state_dict(m3.state_dict())
    with torch.no_grad():
        _call(lg, b, d["neg_item"], False)
        _call(m3, b, d["neg_item"], False)
    E = lg._last.E
    assert torch.allclose(m3.all_users_emb, ((E[1] + E[2] + E[3]) / 3)[:N_USER], rtol=1e-6, atol=1e-7)


def _distinct_batch(B, seed):
    rng = np.random.default_rng(seed)
    b = {k: torch.from_numpy(v) for k, v in synth.random_batch(N_USER, N_ITEM, B, seed=seed).items()}
    b["u_id"] = torch.from_numpy(rng.permutation(N_USER)[:B])
    items = rng.permutation(N_ITEM)[:2 * B]
    b["pos_item"], b["neg_item"] = torch.from_numpy(items[:B]), torch.from_numpy(items[B:])
    return b


@functools.lru_cache(maxsize=None)
def _gowalla():
    n_user, n_item, n_inter, _, _ = synth.SHAPES["gowalla"]
    u, i, r = synth.powerlaw_bipartite(n_user, n_item, n_inter, alpha=0.8, seed=0)
    return n_user, n_item, laplacian.laplacian_coo(u, i, r, n_user, n_item)


@pytest.mark.parametrize("case", ["distinct", "repeats", "gowalla_2048"])
def test_graphed_step_with_adam_equals_the_eager_loop(case):
    """The captured step (noise, both InfoNCE calls, the view-2 gradient at layer cl_layer) against the eager loop:
    on batches of distinct ids, on batches that repeat users and items (first-occurrence masks under capture, zero
    view-2 rows on shared slots), and at XSimGCL's usual batch of 2048 on a graph of Gowalla's size."""
    if case == "gowalla_2048":
        n_user, n_item, L = _gowalla()
        B, steps = 2048, 2
        torch.manual_seed(0)
        m = pkg.XSimGCL(64, 3, [L, L], synth.num_dict_for(n_user, n_item)).to(DEV)
        batches = []
        for s in range(steps):
            bt = {k: torch.from_numpy(v) for k, v in synth.random_batch(n_user, n_item, B, seed=40 + s).items()}
            bt["u_id"][:6] = torch.tensor([0, 1, 0, 1, 2, 1])
            bt["pos_item"][:4] = torch.tensor([7, 7, 9, 9])
            batches.append(bt)
    else:
        B, steps = 128, 4
        m, L = _model(64, 3)
        batches = [(_distinct_batch if case == "distinct" else _batch)(B, 40 + s) for s in range(steps)]
    ref = copy.deepcopy(m)
    torch.manual_seed(9)
    step = pkg.GraphedStep(m, pkg.BPR(1e-3, B), B, optimizer=pkg.Adam(m.parameters(), lr=1e-2))
    losses, layer1 = [], []
    for bt in batches:
        losses.append(float(step(bt)))
        layer1.append(next(iter(step.graphs.values()))[3].E[1].clone())
    assert not torch.equal(layer1[0] - layer1[1], torch.zeros_like(layer1[0]))
    torch.manual_seed(9)
    torch.randint(0, 2 ** 62, (1,))                                    # the warm-up forward's draw
    gen_state = torch.get_rng_state()
    ref._seed_dev = torch.zeros(1, dtype=torch.int64, device=DEV)
    opt = torch.optim.Adam(ref.parameters(), lr=1e-2)
    crit = pkg.BPR(1e-3, B)
    for r, bt in enumerate(batches):
        torch.set_rng_state(gen_state)
        ref._seed_dev.fill_((r + 1) * GRAPH_STEP)
        opt.zero_grad()
        u, p, n = _call(ref, bt, bt["neg_item"].to(DEV))
        if r == 0:                                                     # the replay's noise, reproduced eagerly
            assert _rel(ref._last.E[1], layer1[0]) <= 1e-6
        loss = crit(u, p, n) + ref.cl_loss
        loss.backward()
        opt.step()
        assert abs(float(loss) - losses[r]) <= 1e-5 * abs(losses[r]), (r, float(loss), losses[r])
    for (k, a), (_, b) in zip(m.named_parameters(), ref.named_parameters()):
        err = _rel(a, b)
        assert err <= 1e-4, (k, err)


def _train_rows():
    u, i, _ = _graph()
    return pkg.Interactions.from_pairs(u, i, N_ITEM, rows=torch.arange(N_USER))


def test_hard_negatives_pick_on_the_perturbed_mean():
    B, M = 203, 32
    m, L = _model(64, 3)
    train = _train_rows()
    rows = _rank_ref.rows_of(train)
    b = _batch(B)
    hn = pkg.HardNegatives(train, M, debug=True)
    torch.manual_seed(3)
    with torch.no_grad():
        u, p, n = _call(m, b, hn)
    assert m._last.seed != 0
    cand = H.candidates(m._last.seed, b["u_id"].numpy(), rows, N_ITEM, M)
    assert np.array_equal(hn.cand.cpu().numpy(), cand)
    U, I = m.all_users_emb.double().cpu(), m.all_items_emb.double().cpu()     # this step's perturbed mean(E_1..E_K)
    uid, cnd = b["u_id"], hn.cand.cpu()
    want = torch.einsum("bd,bmd->bm", U[uid], I[cnd])
    scale = U[uid].norm(dim=1)[:, None] * I[cnd].norm(dim=2)
    assert ((hn.score.cpu().double() - want).abs() <= 1e-5 * scale).all()
    assert torch.equal(hn.chosen, hn.cand[torch.arange(B, device=DEV), hn.score.abs().argmax(1)])
    assert torch.equal(n, m.all_items_emb[hn.chosen]) and torch.equal(u, m.all_users_emb[uid.to(DEV)])


def test_experiment_train_and_eval_run():
    B, G = 64, 25
    m, _ = _model(64, 2)
    train_dl = []
    for s in range(3):
        b = _batch(B, seed=50 + s)
        train_dl.append(tuple(b[k] for k in FIELDS + ("neg_item",)))
    test_dl = []
    for s in range(2):
        b = {k: torch.from_numpy(v) for k, v in synth.random_batch(N_USER, N_ITEM, G, seed=60 + s).items()}
        b["u_id"][:] = b["u_id"][0]
        test_dl.append(tuple(b[k] for k in FIELDS[:7]) + (torch.ones(G), b["pos_item"]))
    exp = pkg.Experiment(m, torch.optim.Adam(m.parameters(), lr=1e-3), pkg.BPR(0.025, B), pkg.BPR(0.025, G),
                         train_dl, test_dl, epochs=1, ks=5, device=torch.device(DEV), verbose=False)
    hist = exp.train()
    assert len(hist) == 1 and all(np.isfinite(v) for v in hist[0])


def test_state_dict_round_trip_with_lightgcn():
    m, L = _model(65, 2)
    lg = pkg.LightGCN(65, 2, [L, L], synth.num_dict_for(N_USER, N_ITEM)).to(DEV)
    lg.load_state_dict(m.state_dict())
    m2, _ = _model(65, 2, seed=1)
    m2.load_state_dict(lg.state_dict())
    b = _batch(128)
    outs = []
    for mod in (m, m2):
        torch.manual_seed(8)
        with torch.no_grad():
            outs.append(_call(mod, b, b["neg_item"].to(DEV)))
    for a, c in zip(*outs):
        assert torch.equal(a, c)


def test_short_captured_training_run_raises_recall():
    n_user, n_item, B = 600, 400, 256
    u, i, r = synth.powerlaw_bipartite(n_user, n_item, 12000, seed=7)
    rng = np.random.default_rng(7)
    test_mask = rng.random(u.size) < 0.2
    tu, ti = u[~test_mask], i[~test_mask]
    L = laplacian.laplacian_coo(tu, ti, r[~test_mask], n_user, n_item)
    train = pkg.Interactions.from_pairs(tu, ti, n_item, rows=torch.arange(n_user))
    test = pkg.Interactions.from_pairs(u[test_mask], i[test_mask], n_item, rows=torch.arange(n_user))
    torch.manual_seed(0)
    m = pkg.XSimGCL(64, 3, [L, L], synth.num_dict_for(n_user, n_item)).to(DEV)

    def recall():
        ctx = synth.random_batch(n_user, n_item, 64, seed=1)
        with torch.no_grad():
            m(*(torch.from_numpy(ctx[k]).to(DEV) for k in FIELDS), torch.empty(0), False)
            return pkg.full_rank_eval(m.all_users_emb, m.all_items_emb, train=train.to(DEV),
                                      test=test.to(DEV))["recall@20"]

    r0 = recall()
    step = pkg.GraphedStep(m, pkg.SoftmaxLoss(1e-4, B, 0.2), B, optimizer=pkg.Adam(m.parameters(), lr=5e-3))
    for s in range(150):
        b = {k: torch.from_numpy(v) for k, v in synth.random_batch(n_user, n_item, B, seed=100 + s).items()}
        j = rng.integers(0, tu.size, B)
        b["u_id"], b["pos_item"] = torch.from_numpy(tu[j]), torch.from_numpy(ti[j])
        loss = step(b)
    assert torch.isfinite(loss)
    r1 = recall()
    print(f"recall@20: {r0:.4f} -> {r1:.4f}")
    assert r1 > r0          # (the untrained mean(E_1 .. E_K) already ranks well: E_0's random rows are not in it)
