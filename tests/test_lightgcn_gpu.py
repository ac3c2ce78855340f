"""LightGCN on the GPU against the float64 restatement (tests/_lightgcn_ref.py): forward rows and all_*_emb, table
gradients under BPR and SoftmaxLoss, NGCF's feature mix, GraphedStep + Adam against the eager loop, Experiment, hard
negatives on the mean readout, full-ranking evaluation, state_dict, a short training run, and the refusals."""
import copy
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import laplacian, plgraph, synth
from tests import _hneg_ref as H
from tests import _lightgcn_ref as R
from tests import _rank_ref
from tests import _softmax_ref as S

pytestmark = pytest.mark.gpu
DEV = "cuda"
N_USER, N_ITEM = 700, 500
GRAPH_STEP = 0x9E3779B97F4A7C15 & (2 ** 62 - 1)          # GraphedStep's per-replay seed_dev increment
FIELDS = ("year", "u_id", "age", "sex", "month", "day", "dow", "pos_item")


@functools.lru_cache(maxsize=None)
def _graph(fmt="coo", seed=3):
    u, i, r = synth.powerlaw_bipartite(N_USER, N_ITEM, 20000, seed=seed)
    if fmt == "coo":
        return u, i, laplacian.laplacian_coo(u, i, r, N_USER, N_ITEM)
    return u, i, plgraph.laplacian_csr_device(u, i, r, N_USER, N_ITEM, DEV)


def _model(emb, K, p=0.3, fmt="coo", emb_ratio=0.0, seed=0):
    L = _graph(fmt)[2]
    torch.manual_seed(seed)
    return pkg.LightGCN(emb, K, [L, L], synth.num_dict_for(N_USER, N_ITEM), node_dropout=p,
                        emb_ratio=emb_ratio).to(DEV), L


def _batch(B, seed=4):
    """A batch whose users and items repeat (within and across the positive and negative sets)."""
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


def _keep(m, L):
    st = m._last
    if st.drop_p == 0:
        return None
    key = st.seed + (int(st.seed_dev) if st.seed_dev is not None else 0)
    return R.keep_lists(L, key, st.drop_p, m.n_layer)


@pytest.mark.parametrize("fmt", ["coo", "csr"])
@pytest.mark.parametrize("p", [0.0, 0.3])
@pytest.mark.parametrize("d", [4, 64, 65, 128])
@pytest.mark.parametrize("K", [1, 2, 3, 4])
def test_forward_rows_equal_the_restatement(K, d, p, fmt):
    m, L = _model(d, K, p, fmt)
    b = _batch(203)
    worst = 0.0
    for training, node_flag in ((True, True), (False, True), (False, False)):
        m.train(training)
        torch.manual_seed(5)
        with torch.no_grad():
            u, pp, n = _call(m, b, b["neg_item"].to(DEV), node_flag)
        assert m._last.drop_p == (p if node_flag else 0.0)
        Fr = R.final_rows(L, m.user_embedding.weight, m.item_embedding.weight, K, _keep(m, L))
        ru, rp, rn = R.batch_rows(Fr, N_USER, b["u_id"], b["pos_item"], b["neg_item"])
        assert u.shape == pp.shape == n.shape == (203, d)
        errs = [_rel(u, ru), _rel(pp, rp), _rel(n, rn), _rel(m.all_users_emb, Fr[:N_USER]),
                _rel(m.all_items_emb, Fr[N_USER:])]
        worst = max(worst, *errs)
    print(f"K={K} d={d} p={p} {fmt}: worst max-relative error {worst:.2e}")
    assert worst <= 1e-5


def _bpr64(u, p, n, wd, bs):
    x = (u * p).sum(1).abs() - (u * n).sum(1).abs()
    reg = (u * u).sum() + (p * p).sum() + (n * n).sum()
    return (-F.logsigmoid(x).sum() + wd * reg) / bs


@pytest.mark.parametrize("crit,with_neg", [("bpr", True), ("softmax", True), ("softmax", False)])
@pytest.mark.parametrize("emb,K", [(64, 3), (65, 2)])
def test_table_gradients_equal_float64_autograd(emb, K, crit, with_neg):
    B = 256
    m, L = _model(emb, K, 0.3)
    m.train()
    b = _batch(B)
    d = {k: v.to(DEV) for k, v in b.items()}
    torch.manual_seed(21)
    u, p, n = _call(m, b, d["neg_item"] if with_neg else torch.empty(0))
    if crit == "bpr":
        loss = pkg.BPR(0.025, B)(u, p, n)
    else:
        loss = pkg.SoftmaxLoss(0.025, B, 0.2)(u, p, n, d["pos_item"], d["neg_item"] if with_neg else None)
    loss.backward()
    uw = m.user_embedding.weight.detach().double().cpu().requires_grad_(True)
    iw = m.item_embedding.weight.detach().double().cpu().requires_grad_(True)
    Fr = R.final_rows(L, uw, iw, K, _keep(m, L))
    ru, rp, rn = R.batch_rows(Fr, N_USER, b["u_id"], b["pos_item"], b["neg_item"] if with_neg else None)
    if crit == "bpr":
        ref = _bpr64(ru, rp, rn, 0.025, B)
    else:
        ref = S.loss(ru, rp, rn if with_neg else torch.empty(0), temperature=0.2, weight_decay=0.025, batch_size=B,
                     pos_ids=b["pos_item"], neg_ids=b["neg_item"] if with_neg else None)
    gU, gI = torch.autograd.grad(ref, [uw, iw])
    eu, ei = _rel(m.user_embedding.weight.grad, gU), _rel(m.item_embedding.weight.grad, gI)
    print(f"{crit} neg={with_neg} {emb}x{K}: loss {float(loss):.6f} vs {float(ref):.6f}, grad errors {eu:.2e} {ei:.2e}")
    assert abs(float(loss) - float(ref)) <= 1e-5 * abs(float(ref))
    assert eu <= 1e-4 and ei <= 1e-4


def test_feature_mix_equals_ngcf():
    """emb_ratio = 1 on a Seoul-shaped graph: the user rows LightGCN mixes are the rows NGCF's feature mix writes."""
    n_user, n_item, emb, B = 5840, 100, 65, 512
    u, i, r = synth.powerlaw_bipartite(n_user, n_item, 40000, seed=11)
    L = laplacian.laplacian_coo(u, i, r, n_user, n_item)
    nd = synth.num_dict_for(n_user, n_item)
    torch.manual_seed(0)
    lg = pkg.LightGCN(emb, 2, [L], nd, emb_ratio=1.0).to(DEV)
    ng = pkg.NGCF(emb, [emb, emb], 0.0, [0.0, 0.0], 1.0, [L], nd, B, torch.device(DEV)).to(DEV)
    ng.load_state_dict({**ng.state_dict(), **lg.state_dict()})
    b = {k: torch.from_numpy(v) for k, v in synth.random_batch(n_user, n_item, B, seed=12).items()}
    with torch.no_grad():
        _call(lg, b, torch.empty(0), False)
        _call(ng, b, torch.empty(0), False)
    users = b["u_id"].unique().to(DEV)
    assert torch.equal(lg.user_embedding.weight[users], ng.user_embedding.weight[users])
    assert torch.equal(lg.user_embedding.weight, ng.user_embedding.weight)
    # and the mixed rows are the concat of the five feature rows (emb_ratio = 1)
    cat = torch.cat([lg.age_emb.weight[b["age"].to(DEV)], lg.sex_emb.weight[b["sex"].to(DEV)],
                     lg.month_emb.weight[b["month"].to(DEV)], lg.day_emb.weight[b["day"].to(DEV)],
                     lg.dow_emb.weight[b["dow"].to(DEV)]], 1)
    last = {int(x): j for j, x in enumerate(b["u_id"])}                # the last occurrence of a user wins
    j = torch.tensor(list(last.values()), device=DEV)
    assert torch.equal(lg.user_embedding.weight[torch.tensor(list(last.keys()), device=DEV)], cat[j])


def _distinct_batch(B, seed):
    """Distinct users and distinct items over the positive and negative sets: the row-gradient sums then add one row
    each, so two runs give the same gradient bits."""
    rng = np.random.default_rng(seed)
    b = {k: torch.from_numpy(v) for k, v in synth.random_batch(N_USER, N_ITEM, B, seed=seed).items()}
    b["u_id"] = torch.from_numpy(rng.permutation(N_USER)[:B])
    items = rng.permutation(N_ITEM)[:2 * B]
    b["pos_item"], b["neg_item"] = torch.from_numpy(items[:B]), torch.from_numpy(items[B:])
    return b


def test_graphed_step_with_adam_equals_the_eager_loop():
    B, steps = 128, 4
    m, L = _model(64, 3, 0.3)
    m.train()
    ref = copy.deepcopy(m)
    batches = [_distinct_batch(B, 40 + s) for s in range(steps)]
    torch.manual_seed(9)
    step = pkg.GraphedStep(m, pkg.BPR(1e-3, B), B, optimizer=pkg.Adam(m.parameters(), lr=1e-2))
    losses = [float(step(bt)) for bt in batches]
    # eager: the same per-step keys (the capture's seed + (r+1) * GRAPH_STEP) through the same device counter
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
        loss = crit(u, p, n)
        loss.backward()
        opt.step()
        assert abs(float(loss) - losses[r]) <= 1e-6 * abs(losses[r]), r
    for (k, a), (_, b) in zip(m.named_parameters(), ref.named_parameters()):
        err = _rel(a, b)
        assert err <= 1e-5, (k, err)
    assert step.launches_per_step > 0


def test_experiment_train_and_eval_run():
    B, G = 64, 25
    m, _ = _model(64, 2, 0.1)
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


def _train_rows():
    u, i, _ = _graph()
    keep = u > 1
    tu = np.concatenate([u[keep], np.ones(N_ITEM - 1, dtype=u.dtype)])           # user 0: no items; user 1: all but 123
    ti = np.concatenate([i[keep], np.delete(np.arange(N_ITEM), 123)])
    return pkg.Interactions.from_pairs(tu, ti, N_ITEM, rows=torch.arange(N_USER))


@pytest.mark.parametrize("signed", [False, True])
def test_hard_negatives_on_the_mean_readout(signed):
    B, M = 203, 32
    m, L = _model(64, 3, 0.3)
    train = _train_rows()
    rows = _rank_ref.rows_of(train)
    b = _batch(B)
    hn = pkg.HardNegatives(train, M, signed=signed, debug=True)
    m.eval()
    torch.manual_seed(3)
    with torch.no_grad():
        u, p, n = _call(m, b, hn)
    key = m._last.seed
    cand = H.candidates(key, b["u_id"].numpy(), rows, N_ITEM, M)
    assert np.array_equal(hn.cand.cpu().numpy(), cand)
    assert np.all(cand[b["u_id"].numpy() == 1] == 123)
    U, I = m.all_users_emb.double().cpu(), m.all_items_emb.double().cpu()
    uid, cnd = b["u_id"], hn.cand.cpu()
    want = torch.einsum("bd,bmd->bm", U[uid], I[cnd])
    scale = U[uid].norm(dim=1)[:, None] * I[cnd].norm(dim=2)
    assert ((hn.score.cpu().double() - want).abs() <= 1e-5 * scale).all()
    key_of = hn.score if signed else hn.score.abs()
    assert torch.equal(hn.chosen, hn.cand[torch.arange(B, device=DEV), key_of.argmax(1)])
    assert torch.equal(n, m.all_items_emb[hn.chosen]) and torch.equal(u, m.all_users_emb[uid.to(DEV)])
    # training mode, node dropout on: the DNS step and the plain step given its picks give the same rows, bit for bit
    m.train()
    outs = []
    for neg in (hn, "picks"):
        torch.manual_seed(17)
        with torch.no_grad():
            outs.append([t.clone() for t in _call(m, b, hn if neg is hn else picks)])
        if neg is hn:
            picks = hn.chosen.clone()
            assert m._last.drop_p > 0
    for a, c in zip(*outs):
        assert torch.equal(a, c)


def test_graphed_step_redraws_hard_negatives_every_replay():
    B = 256
    m, _ = _model(64, 3, 0.3)
    m.train()
    train = _train_rows()
    hn = pkg.HardNegatives(train, 16, debug=True)
    step = pkg.GraphedStep(m, pkg.BPR(0.025, B), B, negatives=hn, optimizer=pkg.Adam(m.parameters(), lr=1e-3))
    b = _batch(B)
    batch = {k: v for k, v in b.items() if k != "neg_item"}
    rows = _rank_ref.rows_of(train)
    picks = []
    for _ in range(2):
        assert np.isfinite(float(step(batch)))
        st = next(iter(step.graphs.values()))[3]
        key = (st.seed + int(step.seed_dev) - GRAPH_STEP) % (1 << 64)
        assert np.array_equal(hn.cand.cpu().numpy(), H.candidates(key, b["u_id"].numpy(), rows, N_ITEM, 16))
        assert torch.equal(hn.chosen, hn.cand[torch.arange(B, device=DEV), hn.score.abs().argmax(1)])
        picks.append(hn.cand.clone())
    assert not torch.equal(picks[0], picks[1])


def test_full_rank_eval_on_the_model_rows():
    m, _ = _model(64, 3, 0.0)
    u, i, _ = _graph()
    rng = np.random.default_rng(5)
    held = rng.random(u.size) < 0.2
    train = pkg.Interactions.from_pairs(u[~held], i[~held], N_ITEM, rows=torch.arange(N_USER))
    test = pkg.Interactions.from_pairs(u[held], i[held], N_ITEM, rows=torch.arange(N_USER))
    with torch.no_grad():
        _call(m, _batch(64), torch.empty(0), False)
    out = pkg.full_rank_eval(m.all_users_emb, m.all_items_emb, train=train.to(DEV), test=test.to(DEV), Ks=(10, 20))
    S64 = m.all_users_emb.double().cpu() @ m.all_items_emb.double().cpu().T
    tr = _rank_ref.rows_of(train)
    for r in range(N_USER):
        S64[r, torch.from_numpy(tr[r]).long()] = -float("inf")
    ranked = torch.topk(S64, 20, dim=1).indices.numpy()
    means, n, _ = _rank_ref.metrics(ranked, _rank_ref.rows_of(test), (10, 20))
    assert out["n_users"] == n
    for j, K in enumerate((10, 20)):
        for c, name in enumerate(("recall", "precision", "ndcg", "hit")):
            assert abs(out[f"{name}@{K}"] - means[j, c]) <= 2e-3, (name, K)


@pytest.mark.parametrize("emb_ratio", [0.0, 1.0])
def test_state_dict_round_trip(emb_ratio):
    m, L = _model(65, 2, 0.3, emb_ratio=emb_ratio)
    m2, _ = _model(65, 2, 0.3, emb_ratio=emb_ratio, seed=1)
    assert not torch.equal(m.user_embedding.weight, m2.user_embedding.weight)
    m2.load_state_dict(m.state_dict())
    b = _batch(128)
    outs = []
    for mod in (m, m2):
        torch.manual_seed(8)
        with torch.no_grad():
            outs.append(_call(mod, b, b["neg_item"].to(DEV)))
    for a, c in zip(*outs):
        assert torch.equal(a, c)
    assert torch.equal(m.all_items_emb, m2.all_items_emb)


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
    m = pkg.LightGCN(64, 3, [L, L], synth.num_dict_for(n_user, n_item), node_dropout=0.1).to(DEV)

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
    assert r1 > r0 + 0.02


def test_refusals():
    m, L = _model(64, 2, 0.3)
    b = _batch(64)
    short = pkg.Interactions.from_pairs([0, 3], [1, 2], N_ITEM, rows=torch.arange(N_USER - 1))
    with pytest.raises(ValueError, match="699 rows"):
        _call(m, b, pkg.HardNegatives(short))
    wide = pkg.Interactions.from_pairs([0, 3], [1, 2], N_ITEM + 1, rows=torch.arange(N_USER))
    with pytest.raises(ValueError, match="501 items"):
        _call(m, b, pkg.HardNegatives(wide))
    with pytest.raises(NotImplementedError, match="row-sharded"):
        m.shard()
    other = laplacian.laplacian_coo(np.array([0, 1]), np.array([0, 1]), np.ones(2, np.float32), N_USER - 1, N_ITEM)
    m.lap_list[0] = other                                         # replaced after construction
    with pytest.raises(ValueError, match="n_user \\+ n_item = 1200"):
        _call(m, b, torch.empty(0))
    m.lap_list[0] = L
    with pytest.raises(AttributeError):
        _model(64, 2)[0].all_users_emb                           # no forward yet
    with torch.no_grad():
        _call(m, b, b["neg_item"])
    opt = pkg.Adam(m.parameters(), lr=1e-3)
    _call(m, b, b["neg_item"])[0].sum().backward()
    opt.step()
    with pytest.raises(RuntimeError, match="LightGCN \\(B200\\)"):
        m.all_users_emb                                           # the table changed under the forward's E_0
