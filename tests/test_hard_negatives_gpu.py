"""Dynamic hard-negative sampling on the GPU: the candidates equal the host restatement of the draws, the scores equal
float64 dot products of the forward's own final rows, the pick is the largest |score|, a DNS step is the plain step
with the picks passed as neg_item, and GraphedStep draws fresh candidates on every replay."""
import copy

import numpy as np
import pytest
import torch

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import laplacian, synth
from seoul_tourism_recommendation_ngcf_b200.sharded import RowShards
from tests import _hneg_ref as H
from tests._rank_ref import rows_of

pytestmark = pytest.mark.gpu
DEV = "cuda"
N_USER, N_ITEM = 700, 500
GRAPH_STEP = 0x9E3779B97F4A7C15 & (2 ** 62 - 1)          # GraphedStep's per-replay seed_dev increment


def _setup(emb=64, K=3, B=203, node_p=0.3, mess_p=0.1, seed=3):
    """Model, training Interactions (user 0: no items, user 1: every item but one) and a batch that holds users 0 and
    1 several times."""
    u, i, r = synth.powerlaw_bipartite(N_USER, N_ITEM, 20000, seed=seed)
    L = laplacian.laplacian_coo(u, i, r, N_USER, N_ITEM)
    torch.manual_seed(0)
    m = pkg.NGCF(emb, [emb] * K, node_p, [mess_p] * K, 1.0, [L, L], synth.num_dict_for(N_USER, N_ITEM), B,
                 torch.device(DEV)).to(DEV)
    keep = u > 1
    tu = np.concatenate([u[keep], np.ones(N_ITEM - 1, dtype=u.dtype)])
    ti = np.concatenate([i[keep], np.delete(np.arange(N_ITEM), 123)])
    train = pkg.Interactions.from_pairs(tu, ti, N_ITEM, rows=torch.arange(N_USER))
    b = {k: torch.from_numpy(v) for k, v in synth.random_batch(N_USER, N_ITEM, B, seed=seed + 1).items()}
    b["u_id"][:6] = torch.tensor([0, 1, 0, 1, 2, 1])
    return m, train, b


def _call(m, b, neg, node_flag=True):
    d = {k: v.to(DEV) for k, v in b.items()}
    return m(d["year"], d["u_id"], d["age"], d["sex"], d["month"], d["day"], d["dow"], d["pos_item"], neg, node_flag)


@pytest.mark.parametrize("M,B", [(1, 203), (32, 203), (64, 61)])
def test_candidates_equal_the_restatement(M, B):
    m, train, b = _setup(B=B)
    m.eval()
    rows = rows_of(train)
    hn = pkg.HardNegatives(train, M, debug=True)
    for s, seed_dev in ((1, None), (2, 0), (3, 12345), (4, "carry")):
        torch.manual_seed(s)
        m._seed_dev = None if seed_dev is None else torch.zeros(1, dtype=torch.int64, device=DEV)
        with torch.no_grad():
            if seed_dev == "carry":                              # seed + *seed_dev carries across bit 32: read the
                _call(m, b, hn)                                  # key off a first forward, then set the counter
                key = m._last.seed
                m._seed_dev.fill_((1 << 32) - (key & 0xFFFFFFFF) + 5)
                torch.manual_seed(s)
            elif seed_dev:
                m._seed_dev.fill_(seed_dev)
            _call(m, b, hn)
        key = m._last.seed + (int(m._seed_dev) if m._seed_dev is not None else 0)
        want = H.candidates(key, b["u_id"].numpy(), rows, N_ITEM, M)
        got = hn.cand.cpu().numpy()
        assert np.array_equal(got, want), (s, seed_dev)
        assert np.all(got[b["u_id"].numpy() == 1] == 123)         # the one free item
        assert hn.chosen.shape == (B,) and torch.equal(hn.chosen, hn.cand[torch.arange(B), hn.score.abs().argmax(1)])
    m._seed_dev = None


@pytest.mark.parametrize("M", [1, 32])
def test_scores_and_choice(M):
    m, train, b = _setup(B=203)
    m.eval()
    hn = pkg.HardNegatives(train, M, debug=True)
    with torch.no_grad():
        uu, pp, nn_ = _call(m, b, hn)                            # eval-mode, no_grad forward with node dropout
    U = m.all_users_emb.double().cpu()
    I = m.all_items_emb.double().cpu()
    uid, cand, score, chosen = b["u_id"], hn.cand.cpu(), hn.score.cpu().double(), hn.chosen.cpu()
    want = torch.einsum("bd,bmd->bm", U[uid], I[cand])
    scale = U[uid].norm(dim=1)[:, None] * I[cand].norm(dim=2)
    assert ((score - want).abs() <= 1e-5 * scale).all()
    assert torch.equal(nn_, m.all_items_emb[hn.chosen])          # the negative rows are the picks' final rows
    assert torch.equal(uu, m.all_users_emb[uid.to(DEV)])
    if M == 1:
        assert torch.equal(chosen, cand[:, 0])
    j = (cand == chosen[:, None]).float().argmax(1)
    assert (cand[torch.arange(len(j)), j] == chosen).all()
    best = want.abs().max(1).values
    picked = want.abs()[torch.arange(len(j)), j]
    assert (picked >= best - 1e-5 * scale.max(1).values).all()  # the largest |score|, up to fp32 ties


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp(min=1e-30))


@pytest.mark.parametrize("emb,K", [(64, 3), (128, 4), (65, 2)])
def test_dns_step_is_the_plain_step_with_the_picks(emb, K):
    """Training mode, node and message dropout on: a step with HardNegatives and the plain step given its picks as
    neg_item draw the same dropout key and compute the same outputs bit for bit.  Loss and gradients are summed with
    float atomics (BPR's batch sum, the table and weight gradients), so they are compared at the tolerance the suite
    uses for a repeated step."""
    m, train, b = _setup(emb=emb, K=K, B=256)
    m.train()
    state = copy.deepcopy(m.state_dict())
    hn = pkg.HardNegatives(train, 32)
    crit = pkg.BPR(0.025, 256)
    res = []
    for neg in (hn, None):
        m.load_state_dict(state)                                 # the forward's feature mix rewrites user rows
        m.zero_grad(set_to_none=True)
        torch.manual_seed(17)
        uu, pp, nn_ = _call(m, b, hn if neg is hn else chosen)
        loss = crit(uu, pp, nn_)
        loss.backward()
        if neg is hn:
            chosen = hn.chosen.clone()
            assert m._last.drop_p > 0 and max(m._last.mess_p) > 0
        res.append((uu.detach().clone(), pp.detach().clone(), nn_.detach().clone(), loss.detach().clone(),
                    {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}, m._last.seed))
    (u0, p0, n0, l0, g0, s0), (u1, p1, n1, l1, g1, s1) = res
    assert s0 == s1
    assert torch.equal(u0, u1) and torch.equal(p0, p1) and torch.equal(n0, n1)
    assert abs(float(l0) - float(l1)) <= 1e-6 * abs(float(l1))
    assert g0.keys() == g1.keys() and len(g0) > 0
    for k in g0:
        assert _rel(g0[k], g1[k]) <= 1e-6, k


def test_graphed_step_redraws_candidates_every_replay():
    m, train, b = _setup(B=256)
    m.train()
    hn = pkg.HardNegatives(train, 16, debug=True)
    step = pkg.GraphedStep(m, pkg.BPR(0.025, 256), 256, negatives=hn)
    with pytest.raises(ValueError, match="neg_item"):
        step(b)
    batch = {k: v for k, v in b.items() if k != "neg_item"}
    rows = rows_of(train)
    picks = []
    for _ in range(2):
        loss = float(step(batch))
        assert np.isfinite(loss)
        st = next(iter(step.graphs.values()))[3]
        key = (st.seed + int(step.seed_dev) - GRAPH_STEP) % (1 << 64)   # the counter before this replay's bump
        want = H.candidates(key, b["u_id"].numpy(), rows, N_ITEM, 16)
        assert np.array_equal(hn.cand.cpu().numpy(), want)
        assert torch.equal(hn.chosen, hn.cand[torch.arange(256, device=DEV), hn.score.abs().argmax(1)])
        picks.append((hn.cand.clone(), hn.chosen.clone()))
    assert not torch.equal(picks[0][0], picks[1][0]) and not torch.equal(picks[0][1], picks[1][1])


def test_refusals():
    m, train, b = _setup(B=64)
    m.eval()
    short = pkg.Interactions.from_pairs([0, 3], [1, 2], N_ITEM, rows=torch.arange(N_USER - 1))
    with pytest.raises(ValueError, match="699 rows"):
        _call(m, b, pkg.HardNegatives(short))
    wide = pkg.Interactions.from_pairs([0, 3], [1, 2], N_ITEM + 1, rows=torch.arange(N_USER))
    with pytest.raises(ValueError, match="501 items"):
        _call(m, b, pkg.HardNegatives(wide))
    m._shard = RowShards(N_USER + N_ITEM, 2, 0)
    try:
        with pytest.raises(ValueError, match="row-sharded"):
            _call(m, b, pkg.HardNegatives(train))
    finally:
        m._shard = None
    with torch.no_grad():                                        # and the plain forms still work on the same model
        _call(m, b, b["neg_item"])
        _call(m, b, torch.empty(0))
