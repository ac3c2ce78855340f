"""Sampled-softmax loss on the GPU: loss and gradients against the float64 restatement over batch sizes, widths,
temperatures, weight decays, with and without negatives and ids; masking edge cases; large logits; bit-identical
repeats; CUDA-graph capture; end-to-end parameter gradients of NGCF steps (eager, GraphedStep, signed hard negatives);
and a short training run that raises recall."""
import numpy as np
import pytest
import torch

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import laplacian, synth
from tests import _softmax_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
LOSS_TOL, GRAD_TOL = 1e-5, 1e-4


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


def _inputs(B, D, seed, n_items=None, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    u, p, n = (torch.randn(B, D, generator=g) * scale / D ** 0.5 for _ in range(3))
    n_items = n_items or max(2, B // 2)                   # repeated ids in most batches
    pos = torch.randint(0, n_items, (B,), generator=g)
    neg = torch.randint(0, n_items, (B,), generator=g)
    return [t.to(DEV) for t in (u, p, n, pos, neg)]


def _fused(u, p, n, tau, wd, bs, pos=None, neg=None):
    ts = [t.clone().requires_grad_(True) for t in (u, p)] + [n.clone().requires_grad_(n.numel() > 0)]
    loss = pkg.SoftmaxLoss(wd, bs, tau)(ts[0], ts[1], ts[2], pos, neg)
    loss.backward()
    return loss.detach(), ts[0].grad, ts[1].grad, ts[2].grad


def _check(u, p, n, tau, wd, bs, pos=None, neg=None, worst=None):
    got = _fused(u, p, n, tau, wd, bs, pos, neg)
    want = R.loss_and_grads(u, p, n, temperature=tau, weight_decay=wd, batch_size=bs, pos_ids=pos, neg_ids=neg)
    assert torch.isfinite(got[0])
    lr = abs(float(got[0]) - float(want[0])) / max(abs(float(want[0])), 1e-30)
    assert lr <= LOSS_TOL, (float(got[0]), float(want[0]))
    errs = [lr]
    for k in range(1, 4):
        if want[k] is None:
            assert got[k] is None
            continue
        e = _rel(got[k], want[k])
        assert e <= GRAD_TOL, (("gu", "gp", "gn")[k - 1], e)
        errs.append(e)
    if worst is not None:
        worst.append(max(errs))
    return got


@pytest.mark.parametrize("B", [1, 7, 128, 203, 1024, 4096])
@pytest.mark.parametrize("D", [4, 65, 195, 256, 257, 1152])
def test_loss_and_gradients_equal_the_restatement(B, D):
    u, p, n, pos, neg = _inputs(B, D, seed=B * 10007 + D)
    empty = torch.empty(0, device=DEV)
    worst = []
    for tau in (0.05, 0.2, 1.0):
        for wd in (0.0, 0.025):
            for with_n in (False, True):
                for ids in (False, True):
                    nn_ = n if with_n else empty
                    _check(u, p, nn_, tau, wd, B, pos if ids else None, neg if ids and with_n else None, worst)
    print(f"B={B} D={D}: worst relative error {max(worst):.2e}")


def test_duplicated_positive_ids_and_a_negative_equal_to_a_positive():
    B, D = 203, 65
    u, p, n, pos, neg = _inputs(B, D, seed=5, n_items=1000)
    pos[10:20] = 3                                        # ten rows share item 3
    neg[:5] = pos[100]                                    # five negatives are row 100's positive
    neg[50] = pos[50]                                     # a row's own negative equals its positive
    _check(u, p, n, 0.2, 0.025, B, pos, neg)
    keep = R.mask(pos.cpu(), neg.cpu(), B, True)
    assert not keep[10, 11] and keep[10, 10] and not keep[100, B] and not keep[50, B + 50]


def test_every_other_column_masked_leaves_the_regularisation():
    B, D = 128, 64
    u, p, n, _, _ = _inputs(B, D, seed=6)
    pos = torch.zeros(B, dtype=torch.int64, device=DEV)  # one item everywhere: every column but the own positive
    neg = torch.zeros(B, dtype=torch.int64, device=DEV)
    wd = 0.025
    loss, gu, gp, gn = _check(u, p, n, 0.2, wd, B, pos, neg)
    reg = wd * ((u.double() ** 2).sum() + (p.double() ** 2).sum() + (n.double() ** 2).sum()) / B
    assert abs(float(loss) - float(reg)) <= 1e-5 * float(reg)
    for g, x in ((gu, u), (gp, p), (gn, n)):
        assert _rel(g, 2 * wd / B * x) <= GRAD_TOL


def test_large_logits_are_finite_and_equal_the_restatement():
    # small integers: the 3xTF32 products are exact, so ties between the largest logits stay ties
    B, D = 256, 128
    g = torch.Generator().manual_seed(9)
    u, p, n = (torch.randint(-3, 4, (B, D), generator=g).float().to(DEV) for _ in range(3))
    s = (u @ torch.cat([p, n]).T).abs().max()
    tau = float(s) / 1e4                                   # |s| up to 1e4
    got = _check(u, p, n, tau, 0.0, B)
    assert all(torch.isfinite(t).all() for t in got)


def test_repeat_is_bit_identical_and_forward_only_gives_the_same_loss():
    B, D = 1024, 256
    u, p, n, pos, neg = _inputs(B, D, seed=11)
    a = _fused(u, p, n, 0.2, 0.025, B, pos, neg)
    b = _fused(u, p, n, 0.2, 0.025, B, pos, neg)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    with torch.no_grad():
        fo = pkg.SoftmaxLoss(0.025, B, 0.2)(u, p, n, pos, neg)
    assert torch.equal(fo, a[0])


def test_captured_loss_replays_on_new_inputs():
    B, D = 300, 192
    crit = pkg.SoftmaxLoss(0.025, B, 0.2)
    su, sp, sn = (torch.zeros(B, D, device=DEV, requires_grad=True) for _ in range(3))
    spos = torch.zeros(B, dtype=torch.int64, device=DEV)
    sneg = torch.zeros(B, dtype=torch.int64, device=DEV)
    u, p, n, pos, neg = _inputs(B, D, seed=12)
    with torch.no_grad():
        for s, t in ((su, u), (sp, p), (sn, n), (spos, pos), (sneg, neg)):
            s.copy_(t)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                          # warm-up outside the graph
        crit(su, sp, sn, spos, sneg).backward()
    torch.cuda.current_stream().wait_stream(side)
    for t in (su, sp, sn):
        t.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss = crit(su, sp, sn, spos, sneg)
        loss.backward()
    for seed in (13, 14):
        u, p, n, pos, neg = _inputs(B, D, seed=seed)
        with torch.no_grad():
            for s, t in ((su, u), (sp, p), (sn, n), (spos, pos), (sneg, neg)):
                s.copy_(t)
        graph.replay()
        want = _fused(u, p, n, 0.2, 0.025, B, pos, neg)
        assert torch.equal(loss, want[0])
        for g, w in zip((su.grad, sp.grad, sn.grad), want[1:]):
            assert torch.equal(g, w)


# ---- end to end with NGCF ---------------------------------------------------------------------------------------------
N_USER, N_ITEM = 700, 500


class _RefSoftmax(pkg.SoftmaxLoss):
    """The same loss in float64 torch: a SoftmaxLoss for GraphedStep (it passes the ids), computed by the restatement."""

    def forward(self, u, p, n, pos_ids=None, neg_ids=None):
        return R.loss(u, p, n, temperature=self.temperature, weight_decay=self.weight_decay,
                      batch_size=self.batch_size, pos_ids=pos_ids, neg_ids=neg_ids)


def _model(emb, K, B):
    u, i, r = synth.powerlaw_bipartite(N_USER, N_ITEM, 20000, seed=3)
    L = laplacian.laplacian_coo(u, i, r, N_USER, N_ITEM)
    torch.manual_seed(0)
    m = pkg.NGCF(emb, [emb] * K, 0.3, [0.1] * K, 1.0, [L, L], synth.num_dict_for(N_USER, N_ITEM), B,
                 torch.device(DEV)).to(DEV)
    train = pkg.Interactions.from_pairs(u, i, N_ITEM, rows=torch.arange(N_USER))
    b = {k: torch.from_numpy(v) for k, v in synth.random_batch(N_USER, N_ITEM, B, seed=4).items()}
    return m, train, b


def _grads(m):
    return {k: q.grad.detach().clone() for k, q in m.named_parameters() if q.grad is not None}


def _compare(ga, gb):
    assert ga.keys() == gb.keys() and ga
    for k in ga:
        assert _rel(ga[k], gb[k]) <= GRAD_TOL, (k, _rel(ga[k], gb[k]))


@pytest.mark.parametrize("emb,K", [(64, 3), (65, 2)])
def test_ngcf_step_gradients_equal_a_float64_loss(emb, K):
    B = 256
    m, _, b = _model(emb, K, B)
    d = {k: v.to(DEV) for k, v in b.items()}

    def step(crit):
        m.zero_grad(set_to_none=True)
        torch.manual_seed(21)                              # same dropout masks in both steps
        u, p, n = m(d["year"], d["u_id"], d["age"], d["sex"], d["month"], d["day"], d["dow"], d["pos_item"],
                    d["neg_item"], True)
        crit(u, p, n, d["pos_item"], d["neg_item"]).backward()
        return _grads(m)

    _compare(step(pkg.SoftmaxLoss(0.025, B, 0.2)), step(_RefSoftmax(0.025, B, 0.2)))


def test_ngcf_step_without_negatives():
    """NGCF returns a host torch.empty(0) for n when there are no negatives: the loss takes it as "no negatives"."""
    B = 128
    m, _, b = _model(64, 3, B)
    d = {k: v.to(DEV) for k, v in b.items()}

    def step(crit):
        m.zero_grad(set_to_none=True)
        torch.manual_seed(22)
        u, p, n = m(d["year"], d["u_id"], d["age"], d["sex"], d["month"], d["day"], d["dow"], d["pos_item"],
                    torch.empty(0), True)
        assert n.numel() == 0
        crit(u, p, n, d["pos_item"]).backward()
        return _grads(m)

    _compare(step(pkg.SoftmaxLoss(0.025, B, 0.2)), step(_RefSoftmax(0.025, B, 0.2)))


@pytest.mark.parametrize("emb,K,hard", [(64, 3, False), (65, 2, False), (64, 3, True)])
def test_graphed_step_gradients_equal_a_float64_loss(emb, K, hard):
    B = 256
    m, train, b = _model(emb, K, B)
    batch = dict(b)
    hn = None
    if hard:
        hn = pkg.HardNegatives(train, 16, signed=True)
        del batch["neg_item"]

    def run(crit):
        torch.manual_seed(31)                              # the same per-forward keys for both captures
        step = pkg.GraphedStep(m, crit, B, negatives=hn)
        step(batch)
        picks = None if hn is None else hn.chosen.clone()
        return _grads(m), picks

    ga, pa = run(pkg.SoftmaxLoss(0.025, B, 0.2))
    gb, pb = run(_RefSoftmax(0.025, B, 0.2))
    if hard:
        assert torch.equal(pa, pb)
    _compare(ga, gb)


def test_signed_hard_negatives_pick_the_largest_signed_score():
    B = 203
    m, train, b = _model(64, 3, B)
    m.eval()
    d = {k: v.to(DEV) for k, v in b.items()}
    with torch.no_grad():                                  # a large raw item block: scores of both signs
        m.item_embedding.weight.data.mul_(1000.0)
    hn = pkg.HardNegatives(train, 32, signed=True, debug=True)
    with torch.no_grad():
        m(d["year"], d["u_id"], d["age"], d["sex"], d["month"], d["day"], d["dow"], d["pos_item"], hn, True)
    rows = torch.arange(B, device=DEV)
    assert torch.equal(hn.chosen, hn.cand[rows, hn.score.argmax(1)])
    # the signed pick is not the |score| pick in many rows
    assert (hn.chosen != hn.cand[rows, hn.score.abs().argmax(1)]).sum() > B // 10


def test_short_training_run_raises_recall():
    n_user, n_item, B = 600, 400, 256
    u, i, r = synth.powerlaw_bipartite(n_user, n_item, 12000, seed=7)
    rng = np.random.default_rng(7)
    test_mask = rng.random(u.size) < 0.2
    tu, ti = u[~test_mask], i[~test_mask]
    L = laplacian.laplacian_coo(tu, ti, r[~test_mask], n_user, n_item)
    train = pkg.Interactions.from_pairs(tu, ti, n_item, rows=torch.arange(n_user))
    test = pkg.Interactions.from_pairs(u[test_mask], i[test_mask], n_item, rows=torch.arange(n_user))
    torch.manual_seed(0)
    m = pkg.NGCF(64, [64] * 2, 0.1, [0.1] * 2, 1.0, [L, L], synth.num_dict_for(n_user, n_item), B,
                 torch.device(DEV)).to(DEV)

    def recall():
        m.eval()
        ctx = synth.random_batch(n_user, n_item, n_user, seed=1)
        with torch.no_grad():
            m(*(torch.from_numpy(ctx[k]).to(DEV) for k in ("year", "u_id", "age", "sex", "month", "day", "dow")),
              torch.from_numpy(ctx["pos_item"]).to(DEV), torch.empty(0), False)
            out = pkg.full_rank_eval(m.all_users_emb, m.all_items_emb, train=train.to(DEV), test=test.to(DEV))
        m.train()
        return out["recall@20"]

    r0 = recall()
    opt = pkg.Adam(m.parameters(), lr=5e-3)
    step = pkg.GraphedStep(m, pkg.SoftmaxLoss(1e-4, B, 0.2), B, optimizer=opt)
    for s in range(150):
        b = {k: torch.from_numpy(v) for k, v in synth.random_batch(n_user, n_item, B, seed=100 + s).items()}
        j = rng.integers(0, tu.size, B)
        b["u_id"], b["pos_item"] = torch.from_numpy(tu[j]), torch.from_numpy(ti[j])
        loss = step(b)
    assert torch.isfinite(loss)
    r1 = recall()
    print(f"recall@20: {r0:.4f} -> {r1:.4f}")
    assert r1 > r0 + 0.02
