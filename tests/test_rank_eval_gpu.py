"""Full-ranking evaluation on the GPU: score_topk(exclude=...) on both kernels against float64 U·Iᵀ with the excluded
entries at -inf, rank_metrics against the numpy restatement, and full_rank_eval end to end (model forward, repeat
determinism, CUDA-graph capture)."""
import numpy as np
import pytest
import torch

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import laplacian, synth
from tests import _rank_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
FLT_MAX = float(np.finfo(np.float32).max)


def _assert_masked_topk(val, idx, ref_scores, k, tie=2e-5):
    """As test_parity_gpu._assert_topk (same list as sorting the reference scores apart from ties within `tie`,
    relative), over the finite reference scores only; rows with fewer than k of them end in (-1, -FLT_MAX) slots."""
    finite = np.isfinite(ref_scores)
    scale = np.abs(ref_scores[finite]).max()
    order = np.argsort(-ref_scores, axis=1, kind="stable")[:, :k]
    for r in range(ref_scores.shape[0]):
        nv = min(k, int(finite[r].sum()))
        got = idx[r, :nv]
        assert len(set(got.tolist())) == nv and np.all(got >= 0), (r, got)
        assert np.all(finite[r, got]), (r, "an excluded item was ranked")
        got_ref_scores = ref_scores[r, got]
        want = ref_scores[r, order[r, :nv]]
        assert np.all(np.abs(got_ref_scores - want) <= tie * scale), (r, got, order[r, :nv])
        assert np.all(np.abs(val[r, :nv] - want) <= 1e-4 * scale)
        assert np.all(np.diff(val[r, :nv]) <= 0)
        assert np.all(idx[r, nv:] == -1) and np.all(val[r, nv:] == -FLT_MAX), r


def _exclusion(u, it, density, seed):
    """Power-law pairs plus three kinds of special rows: users 0-4 exclude their true top-50 items, users 5-9 exclude
    nothing, user 10 keeps only k/2 items."""
    U, I = u.shape[0], it.shape[0]
    nnz = max(1, int(U * I * density))
    pu, pi, _ = synth.powerlaw_bipartite(U, I, nnz, seed=seed)
    scores = (u.double() @ it.double().T).numpy()
    top50 = np.argsort(-scores, axis=1)[:, :50]
    keep = (pu < 5) | (pu > 10)
    pu, pi = pu[keep], pi[keep]
    n0 = min(5, U)
    pu = np.concatenate([pu, np.repeat(np.arange(n0), min(50, I))])
    pi = np.concatenate([pi, top50[:n0, :min(50, I)].reshape(-1)])
    return pu, pi, scores


@pytest.mark.parametrize("U,I,D,k,density", [(1000, 20011, 256, 20, 0.01), (129, 1300, 96, 32, 0.05),
                                             (37, 100, 195, 100, 0.1), (300, 4000, 256, 33, 0.02)])
def test_masked_topk_vs_float64(U, I, D, k, density):
    gen = torch.Generator().manual_seed(U * 7 + k)
    u, it = torch.randn(U, D, generator=gen), torch.randn(I, D, generator=gen)
    it[I // 2] = it[I // 3]                                               # an exact tie
    pu, pi, scores = _exclusion(u, it, density, seed=k)
    rest = np.setdiff1d(np.arange(I), np.arange(0, I, I // (k // 2)))      # user 10 keeps ~k/2 items, spread out
    pu, pi = np.concatenate([pu, np.full(rest.size, 10)]), np.concatenate([pi, rest])
    ex = pkg.Interactions.from_pairs(pu, pi, I, rows=np.arange(U))
    lens = np.diff(ex.ptr.numpy())
    assert lens[5:10].sum() == 0 and lens[:5].min() >= min(50, I)
    val, idx = pkg.score_topk(u.to(DEV), it.to(DEV), k, exclude=ex)
    masked = scores.copy()
    masked[ex.ptr.numpy().searchsorted(np.arange(ex.idx.numel()), side="right") - 1, ex.idx.numpy()] = -np.inf
    _assert_masked_topk(val.cpu().numpy(), idx.cpu().numpy(), masked, k)
    assert (idx[10] == -1).sum().item() == k - np.isfinite(masked[10]).sum() > 0   # the short row's tail
    # exclusion changes the answer: none of the unmasked list's leaders of users 0-4 (their true top 50) is left
    plain = pkg.score_topk(u.to(DEV), it.to(DEV), k)[1].cpu().numpy()
    for r in range(5):
        assert not np.intersect1d(plain[r, :min(k, 50)], idx[r].cpu().numpy()).size


def test_masked_topk_unaligned_view_runs_the_fallback():
    gen = torch.Generator().manual_seed(3)
    base_u, base_i = torch.randn(200 * 129 + 1, generator=gen), torch.randn(3000 * 128 + 1, generator=gen)
    u = base_u.to(DEV)[1:].view(200, 129)[:, :128]                        # not 16-byte aligned: CUDA-core kernel
    it = base_i.to(DEV)[1:].view(3000, 128)
    pu, pi, _ = synth.powerlaw_bipartite(200, 3000, 30000, seed=9)
    ex = pkg.Interactions.from_pairs(pu, pi, 3000, rows=np.arange(200))
    val, idx = pkg.score_topk(u, it, 20, exclude=ex)
    scores = (u.cpu().double() @ it.cpu().double().T).numpy()
    scores[pu, pi] = -np.inf
    _assert_masked_topk(val.cpu().numpy(), idx.cpu().numpy(), scores, 20)


@pytest.mark.parametrize("U,I,D,k", [(1000, 20011, 256, 20), (37, 100, 195, 100)])
def test_empty_exclusion_is_bit_identical_to_none(U, I, D, k):
    gen = torch.Generator().manual_seed(11)
    u, it = torch.randn(U, D, generator=gen).to(DEV), torch.randn(I, D, generator=gen).to(DEV)
    empty = pkg.Interactions.from_pairs([], [], I, rows=np.arange(U))
    v0, i0 = pkg.score_topk(u, it, k)
    v1, i1 = pkg.score_topk(u, it, k, exclude=empty)
    assert torch.equal(i0, i1) and torch.equal(v0.view(torch.int32), v1.view(torch.int32))


def test_rank_metrics_match_numpy_restatement():
    rng = np.random.default_rng(2)
    U, n_items, k, Ks = 700, 3000, 40, (1, 5, 20, 40)
    idx = np.stack([rng.choice(n_items, k, replace=False) for _ in range(U)])
    idx[::7, 30:] = -1                                                    # short lists
    tu = np.repeat(np.arange(U), rng.integers(0, 60, U))
    ti = np.where(rng.random(tu.size) < 0.5, idx[tu, rng.integers(0, k, tu.size)].clip(0), rng.integers(0, n_items, tu.size))
    truth = pkg.Interactions.from_pairs(tu, ti, n_items, rows=np.arange(U))
    totals, per = pkg.rank_metrics(torch.from_numpy(idx).to(DEV), truth, Ks)
    means, n, want = R.metrics(idx, R.rows_of(truth), Ks)
    assert n < U                                                          # some users have no truth items
    assert np.abs(per.cpu().numpy() - want).max() <= 1e-6
    t = totals.cpu().numpy()
    assert t[-1] == n and np.abs(t[:-1] - means.reshape(-1)).max() <= 1e-6


def _trained_like_model(n_user=1500, n_item=2200, emb=64, K=3):
    u, i, r = synth.powerlaw_bipartite(n_user, n_item, 40000, seed=4)
    L = laplacian.laplacian_coo(u, i, r, n_user, n_item)
    torch.manual_seed(0)
    m = pkg.NGCF(emb, [emb] * K, 0.3, [0.1] * K, 1.0, [L, L], synth.num_dict_for(n_user, n_item), 128,
                 torch.device(DEV)).to(DEV).eval()
    b = {k: torch.from_numpy(v).to(DEV) for k, v in synth.random_batch(n_user, n_item, 128, seed=1).items()}
    with torch.no_grad():
        m(b["year"], b["u_id"], b["age"], b["sex"], b["month"], b["day"], b["dow"], b["pos_item"], torch.empty(0), False)
    return m, u, i


def test_full_rank_eval_end_to_end():
    m, u, i = _trained_like_model()
    n_item = m.all_items_emb.shape[0]
    rng = np.random.default_rng(0)
    is_test = rng.random(u.size) < 0.2
    rows = torch.from_numpy(np.unique(u[is_test])).to(DEV)
    train = pkg.Interactions.from_pairs(u[~is_test], i[~is_test], n_item, rows=rows)
    test = pkg.Interactions.from_pairs(u[is_test], i[is_test], n_item, rows=rows)
    U, I = m.all_users_emb[rows], m.all_items_emb
    assert U.shape[1] == 256 and I.shape[0] >= 1024                       # the tensor-core ranking
    Ks = (5, 20)
    got, per = pkg.full_rank_eval(U, I, train=train, test=test, Ks=Ks, return_per_user=True)
    assert got["n_users"] == rows.numel()
    # torch: mm + mask + topk, numpy metrics
    s = (U.double() @ I.double().T)
    tr_rows = R.rows_of(train)
    s[torch.from_numpy(np.repeat(np.arange(len(tr_rows)), [len(t) for t in tr_rows])).to(DEV),
      train.idx.to(DEV).long()] = -float("inf")
    ref_idx = torch.topk(s, 20).indices.cpu().numpy()
    means, n, _ = R.metrics(ref_idx, R.rows_of(test), Ks)
    for j, K in enumerate(Ks):
        for q, name in enumerate(("recall", "precision", "ndcg", "hit")):
            assert abs(got[f"{name}@{K}"] - means[j, q]) <= 2e-3, (name, K)   # list differences only at score ties
    # the per-user numbers are exactly the metrics of the returned lists
    _, idx = pkg.score_topk(U, I, 20, exclude=train)
    assert (idx.cpu().numpy() == ref_idx).mean() > 0.99
    _, _, want = R.metrics(idx.cpu().numpy(), R.rows_of(test), Ks)
    assert np.abs(per.cpu().numpy() - want).max() <= 1e-6
    # repeat: identical bits
    again, per2 = pkg.full_rank_eval(U, I, train=train, test=test, Ks=Ks, return_per_user=True)
    assert again == got and torch.equal(per, per2)
    # one CUDA graph of the score and metric launches, replayed, equals the eager call
    train_d, test_d = train.to(DEV), test.to(DEV)
    eager_tot, eager_per = pkg.rank_metrics(pkg.score_topk(U, I, 20, exclude=train_d)[1], test_d, Ks)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                                         # warm-up off the capture
        pkg.rank_metrics(pkg.score_topk(U, I, 20, exclude=train_d)[1], test_d, Ks)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        tot, pu = pkg.rank_metrics(pkg.score_topk(U, I, 20, exclude=train_d)[1], test_d, Ks)
    tot.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(tot, eager_tot) and torch.equal(pu, eager_per)
    assert tot.tolist()[:-1] == [got[f"{n}@{K}"] for K in Ks for n in ("recall", "precision", "ndcg", "hit")]
