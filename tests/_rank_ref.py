"""numpy restatement of the full-ranking metrics (ngcf_rank_metrics, include/ngcf_b200.h), used by the rank-eval tests."""
import numpy as np


def user_metrics(ranked, truth, Ks):
    """[len(Ks), 4] = (recall, precision, ndcg, hit) of one ranked id list against the set ``truth``; zeros when
    ``truth`` is empty.  -1 entries (empty slots) never hit."""
    truth = set(int(t) for t in truth)
    out = np.zeros((len(Ks), 4))
    if not truth:
        return out
    hit = np.array([int(r) >= 0 and int(r) in truth for r in ranked], dtype=bool)
    w = 1.0 / np.log2(np.arange(len(ranked)) + 2.0)
    for j, K in enumerate(Ks):
        h = int(hit[:K].sum())
        idcg = (1.0 / np.log2(np.arange(min(len(truth), K)) + 2.0)).sum()
        out[j] = (h / len(truth), h / K, w[:K][hit[:K]].sum() / idcg, float(h > 0))
    return out


def metrics(ranked_rows, truth_rows, Ks):
    """(means [len(Ks), 4] over the users with truth items, their number, per-user [U, len(Ks), 4])."""
    per = np.stack([user_metrics(r, t, Ks) for r, t in zip(ranked_rows, truth_rows)]) if len(ranked_rows) else \
        np.zeros((0, len(Ks), 4))
    counted = np.array([len(t) > 0 for t in truth_rows], dtype=bool)
    n = int(counted.sum())
    means = per[counted].mean(axis=0) if n else np.zeros((len(Ks), 4))
    return means, n, per


def rows_of(inter):
    """Interactions -> list of numpy item arrays, one per row."""
    ptr, idx = inter.ptr.cpu().numpy(), inter.idx.cpu().numpy()
    return [idx[ptr[r]:ptr[r + 1]] for r in range(inter.n_rows)]
