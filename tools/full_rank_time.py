"""Full-ranking evaluation at the NGCF paper's dataset shapes (synth.SHAPES: all users, item table of width d·(K+1), an
80/20 train/test split of synth.powerlaw_bipartite pairs, k = 20), three ways:

  masked   score_topk(exclude=train) + rank_metrics(test)      (what full_rank_eval launches)
  unmasked score_topk                                          (no exclusion, no metrics)
  torch    per chunk of users: mm + index_put_(-inf) + topk, then the metrics in torch (searchsorted in the test keys)

CUDA events, a 512-MB buffer overwritten before every timed call (cold L2), medians.  Prints the card and its power
limit, and how far the masked lists and metrics agree with torch's.  ``--ab-lib PATH`` also times the unmasked call
through another build of libngcf_b200.so, alternating with this one.  python tools/full_rank_time.py [--ab-lib PATH]"""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import _lib, synth

dev = torch.device("cuda:0")
flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
K = 20


def timed(fns, reps):
    """medians (ms) of each fn in fns, called alternately, cold L2 before each call"""
    for fn in fns:
        fn(); fn()
    ev = [[] for _ in fns]
    for _ in range(reps):
        for j, fn in enumerate(fns):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            ev[j].append((e0, e1))
    torch.cuda.synchronize()
    return [statistics.median(a.elapsed_time(b) for a, b in e) for e in ev]


def raw_score_topk(lib, u, it, k):
    """ngcf_score_topk through an explicitly loaded library (the A/B arm)"""
    need = C.c_size_t(0)
    _lib.check(lib.ngcf_score_topk_workspace(u.shape[0], it.shape[0], u.shape[1], k, C.byref(need)))
    ws = torch.empty(need.value, dtype=torch.uint8, device=dev)
    val = torch.empty(u.shape[0], k, dtype=torch.float32, device=dev)
    idx = torch.empty(u.shape[0], k, dtype=torch.int64, device=dev)
    rc = lib.ngcf_score_topk(u.data_ptr(), u.shape[0], it.data_ptr(), it.shape[0], u.shape[1], k, val.data_ptr(),
                             idx.data_ptr(), ws.data_ptr(), need.value, _lib.current_stream())
    assert rc == 0, lib.ngcf_last_error()
    return val, idx


def torch_pipeline(u, it, train, test, chunk):
    """mm + mask + topk + metrics per chunk of users; returns (totals [recall, precision, ndcg, hit, n], idx)"""
    n_items = it.shape[0]
    tr_row = torch.repeat_interleave(torch.arange(train.n_rows, device=dev), train.ptr.diff())
    te_row = torch.repeat_interleave(torch.arange(test.n_rows, device=dev), test.ptr.diff())
    te_key = te_row * n_items + test.idx.long()                          # ascending
    n_te = test.ptr.diff()
    w = 1.0 / torch.log2(torch.arange(K, device=dev, dtype=torch.float64) + 2)
    cw = torch.cat((w.new_zeros(1), w.cumsum(0)))
    sums = torch.zeros(4, dtype=torch.float64, device=dev)
    out = []
    for r0 in range(0, u.shape[0], chunk):
        r1 = min(u.shape[0], r0 + chunk)
        s = u[r0:r1] @ it.T
        a, b = int(train.ptr[r0]), int(train.ptr[r1])                    # host reads: a user's code would do them too
        s.index_put_((tr_row[a:b] - r0, train.idx[a:b].long()), torch.tensor(-float("inf"), device=dev))
        idx = torch.topk(s, K).indices
        q = torch.arange(r0, r1, device=dev)[:, None] * n_items + idx
        pos = torch.searchsorted(te_key, q).clamp_(max=max(te_key.numel() - 1, 0))
        hit = (te_key[pos] == q).double()
        h = hit.sum(1)
        nt = n_te[r0:r1].double()
        ok = nt > 0
        idcg = cw[nt.clamp(max=K).long()]
        sums += torch.stack(((h / nt.clamp(min=1))[ok].sum(), (h / K)[ok].sum(),
                             ((hit * w).sum(1) / idcg.clamp(min=1e-30))[ok].sum(), (h > 0).double()[ok].sum()))
        out.append(idx)
    n = (n_te > 0).sum()
    return torch.cat((sums / n, n[None].double())), torch.cat(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ab-lib", default=None, help="another libngcf_b200.so to time the unmasked call against")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--chunk", type=int, default=4096, help="users per chunk of the torch pipeline")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {torch.cuda.get_device_name(0)}; nvidia-smi (name, power limit, max SM clock): {q[0] if q else '?'}")
    other = None
    if args.ab_lib:
        other = C.CDLL(os.path.abspath(args.ab_lib))
        for name in ("ngcf_score_topk_workspace", "ngcf_score_topk", "ngcf_last_error"):
            getattr(other, name).argtypes = _lib.SIGNATURES[name]
        other.ngcf_last_error.restype = C.c_char_p
    for shape in ("gowalla", "yelp2018", "amazon-book"):
        n_user, n_item, n_inter, emb, layers = synth.SHAPES[shape]
        D = emb * (layers + 1)
        users, items, _ = synth.powerlaw_bipartite(n_user, n_item, n_inter, seed=0)
        is_test = np.random.default_rng(1).random(users.size) < 0.2
        rows = np.arange(n_user)
        train = pkg.Interactions.from_pairs(users[~is_test], items[~is_test], n_item, rows=rows).to(dev)
        test = pkg.Interactions.from_pairs(users[is_test], items[is_test], n_item, rows=rows).to(dev)
        gen = torch.Generator(device=dev).manual_seed(0)
        u = torch.randn(n_user, D, device=dev, generator=gen) * 0.1
        it = torch.randn(n_item, D, device=dev, generator=gen) * 0.1

        def masked():
            return pkg.rank_metrics(pkg.score_topk(u, it, K, exclude=train)[1], test, (K,))

        fns = [masked, lambda: pkg.score_topk(u, it, K), lambda: torch_pipeline(u, it, train, test, args.chunk)]
        if other is not None:
            fns.append(lambda: raw_score_topk(other, u, it, K))
        t = timed(fns, args.reps)
        _, idx = pkg.score_topk(u, it, K, exclude=train)
        tot = masked()[0].cpu().numpy()
        ref_tot, ref_idx = torch_pipeline(u, it, train, test, args.chunk)
        ref_tot = ref_tot.cpu().numpy()
        same = float((idx == ref_idx).float().mean())
        diff = np.abs(tot[:4] - ref_tot[:4]).max()
        line = (f"{shape:12s} {n_user} users x {n_item} items, D {D}, k {K}, {int(train.ptr[-1])} train / "
                f"{int(test.ptr[-1])} test pairs: masked {t[0]:.3f} ms, unmasked {t[1]:.3f} ms "
                f"(masked/unmasked {t[0] / t[1]:.3f}), torch mm+mask+topk+metrics {t[2]:.3f} ms "
                f"({t[2] / t[0]:.1f}x); same indices as torch {same:.5f}; recall/precision/ndcg/hit@{K} "
                f"{tot[0]:.5f}/{tot[1]:.5f}/{tot[2]:.5f}/{tot[3]:.5f} (torch max |diff| {diff:.2e}), users {int(tot[4])}")
        if other is not None:
            v0, i0 = pkg.score_topk(u, it, K)
            v1, i1 = raw_score_topk(other, u, it, K)
            line += (f"; unmasked with {args.ab_lib}: {t[3]:.3f} ms (this build / that {t[1] / t[3]:.3f}, "
                     f"identical output {bool(torch.equal(i0, i1) and torch.equal(v0, v1))})")
        print(line, flush=True)
        del u, it, train, test


if __name__ == "__main__":
    main()
