"""Dynamic hard-negative sampling at Gowalla shape (synth.SHAPES["gowalla"]: the bench graph, emb 64, 3 layers, so the
final rows are D = 256 wide; batch 1024, node dropout 0.3, message dropout 0.1, training mode):

  kernel      ngcf_hard_negatives alone on the layer outputs of one forward, M in {1, 8, 32, 64}, with an L2 flush
              (512 MB overwrite) before every call; the bytes of candidate rows it must read are printed beside it
  step        GraphedStep replays (forward + BPR + backward) with the batch's own neg_item and with
              negatives=HardNegatives(train, 32), alternating, no L2 flush

CUDA events, medians.  Prints the card and its power limit read in the same run.
python tools/hard_negatives_time.py [--reps N] [--out PATH]"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import _lib, laplacian, synth

dev = torch.device("cuda:0")
B, NODE_P, MESS_P = 1024, 0.3, 0.1


def timed(fns, reps, flush=None):
    """medians (ms) of each fn in fns, called alternately"""
    for fn in fns:
        fn(); fn()
    ev = [[] for _ in fns]
    for _ in range(reps):
        for j, fn in enumerate(fns):
            if flush is not None:
                flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            ev[j].append((e0, e1))
    torch.cuda.synchronize()
    return [statistics.median(a.elapsed_time(b) for a, b in e) for e in ev]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                  "profiles", "r04_hard_negatives_time.txt"))
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    say(f"card: {torch.cuda.get_device_name(0)}; nvidia-smi (name, power limit, max SM clock): {q[0] if q else '?'}")
    n_user, n_item, n_inter, emb, K = synth.SHAPES["gowalla"]
    u, i, r = synth.powerlaw_bipartite(n_user, n_item, n_inter, alpha=0.8, seed=0)
    L = laplacian.laplacian_coo(u, i, r, n_user, n_item)
    train = pkg.Interactions.from_pairs(u, i, n_item, rows=torch.arange(n_user)).to(dev)
    torch.manual_seed(0)
    m = pkg.NGCF(emb, [emb] * K, NODE_P, [MESS_P] * K, 1.0, [L, L], synth.num_dict_for(n_user, n_item), B, dev).to(dev)
    m.train()
    batch = {k: torch.from_numpy(v) for k, v in synth.random_batch(n_user, n_item, B, seed=1).items()}
    D = emb * (K + 1)
    say(f"gowalla shape: {n_user} users x {n_item} items, {n_inter} interactions, emb {emb} x {K} layers (D {D}), "
        f"batch {B}, node dropout {NODE_P}, message dropout {MESS_P}")

    # kernel alone, on the layer outputs of one training-mode forward
    d = {k: v.to(dev) for k, v in batch.items()}
    with torch.no_grad():
        m(d["year"], d["u_id"], d["age"], d["sex"], d["month"], d["day"], d["dow"], d["pos_item"], d["neg_item"], True)
    st, lib = m._last, _lib.load()
    layers, dims = _lib.ptr_array(st.E), _lib.int_array(st.dims)
    chosen = torch.empty(B, dtype=torch.int64, device=dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def kernel(M):
        def run():
            _lib.check(lib.ngcf_hard_negatives(layers, dims, K + 1, n_user, d["u_id"].data_ptr(), B, train.ptr.data_ptr(),
                                               train.idx.data_ptr(), n_item, M, 12345, None, chosen.data_ptr(), None,
                                               None, _lib.current_stream()), "hard_negatives")
        return run

    Ms = (1, 8, 32, 64)
    t = timed([kernel(M) for M in Ms], args.reps, flush)
    for M, ms in zip(Ms, t):
        mb = B * M * D * 4 / 1e6
        say(f"kernel  M {M:2d}: {ms * 1e3:7.1f} us  ({mb:5.1f} MB of candidate rows, {mb / 1e3 / (ms / 1e3):6.0f} GB/s "
            f"effective)")

    # whole training step, CUDA graph, with and without negatives=
    crit = pkg.BPR(0.025, B)
    plain = pkg.GraphedStep(m, crit, B, node_flag=True)
    hn = pkg.HardNegatives(train, 32)
    dns = pkg.GraphedStep(m, crit, B, node_flag=True, negatives=hn)
    nb = {k: v for k, v in batch.items() if k != "neg_item"}
    t_plain, t_dns = timed([lambda: plain(batch), lambda: dns(nb)], args.reps)
    loss_p, loss_d = float(plain(batch)), float(dns(nb))
    say(f"step    GraphedStep (fwd + BPR + bwd): plain neg_item {t_plain:.3f} ms, negatives=HardNegatives(M=32) "
        f"{t_dns:.3f} ms (+{(t_dns - t_plain) * 1e3:.1f} us); launches per step {plain.launches_per_step} vs "
        f"{dns.launches_per_step}; loss plain {loss_p:.5f}, DNS {loss_d:.5f}")
    picked = hn.chosen.cpu().numpy()
    uid = batch["u_id"].numpy()
    ptr, idx = train.ptr.cpu().numpy(), train.idx.cpu().numpy()
    bad = sum(np.isin(picked[b], idx[ptr[uid[b]]:ptr[uid[b] + 1]]) for b in range(B))
    say(f"picks of the last DNS replay: {len(np.unique(picked))} distinct items, {bad} training items among them")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
