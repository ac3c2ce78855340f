"""Accuracy audit at full Gowalla shape: every gradient of one training step (dropout off) from (a) this library,
(b) the fp32 CPU oracle (= the reference's torch path), both measured against the float64 restatement.
  python tools/grad_accuracy.py [shape]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import seoul_tourism_recommendation_ngcf_b200 as pkg
from oracle import ngcf_oracle as O
from seoul_tourism_recommendation_ngcf_b200 import laplacian, synth

shape = sys.argv[1] if len(sys.argv) > 1 else "gowalla"
n_user, n_item, n_edges, emb, K = synth.SHAPES[shape]
u, i, r = synth.powerlaw_bipartite(n_user, n_item, n_edges, seed=0)
L = laplacian.laplacian_coo(u, i, r, n_user, n_item)
nd = synth.num_dict_for(n_user, n_item)
torch.manual_seed(0)
m = pkg.NGCF(emb, [emb] * K, 0.3, [0.1] * K, 1.0, [L, L], nd, 1024, torch.device("cpu"))
params = {k: v.detach().clone() for k, v in m.state_dict().items()}
m = m.to("cuda").eval()
b = {k: torch.from_numpy(v) for k, v in synth.random_batch(n_user, n_item, 1024, seed=1).items()}
loss_ref, grads_ref, mid = O.train_step(params, L, b, emb_ratio=1.0, weight_decay=0.025, batch_size_ctor=1024)
d = {k: v.to("cuda") for k, v in b.items()}
uu, pp, nn_ = m(d["year"], d["u_id"], d["age"], d["sex"], d["month"], d["day"], d["dow"], d["pos_item"], d["neg_item"], False)
loss = pkg.BPR(0.025, 1024)(uu, pp, nn_)
loss.backward()
# float64 truth, evaluated on the LeakyReLU branches this forward took (see oracle.backward_f64)
act_pos = [(e.cpu().numpy() > 0) for e in m._last.E[1:]]
flips = sum(int(((e.cpu().numpy() > 0) != (r.detach().numpy() > 0)).sum()) for e, r in zip(m._last.E[1:], mid["out"]["E"][1:]))
l64, truth, _ = O.train_step_f64(params, L, b, emb_ratio=1.0, weight_decay=0.025, batch_size_ctor=1024, act_pos=act_pos)
print("LeakyReLU branches differing from the fp32 oracle:", flips)
rel = lambda a, t: float(np.abs(np.asarray(a, np.float64) - t).max() / np.abs(t).max())
print(f"loss: ours {float(loss):.8f} oracle32 {float(loss_ref):.8f} f64 {l64:.8f}")
print(f"{'tensor':24s} {'ours vs f64':>12s} {'oracle32 vs f64':>16s} {'ours vs oracle32':>17s}")
P = dict(m.named_parameters())
for k, t in truth.items():
    print(f"{k:24s} {rel(P[k].grad.cpu().numpy(), t):12.2e} {rel(grads_ref[k].numpy(), t):16.2e} "
          f"{rel(P[k].grad.cpu().numpy(), grads_ref[k].double().numpy()):17.2e}")
