"""float64 torch restatement of LightGCN (seoul_tourism_recommendation_ngcf_b200/lightgcn.py), used by the LightGCN
tests.

E_{k+1} = L_k E_k with L_k a float64 sparse copy of the COO entries of the ``lap_list`` element whose layer-k keep flag
is set (all entries without node dropout), and the final rows are (E_0 + ... + E_K) / (K + 1).  Node dropout is
restated through ``tests._dropout_ref.edge_keep`` on the entries' global coordinates, so the keep lists are the device
decisions recomputed on the host.  Gradients come from torch autograd through ``torch.sparse.mm``, not from a
restated backward.  The product package never imports this module.
"""
import numpy as np
import torch

from tests._dropout_ref import edge_keep


def coo_of(L):
    """(row, col, val) of a ``lap_list`` element, a torch sparse COO tensor or a device CSR (plgraph.CsrLaplacian), as
    int64 / int64 / float64 numpy arrays."""
    if getattr(L, "is_sparse", False):
        idx = L._indices().cpu().numpy()
        return idx[0].astype(np.int64), idx[1].astype(np.int64), L._values().double().cpu().numpy()
    rowptr = L.rowptr.cpu().numpy().astype(np.int64)
    row = np.repeat(np.arange(L.n_rows, dtype=np.int64), np.diff(rowptr)) + L.row0
    return row, L.colidx.cpu().numpy().astype(np.int64), L.vals.double().cpu().numpy()


def keep_lists(L, seed: int, p: float, K: int):
    """Per-layer keep flags of L's entries (COO order of ``coo_of``) under device-RNG key ``seed`` (seed + seed_dev)."""
    row, col, _ = coo_of(L)
    return edge_keep(seed, p, K, row, col)


def layers(L, E0, K: int, keep=None):
    """[E_0, ..., E_K] in float64 (E0 is used as given, so autograd reaches it)."""
    row, col, val = coo_of(L)
    N = int(L.shape[0])
    idx = torch.from_numpy(np.stack([row, col]))
    E = [E0]
    for k in range(K):
        v = val * keep[k] if keep is not None else val
        Lk = torch.sparse_coo_tensor(idx, torch.from_numpy(v), (N, N)).coalesce()
        E.append(torch.sparse.mm(Lk, E[-1]))
    return E


def final_rows(L, user_w, item_w, K: int, keep=None):
    """[N, d] float64 layer mean over all rows; user_w / item_w are the tables (any float dtype, any device)."""
    E0 = torch.cat([user_w.double().cpu(), item_w.double().cpu()])
    E = layers(L, E0, K, keep)
    total = E[0]
    for e in E[1:]:
        total = total + e
    return total / (K + 1)


def batch_rows(F, n_user: int, u_id, pos, neg=None):
    """The forward's three outputs from the final rows F: users, positives, negatives (None without)."""
    u = F[torch.as_tensor(u_id).cpu()]
    p = F[n_user + torch.as_tensor(pos).cpu()]
    n = F[n_user + torch.as_tensor(neg).cpu()] if neg is not None else None
    return u, p, n
