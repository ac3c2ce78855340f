"""float64 torch restatement of XSimGCL (seoul_tourism_recommendation_ngcf_b200/lightgcn.py), used by the XSimGCL tests.

Noise (ngcf_perturb_rows): u_c = (hash64(key, row, col, layer, 'NOIS').x >> 8) * 2^-24 with hash64 restated from
csrc/common.cuh on top of ``tests._dropout_ref``'s ``mix`` and ``seed_words``, and E += eps * sign(E) * u / max(|u|, 1e-12).
The propagation takes sign(.) from the device's own post-noise layers when they are given: the noise never flips a
sign (u >= 0), but an fp32 value within rounding of zero may have another sign than its float64 counterpart.
InfoNCE is SELFRec's: rows normalized, logits cos / tau, -mean(diag(log_softmax)), over the table rows of the batch's
distinct ids (torch.unique).  Gradients come from torch autograd.  The product package never imports this module.
"""
import numpy as np
import torch
import torch.nn.functional as F

from tests._dropout_ref import M32, _u32, mix, seed_words
from tests._lightgcn_ref import coo_of

STREAM_NOISE = np.uint64(0x4E4F4953)       # 'NOIS'


def hash64_x(seed: int, a, b, c: int, stream=STREAM_NOISE):
    """ngcf_hash64(seed, a, b, c, stream).x for arrays a, b (uint64 arrays of 32-bit values)."""
    lo, hi = seed_words(seed)
    h = mix(_u32(a) ^ lo ^ stream)
    h = mix(h ^ ((_u32(b) + np.uint64(0x9E3779B9)) & M32) ^ hi)
    return mix((h + np.uint64((c * 0x632BE5AB) & 0xFFFFFFFF) + np.uint64(0x7F4A7C15)) & M32)


def uniforms(seed: int, n_rows: int, d: int, layer: int):
    """float64 [n_rows, d]: the noise's uniforms of `layer`, exactly (24-bit values)."""
    row = np.arange(n_rows, dtype=np.uint64)[:, None]
    col = np.arange(d, dtype=np.uint64)[None, :]
    h = hash64_x(seed, row, col, layer)
    return torch.from_numpy((h >> np.uint64(8)).astype(np.float64) * 2.0 ** -24)


def noise(sign_of, seed: int, layer: int, eps: float):
    """eps * sign(sign_of) * normalize(U) for the rows of sign_of ([N, d], any dtype): float64 [N, d]."""
    u = uniforms(seed, sign_of.shape[0], sign_of.shape[1], layer)
    u = u / u.norm(dim=1, keepdim=True).clamp(min=1e-12)
    return eps * torch.sign(sign_of.detach().double().cpu()) * u


def layers(L, E0, K: int, eps: float = 0.0, seed: int = 0, signs=None):
    """[E_0, ..., E_K] in float64 with the noise after every product (E0 used as given, so autograd reaches it).
    signs: the device's post-noise layers E_1..E_K (sign source), or None to take the float64 product's own signs."""
    row, col, val = coo_of(L)
    N = int(L.shape[0])
    Lk = torch.sparse_coo_tensor(torch.from_numpy(np.stack([row, col])), torch.from_numpy(val), (N, N)).coalesce()
    E = [E0]
    for k in range(K):
        X = torch.sparse.mm(Lk, E[-1])
        if eps > 0:
            X = X + noise(signs[k] if signs is not None else X, seed, k + 1, eps)
        E.append(X)
    return E


def final_rows(E):
    """mean(E_1 .. E_K): XSimGCL's readout (E_0 left out)."""
    total = E[1]
    for e in E[2:]:
        total = total + e
    return total / (len(E) - 1)


def info_nce(a, b, temperature: float):
    """SELFRec's InfoNCE(view1, view2, temperature) with b_cos=True."""
    a, b = F.normalize(a, dim=1), F.normalize(b, dim=1)
    return -torch.diag(F.log_softmax(a @ b.T / temperature, dim=1)).mean()


def cl_loss(Fr, V2, n_user: int, u_id, pos, temperature: float, cl_weight: float):
    """cl_weight * (InfoNCE over the distinct users + InfoNCE over the distinct positive items), on table rows."""
    u = torch.unique(torch.as_tensor(u_id).cpu())
    i = torch.unique(torch.as_tensor(pos).cpu()) + n_user
    return cl_weight * (info_nce(Fr[u], V2[u], temperature) + info_nce(Fr[i], V2[i], temperature))


def first_occurrences(ids):
    """Indices of the first occurrence of every distinct id, ascending by id (np.unique's return_index)."""
    return torch.from_numpy(np.unique(np.asarray(torch.as_tensor(ids).cpu()), return_index=True)[1])
