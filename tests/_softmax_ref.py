"""Float64 torch restatement of the in-batch sampled-softmax loss (ngcf_softmax_loss, include/ngcf_b200.h), masking
included, for the tests to compare against.  The product never imports this module."""
import torch


def mask(pos_ids, neg_ids, B, has_n, device=None):
    """[B, n_cols] bool, True = column kept for the row: j == i, or id(c_j) != pos_ids[i] (all True without ids)."""
    n_cols = 2 * B if has_n else B
    keep = torch.ones(B, n_cols, dtype=torch.bool, device=device)
    if pos_ids is None:
        return keep
    col_ids = torch.cat([pos_ids, neg_ids]) if has_n else pos_ids
    keep = col_ids[None, :].to(device) != pos_ids[:, None].to(device)
    keep.fill_diagonal_(True)                                          # the row's own positive column
    return keep


def loss(u, p, n, *, temperature, weight_decay, batch_size, pos_ids=None, neg_ids=None):
    """The loss as a differentiable float64 function of u, p, n (n: [B, D] or empty)."""
    u, p = u.double(), p.double()
    has_n = n.numel() > 0
    n = n.double() if has_n else None
    B = u.shape[0]
    cols = torch.cat([p, n]) if has_n else p
    s = u @ cols.T / temperature
    keep = mask(pos_ids, neg_ids, B, has_n, device=u.device)
    s_m = s.masked_fill(~keep, float("-inf"))
    lse = torch.logsumexp(s_m, dim=1)
    reg = (u * u).sum(1) + (p * p).sum(1) + ((n * n).sum(1) if has_n else 0.0)
    return (lse - s.diagonal() + weight_decay * reg).sum() / batch_size


def loss_and_grads(u, p, n, **kw):
    """(loss, gu, gp, gn) in float64 (gn None without negatives)."""
    ts = [t.detach().double().requires_grad_(True) for t in (u, p)]
    has_n = n.numel() > 0
    tn = n.detach().double().requires_grad_(True) if has_n else n
    val = loss(ts[0], ts[1], tn, **kw)
    grads = torch.autograd.grad(val, ts + ([tn] if has_n else []))
    return val.detach(), grads[0], grads[1], grads[2] if has_n else None
