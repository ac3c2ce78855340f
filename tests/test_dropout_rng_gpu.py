"""Every device-RNG dropout path against a host restatement of its decisions (tests/_dropout_ref.py).

Node dropout is evaluated inside the SpMM (``drop_p``), as per-step decision bytes (``keep_bits``) or as per-step
compacted survivor lists (``compact``, with static or coordinate-derived keys); message dropout inside the epilogues
of the tcgen05 and FFMA dense kernels, forward and backward, either hashed in the kernel or from precomputed bits.
Each is compared with a float64 product that uses the host's mask, so one wrong decision fails by far more than the
1e-5 bar.  The seeds have non-zero high words, one ``seed + *seed_dev`` carries across bit 32, row shards run with
their row offsets on one GPU, and the SpMM cases use 8 layers, which draw layers 4-7 from the second hash group.
"""
import numpy as np
import pytest
import torch

import seoul_tourism_recommendation_ngcf_b200 as pkg
from oracle import ngcf_oracle as O
from seoul_tourism_recommendation_ngcf_b200 import _lib, laplacian, synth
from seoul_tourism_recommendation_ngcf_b200.plan import LaplacianPlan, node_dropout_bits, node_dropout_compact, spmm
from seoul_tourism_recommendation_ngcf_b200.sharded import BalancedShards, RowShards
from tests import _dropout_ref as R
from tests._golden import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-4
K = 8                                       # NGCF_MAX_LAYERS: layers 4-7 come from the second hash group
N = 3001                                    # 3 equal shards of 1001 rows; no boundary a multiple of 4 or 128
COL_MASK = (1 << 27) - 1
# (p, host seed, device seed offset): high words set; the middle case carries from the low word into the high word
CASES = [(0.1, 0x6A09E667_F3BCC908, 0), (0.5, 0xA5A50001_FFFFFE00, 0x00000002_00000300),
         (0.9, 0x3C6EF372_FE94F82B, 0)]


def _check(got, want, tol=1e-5, what=""):
    """max|got - want| <= tol * max|want|; an all-zero reference (every entry dropped) must be matched exactly."""
    got = got.detach().cpu().double().numpy() if torch.is_tensor(got) else np.asarray(got, np.float64)
    want = want.numpy() if torch.is_tensor(want) else np.asarray(want, np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    scale = np.abs(want).max() if want.size else 0.0
    if scale == 0:
        assert np.all(got == 0), what
    else:
        err = np.abs(got - want).max() / scale
        assert err <= tol, (what, err)


def _seed_dev(off):
    return torch.tensor([off], dtype=torch.int64, device=DEV) if off else None


# ---- graph and plans ------------------------------------------------------------------------------------------
def _hub_graph():
    """Random COO graph (unsorted, with duplicates) with hub rows and hub columns of exactly split-threshold and
    split + 1 entries, and longer ones spread over the three equal row shards."""
    split = int(_lib.load().ngcf_spmm_split_threshold())
    rng = np.random.default_rng(2024)
    row_hubs = {7: 1000, 1500: split, 1501: split + 1, 2999: 300}
    col_hubs = {11: 700, 2000: split, 2001: split + 1}
    row, col = rng.integers(0, N, 24000), rng.integers(0, N, 24000)
    keep = ~np.isin(row, list(row_hubs)) & ~np.isin(col, list(col_hubs))
    row, col = row[keep], col[keep]
    free_rows = np.setdiff1d(np.arange(N), list(row_hubs))
    free_cols = np.setdiff1d(np.arange(N), list(col_hubs))
    rows, cols = [row, row[:60]], [col, col[:60]]                      # duplicated entries
    for h, cnt in row_hubs.items():
        rows.append(np.full(cnt, h)); cols.append(rng.choice(free_cols, cnt))
    for h, cnt in col_hubs.items():
        cols.append(np.full(cnt, h)); rows.append(rng.choice(free_rows, cnt))
    row, col = np.concatenate(rows), np.concatenate(cols)
    perm = rng.permutation(row.size)
    row, col = row[perm], col[perm]
    assert all((row == h).sum() == c for h, c in row_hubs.items()) and all((col == h).sum() == c for h, c in col_hubs.items())
    val = rng.standard_normal(row.size).astype(np.float32)
    return torch.sparse_coo_tensor(torch.from_numpy(np.stack([row, col])), torch.from_numpy(val), (N, N))


@pytest.fixture(scope="module")
def graph():
    L = _hub_graph()
    idx = L._indices().numpy()
    X = torch.randn(N + 2, 65, generator=torch.Generator().manual_seed(3))      # N_pad = 3003 rows for RowShards
    X64 = X[:, :64].contiguous()
    Xd = X[:N].double()
    # float64 references of the masked products, per (case, layer): L_k X and L_k^T X
    ref = {}
    for ci, (p, seed, off) in enumerate(CASES):
        keep = R.edge_keep(seed + off, p, K, idx[0], idx[1])
        for k in range(K):
            m = torch.from_numpy(keep[k])
            Lk = torch.sparse_coo_tensor(L._indices()[:, m], L._values()[m].double(), (N, N))
            ref[ci, k] = (torch.sparse.mm(Lk, Xd), torch.sparse.mm(Lk.t().coalesce(), Xd))
    return dict(L=L, row=idx[0], col=idx[1], X={64: X64.to(DEV), 65: X.to(DEV)}, ref=ref)


def _shards():
    out = [None] + [RowShards(N, 3, r) for r in range(3)]
    starts = [0, 997, 2011, N]
    out += [BalancedShards(N, 3, r, starts) for r in range(3)]
    return out


def _shard_id(sh):
    return "full" if sh is None else f"{type(sh).__name__}-{sh.rank}"


@pytest.fixture(scope="module")
def plans(graph):
    return {_shard_id(sh): (sh, LaplacianPlan(graph["L"], DEV, shard=sh)) for sh in _shards()}


def _entry_coords(side, r0):
    """Global (row, col) of every entry of a CSR side in execution order (ent, then hub_ent), from its own layout."""
    rp = side.rowptr.cpu().numpy().astype(np.int64)
    rows = np.repeat(np.arange(side.n_rows), np.diff(rp))
    if side.n_chunks:
        cp = side.chunk_ptr.cpu().numpy().astype(np.int64)
        rows = np.concatenate([rows, np.repeat(side.chunk_row.cpu().numpy(), np.diff(cp))])
    cols = side.ent[:side.nnz, 0].cpu().numpy().astype(np.int64) & COL_MASK
    return rows + r0, cols


def _sides(plan):
    """(CSR side, whether it holds L^T): L's row block and L^T's row block."""
    return [(plan.fwd, False), (plan.bwd, True)]


# ---- the restatement pinned to the device, byte for byte ---------------------------------------------------------
@pytest.mark.parametrize("sid", [_shard_id(sh) for sh in _shards()])
def test_entry_keys_and_decision_bytes_equal_restatement(graph, plans, sid):
    sh, plan = plans[sid]
    r0 = sh.r0 if sh is not None else 0
    assert plan.fwd.n_hub >= 1 or plan.bwd.n_hub >= 1
    for side, transposed in _sides(plan):
        r, c = _entry_coords(side, r0)
        # the layout's coordinates are the COO entries' (for L^T's CSR: swapped), through the permutation
        perm = side.perm.cpu().numpy().astype(np.int64)
        lr, lc = (graph["col"], graph["row"]) if transposed else (graph["row"], graph["col"])
        assert np.array_equal(r, lr[perm]) and np.array_equal(c, lc[perm])
        side.ensure_keys(r0)
        kl = side.key_l[:side.nnz].cpu().numpy().view(np.uint32)
        kt = side.key_t[:side.nnz].cpu().numpy().view(np.uint32)
        assert np.array_equal(kl, R.node_key(r, c)) and np.array_equal(kt, R.node_key(c, r))
        for p, seed, off in CASES:
            bl, bt = node_dropout_bits(side, p, seed, _seed_dev(off), K, r0, as_L=True, as_Lt=True)
            assert np.array_equal(bl.cpu().numpy(), R.node_keep_bits(seed + off, p, K, r, c)), (p, transposed)
            assert np.array_equal(bt.cpu().numpy(), R.node_keep_bits(seed + off, p, K, c, r)), (p, transposed)


@pytest.mark.parametrize("d_out", [16, 64, 96, 128])
def test_message_dropout_bits_equal_restatement(d_out):
    lib = _lib.load()
    for (p, seed, off), (n, r0) in zip(CASES, [(1, 1 << 30), (4321, 1001), (129, 0)]):
        for layer in (0, 5):
            words = (d_out + 31) // 32
            bits = torch.full((n * words,), -1, dtype=torch.int32, device=DEV)
            sd = _seed_dev(off)
            _lib.check(lib.ngcf_mess_dropout_bits(n, d_out, p, seed, _lib.ptr(sd), layer, r0, bits.data_ptr(),
                                                  _lib.current_stream()), "mess_dropout_bits")
            want = R.pack_mess_bits(R.mess_keep(seed + off, p, layer, n, d_out, r0))
            assert np.array_equal(bits.cpu().numpy().reshape(n, words), want), (p, layer, n, r0)


# ---- SpMM with node dropout against float64 products of the host-masked L ------------------------------------------
@pytest.mark.parametrize("sid", [_shard_id(sh) for sh in _shards()])
@pytest.mark.parametrize("d", [64, 65])
def test_spmm_node_dropout_vs_float64(graph, plans, sid, d):
    sh, plan = plans[sid]
    r0, valid = (sh.r0, sh.valid) if sh is not None else (0, N)
    X = graph["X"][d]
    for ci, (p, seed, off) in enumerate(CASES):
        sd = _seed_dev(off)
        for side, transposed in _sides(plan):
            lrow, lcol = _entry_coords(side, r0)
            if transposed:
                lrow, lcol = lcol, lrow                           # this CSR holds L^T: entry (r, c) is (c, r) of L
            host_bits = R.node_keep_bits(seed + off, p, K, lrow, lcol)
            bl, bt = node_dropout_bits(side, p, seed, sd, K, r0, as_L=not transposed, as_Lt=transposed)
            bits = bt if transposed else bl
            outs = {}
            for k in range(K):
                outs["inkernel", k] = spmm(side, None, X, d, drop_p=p, seed=seed, seed_dev=sd, layer=k,
                                           transposed=transposed, row_offset=r0)
                outs["bits", k] = spmm(side, None, X, d, layer=k, transposed=transposed, row_offset=r0, keep_bits=bits)
            if d % 4 == 0:                                        # compacted survivors: streaming kernel only
                for static in (True, False):
                    cl, ct = node_dropout_compact(side, p, seed, sd, K, r0, as_L=not transposed, as_Lt=transposed,
                                                  static_keys=static)
                    comp = ct if transposed else cl
                    _check_compaction(side, comp, host_bits)
                    for k in range(K):
                        outs[("compact", static), k] = spmm(side, None, X, d, transposed=transposed, row_offset=r0,
                                                            compact=comp[k])
            for (mode, k), got in outs.items():
                want = graph["ref"][ci, k][1 if transposed else 0][r0:r0 + valid, :d]
                what = (mode, k, p, transposed)
                _check(got[:valid], want, what=what)
                if valid < got.shape[0]:                          # padding rows of the last equal shard
                    assert float(got[valid:].abs().max()) == 0.0, what


def _check_compaction(side, comp, host_bits):
    """Per tile and layer: the count equals the host's survivors, and the survivors are the tile's entries in order."""
    tiles = [(side.tiles.cpu().numpy(), 0)]
    if side.n_chunks:
        tiles.append((side.chunk_tiles.cpu().numpy(), side.nnz_short))
    ent = side.ent[:side.nnz].cpu().numpy()
    for k, (c_ent, c_cnt) in enumerate(comp):
        keep = ((host_bits >> np.uint64(k)) & np.uint64(1)).astype(bool)
        cnt, c_ent = c_cnt.cpu().numpy(), c_ent.cpu().numpy()
        t_base = 0
        for tl, e_base in tiles:
            for t, (_, _, e0, e1) in enumerate(tl):
                e0, e1 = e0 + e_base, e1 + e_base
                n = int(keep[e0:e1].sum())
                assert cnt[t_base + t] == n, (k, t_base + t)
                assert np.array_equal(c_ent[e0:e0 + n], ent[e0:e1][keep[e0:e1]]), (k, t_base + t)
            t_base += len(tl)


# ---- dense layers with device message dropout against the float64 restatement -------------------------------------
def _fwd64(S, E, W1, b1, W2, b2, mult):
    """Per-layer epilogue (NGCF.py:131-142) in float64, as test_dense_forward_vs_float64 states it."""
    Sd, Ed = S.double(), E.double()
    M = (Sd + Ed) @ W1.double().T + (Sd * Ed) @ W2.double().T + 2 * b1.double() + b2.double()
    return torch.where(M > 0, M, 0.2 * M) * mult.double()


def _bwd64(S, E, W1, W2, E_out, gE_next, mult, rows, gsum, col_off, normalized):
    """Row-local backward of one layer in float64, as test_dense_backward_vs_float64 states it; ``normalized``: gsum
    already holds the normalize-backwarded row gradients (gh_normalized = 1)."""
    N, d_out = E_out.shape
    Eo, Sd, Ed = E_out.double(), S.double(), E.double()
    gH = torch.zeros(N, d_out, dtype=torch.float64)
    gH[rows] = gsum[:, col_off:col_off + d_out].double()
    if normalized:
        gEp = gE_next.double() + gH
    else:
        n = Eo.norm(dim=1, keepdim=True).clamp_min(1e-12)
        H = Eo / n
        gEp = gE_next.double() + (gH - H * (H * gH).sum(1, keepdim=True)) / n
    gM = gEp * mult.double() * torch.where(Eo > 0, 1.0, 0.2)
    T1, T2 = gM @ W1.double(), gM @ W2.double()
    return dict(gS=T1 + T2 * Ed, gEl=T1 + T2 * Sd, gW1=gM.T @ (Sd + Ed), gW2=gM.T @ (Sd * Ed), gb1=2 * gM.sum(0),
                gb2=gM.sum(0))


# every (d_in, d_out) the tcgen05 dispatch takes (ngcf_dense_fwd_tc_eligible / ngcf_dense_bwd_tc_eligible; 128-wide
# sides run as 64-wide blocks, a 128-wide backward d_out with gh_normalized = 1), then FFMA-only pairs
FWD_TC = [(i, o) for i in (32, 64, 128) for o in (16, 32, 48, 64, 128)]
BWD_TC = [(64, 32), (64, 64), (64, 128), (128, 64), (128, 128)]
FFMA = [(65, 64), (64, 65), (20, 36)]
# (N, row_offset, p, seed, device seed offset): every pair meets non-zero offsets and partial last 128-row tiles;
# 2^30 rows * d_out >= 2^36 elements, so the quad index needs its high word
DENSE_CASES = [(129, 1001, 0.3, 0x9B05688C_2B3E6C1F, 0), (4321, 1 << 30, 0.25, 0xA5A50001_FFFFFE00, 0x2_00000300),
               (1, 1 << 30, 0.5, 0x1F83D9AB_FB41BD6B, 0), (127, 0, 0.6, 0x5BE0CD19_137E2179, 0)]


def _dense_inputs(N, d_in, d_out, seed):
    g = torch.Generator().manual_seed(seed)
    t = dict(S=torch.randn(N, d_in, generator=g), E=torch.randn(N, d_in, generator=g),
             W1=torch.randn(d_out, d_in, generator=g) * 0.2, W2=torch.randn(d_out, d_in, generator=g) * 0.2,
             b1=torch.randn(d_out, generator=g), b2=torch.randn(d_out, generator=g),
             E_out=torch.randn(N, d_out, generator=g), gE_next=torch.randn(N, d_out, generator=g))
    n_slot = max(1, min(N // 3, 700))
    t["rows"] = torch.randperm(N, generator=g)[:n_slot]
    slot = torch.full((N,), -1, dtype=torch.int32)
    slot[t["rows"]] = torch.arange(n_slot, dtype=torch.int32)
    t["slot"] = slot
    t["gsum"] = torch.randn(n_slot, d_out + 24, generator=g)
    return t


def _mess_modes(d_out, p, seed, layer, N, r0):
    """(name, mess_bits device tensor or None): in-kernel hash, and the host's decisions packed as bits."""
    modes = [("hash", None)]
    if d_out % 4 == 0:                                            # ngcf_mess_dropout_bits' widths
        bits = R.pack_mess_bits(R.mess_keep(seed, p, layer, N, d_out, r0))
        modes.append(("bits", torch.from_numpy(bits.reshape(-1).copy()).to(DEV)))
    return modes


@pytest.mark.parametrize("d_in,d_out", FWD_TC + FFMA)
def test_dense_forward_device_dropout_vs_float64(d_in, d_out):
    lib = _lib.load()
    st = _lib.current_stream()
    for ci, (n, r0, p, seed, off) in enumerate(DENSE_CASES):
        t = _dense_inputs(n, d_in, d_out, n + d_in * 7 + d_out)
        layer = (ci + d_out) % K
        mult = torch.from_numpy(R.mess_mult(seed + off, p, layer, n, d_out, r0))
        want = _fwd64(t["S"], t["E"], t["W1"], t["b1"], t["W2"], t["b2"], mult)
        d = {k: v.to(DEV).contiguous() for k, v in t.items()}
        wcat = torch.empty(2 * d_in * d_out, device=DEV)
        bias = torch.empty(d_out, device=DEV)
        _lib.check(lib.ngcf_pack_weights(d["W1"].data_ptr(), d["b1"].data_ptr(), d["W2"].data_ptr(), d["b2"].data_ptr(),
                                         d_in, d_out, wcat.data_ptr(), bias.data_ptr(), st), "pack_weights")
        sd = _seed_dev(off)
        for mode, bits in _mess_modes(d_out, p, seed + off, layer, n, r0):
            out = torch.full((n, d_out), float("nan"), device=DEV)
            _lib.check(lib.ngcf_dense_fwd(d["S"].data_ptr(), d["E"].data_ptr(), n, d_in, d_out, wcat.data_ptr(),
                                          bias.data_ptr(), 0.2, None, _lib.ptr(bits), p, seed, _lib.ptr(sd), layer, r0,
                                          out.data_ptr(), st), "dense_fwd")
            _check(out, want, 1e-5, (mode, n, r0, layer))


@pytest.mark.parametrize("d_in,d_out", BWD_TC + FFMA)
def test_dense_backward_device_dropout_vs_float64(d_in, d_out):
    lib = _lib.load()
    st = _lib.current_stream()
    normalized = int(d_out == 128)                                # a blocked d_out needs gh_normalized
    col_off = 8
    for ci, (n, r0, p, seed, off) in enumerate(DENSE_CASES):
        t = _dense_inputs(n, d_in, d_out, n + d_in + d_out * 5)
        layer = (ci + d_in) % K
        mult = torch.from_numpy(R.mess_mult(seed + off, p, layer, n, d_out, r0))
        want = _bwd64(t["S"], t["E"], t["W1"], t["W2"], t["E_out"], t["gE_next"], mult, t["rows"], t["gsum"], col_off,
                      normalized)
        d = {k: v.to(DEV).contiguous() for k, v in t.items()}
        sd = _seed_dev(off)
        for mode, bits in _mess_modes(d_out, p, seed + off, layer, n, r0):
            gS, gEl = torch.full((n, d_in), float("nan"), device=DEV), torch.full((n, d_in), float("nan"), device=DEV)
            gW1, gW2 = torch.zeros(d_out, d_in, device=DEV), torch.zeros(d_out, d_in, device=DEV)
            gb1, gb2 = torch.zeros(d_out, device=DEV), torch.zeros(d_out, device=DEV)
            scratch = torch.empty(n, d_out, device=DEV)
            _lib.check(lib.ngcf_dense_bwd(d["gE_next"].data_ptr(), d["slot"].data_ptr(), d["gsum"].data_ptr(),
                                          d_out + 24, col_off, d["E_out"].data_ptr(), d["S"].data_ptr(), d["E"].data_ptr(),
                                          n, d_in, d_out, d["W1"].data_ptr(), d["W2"].data_ptr(), 0.2, None,
                                          _lib.ptr(bits), p, seed, _lib.ptr(sd), layer, r0, normalized, gS.data_ptr(),
                                          gEl.data_ptr(), gW1.data_ptr(), gb1.data_ptr(), gW2.data_ptr(), gb2.data_ptr(),
                                          scratch.data_ptr(), st), "dense_bwd")
            got = dict(gS=gS, gEl=gEl, gW1=gW1, gW2=gW2, gb1=gb1, gb2=gb2)
            for k in want:
                _check(got[k], want[k], 2e-5, (k, mode, n, r0, layer))


# ---- one eager training step per node-dropout mode, against the CPU oracle given the host's masks ------------------
MODELS = {"A": [64, 32, 128, 48, 64],                 # every width a multiple of 4: compacted survivor lists apply
          "B": [48, 16, 65, 64, 32, 64]}              # width 65: per-step decision bytes and FFMA kernels
STEP_CASES = [("A", mode, mb) for mode in ("compact", "bits", "inkernel") for mb in (False, True)] + \
             [("B", mode, mb) for mode in ("bits", "inkernel") for mb in (False, True)]


@pytest.fixture(scope="module")
def step_graph():
    n_user, n_item, B = 700, 500, 256
    u, i, r = synth.powerlaw_bipartite(n_user, n_item, 30000, seed=9)
    L = laplacian.laplacian_coo(u, i, r, n_user, n_item)
    b = {k: torch.from_numpy(v) for k, v in synth.random_batch(n_user, n_item, B, seed=4).items()}
    return n_user, n_item, B, L, b


@pytest.mark.parametrize("model,node_mode,mess_bits", STEP_CASES)
def test_training_step_device_dropout_vs_host_masks(step_graph, model, node_mode, mess_bits):
    n_user, n_item, B, L, b = step_graph
    layers = MODELS[model]
    nK, N_ = len(layers), n_user + n_item
    node_p, mess_p = 0.3, 0.2
    torch.manual_seed(0)
    m = pkg.NGCF(64, layers, node_p, [mess_p] * nK, 1.0, [L, L], synth.num_dict_for(n_user, n_item), B,
                 torch.device("cpu"))
    params = {k: v.detach().clone() for k, v in m.state_dict().items()}
    m = m.to(DEV)
    m._node_mode, m._mess_bits = node_mode, mess_bits
    m.train()
    torch.manual_seed(77)
    d = {k: v.to(DEV) for k, v in b.items()}
    uu, pp, nn_ = m(year=d["year"], u_id=d["u_id"], age=d["age"], sex=d["sex"], month=d["month"], day=d["day"],
                    dow=d["dow"], pos_item=d["pos_item"], neg_item=d["neg_item"], node_flag=True)
    all_u, all_i = m.all_users_emb.clone(), m.all_items_emb.clone()
    loss = pkg.BPR(0.025, B)(uu, pp, nn_)
    loss.backward()
    st = m._last
    assert st.node_mode == node_mode and st.drop_p == pytest.approx(node_p) and st.plan.fwd.n_hub > 0
    assert [x is not None for x in st.mess_bits] == [mess_bits and w % 4 == 0 for w in layers]
    idx = L._indices().numpy()
    keep = R.edge_keep(st.seed, node_p, nK, idx[0], idx[1])
    mult = [torch.from_numpy(R.mess_mult(st.seed, mess_p, k, N_, layers[k])) for k in range(nK)]
    loss_ref, grads_ref, mid = O.train_step(params, L, b, emb_ratio=1.0, weight_decay=0.025, batch_size_ctor=B,
                                            edge_keep=keep, mess_mult=mult)
    for got, want in ((uu, mid["u"]), (pp, mid["pos"]), (nn_, mid["neg"]),
                      (all_u, mid["out"]["all_E"][:n_user]), (all_i, mid["out"]["all_E"][n_user:])):
        assert rel_err(got.detach().cpu().numpy(), want.detach().numpy()) <= TOL
    assert abs(float(loss) - float(loss_ref)) <= TOL * abs(float(loss_ref))
    named = dict(m.named_parameters())
    for k, gr in grads_ref.items():
        if gr is None:
            assert named[k].grad is None, k
        else:
            assert rel_err(named[k].grad.cpu().numpy(), gr.numpy()) <= TOL, k
