"""Every ngcf_spmm path and operand form against a float64 product (the contract in include/ngcf_b200.h).

One non-symmetric random graph with duplicates carries every structural edge the kernels special-case: empty rows and
columns, rows of exactly split and split + 1 entries, a tile whose 16 rows are all hubs, a hub in the last row, and a
hub row and a hub column of more than 512 chunks (hub_finish_kernel's 4-deep loop at G = 1).  Each product runs as L
and as L^T, at widths that take every branch of launch_any (the scalar kernel and G = 1, 2, 4, 8, 16, 32, with full
and partial last lane groups), with plain, out-of-place, in-place, strided and misaligned operands and with the
slot/gsum row addend of the backward's last product.  After every call: the inputs are unchanged, the hub counters are
back at zero, and a repeated call is bitwise identical.  Node dropout (all three device modes and an explicit COO mask)
meets the same operands at layers 0 and 7 of p = 0.9; the vector row-per-warp kernel, CUDA-graph replay and the
index limits (27-bit column ids, the 32-bit byte stride of the gathers) have tests of their own.
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from seoul_tourism_recommendation_ngcf_b200 import _lib
from seoul_tourism_recommendation_ngcf_b200.plan import (LaplacianPlan, greedy_tiles, node_dropout_bits,
                                                         node_dropout_compact, spmm)
from tests import _dropout_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
N = 4093                                    # not a multiple of the 16-row tile
K = 8                                       # NGCF_MAX_LAYERS
BIG_ROW, ROW_SPLIT, ROW_SPLIT1, LAST = 5, 777, 778, N - 1
BIG_COL, COL_SPLIT, COL_SPLIT1, COL_HUB = 9, 1234, 1235, 3001
REG = range(2048, 2048 + 48)                # no ordinary entries: 16 of these rows become the all-hub tile
EMPTY_ROWS = [1, 1999, N - 2]
EMPTY_COLS = [2, 600, N - 3]


def _check(got, want, what=""):
    """max|got - want| <= 1e-5 * max|want|; an all-zero reference must be matched exactly."""
    got = got.detach().cpu().double().numpy() if torch.is_tensor(got) else np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    scale = np.abs(want).max() if want.size else 0.0
    if scale == 0:
        assert np.all(got == 0), what
    else:
        err = np.abs(got - want).max() / scale
        assert err <= 1e-5, (what, err)


def _lib_sizes():
    lib = _lib.load()
    return lib.ngcf_spmm_split_threshold(), lib.ngcf_spmm_tile_rows(), lib.ngcf_spmm_tile_entries()


def _hub_graph():
    split, tr, te = _lib_sizes()
    big = 4 * 128 * split + 38 * split + 7              # 551 chunks: > 4 * (128 threads / G = 1) of hub_finish_kernel
    rng = np.random.default_rng(2025)
    row_hubs = {BIG_ROW: big, ROW_SPLIT: split, ROW_SPLIT1: split + 1, LAST: 300}
    col_hubs = {BIG_COL: big, COL_SPLIT: split, COL_SPLIT1: split + 1, COL_HUB: 400}
    free_rows = np.setdiff1d(np.arange(N), list(row_hubs) + list(REG) + EMPTY_ROWS)
    free_cols = np.setdiff1d(np.arange(N), list(col_hubs) + EMPTY_COLS)
    row, col = rng.choice(free_rows, 30000), rng.choice(free_cols, 30000)
    rows, cols = [row, row[:300]], [col, col[:300]]                 # duplicated entries
    for h, cnt in row_hubs.items():
        rows.append(np.full(cnt, h)); cols.append(rng.choice(free_cols, cnt))
    for h, cnt in col_hubs.items():
        cols.append(np.full(cnt, h)); rows.append(rng.choice(free_rows, cnt))
    # the row CSR holds no hub entries, so its tiles are known before the hub block is placed: 16 rows of REG that
    # start a tile become hubs
    deg = np.bincount(np.concatenate(rows), minlength=N)
    rp = np.concatenate([[0], np.cumsum(np.where(deg > split, 0, deg))])
    starts = greedy_tiles(rp, tr, te)[:, 0]
    r0 = int(starts[(starts >= REG[0]) & (starts + tr <= REG[-1] + 1)][0])
    block = list(range(r0, r0 + tr))
    for i, h in enumerate(block):
        rows.append(np.full(split + 1 + 13 * i, h)); cols.append(rng.choice(free_cols, split + 1 + 13 * i))
    row, col = np.concatenate(rows), np.concatenate(cols)
    perm = rng.permutation(row.size)
    row, col = row[perm], col[perm]
    val = rng.standard_normal(row.size).astype(np.float32)
    return row, col, val, block


@pytest.fixture(scope="module")
def g():
    split, tr, _ = _lib_sizes()
    row, col, val, block = _hub_graph()
    L = torch.sparse_coo_tensor(torch.from_numpy(np.stack([row, col])), torch.from_numpy(val), (N, N))
    A = sp.csr_matrix((val.astype(np.float64), (row, col)), shape=(N, N))      # duplicates summed
    plan = LaplacianPlan(L, DEV)
    assert not plan.symmetric and N % tr != 0
    # the structure this file relies on, asserted on the built plan
    rdeg, cdeg = np.bincount(row, minlength=N), np.bincount(col, minlength=N)
    assert rdeg[ROW_SPLIT] == split and rdeg[ROW_SPLIT1] == split + 1
    assert cdeg[COL_SPLIT] == split and cdeg[COL_SPLIT1] == split + 1
    assert np.all(rdeg[EMPTY_ROWS] == 0) and np.all(cdeg[EMPTY_COLS] == 0)
    for side, hubs, empty in ((plan.fwd, [BIG_ROW, ROW_SPLIT1, LAST] + block, EMPTY_ROWS),
                              (plan.bwd, [BIG_COL, COL_SPLIT1, COL_HUB], EMPTY_COLS)):
        hub_of = side.hub_of_row.cpu().numpy()
        assert sorted(np.nonzero(hub_of >= 0)[0].tolist()) == sorted(hubs)
        assert np.diff(side.hub_chunk_ptr.cpu().numpy()).max() > 4 * 128
        assert np.all(np.diff(side.rowptr.cpu().numpy())[empty] == 0) and np.all(hub_of[empty] < 0)
    mask = plan.fwd.tile_hubmask.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    full = np.nonzero(mask == (1 << tr) - 1)[0]
    assert full.size == 1 and plan.fwd.tiles[int(full[0]), 0].item() == block[0]
    assert (mask[-1] >> (N - 1 - plan.fwd.tiles[-1, 0].item())) & 1          # the hub in the last row
    # rows that get a gsum row: hubs of L and of L^T, the all-hub tile, empty rows, the last row, ordinary rows
    rng = np.random.default_rng(5)
    special = [BIG_ROW, ROW_SPLIT, ROW_SPLIT1, LAST, BIG_COL, COL_SPLIT, COL_SPLIT1, COL_HUB, REG[-1]]
    special += block + EMPTY_ROWS + EMPTY_COLS
    others = rng.choice(np.setdiff1d(np.arange(N), special), 60, replace=False).tolist()
    slot_rows = np.array(special + others)
    n_gs = slot_rows.size + 7
    slot = np.full(N, -1, dtype=np.int32)
    slot[slot_rows] = rng.permutation(n_gs)[:slot_rows.size]
    gen = torch.Generator().manual_seed(11)
    return dict(plan=plan, row=row, col=col, val=val, A={False: A, True: A.T.tocsr()}, block=block,
                X=torch.randn(N, 128, generator=gen), ADD=torch.randn(N, 128, generator=gen),
                GS=torch.randn(n_gs, 128 + 24, generator=gen), slot=torch.from_numpy(slot))


def _ceil4(x):
    return (x + 3) // 4 * 4


class Ops:
    """The operands of one product and what the reference needs of them.  ``ybuf`` is the storage of Y (Y may be a
    column slice of it); ``reset`` refills it (NaN, or the addend for an in-place addend)."""

    def __init__(self, g, d, form, with_slot=None):
        self.d, self.form = d, form
        Xh = g["X"][:, :d]
        self.pad = None
        if form == "strided":
            ldx = _ceil4(d) + 12
            xb = torch.zeros(N, ldx)
            xb[:, 4:4 + d] = Xh
            self.X = xb.to(DEV)[:, 4:4 + d]
        elif form == "misaligned":
            flat = torch.empty(N * d + 1, device=DEV)
            flat[1:] = Xh.reshape(-1).to(DEV)
            self.X = flat[1:].view(N, d)
            assert self.X.data_ptr() % 16 != 0
        else:
            self.X = Xh.contiguous().to(DEV)
        # Y
        if form == "strided":
            ldy = _ceil4(d) + 8
            self.ybuf = torch.full((N, ldy), float("nan"), device=DEV)
            self.c0 = 4
            self.Y = self.ybuf[:, 4:4 + d]
            self.pad = torch.ones(ldy, dtype=torch.bool, device=DEV)
            self.pad[4:4 + d] = False
        else:
            self.ybuf = torch.full((N, d), float("nan"), device=DEV)
            self.c0 = 0
            self.Y = self.ybuf
        self.y_init = torch.full_like(self.ybuf, float("nan"))
        # addend
        self.add_h = None
        self.addend = None
        if form in ("add_out", "add_in", "strided", "misaligned", "bwd_last"):
            self.add_h = g["ADD"][:, :d]
            if form in ("add_in", "bwd_last"):
                self.addend = self.Y
                self.y_init[:, self.c0:self.c0 + d] = self.add_h.to(DEV)
            elif form == "strided":
                lda = _ceil4(d) + 16
                ab = torch.zeros(N, lda)
                ab[:, 8:8 + d] = self.add_h
                self.addend = ab.to(DEV)[:, 8:8 + d]
            else:
                self.addend = self.add_h.contiguous().to(DEV)
        # slot / gsum: d + 24 floats per gsum row, as NGCF passes the D-wide concat rows and reads d of them
        self.slot = self.gsum = None
        self.gs_rows = None
        if with_slot is None:
            with_slot = form in ("slot", "misaligned", "bwd_last")
        if with_slot:
            gsum_col = 0 if form == "slot" else 8                  # a gsum view that starts at column 8
            gb = g["GS"][:, :d + 24].contiguous().to(DEV)
            self.gsum = gb[:, gsum_col:]
            self.slot = g["slot"].to(DEV)
            s = g["slot"].numpy()
            self.gs_rows = np.zeros((N, d))
            self.gs_rows[s >= 0] = g["GS"][:, gsum_col:gsum_col + d].double().numpy()[s[s >= 0]]
        self.guards = [(t, t.clone()) for t in (self.X, self.gsum, self.slot) if t is not None]
        if self.addend is not None and self.addend is not self.Y:
            self.guards.append((self.addend, self.addend.clone()))

    def reset(self):
        self.ybuf.copy_(self.y_init)

    def empty_value(self):
        """float32 value of a row whose product is empty: addend + gsum row, rounded once."""
        a = self.add_h.clone() if self.add_h is not None else torch.zeros(N, self.d)
        if self.gs_rows is not None:
            a = a + torch.from_numpy(self.gs_rows).float()
        return a


def _bits(t):
    return t.contiguous().view(torch.int32)


def _run(ops, side, transposed, ent=None, **kw):
    """Calls the product twice and checks the call's invariants; returns Y."""
    def call():
        ops.reset()
        spmm(side, ent, ops.X, ops.d, out=ops.Y, addend=ops.addend, slot=ops.slot, gsum=ops.gsum,
             transposed=transposed, **kw)
        return ops.ybuf.clone()

    first = call()
    what = (ops.form, ops.d, transposed)
    if side.hub_done is not None:
        assert int(torch.count_nonzero(side.hub_done)) == 0, what
    for t, t0 in ops.guards:
        assert torch.equal(_bits(t), _bits(t0)), what
    second = call()
    assert torch.equal(_bits(first), _bits(second)), ("repeat", what)
    if ops.pad is not None:                                       # nothing written past column d
        assert torch.equal(_bits(first[:, ops.pad]), _bits(ops.y_init[:, ops.pad])), what
    return first[:, ops.c0:ops.c0 + ops.d]


def _want(P, ops):
    w = P @ ops.X.cpu().double().numpy()
    if ops.add_h is not None:
        w = w + ops.add_h.double().numpy()
    if ops.gs_rows is not None:
        w = w + ops.gs_rows
    return w


def _compare(got, P, ops, what):
    _check(got, _want(P, ops), what)
    empty = np.nonzero(P.getnnz(axis=1) == 0)[0]
    assert empty.size > 0
    e = torch.from_numpy(empty)
    assert torch.equal(got.cpu()[e], ops.empty_value()[e]), ("empty rows", what)


def _side(g, transposed):
    plan = g["plan"]
    return plan.bwd if transposed else plan.fwd


# ---- every width, operand form and direction ------------------------------------------------------------------------
WIDTHS = [1, 3, 4, 8, 12, 16, 20, 32, 36, 64, 65, 100, 127, 128]
FULL = (4, 8, 64, 65, 128)
FORMS = ["plain", "add_out", "add_in", "slot", "strided", "misaligned", "bwd_last"]
CASES = [(d, f) for d in WIDTHS for f in FORMS if d in FULL or f in ("plain", "slot", "misaligned")]


@pytest.mark.parametrize("d,form", CASES)
def test_spmm_operand_forms_vs_float64(g, d, form):
    for transposed in (False, True):
        side = _side(g, transposed)
        ops = Ops(g, d, form)
        got = _run(ops, side, transposed)
        _compare(got, g["A"][transposed], ops, (form, d, transposed))
        if form in ("add_in", "bwd_last"):                        # the same addend out of place: bitwise equal
            out = Ops(g, d, form)
            out.addend = out.add_h.contiguous().to(DEV)
            out.y_init.fill_(float("nan"))
            out.guards.append((out.addend, out.addend.clone()))
            assert torch.equal(_bits(_run(out, side, transposed)), _bits(got)), (form, d, transposed)


# ---- node dropout on the backward's last product --------------------------------------------------------------------
P_DROP, SEED, SEED_OFF = 0.9, 0x3C6EF372_FE94F82B, 0x00000002_00000300


@pytest.mark.parametrize("d", [64, 65])
def test_spmm_node_dropout_with_addend_and_slot_vs_float64(g, d):
    plan = g["plan"]
    sd = torch.tensor([SEED_OFF], dtype=torch.int64, device=DEV)
    keep = R.edge_keep(SEED + SEED_OFF, P_DROP, K, g["row"], g["col"])
    for transposed in (False, True):
        side = _side(g, transposed)
        bl, bt = node_dropout_bits(side, P_DROP, SEED, sd, K, 0, as_L=not transposed, as_Lt=transposed)
        bits = bt if transposed else bl
        comp = None
        if d % 4 == 0:
            cl, ct = node_dropout_compact(side, P_DROP, SEED, sd, K, 0, as_L=not transposed, as_Lt=transposed)
            comp = ct if transposed else cl
        for k in (0, 7):
            m = keep[k]
            P = sp.csr_matrix((g["val"][m].astype(np.float64), (g["row"][m], g["col"][m])), shape=(N, N))
            if transposed:
                P = P.T.tocsr()
            modes = {"inkernel": dict(drop_p=P_DROP, seed=SEED, seed_dev=sd, layer=k),
                     "bits": dict(keep_bits=bits, layer=k),
                     "reference": dict(ent=plan.entries(side, torch.from_numpy(m.astype(np.uint8)).to(DEV)))}
            if comp is not None:
                modes["compact"] = dict(compact=comp[k])
            for mode, kw in modes.items():
                ops = Ops(g, d, "bwd_last")
                got = _run(ops, side, transposed, **kw)
                _compare(got, P, ops, (mode, k, d, transposed))


# ---- the vector row-per-warp kernel: hubs without the streaming kernel's per-tile hub masks -------------------------
@pytest.mark.parametrize("d", [8, 64, 128])
def test_spmm_vector_row_per_warp_kernel_vs_float64(g, d):
    for transposed in (False, True):
        side = _side(g, transposed)
        saved = side.tile_hubmask
        side.tile_hubmask = None                                  # descriptor without tile_hubmask: spmm_tile_kernel<G>
        side._struct_cache.clear()
        try:
            for form in ("bwd_last", "strided"):                  # in-place addend; strided out-of-place addend
                ops = Ops(g, d, form, with_slot=True)
                got = _run(ops, side, transposed)
                _compare(got, g["A"][transposed], ops, ("rows", form, d, transposed))
        finally:
            side.tile_hubmask = saved
            side._struct_cache.clear()


# ---- CUDA graph replay ----------------------------------------------------------------------------------------------
def test_spmm_graph_replay_matches_eager(g):
    plan = g["plan"]
    cl, _ = node_dropout_compact(plan.fwd, 0.3, 0x5BE0CD19_137E2179, None, 2, 0)
    products = [("stream", plan.bwd, True, Ops(g, 64, "bwd_last"), {}),
                ("rows65", plan.fwd, False, Ops(g, 65, "bwd_last"), {}),
                ("compact", plan.fwd, False, Ops(g, 64, "bwd_last"), dict(compact=cl[1]))]
    for name, side, transposed, ops, kw in products:
        eager = _run(ops, side, transposed, **kw)                 # allocates hub_partial before the capture
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            ops.reset()                                           # re-seeds Y from the saved addend: replays repeat
            spmm(side, None, ops.X, ops.d, out=ops.Y, addend=ops.addend, slot=ops.slot, gsum=ops.gsum,
                 transposed=transposed, **kw)
        for _ in range(3):
            ops.ybuf.fill_(float("nan"))
            graph.replay()
            torch.cuda.synchronize()
            assert torch.equal(_bits(ops.Y), _bits(eager)), name
            assert side.hub_done is None or int(torch.count_nonzero(side.hub_done)) == 0, name
        del graph


# ---- index limits ----------------------------------------------------------------------------------------------------
def test_spmm_at_the_27_bit_column_limit():
    """N = 2^27 - 1 nodes: the largest column id, 2^27 - 2, in tile-local row 15 packs to 0x7FFFFFFE."""
    n = (1 << 27) - 1
    rng = np.random.default_rng(8)
    lo, hi = np.arange(0, 200), np.arange(n - 200, n)
    ends = np.concatenate([lo, hi])
    row = np.concatenate([rng.choice(ends, 400), [n - 16, n - 16, n - 1]])
    col = np.concatenate([rng.choice(ends, 400), [n - 1, 0, n - 1]])
    val = rng.standard_normal(row.size).astype(np.float32)
    L = torch.sparse_coo_tensor(torch.from_numpy(np.stack([row, col])), torch.from_numpy(val), (n, n))
    with pytest.raises(ValueError):
        LaplacianPlan(torch.sparse_coo_tensor(torch.tensor([[0], [1]]), torch.ones(1), (1 << 27, 1 << 27)), DEV)
    plan = LaplacianPlan(L, DEV)
    try:
        side = plan.fwd
        a, b = side.rowptr[n - 16].item(), side.rowptr[n - 15].item()
        assert (n - 16) % 16 == 15 and side.tiles[(n - 16) // 16, 0].item() == n - 31
        assert 0x7FFFFFFE in side.ent[a:b, 0].tolist()
        gen = torch.Generator(device=DEV).manual_seed(3)
        for d in (4, 1):                                          # the streaming kernel, G = 1; the scalar kernel
            X = torch.randn(n, d, device=DEV, generator=gen)
            for transposed in (False, True):
                r, c = (col, row) if transposed else (row, col)
                touched, cols = np.unique(r), np.unique(c)            # the product restricted to what it touches
                Pc = sp.csr_matrix((val.astype(np.float64), (np.searchsorted(touched, r), np.searchsorted(cols, c))),
                                   shape=(touched.size, cols.size))
                Xc = X[torch.from_numpy(cols).to(DEV)].cpu().double().numpy()
                Y = torch.full((n, d), float("nan"), device=DEV)
                spmm(plan.bwd if transposed else plan.fwd, None, X, d, out=Y, transposed=transposed)
                t = torch.from_numpy(touched).to(DEV)
                _check(Y[t], Pc @ Xc, (d, transposed))
                Y[t] = 0
                assert int(torch.count_nonzero(Y)) == 0, (d, transposed)    # every other row written, and zero
                del Y
            del X
    finally:
        del plan
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def test_spmm_row_stride_at_the_32_bit_byte_limit():
    """ldx = 2^30 - 4 (byte stride 2^32 - 16) runs on the vector path; ldx = 2^30 + 4 would wrap and is refused."""
    row, col = np.array([0, 0, 1, 1, 1]), np.array([0, 1, 0, 1, 1])
    val = np.array([0.5, -2.0, 1.5, 3.0, 0.25], dtype=np.float32)
    L = torch.sparse_coo_tensor(torch.from_numpy(np.stack([row, col])), torch.from_numpy(val), (2, 2))
    plan = LaplacianPlan(L, DEV)
    A = sp.csr_matrix((val.astype(np.float64), (row, col)), shape=(2, 2))
    buf = torch.zeros((1 << 30) + 8, device=DEV)                 # 4 GiB + 32 bytes
    try:
        x = torch.tensor([[1.0, 2.0, 3.0, 4.0], [-5.0, 7.0, 0.125, 9.0]])
        X = buf.as_strided((2, 4), ((1 << 30) - 4, 1))
        X.copy_(x.to(DEV))
        buf[4:8] = 100.0                                         # what a wrapped stride of 16 bytes would read
        for transposed in (False, True):
            P = A.T.toarray() if transposed else A.toarray()
            got = spmm(plan.bwd if transposed else plan.fwd, None, X, 4, transposed=transposed)
            _check(got, P @ x.double().numpy(), ("ldx 2^30 - 4", transposed))
        bad = buf.as_strided((2, 4), ((1 << 30) + 4, 1))
        with pytest.raises(RuntimeError, match="2\\^30"):
            spmm(plan.fwd, None, bad, 4)
    finally:
        del buf
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
