"""Device-resident execution plan for one ``lap_list`` element.

The reference keeps each Laplacian as an uncoalesced int64 ``torch.sparse_coo`` (matrix.py:79-83) and lets
``torch.mm`` re-sort it on every call (NGCF.py:130; again, transposed, in the backward).  The plan converts it
ONCE into the layout the kernels execute (``ngcf_csr`` in include/ngcf_b200.h), for L and for L^T:

* int32 CSR with interleaved (col, value) entry pairs;
* rows longer than the split threshold (the hubs of a power-law graph) moved out of the row CSR into
  fixed-size chunks that are reduced separately and summed in order (deterministic, no float atomics);
* row tiles (bounded rows and entries) that a CTA stages in shared memory in one go;
* the permutation back to COO order, so a per-edge node-dropout mask generated in COO order (the reference's
  host RNG stream, NGCF.py:93-100) serves both directions.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib


def greedy_tiles(rowptr: np.ndarray, max_rows: int, max_ent: int) -> np.ndarray:
    """Cuts rows [0, n) into consecutive tiles of at most ``max_rows`` rows and ``max_ent`` entries (a single
    row longer than ``max_ent`` gets a tile of its own).  Returns int32 [n_tiles, 4] = (r0, r1, e0, e1)."""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    n = rowptr.size - 1
    out = []
    r = 0
    while r < n:
        k = int(np.searchsorted(rowptr, rowptr[r] + max_ent, side="right")) - 1   # last k with rowptr[k] <= limit
        r1 = max(r + 1, min(r + max_rows, k, n))
        out.append((r, r1, rowptr[r], rowptr[r1]))
        r = r1
    return np.asarray(out, dtype=np.int32).reshape(-1, 4)


def device_tiles(rowptr: torch.Tensor, max_rows: int, max_ent: int) -> torch.Tensor:
    """``greedy_tiles`` evaluated on the device (``ngcf_build_tiles``): same tiles, no host loop — a 1 B-edge graph has
    millions of them.  rowptr: int32 [n + 1] CUDA tensor.  Returns int32 [n_tiles, 4] on the device."""
    lib = _lib.load()
    dev = rowptr.device
    n = int(rowptr.numel()) - 1
    if n <= 0:
        return torch.zeros(0, 4, dtype=torch.int32, device=dev)
    nxt = torch.empty(n, dtype=torch.int32, device=dev)
    cap = n                                               # at most one tile per row
    count = torch.zeros(1, dtype=torch.int32, device=dev)
    # worst case one tile per row; allocate for the entry bound first and fall back to the row bound if it overflows
    guess = int(min(n, int(rowptr[-1]) // max(1, max_ent // 2) + n // max_rows + 16))
    for capacity in (guess, cap):
        tiles = torch.empty(capacity, 4, dtype=torch.int32, device=dev)
        _lib.check(lib.ngcf_build_tiles(rowptr.data_ptr(), n, int(max_rows), int(max_ent), nxt.data_ptr(),
                                        tiles.data_ptr(), capacity, count.data_ptr(), _lib.current_stream()),
                   "build_tiles")
        if int(count) <= capacity:
            return tiles[:int(count)].contiguous()
    raise RuntimeError("tile builder overflow")


DEVICE_TILE_ROWS = 1 << 18        # CSRs with more rows than this get their tiles built on the device


class CsrSide:
    """One direction (L or L^T) in execution layout; owns the device arrays behind an ``ngcf_csr`` struct."""

    def __init__(self, rowptr: torch.Tensor, colidx: torch.Tensor, perm, n_rows: int, nnz: int, vals=None):
        """perm: position of each entry in the COO value array (reference-format Laplacians), or None with ``vals`` =
        the entries' values in CSR order (device-built CSR Laplacians, plgraph.py)."""
        lib = _lib.load()
        dev = rowptr.device
        self.n_rows, self.nnz = int(n_rows), int(nnz)
        split = lib.ngcf_spmm_split_threshold()
        i32 = dict(dtype=torch.int32, device=dev)
        deg = (rowptr[1:] - rowptr[:-1]).to(torch.int64)
        hub_mask = deg > split
        hub = torch.nonzero(hub_mask).flatten()
        self.n_hub = int(hub.numel())
        colidx = colidx[:self.nnz]
        perm = perm[:self.nnz] if perm is not None else None
        self.vals = vals
        if self.n_hub:
            row_of_entry = torch.repeat_interleave(torch.arange(self.n_rows, device=dev), deg)
            ent_is_hub = hub_mask[row_of_entry]
            order = torch.cat([torch.nonzero(~ent_is_hub).flatten(), torch.nonzero(ent_is_hub).flatten()])
            self.colidx = colidx[order].contiguous()
            self.perm = perm[order].contiguous() if perm is not None else None
            if vals is not None:
                self.vals = vals[order].contiguous()
            del row_of_entry, ent_is_hub, order
            hdeg = deg[hub]
            self.nnz_hub = int(hdeg.sum())
            short_deg = torch.where(hub_mask, torch.zeros_like(deg), deg)
            nch = (hdeg + split - 1) // split
            cptr = torch.zeros(self.n_hub + 1, dtype=torch.int64, device=dev)
            cptr[1:] = torch.cumsum(nch, 0)
            self.n_chunks = int(cptr[-1])
            hub_base = torch.zeros(self.n_hub + 1, dtype=torch.int64, device=dev)
            hub_base[1:] = torch.cumsum(hdeg, 0)
            owner = torch.repeat_interleave(torch.arange(self.n_hub, device=dev), nch)
            local = torch.arange(self.n_chunks, device=dev) - cptr[owner]
            chunk_ptr = torch.empty(self.n_chunks + 1, dtype=torch.int64, device=dev)
            chunk_ptr[:-1] = hub_base[owner] + local * split
            chunk_ptr[-1] = self.nnz_hub
            self.hub_of_row = torch.full((self.n_rows,), -1, **i32)
            self.hub_of_row[hub] = torch.arange(self.n_hub, **i32)
            self.hub_chunk_ptr = cptr.to(torch.int32)
            self.chunk_ptr = chunk_ptr.to(torch.int32)
            self.chunk_row = hub[owner].to(torch.int32)
            self.hub_rows = hub.to(torch.int32).contiguous()
            self.hub_done = torch.zeros(self.n_hub, **i32)   # completion counters of the product in flight
        else:
            self.colidx, self.perm = colidx.contiguous(), (perm.contiguous() if perm is not None else None)
            self.nnz_hub, self.n_chunks = 0, 0
            short_deg = deg
            self.hub_of_row = self.hub_chunk_ptr = self.chunk_ptr = self.chunk_row = self.hub_rows = self.hub_done = None
        self.nnz_short = self.nnz - self.nnz_hub
        self.rowptr = torch.zeros(self.n_rows + 1, **i32)
        self.rowptr[1:] = torch.cumsum(short_deg, 0).to(torch.int32)
        tr, te = lib.ngcf_spmm_tile_rows(), lib.ngcf_spmm_tile_entries()
        if self.n_rows > DEVICE_TILE_ROWS:
            self.tiles = device_tiles(self.rowptr, tr, te)
            self.chunk_tiles = device_tiles(self.chunk_ptr, tr, te) if self.n_chunks else None
        else:
            self.tiles = torch.from_numpy(greedy_tiles(self.rowptr.cpu().numpy(), tr, te)).to(dev)
            self.chunk_tiles = torch.from_numpy(greedy_tiles(self.chunk_ptr.cpu().numpy(), tr, te)).to(dev) \
                if self.n_chunks else None
        self._pack_local_rows()
        # per row tile: which of its rows are hubs (the streaming kernel must not write those: hub_finish_kernel does)
        if self.n_hub and self.tiles.shape[0]:
            hm = torch.zeros(self.n_rows + 32, dtype=torch.int64, device=dev)
            hm[:self.n_rows] = hub_mask.to(torch.int64)
            t0 = self.tiles[:, 0].to(torch.int64)
            nr = (self.tiles[:, 1] - self.tiles[:, 0]).to(torch.int64)
            bits = torch.zeros(self.tiles.shape[0], dtype=torch.int64, device=dev)
            for i in range(int(lib.ngcf_spmm_tile_rows())):
                bits |= (hm[t0 + i] * (i < nr).to(torch.int64)) << i
            self.tile_hubmask = (bits & 0xFFFFFFFF).to(torch.int32)      # bit pattern of a uint32
        else:
            self.tile_hubmask = None
        self.ent = None          # base entry pairs, set by LaplacianPlan
        self.key_l = self.key_t = None   # static node-dropout keys (ensure_keys)
        self.key_row_offset = 0
        self._partial = {}
        self._struct_cache = {}

    LR_SHIFT = 27            # spmm_core.cuh: column ids have 27 bits, the 5 bits above them name the entry's row in its tile

    def _pack_local_rows(self):
        """Writes, into the top bits of every entry's column word, the index of the entry's row inside its SpMM tile
        (hub entries: of its chunk inside its chunk tile).  The streaming SpMM kernel reads a tile's entries as one
        stream and needs no row pointers; the per-step node-dropout compaction copies entries verbatim, so the tag
        survives it."""
        dev = self.rowptr.device
        if self.nnz_short:
            pos = torch.arange(self.nnz_short, device=dev)
            row = torch.searchsorted(self.rowptr.to(torch.int64), pos, right=True) - 1
            t0 = self.tiles[:, 0].to(torch.int64).contiguous()
            lr = row - t0[torch.searchsorted(t0, row, right=True) - 1]
            self.colidx[:self.nnz_short] |= (lr << self.LR_SHIFT).to(torch.int32)
        if self.n_chunks:
            pos = torch.arange(self.nnz_hub, device=dev)
            chunk = torch.searchsorted(self.chunk_ptr.to(torch.int64), pos, right=True) - 1
            t0 = self.chunk_tiles[:, 0].to(torch.int64).contiguous()
            lr = chunk - t0[torch.searchsorted(t0, chunk, right=True) - 1]
            self.colidx[self.nnz_short:self.nnz] |= (lr << self.LR_SHIFT).to(torch.int32)

    def descriptor(self, ent: torch.Tensor | None = None) -> "_lib.NgcfCsr":
        """``ngcf_csr`` over this side's arrays; ``ent`` = alternative [nnz, 2] entry pairs (masked values)."""
        ent = self.ent if ent is None else ent
        key = ent.data_ptr()
        s = self._struct_cache.get(key)
        if s is None:
            if len(self._struct_cache) > 64:
                self._struct_cache.clear()
            s = _lib.NgcfCsr()
            s.n_rows = self.n_rows
            s.rowptr = self.rowptr.data_ptr()
            s.ent = ent.data_ptr()
            s.tiles = self.tiles.data_ptr()
            s.hub_of_row = _lib.ptr(self.hub_of_row)
            s.hub_chunk_ptr = _lib.ptr(self.hub_chunk_ptr)
            s.chunk_ptr = _lib.ptr(self.chunk_ptr)
            s.hub_ent = ent.data_ptr() + 8 * self.nnz_short
            s.chunk_row = _lib.ptr(self.chunk_row)
            s.chunk_tiles = _lib.ptr(self.chunk_tiles)
            s.hub_rows = _lib.ptr(self.hub_rows)
            s.hub_done = _lib.ptr(self.hub_done)
            s.key_l = _lib.ptr(self.key_l)
            s.key_t = _lib.ptr(self.key_t)
            s.key_row_offset = self.key_row_offset
            s.n_tiles = int(self.tiles.shape[0])
            s.n_hub = self.n_hub
            s.n_chunks = self.n_chunks
            s.n_chunk_tiles = int(self.chunk_tiles.shape[0]) if self.chunk_tiles is not None else 0
            s.rowptr_nnz = self.nnz_short
            s.tile_hubmask = _lib.ptr(self.tile_hubmask)
            self._struct_cache[key] = s
        return s

    def ensure_keys(self, row_offset: int = 0):
        """Static node-dropout keys of every entry (once per side): the per-step compaction then needs no row search."""
        if self.key_l is None or self.key_row_offset != row_offset:
            lib = _lib.load()
            dev = self.rowptr.device
            kl = torch.empty(max(self.nnz, 1), dtype=torch.int32, device=dev)
            kt = torch.empty(max(self.nnz, 1), dtype=torch.int32, device=dev)
            _lib.check(lib.ngcf_entry_keys(C.byref(self.descriptor(None)), int(row_offset), kl.data_ptr(), kt.data_ptr(),
                                           _lib.current_stream()), "entry_keys")
            self.key_l, self.key_t, self.key_row_offset = kl, kt, int(row_offset)
            self._struct_cache.clear()

    def hub_partial(self, d: int):
        if not self.n_hub:
            return None
        buf = self._partial.get(d)
        if buf is None:
            buf = torch.empty(self.n_chunks * d, dtype=torch.float32, device=self.rowptr.device)
            self._partial[d] = buf
        return buf


class LaplacianPlan:
    """Execution plan of one ``lap_list`` element; ``shard`` (a sharded.RowShards) restricts it to this rank's row
    block of L and of L^T (``rows x N_pad`` matrices whose column ids stay global)."""

    def __init__(self, L, device, shard=None):
        from .plgraph import CsrLaplacian
        if isinstance(L, CsrLaplacian):
            self._init_from_csr(L, torch.device(device), shard)
            return
        if not (L.is_sparse and L.dim() == 2 and L.shape[0] == L.shape[1]):
            raise ValueError("lap_list entries must be square torch.sparse_coo tensors (matrix.py:79-83)")
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("LaplacianPlan needs a CUDA device: the NGCF B200 path has no CPU fallback")
        lib = _lib.load()
        self.src = L
        self.N = int(L.shape[0])
        self.shard = shard
        idx = L._indices().to(device=device, dtype=torch.int64).contiguous()
        self.coo_val = L._values().to(device=device, dtype=torch.float32).contiguous()
        self.nnz = int(self.coo_val.numel())
        if self.nnz and (int(idx.min()) < 0 or int(idx.max()) >= self.N):
            raise ValueError("Laplacian indices out of range")
        if (shard.N_pad if shard is not None else self.N) >= (1 << CsrSide.LR_SHIFT):
            raise ValueError(f"graphs of up to {1 << CsrSide.LR_SHIFT} nodes are supported (27-bit column ids)")
        if lib.ngcf_spmm_tile_rows() > 32:
            raise RuntimeError("the local row tag of an entry assumes SpMM tiles of at most 32 rows")
        if shard is None:
            n_rows = n_cols = self.N
            pos = torch.arange(self.nnz, device=device)
            parts = [(idx[0], idx[1], pos), (idx[1], idx[0], pos)]            # L, L^T
        else:
            from .sharded import shard_coo
            if shard.N != self.N:
                raise ValueError("shard descriptor and Laplacian disagree on N")
            n_rows, n_cols = shard.rows, shard.N_pad
            Ld = torch.sparse_coo_tensor(idx, self.coo_val, L.shape, is_coalesced=False, check_invariants=False)
            parts = list(shard_coo(Ld, shard))
        sides = []
        for row, col, pos in parts:
            nnz = int(row.numel())
            row, col = row.contiguous(), col.contiguous()
            need = C.c_size_t(0)
            _lib.check(lib.ngcf_coo_to_csr_workspace(nnz, n_rows, C.byref(need)), "coo_to_csr_workspace")
            ws = torch.empty(need.value, dtype=torch.uint8, device=device)
            rowptr = torch.empty(n_rows + 1, dtype=torch.int32, device=device)
            colidx = torch.empty(max(nnz, 1), dtype=torch.int32, device=device)
            perm = torch.empty(max(nnz, 1), dtype=torch.int32, device=device)
            _lib.check(lib.ngcf_coo_to_csr(row.data_ptr(), col.data_ptr(), nnz, n_rows, n_cols, 0,
                                           rowptr.data_ptr(), colidx.data_ptr(), perm.data_ptr(), ws.data_ptr(),
                                           need.value, _lib.current_stream()), "coo_to_csr")
            # perm indexes this side's entry list; compose with `pos` so it addresses the ORIGINAL COO order
            perm = pos[perm[:nnz].to(torch.int64)].to(torch.int32) if nnz else perm
            side = CsrSide(rowptr, colidx, perm, n_rows, nnz)
            side.ent = self.entries(side, None)
            sides.append(side)
            torch.cuda.current_stream().synchronize()
            del ws
        self.fwd, self.bwd = sides
        # L = D^-1/2 A D^-1/2 is symmetric (matrix.py:48-62): then L^T's layout is L's, and sharing the arrays
        # halves the distinct bytes a training step touches.  Node dropout breaks the symmetry per step, which
        # is handled by giving the two directions separate masked entry arrays.
        self.symmetric = bool(self.fwd.nnz == self.bwd.nnz and torch.equal(self.fwd.rowptr, self.bwd.rowptr) and
                              torch.equal(self.fwd.ent, self.bwd.ent))

    def _init_from_csr(self, L, device, shard):
        """A device-built CSR row shard (plgraph.CsrLaplacian) of a SYMMETRIC Laplacian: the execution layout is derived
        from it directly (no COO, no sort), and L^T's row shard is the same matrix."""
        if device.type != "cuda":
            raise RuntimeError("LaplacianPlan needs a CUDA device: the NGCF B200 path has no CPU fallback")
        self.src, self.N, self.shard = L, int(L.shape[0]), shard
        n_cols = shard.N_pad if shard is not None else self.N
        if n_cols >= (1 << CsrSide.LR_SHIFT):
            raise ValueError(f"graphs of up to {1 << CsrSide.LR_SHIFT} nodes are supported (27-bit column ids)")
        if shard is not None and (L.row0 != shard.r0 or L.n_rows != shard.rows):
            raise ValueError("the CSR shard does not cover this rank's row block")
        if shard is None and L.n_rows != self.N:
            raise ValueError("an unsharded plan needs all rows of the Laplacian")
        self.nnz = L.nnz
        self.coo_val = L.vals                                      # (device marker for NGCF._plan; not COO-ordered)
        side = CsrSide(L.rowptr.to(device), L.colidx.to(device), None, L.n_rows, L.nnz, vals=L.vals.to(device))
        side.ent = self.entries(side, None)
        side.vals = None                                           # folded into ent
        torch.cuda.current_stream().synchronize()
        self.fwd = self.bwd = side
        self.symmetric = True

    def side(self, transposed: bool, masked: bool) -> CsrSide:
        if transposed and not (self.symmetric and not masked):
            return self.bwd
        return self.fwd

    def entries(self, side: CsrSide, keep_mask):
        """Entry pairs in execution order, optionally with an explicit COO-order node-dropout mask folded in
        (NGCF.py:93-100).  Two trailing pad pairs keep vector reads in bounds."""
        lib = _lib.load()
        if side.perm is None:                                      # device-built CSR: values are already in entry order
            if keep_mask is not None:
                raise ValueError("explicit COO-order edge masks need a reference-format (COO) Laplacian")
            out = torch.zeros(side.nnz + 2, 2, dtype=torch.int32, device=side.colidx.device)
            out[:side.nnz, 0] = side.colidx
            out[:side.nnz, 1] = side.vals.view(torch.int32)
            return out
        out = torch.zeros(side.nnz + 2, 2, dtype=torch.int32, device=self.coo_val.device)
        _lib.check(lib.ngcf_edge_entries(side.colidx.data_ptr(), self.coo_val.data_ptr(), side.perm.data_ptr(),
                                         _lib.ptr(keep_mask), out.data_ptr(), side.nnz, _lib.current_stream()),
                   "edge_entries")
        return out


def node_dropout_bits(side: CsrSide, drop_p: float, seed: int, seed_dev, n_layers: int, row_offset: int = 0,
                      as_L: bool = True, as_Lt: bool = False):
    """One step's node-dropout decisions for every entry of ``side`` (uint8 per entry, bit k = survives layer k),
    for the CSR read as L and/or as L^T.  Returns (bits_as_L or None, bits_as_Lt or None)."""
    lib = _lib.load()
    dev = side.rowptr.device
    bl = torch.empty(side.nnz, dtype=torch.uint8, device=dev) if as_L else None
    bt = torch.empty(side.nnz, dtype=torch.uint8, device=dev) if as_Lt else None
    _lib.check(lib.ngcf_node_dropout_bits(C.byref(side.descriptor(None)), float(drop_p), int(seed) & (2 ** 64 - 1),
                                          _lib.ptr(seed_dev), int(n_layers), int(row_offset), _lib.ptr(bl), _lib.ptr(bt),
                                          _lib.current_stream()), "node_dropout_bits")
    return bl, bt


def node_dropout_compact(side: CsrSide, drop_p: float, seed: int, seed_dev, n_layers: int, row_offset: int = 0,
                         as_L: bool = True, as_Lt: bool = False, static_keys: bool = True):
    """One step's node dropout applied like the reference does it (entries deleted, cumulatively per layer,
    NGCF.py:93-100): per layer the surviving entries of every SpMM tile, compacted, for ``side`` read as L and/or as
    L^T.  Returns (per-layer list of (ent, cnt) or None, same for L^T): the survivors of tile t, in order, at the front of
    the tile's slot range of ``ent`` and their number in ``cnt[t]``; pass one pair to ``spmm(compact=...)``."""
    lib = _lib.load()
    dev = side.rowptr.device
    if static_keys:
        side.ensure_keys(row_offset)
    elif side.key_l is not None:                     # (tests) the pass then derives the keys from the coordinates
        side.key_l = side.key_t = None
        side._struct_cache.clear()
    n_t = int(side.tiles.shape[0]) + (int(side.chunk_tiles.shape[0]) if side.chunk_tiles is not None else 0)

    def alloc():
        return [(torch.empty(side.nnz + 2, 2, dtype=torch.int32, device=dev),
                 torch.empty(max(n_t, 1), dtype=torch.int32, device=dev)) for _ in range(n_layers)]

    cl = alloc() if as_L else None
    ct = alloc() if as_Lt else None

    def arrs(c):
        if c is None:
            return None, None
        return _lib.ptr_array([e for e, _ in c]), _lib.ptr_array([t for _, t in c])

    el, tl = arrs(cl)
    et, tt = arrs(ct)
    _lib.check(lib.ngcf_node_dropout_compact(C.byref(side.descriptor(None)), float(drop_p), int(seed) & (2 ** 64 - 1),
                                             _lib.ptr(seed_dev), int(n_layers), int(row_offset), el, tl, et, tt,
                                             _lib.current_stream()), "node_dropout_compact")
    return cl, ct


def spmm(side: CsrSide, ent, X, d: int, out=None, addend=None, slot=None, gsum=None, drop_p: float = 0.0,
         seed: int = 0, seed_dev=None, layer: int = 0, transposed: bool = False, row_offset: int = 0, keep_bits=None,
         compact=None):
    """Y = L·X (+ addend) (+ gsum[slot] rows) through ngcf_spmm; drop_p > 0 = in-kernel device-RNG node dropout;
    compact = this layer's (ent, cnt) pair from node_dropout_compact.  With ``addend`` and no ``out`` the product is
    accumulated IN PLACE into ``addend`` (which is returned): the streaming kernel adds its row sums to a Y that already
    holds the addend, so a separate output would cost a copy."""
    lib = _lib.load()
    if out is None:
        if addend is not None and d % 4 == 0 and addend.shape[0] == side.n_rows and addend.stride(0) % 4 == 0:
            out = addend
        else:
            out = torch.empty(side.n_rows, d, dtype=torch.float32, device=X.device)
    _lib.check(lib.ngcf_spmm(C.byref(side.descriptor(ent)), X.data_ptr(), X.stride(0), d,
                             _lib.ptr(addend), addend.stride(0) if addend is not None else 0,
                             _lib.ptr(slot), _lib.ptr(gsum), gsum.stride(0) if gsum is not None else 0,
                             _lib.ptr(side.hub_partial(d)),
                             float(drop_p), int(seed) & (2 ** 64 - 1), _lib.ptr(seed_dev), int(layer), int(transposed),
                             int(row_offset), _lib.ptr(keep_bits),
                             _lib.ptr(compact[0]) if compact is not None else None,
                             _lib.ptr(compact[1]) if compact is not None else None,
                             out.data_ptr(), out.stride(0), _lib.current_stream()), "spmm")
    return out


def node_dropout_mode(mode: str, widths) -> str:
    """The node-dropout mode a step runs for the requested ``mode``: survivor lists ("compact") are read by the
    streaming SpMM, which needs every width to be a multiple of 4 (the last one too: the batch-row gradient rows of the
    final backward product are D_total wide); other widths take per-step decision bytes ("bits")."""
    return "bits" if mode == "compact" and any(d % 4 for d in widths) else mode


class NodeDropout:
    """One step's device-RNG node dropout for the K products over L and the K transposed products over L^T.

    ``mode`` "compact" deletes the dropped entries like NGCF.sparse_dropout does (per-step survivor lists, so layer k
    gathers (1-p)^(k+1) of the rows); "bits" draws per-step decision bytes; "inkernel" hashes every entry inside each
    product; ``node_dropout_mode`` turns "compact" into "bits" for widths the survivor lists cannot serve.  The
    decisions of all K layers are drawn once, on construction, and a symmetric L serves L^T from the same pass;
    otherwise ``draw_transposed()`` draws L^T's where the backward calls it.  (L^T's half on a second stream, beside
    the forward or behind its last layer, measured slower on one B200: 0.518 / 0.509-0.513 vs 0.502-0.510 ms per step,
    two more launches and the entries read twice cost more than the overlap hides.)  ``args(layer, transposed)`` are
    the dropout arguments of one ``spmm`` call."""

    def __init__(self, plan: LaplacianPlan, mode: str, drop_p: float, seed: int, seed_dev, n_layers: int,
                 row_offset: int, widths):
        mode = node_dropout_mode(mode, widths)
        self.plan, self.mode, self.drop_p, self.seed, self.seed_dev = plan, mode, drop_p, seed, seed_dev
        self.n_layers, self.row_offset = n_layers, row_offset
        self.fwd = self.bwd = None          # per-layer (ent, cnt) pairs ("compact") or one uint8 array ("bits")
        if self._drawn():
            shared = plan.side(True, False) is plan.fwd
            self.fwd, bwd = self._draw(plan.fwd, as_L=True, as_Lt=shared)
            if shared:
                self.bwd = bwd

    def _drawn(self) -> bool:
        return self.drop_p > 0 and self.mode in ("compact", "bits")

    def _draw(self, side: CsrSide, as_L: bool, as_Lt: bool):
        draw = node_dropout_compact if self.mode == "compact" else node_dropout_bits
        return draw(side, self.drop_p, self.seed, self.seed_dev, self.n_layers, self.row_offset, as_L=as_L, as_Lt=as_Lt)

    def draw_transposed(self):
        """L^T's decisions, unless the forward's pass drew them with L's."""
        if self._drawn() and self.bwd is None:
            _, self.bwd = self._draw(self.plan.side(True, False), as_L=False, as_Lt=True)

    def args(self, layer: int, transposed: bool = False) -> dict:
        lists = self.bwd if transposed else self.fwd
        return dict(drop_p=self.drop_p, seed=self.seed, seed_dev=self.seed_dev, layer=layer, transposed=transposed,
                    row_offset=self.row_offset, keep_bits=lists if self.mode == "bits" else None,
                    compact=lists[layer] if self.mode == "compact" and lists is not None else None)
