/* ngcf_b200.h — C ABI of the B200-native NGCF embedding-propagation hot path.
 *
 * The reference (haesungpyun/seoul_tourism_recommendation_NGCF) is pure Python/PyTorch and has no
 * FFI of its own; the boundary it offers is the Python class surface of model/NGCF.py and
 * model/bprloss.py.  This library is what the drop-in NGCF / BPR modules
 * (seoul_tourism_recommendation_ngcf_b200/NGCF.py, bprloss.py) bind through ctypes; every entry
 * point names the reference lines whose torch calls it replaces (paths relative to
 * /root/reference/model/).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name ends in
 *     _host; the caller (torch) allocates and owns every buffer, the library keeps no pointer past
 *     return and allocates nothing;
 *   - all dense matrices are row-major fp32; `ld*` is the row stride in elements;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*), nothing synchronises, every
 *     call is CUDA-graph capturable unless stated;
 *   - return 0 on success, negative ngcf_status otherwise; ngcf_last_error() gives a thread-local
 *     message.  There is no CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef NGCF_B200_H
#define NGCF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NGCF_B200_ABI_VERSION 4
#define NGCF_MAX_LAYERS 8
#define NGCF_MAX_WIDTH 128          /* widest embedding / layer size the kernels accept */
#define NGCF_ADAM_MAX_TENSORS 32     /* parameter tensors one ngcf_adam_step call updates */

typedef enum {
    NGCF_OK = 0,
    NGCF_ERR_INVALID = -1,          /* bad argument (null pointer, width > NGCF_MAX_WIDTH, ...) */
    NGCF_ERR_CUDA = -2,             /* a CUDA runtime call or launch failed */
    NGCF_ERR_WORKSPACE = -3         /* caller-provided workspace too small */
} ngcf_status;

int ngcf_abi_version(void);
const char* ngcf_last_error(void);
uint64_t ngcf_launch_count(void);   /* kernels this library has launched in this process (bench accounting) */

/* ---- Laplacian format: lap_list[i] (matrix.py:79-83, consumed NGCF.py:117-118,130) ------------
 * One-off conversion of the reference's uncoalesced int64 COO into int32 CSR.  Entries are sorted by
 * (row, col) — or by (col, row) when `transpose` != 0, giving the CSR of L^T that the backward's
 * MmBackward0 needs — and duplicates are kept (their products sum, like coalesce()).  perm[t] is the
 * COO position of CSR entry t, so one edge mask in COO order serves both directions.
 * Not graph-capturable (uses a sort).  nnz < 2^31. */
int ngcf_coo_to_csr_workspace(int64_t nnz, int64_t n_rows, size_t* bytes_host);
int ngcf_coo_to_csr(const int64_t* coo_row, const int64_t* coo_col, int64_t nnz,
                    int64_t n_rows, int64_t n_cols, int transpose,
                    int32_t* rowptr /*[n+1], n = transpose ? n_cols : n_rows*/,
                    int32_t* colidx /*[nnz]*/, int32_t* perm /*[nnz]*/,
                    void* workspace, size_t workspace_bytes, void* stream);

/* ---- execution layout of one Laplacian direction (built once by plan.py from the CSR above) ----------------
 * ngcf_csr is a HOST struct of DEVICE pointers.  Entries are interleaved (col, float-bits) int32 pairs.  Rows
 * with more than ngcf_spmm_split_threshold() entries ("hubs") are empty in rowptr/ent and live in hub_ent, cut
 * into chunks of at most that many entries; chunk c covers hub_ent[chunk_ptr[c] .. chunk_ptr[c+1]) and belongs
 * to row chunk_row[c]; hub row with id h = hub_of_row[row] owns chunks hub_chunk_ptr[h] .. hub_chunk_ptr[h+1].
 * Tiles are int32 quadruples {r0, r1, e0, e1}: rows [r0, r1) with entries [e0, e1) of ent (tiles) or
 * chunks [r0, r1) with entries [e0, e1) of hub_ent (chunk_tiles); at most ngcf_spmm_tile_rows() rows and
 * ngcf_spmm_tile_entries() entries each. */
typedef struct ngcf_csr {
    int64_t n_rows;
    const int32_t* rowptr;          /* [n_rows+1], hub rows empty */
    const int32_t* ent;             /* [2*nnz_short] */
    const int32_t* tiles;           /* [4*n_tiles] */
    const int32_t* hub_of_row;      /* [n_rows] hub id or -1; may be NULL when n_hub == 0 */
    const int32_t* hub_chunk_ptr;   /* [n_hub+1] */
    const int32_t* chunk_ptr;       /* [n_chunks+1] */
    const int32_t* hub_ent;         /* [2*nnz_hub] */
    const int32_t* chunk_row;       /* [n_chunks] */
    const int32_t* chunk_tiles;     /* [4*n_chunk_tiles] */
    const int32_t* hub_rows;        /* [n_hub] row of hub h */
    int32_t* hub_done;              /* [n_hub] completion counters of a product in flight: all zero between calls
                                       (ngcf_spmm leaves them zero); one product per csr at a time */
    const uint32_t* key_l;          /* optional [nnz] static node-dropout keys (ngcf_entry_keys), CSR read as L ... */
    const uint32_t* key_t;          /* ... and read as L^T; NULL: the per-step pass derives them from the coordinates */
    int64_t key_row_offset;         /* the row_offset the keys were computed for */
    int32_t n_tiles, n_hub, n_chunks, n_chunk_tiles;
    int32_t rowptr_nnz;             /* entries in `ent` (= rowptr[n_rows]); per-entry side arrays continue with hub_ent */
    const uint32_t* tile_hubmask;   /* [n_tiles] bit i = row r0 + i of the tile is a hub row; may be NULL when n_hub == 0 */
} ngcf_csr;

int ngcf_spmm_split_threshold(void);
int ngcf_spmm_tile_rows(void);
int ngcf_spmm_tile_entries(void);

/* ent_out[t] = (colidx[t], coo_val[perm[t]] * keep_mask[perm[t]]): entry pairs in execution order (ordinary rows
 * first, then hub chunks; colidx/perm in that order), optionally with an explicit node-dropout mask folded in.
 * Replaces NGCF.sparse_dropout (NGCF.py:93-100) for masks given in COO order (the reference's host RNG stream, or
 * a mask injected by a test): dropped entries are zeroed over the fixed structure instead of deleted (identical
 * sums).  keep_mask: optional uint8[nnz].  (Device-RNG node dropout needs no pass at all: see ngcf_spmm.) */
int ngcf_edge_entries(const int32_t* colidx, const float* coo_val, const int32_t* perm, const uint8_t* keep_mask,
                      int32_t* ent_out, int64_t nnz, void* stream);

/* ---- feature mix: NGCF.py:103-115 ----------------------------------------------------------------
 * user_w[u_id[b], :] = user_w[u_id[b], :]*(1-ratio) + concat(age,sex,month,day,dow rows)*ratio,
 * in place.  Duplicate u_id: the LAST occurrence in the batch wins (the reference's deterministic
 * single-thread CPU behaviour).  tables/idx are host arrays of 5 device pointers in concat order
 * age, sex, month, day, dow (NGCF.py:110); widths[5] must sum to d.  winner is int32[n_user] scratch
 * that must be all -1 on entry and is restored to all -1 before return. */
int ngcf_feature_mix(float* user_w, int64_t n_user, int d,
                     const float* const* tables_host, const int* widths_host,
                     const int64_t* const* idx_host, const int64_t* u_id, int64_t batch,
                     float ratio, int32_t* winner, void* stream);

/* ---- SpMM: torch.mm(L, E), NGCF.py:130, and its backward L^T·gS (autograd MmBackward0) ----------
 * Y[i,:] = sum_t val[t] * X[col[t],:]  (+ addend[i,:])  (+ rowgrad rows, see below), d <= 128.
 * Hub rows are pre-reduced chunk-wise into hub_partial (scratch [n_chunks, d]) and summed in chunk order, so the
 * result is deterministic (no float atomics on shared sums).  Widths that are multiples of 4 run the
 * streaming kernel: it ADDS its row sums to Y after Y := addend (pass addend == Y to accumulate in place and
 * save the copy); other widths run the row-per-warp kernel.  The column word of an entry carries, above its 27-bit
 * column id, the index of the entry's row inside its tile (see plan.py).
 *   ldx, ldy, ld_add, ld_gsum: row pitches in floats, ldx and ldy >= d; ldx < 2^30 (the gathers address rows of X
 *               with a 32-bit byte stride).  An in-place addend (addend == Y) needs ld_add == ldy.
 *   slot/gsum : optional sparse row addend — if slot[i] >= 0, Y[i,:] += gsum[slot[i]*ld_gsum + 0..d)
 *               (the IndexBackward scatter of NGCF.py:151-155 folded into the last backward SpMM).
 *   drop_p > 0: device-RNG node dropout (NGCF.py:93-100,124-126) evaluated in-kernel: entry (r,c) of L survives
 *               layer `layer` iff its counter-based draws keyed on (seed + *seed_dev, r, c) for layers 0..layer are all
 *               >= drop_p (cumulative over layers, unscaled — the reference's semantics).  `transposed` != 0 says
 *               this CSR holds L^T, so both directions drop the same entries of L.
 *               seed_dev: optional device uint64 added to seed (graph-replay safe).
 *   keep_bits : optional output of ngcf_node_dropout_bits for this direction; when given, drop_p/seed are unused.
 *   c_ent/c_cnt: optional output of ngcf_node_dropout_compact for this direction AND layer (the step's surviving
 *               entries, compacted per tile, and their number per tile); when given, keep_bits/drop_p/seed are unused
 *               and only survivors are staged and gathered (width % 4 == 0 only).
 *   row_offset: global index of row 0 of this CSR.  RNG keys use global coordinates, so a row shard (rows
 *               [row_offset, row_offset + n_rows) of L, all columns) draws exactly the single-GPU decisions. */
int ngcf_spmm(const ngcf_csr* csr_host, const float* X, int64_t ldx, int d,
              const float* addend, int64_t ld_add,
              const int32_t* slot, const float* gsum, int64_t ld_gsum,
              float* hub_partial,
              float drop_p, uint64_t seed, const uint64_t* seed_dev, int layer, int transposed, int64_t row_offset,
              const uint8_t* keep_bits, const int32_t* c_ent, const int32_t* c_cnt,
              float* Y, int64_t ldy, void* stream);

/* One step's node-dropout decisions for every entry and every layer at once (bit k of a byte = the entry survives
 * layer k; cumulative).  Entry order = ent then hub_ent.  bits_as_L: this CSR read as L (keys (row, col));
 * bits_as_Lt: the same CSR read as L^T (keys (col, row)) — a symmetric L shares one CSR for both directions.
 * Passing the result to ngcf_spmm as keep_bits replaces its in-kernel hash evaluation by one byte load per
 * entry (same decisions, ~10 us less per product at Gowalla shape). */
int ngcf_node_dropout_bits(const ngcf_csr* csr_host, float drop_p, uint64_t seed, const uint64_t* seed_dev,
                           int n_layers, int64_t row_offset, uint8_t* bits_as_L, uint8_t* bits_as_Lt, void* stream);

/* The same decisions applied the way the reference applies them (NGCF.sparse_dropout, NGCF.py:93-100, DELETES the
 * dropped entries, cumulatively over the layers): one pass per step writes, for every layer k and for the CSR read
 * as L and/or as L^T, the surviving (col, value) pairs of each SpMM tile {r0,r1,e0,e1} compacted in their original
 * order at [e0, e0 + kept) of ent_*[k] (int32[2*nnz], indexed like ent then hub_ent) and `kept` to
 * cnt_*[k][tile] (tiles first, then chunk_tiles).
 * ent_*_host / cnt_*_host are HOST arrays of n_layers device pointers; pass NULL for a direction that is not needed.
 * Products given these arrays gather only the survivors: (1-p)^(k+1) of the entries at layer k. */
int ngcf_node_dropout_compact(const ngcf_csr* csr_host, float drop_p, uint64_t seed, const uint64_t* seed_dev,
                              int n_layers, int64_t row_offset,
                              int32_t* const* ent_as_L_host, int32_t* const* cnt_as_L_host,
                              int32_t* const* ent_as_Lt_host, int32_t* const* cnt_as_Lt_host, void* stream);

/* Static per-entry node-dropout keys (plan time, once per csr): key_l[t] / key_t[t] for entry t in execution order
 * (ent then hub_ent), the CSR read as L / as L^T.  With them in the descriptor ngcf_node_dropout_compact needs no row
 * search and one hash per direction and entry. */
int ngcf_entry_keys(const ngcf_csr* csr_host, int64_t row_offset, uint32_t* key_l, uint32_t* key_t, void* stream);

/* ---- graph construction on the device (matrix.py:41-83 for graphs the reference's dense builder cannot hold) --------
 * ngcf_plgraph_entries: adjacency entries of a synthetic power-law bipartite graph (Zipf(alpha) user activity and item
 * popularity, edge e a pure function of (seed, e)) for the rows [row0, row0 + n_rows) of the (n_user + n_item)-node
 * graph, both directions of every edge, as unsorted 64-bit keys (row - row0) << 32 | col appended through *total_dev
 * (zero on entry; keys_or_null == NULL only counts).  Sorting + deduplicating the keys gives the shard's CSR.
 * ngcf_build_tiles: the SpMM tile list {r0, r1, e0, e1} (greedy: <= max_rows rows, <= max_ent entries) of a CSR;
 * next_scratch is int32[n_rows]; *count_out receives the number of tiles (tiles beyond capacity are not written). */
int ngcf_plgraph_entries(int64_t n_user, int64_t n_item, int64_t n_edges, double alpha, uint64_t seed,
                         int64_t row0, int64_t n_rows, unsigned long long* total_dev,
                         unsigned long long* keys_or_null, int64_t capacity, void* stream);
int ngcf_build_tiles(const int32_t* rowptr, int64_t n_rows, int max_rows, int max_ent, int32_t* next_scratch,
                     int32_t* tiles_out, int64_t capacity, int32_t* count_out, void* stream);

/* ---- row-shard exchange over peer memory (multi-GPU row partition; the reference has no multi-device code) ----------
 * Every rank holds a full [N_pad, d] copy of a matrix in peer-mapped (symmetric) memory and owns rows
 * [row0, row0 + n_rows) of it.  ngcf_push_rows stores the owner's rows into every peer's copy and returns (in stream
 * order) once every peer's rows have landed in the local copy: an all-gather without a library collective, one launch.
 *   matrix_on_rank_host[r] : base address of rank r's copy as mapped into THIS process (r == rank: the local one)
 *   flags_on_rank_host[r]  : rank r's flag block, ngcf_exchange_flag_words() uint32, zero before the first exchange
 *   local_state            : uint32[2] in local device memory, zero before the first exchange
 * Every rank must issue the same sequence of exchanges on the same flag blocks.
 *   multicast_or_null      : the NVLS multicast mapping of the matrix (one multimem.st reaches every rank's copy through
 *                            the NVSwitch), when the platform offers one; NULL: one store per peer
 * ngcf_push_selected_rows does the same for the rows list[q][j] + list_offsets[q] only (those this rank owns): the
 * last layer's output is needed on other ranks for the <= 3 B batch rows alone (NGCF.py:151-155). */
int ngcf_exchange_flag_words(void);
int ngcf_push_rows(float* const* matrix_on_rank_host, uint32_t* const* flags_on_rank_host, uint32_t* local_state,
                   int world, int rank, int64_t row0, int64_t n_rows, int d, float* multicast_or_null, void* stream);
int ngcf_push_selected_rows(float* const* matrix_on_rank_host, uint32_t* const* flags_on_rank_host, uint32_t* local_state,
                            int world, int rank, int64_t row0, int64_t n_rows, int d,
                            const int64_t* const* lists_host, const int64_t* list_offsets_host,
                            const int64_t* list_sizes_host, int n_lists, float* multicast_or_null, void* stream);

/* ---- per-layer epilogue: NGCF.py:131-142 ------------------------------------------------------------
 * pack:  wcat[k, o] = W1[o,k] (k < d_in), W2[o,k-d_in] (k >= d_in);  bias_eff = 2*b1 + b2
 *        (the reference applies w1_list[i] twice, NGCF.py:131,133, so its bias counts twice). */
int ngcf_pack_weights(const float* W1, const float* b1, const float* W2, const float* b2,
                      int d_in, int d_out, float* wcat /*[2*d_in, d_out]*/, float* bias_eff /*[d_out]*/,
                      void* stream);
/* The same for every layer of a step in one launch (host arrays of n_layers pointers / widths). */
int ngcf_pack_weights_all(const float* const* W1_host, const float* const* b1_host, const float* const* W2_host,
                          const float* const* b2_host, const int* d_in_host, const int* d_out_host, int n_layers,
                          float* const* wcat_host, float* const* bias_host, void* stream);
/* E_out = Dropout(LeakyReLU_slope((S+E)·W1^T + (S*E)·W2^T + bias_eff)).
 *   mess_mult : optional [n_rows, d_out] multipliers standing in for nn.Dropout (mask injection);
 *   mess_p>0  : device-RNG inverted dropout keyed on (seed + *seed_dev, layer, element); ignored with mess_mult.
 *   mess_bits : optional output of ngcf_mess_dropout_bits for this layer (the same decisions, drawn once per step
 *               by a full-GPU pass instead of inside the 4 epilogue warps of each CTA); needs mess_p for 1/(1-p).
 *   row_offset: global index of row 0 (RNG keys only; 0 unless the rows are a shard of the full table). */
int ngcf_dense_fwd(const float* S, const float* E, int64_t n_rows, int d_in, int d_out,
                   const float* wcat, const float* bias_eff, float slope,
                   const float* mess_mult, const uint32_t* mess_bits, float mess_p, uint64_t seed,
                   const uint64_t* seed_dev, int layer, int64_t row_offset, float* E_out, void* stream);

/* Message-dropout decisions of one layer for a whole step: bits[row, col >> 5] bit (col & 31) = keep, for a
 * [n_rows, ceil(d_out/32)] uint32 array; same RNG stream as the in-kernel path (keyed on global rows). */
int ngcf_mess_dropout_bits(int64_t n_rows, int d_out, float mess_p, uint64_t seed, const uint64_t* seed_dev, int layer,
                           int64_t row_offset, uint32_t* bits, void* stream);

/* ---- output rows: NGCF.py:144-156 -------------------------------------------------------------------
 * out[b,:] = [ E0[r,:] | E1[r,:]/max(||E1[r,:]||,1e-12) | ... | EK[r,:]/max(...) ],  r = rows[b]+row_offset
 * (rows == NULL: r = b + row_offset, i.e. materialise all_E).  layers_host: K+1 device pointers
 * (E0, E'_1..E'_K, each contiguous [N, dims[k]]); dims_host: K+1 widths. */
int ngcf_gather_concat(const float* const* layers_host, const int* dims_host, int n_layers_plus1,
                       const int64_t* rows, int64_t row_offset, int64_t n_out,
                       float* out, int64_t ld_out, void* stream);
/* The same for up to four row sets at once (the user / positive / negative rows of a batch, NGCF.py:151-155): one launch;
 * set j gathers rows rows_host[j][i] + offsets_host[j] into outs_host[j] ([sizes_host[j], ld_out]). */
int ngcf_gather_concat_sets(const float* const* layers_host, const int* dims_host, int n_layers_plus1,
                            const int64_t* const* rows_host, const int64_t* offsets_host, const int64_t* sizes_host,
                            float* const* outs_host, int n_sets, int64_t ld_out, void* stream);

/* ---- LightGCN readout and its backward (lightgcn.py) -----------------------------------------------------------------
 * ngcf_layer_mean: out[b, :] = (E_0[r, :] + E_1[r, :] + ... + E_K[r, :]) * (1/(K+1)), summed in that order in fp32,
 * r = rows[b] + row_offset (rows == NULL: r = b + row_offset, i.e. all_users_emb / all_items_emb).  layers_host: K+1
 * device pointers to contiguous [N, d] layers, 1 <= d <= NGCF_MAX_WIDTH; out is [n_out, ld_out], ld_out >= d.
 * ngcf_layer_mean_sets: the same for up to four row sets at once (users / positives / negatives of a batch): set j
 * gathers rows rows_host[j][i] + offsets_host[j] into outs_host[j] ([sizes_host[j], ld_out]). */
int ngcf_layer_mean(const float* const* layers_host, int n_layers_plus1, int d, const int64_t* rows, int64_t row_offset,
                    int64_t n_out, float* out, int64_t ld_out, void* stream);
int ngcf_layer_mean_sets(const float* const* layers_host, int n_layers_plus1, int d, const int64_t* const* rows_host,
                         const int64_t* offsets_host, const int64_t* sizes_host, float* const* outs_host, int n_sets,
                         int64_t ld_out, void* stream);
/* The dense gradient of the last layer from a slot map (ngcf_rowgrad_scatter's slot / gsum):
 *   out[i, :] = slot[i] >= 0 ? scale * gsum[slot[i], :] : 0      for i < n_rows, and gsum[slot[i], :] *= scale in place,
 * so that ngcf_spmm's slot/gsum addend then adds the same scaled rows (LightGCN: scale = 1/(K+1), the readout's
 * weight).  Every slot must belong to one row only, as ngcf_rowgrad_scatter leaves them.  n_rows < 2^31,
 * 1 <= d <= NGCF_MAX_WIDTH, ld_gsum and ld_out >= d (row pitches in floats). */
int ngcf_rowgrad_expand(const int32_t* slot, int64_t n_rows, float* gsum, int64_t ld_gsum, int d, float scale,
                        float* out, int64_t ld_out, void* stream);

/* ---- BPR loss: bprloss.py:15-22, forward and row gradients in one kernel ------------------------------
 * loss = (-sum_b logsigmoid(|u_b.p_b| - |u_b.n_b|)
 *         + wd (reg_w_u sum|u_b|^2 + reg_w_p sum|p_b|^2 + reg_w_n sum|n_b|^2)) / batch_size_ctor  -> *loss (device)
 * reg_w_* are 1 except for an operand the caller broadcast from one row to `batch` rows
 * (experiment.py:96-100 passes pos_i_embeds[:1]), where it is 1/batch so the row is regularised once.
 * gu/gp/gn = dloss/du, /dp, /dn (each [batch, D]); pass all three NULL to skip the gradients. */
int ngcf_bpr_fwd_bwd(const float* u, const float* p, const float* n, int64_t batch, int D,
                     float weight_decay, float batch_size_ctor, float reg_w_u, float reg_w_p, float reg_w_n,
                     float* loss, float* gu, float* gp, float* gn, void* stream);

/* ---- backward of the row gather (IndexBackward, NGCF.py:151-155) as a slot map ----------------------
 * For the n_sets (<= 4) index sets (row ids rows[j][b] + offsets[j]) and their row gradients g[j]
 * ([batch_j, D]): pick one slot per distinct row
 * (slot[row] = index into gsum), and gsum[slot] = sum of that row's gradients.  slot must be all -1 on
 * entry ([N] int32); gsum is [sum batch_j, D] and is zeroed here.  ngcf_rowgrad_reset restores slot. */
int ngcf_rowgrad_scatter(const int64_t* const* rows_host, const int64_t* offsets_host,
                         const float* const* g_host, const int64_t* batch_host, int n_sets, int D,
                         int32_t* slot, float* gsum, void* stream);
/* In place, for every distinct row r of the sets (its slot s = slot[r]) and every block k >= 1 of the output row
 * (widths dims_host[k], layer k's stored E'_k in layers_host[k], as in ngcf_gather_concat):
 *   gsum[s, block k] <- (gH - H (H.gH)) / n,   n = max(||E'_k[r]||, 1e-12), H = E'_k[r] / n
 * i.e. the backward of F.normalize (NGCF.py:144) for the <= 3B rows that have an output-row gradient at all, done once
 * instead of inside every row tile of ngcf_dense_bwd (which is then called with gh_normalized = 1). */
int ngcf_rowgrad_normalize(const int64_t* const* rows_host, const int64_t* offsets_host,
                           const int64_t* batch_host, int n_sets, const float* const* layers_host,
                           const int* dims_host, int n_layers_plus1, const int32_t* slot, float* gsum, int D,
                           void* stream);
int ngcf_rowgrad_reset(const int64_t* const* rows_host, const int64_t* offsets_host,
                       const int64_t* batch_host, int n_sets, int32_t* slot, void* stream);

/* ---- row-local backward of one layer (AddmmBackward/LeakyReluBackward/normalize backward) -----------
 * With gH = gsum[slot[i], col_off .. col_off+d_out) (0 when slot[i] < 0), n = max(||E_out[i]||,1e-12),
 * H = E_out[i]/n:
 *   gE' = gE_next[i] (0 if NULL) + (gH - H (H.gH)) / n       (gh_normalized != 0: + gH as it is, see
 *                                                            ngcf_rowgrad_normalize)
 *   gM  = gE' * mess_mult * (E_out > 0 ? 1 : slope)         (sign(E_out) = sign(M); dropped -> 0)
 *   gS[i]  = gM·W1 + (gM·W2) * E[i]      gEl[i] = gM·W1 + (gM·W2) * S[i]
 *   gW1 += gM^T (S+E)   gb1 += 2 colsum(gM)   gW2 += gM^T (S*E)   gb2 += colsum(gM)   (atomic accumulate
 *   into caller-zeroed buffers).  W1/W2 are the nn.Linear weights, [d_out, d_in] row-major.
 *   gM_scratch: optional [n_rows, d_out] scratch; when given the tcgen05 path runs for d_in = 64 with d_out in
 *   {32, 64}, and for widths 64 / 128 on either side as 64-wide blocks (a 128-wide d_out needs gh_normalized): both
 *   GEMMs as 3xTF32 tensor-core products, the weight gradients accumulated in TMEM. */
/* Optional: the tensor-core weight-gradient launches of the following ngcf_dense_bwd calls (this thread) go to this
 * stream, ordered after the backward kernel by an event; the caller joins it before reading gW / gb and must not reuse
 * gM_scratch before then.  NULL restores single-stream operation. */
int ngcf_set_wgrad_stream(void* stream_or_null);
/* 1 if a weight-gradient launch went to that stream since the last call of this function (this thread), else 0: only
 * then is there anything to join (a layer on the FFMA kernels never forks; under CUDA-graph capture waiting on a
 * stream that holds no captured work is an error). */
int ngcf_wgrad_stream_forked(void);
int ngcf_dense_bwd(const float* gE_next, const int32_t* slot, const float* gsum, int64_t ld_gsum, int col_off,
                   const float* E_out, const float* S, const float* E, int64_t n_rows, int d_in, int d_out,
                   const float* W1, const float* W2, float slope,
                   const float* mess_mult, const uint32_t* mess_bits, float mess_p, uint64_t seed,
                   const uint64_t* seed_dev, int layer, int64_t row_offset, int gh_normalized, float* gS, float* gEl,
                   float* gW1, float* gb1, float* gW2, float* gb2, float* gM_scratch, void* stream);

/* ---- scoring: demo.py:234-235, experiment.py:93,104,109 ----------------------------------------------
 * scores = U·I^T without materialising them; per user row the k largest (descending; ties by lower item
 * id).  k <= 128.  workspace: ngcf_score_topk_workspace bytes. */
int ngcf_score_topk_workspace(int64_t n_users, int64_t n_items, int D, int k, size_t* bytes_host);
int ngcf_score_topk(const float* U, int64_t n_users, const float* I, int64_t n_items, int D, int k,
                    float* out_val /*[n_users,k]*/, int64_t* out_idx /*[n_users,k]*/,
                    void* workspace, size_t workspace_bytes, void* stream);
/* The same ranking with items removed per user (full-ranking evaluation: a user's training items are never
 * recommended).  Row u's items excl_idx[excl_ptr[u] .. excl_ptr[u+1]) must be ascending and unique (excl_idx may be
 * NULL when every row is empty); n_items < 2^31.  A row with fewer than k items left ends in slots of idx = -1,
 * val = -FLT_MAX.  workspace: ngcf_score_topk_workspace bytes.  k <= 32 with n_items >= 1024 and D % 4 == 0 runs on
 * the tensor cores like ngcf_score_topk; other shapes (k > 32 among them) run the much slower CUDA-core kernel. */
int ngcf_score_topk_excluding(const float* U, int64_t n_users, const float* I, int64_t n_items, int D, int k,
                              const int64_t* excl_ptr /*[n_users+1]*/, const int32_t* excl_idx,
                              float* out_val /*[n_users,k]*/, int64_t* out_idx /*[n_users,k]*/,
                              void* workspace, size_t workspace_bytes, void* stream);

/* ---- full-ranking metrics against held-out items ------------------------------------------------------------------
 * topk_idx [n_users,k]: ranked item ids per user (-1 = empty slot), e.g. from ngcf_score_topk_excluding; truth_ptr
 * [n_users+1] / truth_idx: per user the ascending unique held-out item ids.  For each of the n_K cut-offs Ks_host
 * (strictly ascending, 1 <= K <= k <= 128, n_K <= 8), with hits = how many of the first K ids are held out:
 *   recall = hits / |T|,  precision = hits / K,  hit = hits > 0,
 *   ndcg = sum over hit positions p < K of 1/log2(p+2)  /  sum over p < min(|T|, K) of 1/log2(p+2).
 * per_user [n_users, n_K, 4] = (recall, precision, ndcg, hit) per K; users with an empty T get zeros and are not
 * counted.  totals [n_K*4 + 1]: the means over the counted users (double sums in a fixed order: bit-reproducible;
 * 0 when none is counted), then the counted users' number. */
int ngcf_rank_metrics(const int64_t* topk_idx, int64_t n_users, int k, const int64_t* truth_ptr,
                      const int32_t* truth_idx, const int* Ks_host, int n_K, float* per_user, float* totals,
                      void* stream);

/* ---- optimizer step: torch.optim.Adam(model.parameters(), lr) of main.py:74, stepped at experiment.py:58 -----------
 * One launch over up to NGCF_ADAM_MAX_TENSORS parameter tensors (host arrays of device pointers, sizes in elements):
 *   g' = g + weight_decay p;  m = beta1 m + (1-beta1) g';  v = beta2 v + (1-beta2) g'^2;
 *   p -= lr / (1 - beta1^t) * m / (sqrt(v) / sqrt(1 - beta2^t) + eps)          (torch's non-amsgrad Adam)
 * t = step + *step_dev (step_dev: optional device counter, for CUDA-graph replay; t counts from 1).  zero_grads != 0
 * also clears the gradients (optimizer.zero_grad(), experiment.py:55) in the same pass.  Hyper-parameters are doubles:
 * 1 - beta and the bias corrections are formed in double like torch's Python floats, the element math is fp32. */
int ngcf_adam_step(float* const* params_host, float* const* grads_host, float* const* exp_avg_host,
                   float* const* exp_avg_sq_host, const int64_t* sizes_host, int n_tensors, double lr, double beta1,
                   double beta2, double eps, double weight_decay, int64_t step, const int64_t* step_dev,
                   int zero_grads, void* stream);

/* ---- evaluation metrics: the per-batch block of Experiment.eval, experiment.py:92-116, for all test groups at once
 * (SURVEY.md section 8(f) #4).  Rows g*group .. g*group+group-1 (group_ptr == NULL) or group_ptr[g] .. group_ptr[g+1]-1
 * (ragged batches, e.g. a DataLoader without drop_last; then `group` = the smallest group size, which the k's are
 * checked against, and every size must lie in [2, 128]) of u / items are what NGCF.forward returned for test
 * batch g (u_embeds, pos_i_embeds: row 0 the positive, rows 1.. the sampled negatives); item_ids / rating are the
 * batch's pos_item / rating columns (rating read at row 0 of each group).  Per group:
 *   scores[b] = u[0].items[b]                                   (pred_ratings[0], :93)
 *   bpr  = BPR(weight_decay, batch_size_ctor)(u, items[:1], cat(items[1:], items[1:2]))      (:95-101, bprloss.py:15-22)
 *   hit  = item_ids[0] among the ids of the k_hr best scores    (:104-106; the reference uses 3)
 *   ndcg = 1/log2(pos+2) if its position pos < k_ndcg else 0     (:109-111, :120-126)
 *   rmse = |scores[0] - rating[0]|                               (:114-116)
 * bpr/hit/ndcg/rmse: [n_groups] outputs; scores: optional [n_groups*group]; totals: optional float[4] =
 * {sum(bpr)/G, mean(hit), mean(ndcg), sum(rmse)/G}, the tuple eval() returns (:119).  2 <= group <= 128. */
int ngcf_eval_groups(const float* u, const float* items, const int64_t* item_ids, const float* rating,
                     const int64_t* group_ptr, int64_t n_groups, int group, int D, int k_hr, int k_ndcg, float weight_decay,
                     float batch_size_ctor, float* bpr, float* hit, float* ndcg, float* rmse, float* scores,
                     float* totals, void* stream);

/* ---- triple sampler: TourDataset._negative_sampling, utils.py:213-275 (SURVEY.md section 8(f) #3) --------------------
 * For positive row r of user row_user[r]: out[r, 0..ng_ratio) = ng_ratio DISTINCT candidates the user has no positive
 * feedback for, an ordered uniform sample without replacement (np.random.choice(neg_items, ng_ratio, replace=False),
 * utils.py:258).  candidates: the sorted unique item ids (np.setxor1d's universe, utils.py:224,240);
 * pos_ptr [n_user+1] / pos_idx: per user the ascending unique candidate INDICES of the positives.  Counter-based RNG
 * keyed on (seed, r, draw): reproducible, order-independent, not numpy's MT19937 stream.  *n_short counts rows
 * with fewer than ng_ratio free candidates (numpy raises there; their outputs are -1); caller zeroes it. */
int ngcf_sample_negatives(const int32_t* pos_ptr, const int32_t* pos_idx, const int64_t* row_user, int64_t n_rows,
                          const int64_t* candidates, int n_candidates, int ng_ratio, uint64_t seed, int64_t* out,
                          int32_t* n_short, void* stream);

/* ---- dynamic hard-negative sampling (DNS): the negative of each training row chosen on the device ----------------------
 * Layers / dims / n_layers_plus1 as ngcf_gather_concat takes them (E_0..E_K, [N, d_k] each, N = n_user + n_items).  For
 * batch row b of user u = u_id[b]: the user's final row is built as ngcf_gather_concat builds it (E_0 raw, blocks k >= 1
 * divided by max(||E_k row||, 1e-12)); then M candidates j = 0..M-1 are drawn with replacement, uniformly over the items
 * outside u's exclusion list excl_idx[excl_ptr[u] .. excl_ptr[u+1]) (ascending, unique item ids; excl_idx may be NULL
 * when every list is empty):  h = hash64(seed + *seed_dev, b, b >> 32, j, 'HNEG'),  r = (h.x * n_free) >> 32,
 * item = the r-th item not in the list.  Each candidate is scored as the dot product of the two final rows, and
 * chosen[b] = the candidate of largest |score| (ties: lowest j), an item id without the n_user offset.  |score| because
 * the BPR loss compares |u.p| with |u.n| (ngcf_bpr_fwd_bwd).  Every user in u_id must have a free item (n_free >= 1);
 * the caller checks that once (a row without one gets chosen = -1).  cand [batch, M] (int64) and score [batch, M]
 * (fp32) are optional debug outputs.  1 <= M <= 64, n_items < 2^31.  Allocates nothing, never synchronises
 * (capturable; seed_dev optional, as for dropout). */
int ngcf_hard_negatives(const float* const* layers_host, const int* dims_host, int n_layers_plus1, int64_t n_user,
                        const int64_t* u_id, int64_t batch, const int64_t* excl_ptr /*[n_user+1]*/,
                        const int32_t* excl_idx, int64_t n_items, int M, uint64_t seed, const uint64_t* seed_dev,
                        int64_t* chosen /*[batch]*/, int64_t* cand, float* score, void* stream);

/* Same draws, but chosen[b] = the candidate of largest SIGNED score (ties: lowest j): the hard negative of a softmax
 * loss (ngcf_softmax_loss), where a large negative score is an easy negative.  Same arguments and rules. */
int ngcf_hard_negatives_signed(const float* const* layers_host, const int* dims_host, int n_layers_plus1,
                               int64_t n_user, const int64_t* u_id, int64_t batch, const int64_t* excl_ptr,
                               const int32_t* excl_idx, int64_t n_items, int M, uint64_t seed, const uint64_t* seed_dev,
                               int64_t* chosen, int64_t* cand, float* score, void* stream);

/* Same draws and picks (signed_pick != 0: the largest signed score, else the largest |score|) on LightGCN's final rows:
 * the layer mean (E_0 + ... + E_K) / (K+1) of n_layers_plus1 layers of width d each, summed in ngcf_layer_mean's order,
 * for the user and for every candidate.  Other arguments and rules as ngcf_hard_negatives; 1 <= d <= NGCF_MAX_WIDTH. */
int ngcf_hard_negatives_mean(const float* const* layers_host, int d, int n_layers_plus1, int64_t n_user,
                             const int64_t* u_id, int64_t batch, const int64_t* excl_ptr, const int32_t* excl_idx,
                             int64_t n_items, int M, int signed_pick, uint64_t seed, const uint64_t* seed_dev,
                             int64_t* chosen, int64_t* cand, float* score, void* stream);

/* ---- in-batch sampled-softmax (InfoNCE) loss with its row gradients ---------------------------------------------------
 * u, p: [batch, D] fp32; n: [batch, D] or NULL (no explicit negatives).  Columns c_j = p_j (j < batch), then
 * c_{batch+j} = n_j; logits s_ij = u_i.c_j / temperature.  With item ids (pos_ids [batch], and neg_ids [batch] when n is
 * given; both NULL: no masking) column j is masked for row i iff j != i and id(c_j) == pos_ids[i]; repeated items
 * are not de-duplicated.
 *   loss[0] = (1/batch_size) sum_i [ logsumexp_{unmasked j} s_ij - s_ii + weight_decay (|u_i|^2 + |p_i|^2 + |n_i|^2) ]
 * and, when gu / gp (/ gn with n) are given, its gradients with respect to u, p and n (all NULL: forward only).
 * 1 <= batch <= 4096, 1 <= D <= 1152, temperature > 0, weight_decay >= 0, batch_size > 0.  The three products run on
 * the tensor cores (3xTF32); no atomics, the loss is summed in a fixed order in double: two calls on the same inputs
 * give the same bits.  workspace: ngcf_softmax_loss_workspace bytes for n_cols = batch (no n) or 2 * batch (a short
 * one: NGCF_ERR_WORKSPACE).  Allocates nothing, never synchronises (capturable). */
int ngcf_softmax_loss_workspace(int64_t batch, int n_cols, int D, size_t* bytes_host);
int ngcf_softmax_loss(const float* u, const float* p, const float* n, int64_t batch, int D, const int64_t* pos_ids,
                      const int64_t* neg_ids, float temperature, float weight_decay, float batch_size,
                      float* loss /*[1]*/, float* gu, float* gp, float* gn, void* workspace, size_t workspace_bytes,
                      void* stream);

/* ---- XSimGCL (xsimgcl.py): layer noise, cosine InfoNCE over distinct ids, view-2 row gradients --------------------
 * ngcf_perturb_rows, in place on rows r < n_rows of E ([n_rows, ld], 1 <= d <= NGCF_MAX_WIDTH, ld >= d):
 *   u_c = (hash64(seed + *seed_dev, r, c, layer, 'NOIS').x >> 8) * 2^-24            (uniform on [0, 1), c < d)
 *   E[r, c] += eps * sign(E[r, c]) * u_c / max(|u|, 1e-12)                         (sign(0) = 0)
 * One warp per row.  eps >= 0, 0 <= layer <= NGCF_MAX_LAYERS, n_rows < 2^31; seed_dev optional, as for dropout. */
int ngcf_perturb_rows(float* E, int64_t n_rows, int d, int64_t ld, float eps, uint64_t seed, const uint64_t* seed_dev,
                      int layer, void* stream);
/* ngcf_infonce: x1, x2 [batch, D] fp32, ids [batch].  Row i is valid iff ids[i] occurs in no earlier row (torch.unique
 * semantics at a fixed shape); U = the number of valid rows, found on the device.  With z = x / max(|x|, 1e-12) per row:
 *   loss[0] = (1/U) sum_{valid i} [ logsumexp_{valid j} (z1_i . z2_j / temperature) - z1_i . z2_i / temperature ]
 * and, when g1 / g2 are given, its gradients with respect to x1 and x2 (zero on the rows that are not valid).  The
 * products run on the softmax loss's tensor-core path; no atomics: two calls give the same bits.  1 <= batch <= 4096,
 * 1 <= D <= 1152, temperature > 0.  workspace: ngcf_infonce_workspace bytes (a short one: NGCF_ERR_WORKSPACE).
 * Allocates nothing, never synchronises (capturable). */
int ngcf_infonce_workspace(int64_t batch, int D, size_t* bytes_host);
int ngcf_infonce(const float* x1, const float* x2, int64_t batch, int D, const int64_t* ids, float temperature,
                 float* loss /*[1]*/, float* g1, float* g2, void* workspace, size_t workspace_bytes, void* stream);
/* ngcf_rowgrad_add: for each of the n_sets (<= 2) row sets (rows rows_host[j][b] + offsets_host[j], gradient rows
 * g_host[j] [batch_host[j], d]):  dst[t, :] += g_host[j][b, :]  with t = slot[row] (a slot map that ngcf_rowgrad_scatter
 * built over these rows), or t = row when slot is NULL (dst a dense [N, ld_dst] matrix).  Rows sharing a destination
 * are added with atomics, in no fixed order: the result is exact when at most one of them is non-zero, as with
 * ngcf_infonce's gradients.  1 <= d <= NGCF_MAX_WIDTH, ld_dst >= d. */
int ngcf_rowgrad_add(const int64_t* const* rows_host, const int64_t* offsets_host, const float* const* g_host,
                     const int64_t* batch_host, int n_sets, int d, const int32_t* slot, float* dst, int64_t ld_dst,
                     void* stream);

/* ---- Laplacian builder on the device: matrix.py:41-62 restricted to the non-zeros (SURVEY.md section 8(f) #2) ----------
 * From n_pairs DISTINCT (user, item, rating != 0) pairs: deg[N] = number of non-zeros per row of A = [[0,R],[R^T,0]]
 * (matrix.py:55), then the 2*n_pairs entries of L = D^-1/2 A D^-1/2 (matrix.py:56-62): entry e -> (user, n_user+item),
 * entry n_pairs+e -> (n_user+item, user), value = float(d_row * (rating * d_col)) with d = float32(deg^-1/2), the product
 * in double like the reference's float64 multi_dot.  Unsorted; the caller sorts row-major (matrix.py:79-83 emits sorted
 * indices) or feeds ngcf_coo_to_csr directly.  deg is cleared by the call. */
int ngcf_laplacian_entries(const int64_t* user, const int64_t* item, const float* rating, int64_t n_pairs,
                           int64_t n_user, int64_t n_item, int32_t* deg, int64_t* row, int64_t* col, float* val,
                           void* stream);

/* ---- debugging aids (tools/bwd_timeline.py, fwd_timeline.py, spmm_timeline.py); not part of the product path --------
 * ngcf_debug_bwd_timeline: switches the in-kernel SM-clock stamps of CTA 0 of the tcgen05 dense kernels on/off and
 * copies them back (out_host: int64[4*8*8] or NULL).  ngcf_debug_spmm_timeline: device buffer uint64[n_ctas*4]
 * ({start, staged, done, smid} in globaltimer ns) that every SpMM CTA stamps while it is set; NULL switches it off. */
int ngcf_debug_bwd_timeline(int enable, long long* out_host);
int ngcf_debug_spmm_timeline(unsigned long long* dev_buf_or_null);
int ngcf_debug_compact_timeline(unsigned long long* dev_buf_or_null);   /* same, row launch of the compaction pass */

#ifdef __cplusplus
}
#endif
#endif /* NGCF_B200_H */
