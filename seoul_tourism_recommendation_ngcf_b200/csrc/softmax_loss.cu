// In-batch sampled-softmax (InfoNCE) loss with its row gradients, on the tensor cores.
//
// Columns c_j: p_j (j < B), then n_j (when negatives are given).  The column space is laid out in 128-column tiles:
// p occupies columns [0, Bp) and n columns [Bp, 2 Bp), Bp = B rounded up to 128, so every tile and every 32-column K
// block holds one of the two; padded columns are masked.  s_ij = u_i·c_j / tau; with item ids, column j is masked for
// row i iff j != i and id(c_j) == pos_ids[i].
//   loss = (1/bs) sum_i [ logsumexp_{j unmasked} s_ij - s_ii + wd (|u_i|^2 + |p_i|^2 + |n_i|^2) ]
//   G_ij = (P_ij - delta_ij) / (tau bs),  P_ij = m_ij exp(s_ij - LSE_i)
//   dL/du = G C + (2 wd / bs) u,   dL/d[p; n] = G^T U + (2 wd / bs) [p; n]
// Launches (one stream, no atomics, nothing allocated):
//   1. operand images of U and C (score_pack_kernel, tc_gemm.cuh, with the round-to-nearest 3xTF32 split: the
//      gradient products contract over up to 8192 terms), K-major along D, D zero-padded to 32;
//   2. S = U C^T on the tensor cores; the epilogue writes the masked logits (masked: -inf) and, per (row, column tile),
//      the running max and sum of exp;
//   3. softmax_row_kernel: per row, LSE from the partials in a fixed order, the row's loss term (double), and G in
//      place of S;  softmax_sum_kernel: the loss, summed in a fixed order in double;
//   4. images of G, G^T, C^T and U^T, then gU = G·C and [gP; gN] = G^T·U, the same main loop, tiled over D in
//      128-column blocks; the epilogue adds (2 wd / bs) x and stores each output row once.
// Forward only (no gradient buffers): steps 1-3 without G.
// softmax_run is shared with the cosine InfoNCE of xsimgcl.cu, which adds a validity mask (rows and columns outside it
// take no part: no loss term, masked as a column, zero gradient) and divides by the number of valid rows.
#include <math.h>

#include "softmax_core.cuh"
#include "tc_gemm.cuh"

namespace {

constexpr int SL_MAX_B = 4096;
constexpr int SL_MAX_D = 1152;
constexpr int SL_ROW_THREADS = 256;

enum { SL_LOGITS = 0, SL_GRAD_U = 1, SL_GRAD_C = 2 };

struct LossGemmArgs {
    const uint8_t* Aimg;       // operand images (tc_gemm.cuh)
    const uint8_t* Bimg;
    int KB;                    // K blocks of 32
    int n_b_tiles, tiles_per_split;
    int64_t B;
    int Bp;                    // B rounded up to 128: first column (SL_LOGITS) / row (SL_GRAD_C) of the negatives
    int ld;                    // SL_LOGITS: row pitch of S (n_col_tiles * 128)
    float inv_tau;
    const int64_t* pos_ids;    // NULL: no masking
    const int64_t* neg_ids;
    const uint8_t* valid;      // NULL: every column < B takes part
    float* S;                  // [B][ld]
    float2* part;              // [B][n_b_tiles]: (max, sum of exp) of the row's unmasked logits in the tile
    int D;
    float reg;                 // 2 wd / bs
    const float* x0;           // SL_GRAD_U: u -> out0 = gu;  SL_GRAD_C: p -> out0 = gp, n -> out1 = gn
    const float* x1;
    float* out0;
    float* out1;
};

template <int kMode>
__global__ void __launch_bounds__(ST_THREADS, 1) softmax_gemm_kernel(LossGemmArgs a) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* ring = smem_raw + (base - smem_u32(smem_raw));
    GemmBars* bars = reinterpret_cast<GemmBars*>(ring + ST_STAGES * ST_STAGE_BYTES);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int at = blockIdx.x;
    const int t0 = blockIdx.y * a.tiles_per_split, n_t = max(0, min(a.n_b_tiles, t0 + a.tiles_per_split) - t0);
    const uint32_t tmem_base = gemm_setup(bars, warp);

    if (warp < ST_EPI_WARPS) {
        const int64_t r = (int64_t)at * ST_ROWS + warp * 32 + lane;      // TMEM lane = row of A
        // the output row and its addend (row of x) of this thread, or none
        const float* xr = nullptr;
        float* orow = nullptr;
        bool live;
        int64_t my_id = 0;
        if (kMode == SL_LOGITS) {
            live = r < a.B;
            if (live && a.pos_ids) my_id = a.pos_ids[r];
        } else if (kMode == SL_GRAD_U) {
            live = r < a.B;
            if (live) { xr = a.x0 + r * a.D; orow = a.out0 + r * a.D; }
        } else {
            const int64_t q = r < a.Bp ? r : r - a.Bp;
            live = q < a.B;
            if (live) {
                xr = (r < a.Bp ? a.x0 : a.x1) + q * a.D;
                orow = (r < a.Bp ? a.out0 : a.out1) + q * a.D;
            }
        }
        for (int it = 0; it < n_t; ++it) {
            const int buf = it & 1, bt = t0 + it;
            mbar_wait(&bars->tmem_full[buf], (it >> 1) & 1);
            tc_fence_after_sync();
            float m = -INFINITY, sum = 0.f;
#pragma unroll 1
            for (int c = 0; c < ST_ROWS / 32; ++c) {
                float v[32];
                tmem_ld_32x32(tmem_base + ((uint32_t)(warp * 32) << 16) + buf * ST_ROWS + c * 32, v);
                if (c == ST_ROWS / 32 - 1) {                              // accumulator fully read
                    tc_fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars->tmem_empty[buf]);
                }
                const int j0 = bt * ST_ROWS + c * 32;
                if (kMode == SL_LOGITS) {
                    // the 32 columns lie on one side of Bp: all positives or all negatives
                    const bool neg = j0 >= a.Bp;
                    const int q0 = neg ? j0 - a.Bp : j0;
                    const int64_t* ids = neg ? a.neg_ids : a.pos_ids;
                    float cm = -INFINITY;
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) {
                        const int q = q0 + jj;
                        bool masked = q >= a.B;
                        if (!masked && a.pos_ids && (neg || q != r)) masked = ids[q] == my_id;
                        if (!masked && a.valid) masked = !a.valid[q];
                        v[jj] = masked ? -INFINITY : v[jj] * a.inv_tau;
                        cm = fmaxf(cm, v[jj]);
                    }
                    if (!live) continue;
                    float* srow = a.S + r * a.ld + j0;
#pragma unroll
                    for (int jj = 0; jj < 32; jj += 4) st_f4(srow + jj, make_float4(v[jj], v[jj + 1], v[jj + 2], v[jj + 3]));
                    if (cm == -INFINITY) continue;                        // every column of the chunk masked
                    const float mn = fmaxf(m, cm);
                    float s = sum * expf(m - mn);                         // m = -inf: exp(-inf) = 0
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) s += expf(v[jj] - mn);
                    m = mn;
                    sum = s;
                } else {
                    if (!live) continue;
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) {
                        const int d = j0 + jj;
                        if (d < a.D) orow[d] = fmaf(a.reg, xr[d], v[jj]);
                    }
                }
            }
            if (kMode == SL_LOGITS && live) a.part[r * a.n_b_tiles + bt] = make_float2(m, sum);
        }
    } else if (warp == ST_EPI_WARPS) {
        gemm_issue(n_t, a.KB, ring, bars, tmem_base, lane);
    } else if (lane == 0) {
        gemm_produce(a.Aimg, a.Bimg, at, t0, n_t, a.KB, ring, bars);
    }
    gemm_teardown(tmem_base, warp);
}

// fixed-order block sum (every thread gets it)
__device__ __forceinline__ float block_sum(float v, float* red) {
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < SL_ROW_THREADS / 32; ++w) s += red[w];
    return s;
}

// one block per row i: LSE_i from the per-tile partials (in tile order), the row's loss term, and (kGrad) G in place of S;
// a row outside `valid` has no loss term and a zero row of G
template <bool kGrad>
__global__ void __launch_bounds__(SL_ROW_THREADS) softmax_row_kernel(float* __restrict__ S, const float2* __restrict__ part,
                                                                     int n_tiles, int ld, const float* __restrict__ u,
                                                                     const float* __restrict__ p,
                                                                     const float* __restrict__ n, int D, float wd,
                                                                     float g_scale, const uint8_t* __restrict__ valid,
                                                                     double* __restrict__ row_loss) {
    __shared__ float red[SL_ROW_THREADS / 32];
    const int64_t i = blockIdx.x;
    float* srow = S + i * ld;
    if (valid && !valid[i]) {
        if (threadIdx.x == 0) row_loss[i] = 0.0;
        if (kGrad)
            for (int j = threadIdx.x * 4; j < ld; j += SL_ROW_THREADS * 4) st_f4(srow + j, make_float4(0.f, 0.f, 0.f, 0.f));
        return;
    }
    float m = -INFINITY;
    for (int t = 0; t < n_tiles; ++t) m = fmaxf(m, part[i * n_tiles + t].x);
    float sum = 0.f;
    for (int t = 0; t < n_tiles; ++t) {
        const float2 q = part[i * n_tiles + t];
        if (q.x != -INFINITY) sum += q.y * expf(q.x - m);
    }
    // LSE = m + lsum, kept apart: at |s| ~ 1e4 an fp32 LSE would round by 1e-3, and that error would enter every P
    const float lsum = logf(sum);                                         // the row's own positive keeps sum >= 1
    const float s_ii = srow[i];
    float su = 0.f, sp = 0.f, sn = 0.f;
    for (int c = threadIdx.x; c < D; c += SL_ROW_THREADS) {
        const float a = u[i * D + c], b = p[i * D + c];
        su = fmaf(a, a, su);
        sp = fmaf(b, b, sp);
        if (n) sn = fmaf(n[i * D + c], n[i * D + c], sn);
    }
    su = block_sum(su, red);                                              // (its barriers also order the read of s_ii
    sp = block_sum(sp, red);                                              //  before the write of G_ii below)
    sn = block_sum(sn, red);
    if (threadIdx.x == 0)
        row_loss[i] = ((double)m - (double)s_ii + (double)lsum) + (double)wd * ((double)su + (double)sp + (double)sn);
    if (kGrad) {
        for (int j = threadIdx.x * 4; j < ld; j += SL_ROW_THREADS * 4) {
            float4 s = ld_f4(srow + j);
            s.x = (expf((s.x - m) - lsum) - (j == i ? 1.f : 0.f)) * g_scale;
            s.y = (expf((s.y - m) - lsum) - (j + 1 == i ? 1.f : 0.f)) * g_scale;
            s.z = (expf((s.z - m) - lsum) - (j + 2 == i ? 1.f : 0.f)) * g_scale;
            s.w = (expf((s.w - m) - lsum) - (j + 3 == i ? 1.f : 0.f)) * g_scale;
            st_f4(srow + j, s);
        }
    }
}

// fixed-order sum of v over the block (strided partials, then a tree), in double; thread 0 gets it
__device__ __forceinline__ double block_sum_fixed(double v, double* red) {
    red[threadIdx.x] = v;
    __syncthreads();
    for (int w = SL_ROW_THREADS / 2; w > 0; w >>= 1) {
        if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
        __syncthreads();
    }
    return red[0];
}

// loss = sum_i row_loss[i] / bs, in a fixed order in double.  With `valid`, bs = the number of valid rows, and 1 / bs
// goes to *inv_count as well.
__global__ void __launch_bounds__(SL_ROW_THREADS) softmax_sum_kernel(const double* __restrict__ row_loss, int64_t B,
                                                                     double bs, const uint8_t* __restrict__ valid,
                                                                     float* __restrict__ loss,
                                                                     float* __restrict__ inv_count) {
    __shared__ double red[SL_ROW_THREADS];
    double s = 0.0, c = 0.0;
    for (int64_t i = threadIdx.x; i < B; i += SL_ROW_THREADS) {
        s += row_loss[i];
        if (valid) c += valid[i];
    }
    const double total = block_sum_fixed(s, red);
    if (valid) {
        __syncthreads();
        bs = block_sum_fixed(c, red);
    }
    if (threadIdx.x == 0) {
        *loss = (float)(total / bs);
        if (valid) *inv_count = (float)(1.0 / bs);
    }
}

// workspace layout; every region starts on a 1024-byte boundary (the operand images are read by bulk copies into
// 1024-byte-aligned swizzle atoms)
struct LossLayout {
    int64_t B;
    int Bp, n_col_tiles, n_cols_pad, KBd, Dt;
    size_t S, part, row_loss, U, C, G, GT, CT, UT, total;
};

inline size_t align1k(size_t x) { return (x + 1023) & ~(size_t)1023; }

LossLayout loss_layout(int64_t B, bool has_n, int D) {
    LossLayout L;
    L.B = B;
    L.Bp = (int)ceil_div64(B, ST_ROWS) * ST_ROWS;
    L.n_col_tiles = (has_n ? 2 : 1) * L.Bp / ST_ROWS;
    L.n_cols_pad = L.n_col_tiles * ST_ROWS;
    L.KBd = (D + 31) / 32;
    L.Dt = (int)ceil_div64(D, ST_ROWS);
    const size_t img = 2 * ST_BLOCK;                                      // bytes per (row tile, K block)
    const int bt = L.Bp / ST_ROWS;
    size_t o = 0;
    L.S = o;        o = align1k(o + (size_t)B * L.n_cols_pad * sizeof(float));
    L.part = o;     o = align1k(o + (size_t)B * L.n_col_tiles * sizeof(float2));
    L.row_loss = o; o = align1k(o + (size_t)B * sizeof(double));
    L.U = o;        o += (size_t)bt * L.KBd * img;
    L.C = o;        o += (size_t)L.n_col_tiles * L.KBd * img;
    L.G = o;        o += (size_t)bt * (L.n_cols_pad / 32) * img;
    L.GT = o;       o += (size_t)L.n_col_tiles * (L.Bp / 32) * img;
    L.CT = o;       o += (size_t)L.Dt * (L.n_cols_pad / 32) * img;
    L.UT = o;       o += (size_t)L.Dt * (L.Bp / 32) * img;
    L.total = o + 1024;                                                   // slack to align the caller's base
    return L;
}

template <int kMode>
int launch_gemm(LossGemmArgs a, int a_tiles, cudaStream_t st) {
    int64_t splits = ngcf_num_sms() / a_tiles;                            // one wave of CTAs
    if (splits > a.n_b_tiles) splits = a.n_b_tiles;
    if (splits < 1) splits = 1;
    a.tiles_per_split = (int)ceil_div64(a.n_b_tiles, splits);
    splits = ceil_div64(a.n_b_tiles, a.tiles_per_split);
    const size_t smem = 1024 + (size_t)ST_STAGES * ST_STAGE_BYTES + sizeof(GemmBars);
    NGCF_CUDA(cudaFuncSetAttribute(softmax_gemm_kernel<kMode>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    softmax_gemm_kernel<kMode><<<dim3((unsigned)a_tiles, (unsigned)splits), ST_THREADS, smem, st>>>(a);
    NGCF_LAUNCH_OK(kMode == SL_LOGITS ? "softmax_gemm_kernel<logits>" : "softmax_gemm_kernel<grad>");
    return NGCF_OK;
}

}  // namespace

size_t softmax_run_bytes(int64_t batch, bool has_n, int D) { return loss_layout(batch, has_n, D).total - 1024; }

extern "C" int ngcf_softmax_loss_workspace(int64_t batch, int n_cols, int D, size_t* bytes_host) {
    NGCF_REQUIRE(bytes_host, "softmax_loss_workspace: null pointer");
    NGCF_REQUIRE(batch >= 1 && batch <= SL_MAX_B, "softmax_loss_workspace: batch %lld not in [1, %d]", (long long)batch,
                 SL_MAX_B);
    NGCF_REQUIRE(D >= 1 && D <= SL_MAX_D, "softmax_loss_workspace: D %d not in [1, %d]", D, SL_MAX_D);
    NGCF_REQUIRE(n_cols == batch || n_cols == 2 * batch, "softmax_loss_workspace: n_cols %d is neither B nor 2B", n_cols);
    *bytes_host = loss_layout(batch, n_cols == 2 * batch, D).total;
    return NGCF_OK;
}

extern "C" int ngcf_softmax_loss(const float* u, const float* p, const float* n, int64_t batch, int D,
                                 const int64_t* pos_ids, const int64_t* neg_ids, float temperature, float weight_decay,
                                 float batch_size, float* loss, float* gu, float* gp, float* gn, void* workspace,
                                 size_t workspace_bytes, void* stream) {
    NGCF_REQUIRE(u && p && loss, "softmax_loss: null u, p or loss");
    NGCF_REQUIRE(batch >= 1 && batch <= SL_MAX_B, "softmax_loss: batch %lld not in [1, %d]", (long long)batch, SL_MAX_B);
    NGCF_REQUIRE(D >= 1 && D <= SL_MAX_D, "softmax_loss: D %d not in [1, %d]", D, SL_MAX_D);
    NGCF_REQUIRE(temperature > 0.f && isfinite(temperature), "softmax_loss: temperature %g is not > 0", temperature);
    NGCF_REQUIRE(weight_decay >= 0.f && isfinite(weight_decay), "softmax_loss: weight_decay %g is not >= 0", weight_decay);
    NGCF_REQUIRE(batch_size > 0.f && isfinite(batch_size), "softmax_loss: batch_size %g is not > 0", batch_size);
    NGCF_REQUIRE(!gn || n, "softmax_loss: gn given without n");
    NGCF_REQUIRE((gu && gp && (gn || !n)) || (!gu && !gp && !gn),
                 "softmax_loss: give every gradient buffer (gu, gp, and gn with n) or none");
    NGCF_REQUIRE(pos_ids || !neg_ids, "softmax_loss: neg_ids given without pos_ids");
    NGCF_REQUIRE(n || !neg_ids, "softmax_loss: neg_ids given without n");
    NGCF_REQUIRE(!pos_ids || !n || neg_ids, "softmax_loss: pos_ids and n given without neg_ids");
    const LossLayout L = loss_layout(batch, n != nullptr, D);
    if (!workspace || workspace_bytes < L.total) {
        ngcf_set_error("softmax_loss: workspace of %zu bytes, %zu needed", workspace ? workspace_bytes : (size_t)0,
                       L.total);
        return NGCF_ERR_WORKSPACE;
    }
    SoftmaxRun r{};
    r.u = u; r.p = p; r.n = n; r.batch = batch; r.D = D; r.pos_ids = pos_ids; r.neg_ids = neg_ids;
    r.temperature = temperature; r.weight_decay = weight_decay; r.batch_size = batch_size;
    r.loss = loss; r.gu = gu; r.gp = gp; r.gn = gn;
    return softmax_run(r, reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 1023) & ~(uintptr_t)1023),
                       as_stream(stream));
}

int softmax_run(const SoftmaxRun& r, uint8_t* ws, cudaStream_t st) {
    const float *u = r.u, *p = r.p, *n = r.n;
    const int64_t batch = r.batch;
    const int D = r.D;
    const bool grad = r.gu != nullptr;
    const LossLayout L = loss_layout(batch, n != nullptr, D);
    float* S = reinterpret_cast<float*>(ws + L.S);
    float2* part = reinterpret_cast<float2*>(ws + L.part);
    double* row_loss = reinterpret_cast<double*>(ws + L.row_loss);
    const int bt = L.Bp / ST_ROWS, KBc = L.n_cols_pad / 32, KBb = L.Bp / 32;

    // 1-2. S = U C^T with its per-tile (max, sum of exp)
    int rc = gemm_pack<true>(false, u, batch, D, D, L.KBd, 0, L.KBd, ws + L.U, st);
    if (rc == NGCF_OK) rc = gemm_pack<true>(false, p, batch, D, D, L.KBd, 0, L.KBd, ws + L.C, st);
    if (rc == NGCF_OK && n) rc = gemm_pack<true>(false, n, batch, D, D, L.KBd, 0, L.KBd, ws + L.C + (size_t)bt * L.KBd * 2 * ST_BLOCK, st);
    if (rc != NGCF_OK) return rc;
    LossGemmArgs a{};
    a.B = batch; a.Bp = L.Bp; a.D = D;
    a.Aimg = ws + L.U; a.Bimg = ws + L.C; a.KB = L.KBd; a.n_b_tiles = L.n_col_tiles;
    a.ld = L.n_cols_pad; a.inv_tau = 1.f / r.temperature; a.pos_ids = r.pos_ids; a.neg_ids = r.neg_ids;
    a.valid = r.valid; a.S = S; a.part = part;
    rc = launch_gemm<SL_LOGITS>(a, bt, st);
    if (rc != NGCF_OK) return rc;

    // 3. LSE, the row terms and G; the loss
    const float g_scale = 1.f / (r.temperature * r.batch_size);
    if (grad)
        softmax_row_kernel<true><<<(unsigned)batch, SL_ROW_THREADS, 0, st>>>(S, part, L.n_col_tiles, L.n_cols_pad, u, p, n,
                                                                             D, r.weight_decay, g_scale, r.valid,
                                                                             row_loss);
    else
        softmax_row_kernel<false><<<(unsigned)batch, SL_ROW_THREADS, 0, st>>>(S, part, L.n_col_tiles, L.n_cols_pad, u, p,
                                                                              n, D, r.weight_decay, g_scale, r.valid,
                                                                              row_loss);
    NGCF_LAUNCH_OK("softmax_row_kernel");
    softmax_sum_kernel<<<1, SL_ROW_THREADS, 0, st>>>(row_loss, batch, (double)r.batch_size, r.valid, r.loss,
                                                     r.inv_count);
    NGCF_LAUNCH_OK("softmax_sum_kernel");
    if (!grad) return NGCF_OK;

    // 4. images of G (rows i, K = j), G^T (rows j, K = i), C^T (rows d, K = j) and U^T (rows d, K = i); two GEMMs
    rc = gemm_pack<true>(false, S, batch, L.n_cols_pad, L.n_cols_pad, KBc, 0, KBc, ws + L.G, st);
    if (rc == NGCF_OK) rc = gemm_pack<true>(true, S, L.n_cols_pad, (int)batch, L.n_cols_pad, KBb, 0, KBb, ws + L.GT, st);
    if (rc == NGCF_OK) rc = gemm_pack<true>(true, p, D, (int)batch, D, KBb, 0, KBc, ws + L.CT, st);
    if (rc == NGCF_OK && n) rc = gemm_pack<true>(true, n, D, (int)batch, D, KBb, KBb, KBc, ws + L.CT, st);
    if (rc == NGCF_OK) rc = gemm_pack<true>(true, u, D, (int)batch, D, KBb, 0, KBb, ws + L.UT, st);
    if (rc != NGCF_OK) return rc;
    a.reg = 2.f * r.weight_decay / r.batch_size;
    a.n_b_tiles = L.Dt;
    a.Aimg = ws + L.G; a.Bimg = ws + L.CT; a.KB = KBc;
    a.x0 = u; a.out0 = r.gu;
    rc = launch_gemm<SL_GRAD_U>(a, bt, st);
    if (rc != NGCF_OK) return rc;
    a.Aimg = ws + L.GT; a.Bimg = ws + L.UT; a.KB = KBb;
    a.x0 = p; a.x1 = n; a.out0 = r.gp; a.out1 = r.gn;
    return launch_gemm<SL_GRAD_C>(a, L.n_col_tiles, st);
}
