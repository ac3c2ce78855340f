// The two callers either side of the propagation path (SURVEY.md section 8(f) #3 and #4):
//   * ngcf_eval_groups    — Experiment.eval's per-batch metric block (experiment.py:92-116) for ALL test groups in
//                           one launch: scores of row 0 against the group's items, test BPR, HR@3, NDCG@ks, RMSE;
//   * ngcf_sample_negatives — TourDataset._negative_sampling (utils.py:213-275): for every positive row, ng_ratio
//                           distinct items the user has no positive feedback for, uniformly, without replacement.
//   * ngcf_laplacian_entries — the non-zeros of L = D^-1/2 A D^-1/2 from the rating pairs (matrix.py:41-62),
//                           section 8(f) #2.
//   * ngcf_hard_negatives  — dynamic hard-negative sampling inside a training step: per batch row, M free items
//                           scored against the user with the current layer outputs, the hardest one kept
//                           (ngcf_hard_negatives_mean: the same on LightGCN's layer-mean rows).
// All are small latency/HBM-bound integer + dot-product kernels; no tensor cores.
#include <limits.h>

#include "common.cuh"

namespace {

constexpr int EV_THREADS = 256;
constexpr int EV_WARPS = EV_THREADS / 32;
constexpr int EV_MAX_GROUP = 128;

// One CTA per test group (grid-stride).  Rows base .. base+group-1 of `u` / `it` (base = g*group, or group_ptr[g]
// for ragged groups) are what NGCF.forward returned for the group's batch: u_embeds and pos_i_embeds, row 0 = the
// positive, rows 1.. = the negatives.
template <bool VEC4>
__global__ void __launch_bounds__(EV_THREADS)
eval_groups_kernel(const float* __restrict__ u, const float* __restrict__ it, const int64_t* __restrict__ ids,
                   const float* __restrict__ rating, const int64_t* __restrict__ group_ptr, int64_t n_groups,
                   int group_fixed, int D, int k_hr, int k_ndcg,
                   float wd, float inv_bs, float* __restrict__ bpr, float* __restrict__ hit,
                   float* __restrict__ ndcg, float* __restrict__ rmse, float* __restrict__ scores) {
    __shared__ float s_score[EV_MAX_GROUP], s_up[EV_MAX_GROUP], s_un[EV_MAX_GROUP], s_nu[EV_MAX_GROUP],
        s_ni[EV_MAX_GROUP];
    __shared__ int s_pos;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int64_t g = blockIdx.x; g < n_groups; g += gridDim.x) {
        const int64_t base = group_ptr ? group_ptr[g] : g * group_fixed;
        const int group = group_ptr ? (int)(group_ptr[g + 1] - base) : group_fixed;
        if (group < 2 || group > EV_MAX_GROUP || k_hr > group || k_ndcg > group) {   // caller's contract broken
            if (threadIdx.x == 0) bpr[g] = hit[g] = ndcg[g] = rmse[g] = __int_as_float(0x7fc00000);
            continue;
        }
        const float* u0 = u + base * D;
        const float* p0 = it + base * D;
        if (threadIdx.x == 0) s_pos = INT_MAX;
        for (int b = warp; b < group; b += EV_WARPS) {
            // experiment.py:96-98: negatives = [p_1 .. p_{group-1}, p_1]
            const int nb = (b + 1 < group) ? b + 1 : 1;
            const float* ub = u + (base + b) * D;
            const float* pb = it + (base + b) * D;
            const float* nbp = it + (base + nb) * D;
            float sc = 0.f, up = 0.f, un = 0.f, nu = 0.f, ni = 0.f;
            // sc: pred_ratings[0, b], experiment.py:93; up: x_upos, bprloss.py:16 (positive row broadcast);
            // un: x_uneg, bprloss.py:17; nu / ni: the squared norms of bprloss.py:20-21
            if (VEC4) {                             // D % 4 == 0 and 16-byte aligned rows: 128-bit loads
                for (int c = lane; c < (D >> 2); c += 32) {
                    const float4 x = ld_stream_f4(ub + 4 * c), y = ld_f4(pb + 4 * c);
                    const float4 a = ld_f4(u0 + 4 * c), p = ld_f4(p0 + 4 * c), n = ld_f4(nbp + 4 * c);
                    sc = fmaf(a.x, y.x, fmaf(a.y, y.y, fmaf(a.z, y.z, fmaf(a.w, y.w, sc))));
                    up = fmaf(x.x, p.x, fmaf(x.y, p.y, fmaf(x.z, p.z, fmaf(x.w, p.w, up))));
                    un = fmaf(x.x, n.x, fmaf(x.y, n.y, fmaf(x.z, n.z, fmaf(x.w, n.w, un))));
                    nu = fmaf(x.x, x.x, fmaf(x.y, x.y, fmaf(x.z, x.z, fmaf(x.w, x.w, nu))));
                    ni = fmaf(y.x, y.x, fmaf(y.y, y.y, fmaf(y.z, y.z, fmaf(y.w, y.w, ni))));
                }
            } else {
                for (int c = lane; c < D; c += 32) {
                    const float x = ub[c], y = pb[c];
                    sc = fmaf(u0[c], y, sc);
                    up = fmaf(x, p0[c], up);
                    un = fmaf(x, nbp[c], un);
                    nu = fmaf(x, x, nu);
                    ni = fmaf(y, y, ni);
                }
            }
            sc = warp_sum(sc); up = warp_sum(up); un = warp_sum(un); nu = warp_sum(nu); ni = warp_sum(ni);
            if (lane == 0) { s_score[b] = sc; s_up[b] = up; s_un[b] = un; s_nu[b] = nu; s_ni[b] = ni; }
        }
        __syncthreads();
        // position of the ground-truth item id in the descending ranking (`pred_items.index(gt_item)`,
        // experiment.py:124-125): the best-ranked row whose id equals row 0's; ties rank the lower row first
        if ((int)threadIdx.x < group && ids[base + threadIdx.x] == ids[base]) {
            const float s = s_score[threadIdx.x];
            int r = 0;
            for (int i = 0; i < group; ++i) r += (s_score[i] > s) || (s_score[i] == s && i < (int)threadIdx.x);
            atomicMin(&s_pos, r);
        }
        if (scores)
            for (int b = threadIdx.x; b < group; b += EV_THREADS) scores[base + b] = s_score[b];
        __syncthreads();
        if (threadIdx.x == 0) {
            float logp = 0.f, reg = s_ni[0];                                  // ||pos[:1]||^2 once
            for (int b = 0; b < group; ++b) {
                const float x = fabsf(s_up[b]) - fabsf(s_un[b]);              // bprloss.py:18
                logp += fminf(x, 0.f) - log1pf(expf(-fabsf(x)));              // F.logsigmoid
                reg += s_nu[b] + s_ni[(b + 1 < group) ? b + 1 : 1];
            }
            bpr[g] = (-logp + wd * reg) * inv_bs;                             // bprloss.py:20-22
            const int pos = s_pos;
            hit[g] = pos < k_hr ? 1.f : 0.f;                                  // experiment.py:104-106, 127-130
            ndcg[g] = pos < k_ndcg ? 1.f / log2f((float)(pos + 2)) : 0.f;     // experiment.py:109-111, 120-126
            rmse[g] = fabsf(s_score[0] - rating[base]);                       // sqrt(mse(scalar, scalar)), :114-116
        }
        __syncthreads();
    }
}

// totals = {sum(bpr)/G, mean(hit), mean(ndcg), sum(rmse)/G} (experiment.py:119), fixed summation order
__global__ void __launch_bounds__(256)
eval_reduce_kernel(const float* __restrict__ bpr, const float* __restrict__ hit, const float* __restrict__ ndcg,
                   const float* __restrict__ rmse, int64_t n, float* __restrict__ totals) {
    __shared__ double sh[4][256];
    const float* src[4] = {bpr, hit, ndcg, rmse};
    for (int m = 0; m < 4; ++m) {
        double a = 0.0;
        for (int64_t i = threadIdx.x; i < n; i += 256) a += (double)src[m][i];
        sh[m][threadIdx.x] = a;
    }
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o)
            for (int m = 0; m < 4; ++m) sh[m][threadIdx.x] += sh[m][threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x < 4) totals[threadIdx.x] = (float)(sh[threadIdx.x][0] / (double)n);
}

// ---- negative sampler ------------------------------------------------------------------------------------------------
constexpr int NS_MAX = 64;                               // ng_ratio cap (reference: 1 for train, 24 for test)
#define NGCF_STREAM_SAMP 0x53414d50u                     // 'SAMP'

// index (in the candidate list) of the r-th candidate that is NOT one of the user's positives; p[0..deg) are the
// positives' candidate indices, ascending and unique: p[k]-k candidates below p[k] are free, so the answer is
// r + (number of k with p[k]-k <= r)
__device__ __forceinline__ int nth_free(const int32_t* __restrict__ p, int deg, int r) {
    int lo = 0, hi = deg;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (p[mid] - mid <= r) lo = mid + 1; else hi = mid;
    }
    return r + lo;
}

// One thread per positive row: an ordered uniform sample without replacement (what np.random.choice(neg, ng,
// replace=False) returns, utils.py:258) by a partial Fisher-Yates shuffle over the free-candidate index space
// [0, n_free), the displaced indices kept in a small per-thread map.
__global__ void __launch_bounds__(128)
sample_negatives_kernel(const int32_t* __restrict__ pos_ptr, const int32_t* __restrict__ pos_idx,
                        const int64_t* __restrict__ row_user, int64_t n_rows, const int64_t* __restrict__ cand,
                        int n_cand, int ng, uint64_t seed, int64_t* __restrict__ out, int32_t* __restrict__ n_short) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    const int64_t usr = row_user[row];
    const int32_t p0 = pos_ptr[usr];
    const int deg = pos_ptr[usr + 1] - p0;
    const int n_free = n_cand - deg;
    if (n_free < ng) {                                   // numpy: "Cannot take a larger sample than population"
        atomicAdd(n_short, 1);
        for (int j = 0; j < ng; ++j) out[row * ng + j] = -1;
        return;
    }
    int key[NS_MAX], val[NS_MAX];
    int n_map = 0;
    for (int j = 0; j < ng; ++j) {
        const uint2 h = ngcf_hash64(seed, (uint32_t)row, (uint32_t)(row >> 32), (uint32_t)j, NGCF_STREAM_SAMP);
        const int t = j + (int)(((uint64_t)h.x * (uint64_t)(n_free - j)) >> 32);     // uniform in [j, n_free)
        int vt = t, vj = j, it = -1;
        for (int m = 0; m < n_map; ++m) {
            if (key[m] == t) { vt = val[m]; it = m; }
            if (key[m] == j) vj = val[m];
        }
        if (it >= 0) val[it] = vj; else { key[n_map] = t; val[n_map] = vj; ++n_map; }   // a[t] = a[j]
        out[row * ng + j] = cand[nth_free(pos_idx + p0, deg, vt)];                     // pick a[t]
    }
}

// ---- dynamic hard negatives (DNS) -------------------------------------------------------------------------------------
constexpr int HN_WARPS = 4;                              // rows per CTA
constexpr int HN_MAX_M = 64;                             // candidates per row
constexpr int HN_GROUP = 4;                              // candidates scored together (loads in flight per lane)
constexpr int HN_Q = NGCF_MAX_WIDTH / 32;                // columns per lane of one layer block
#define NGCF_STREAM_HNEG 0x484e4547u                     // 'HNEG'

struct HardNegArgs {
    const float* layer[NGCF_MAX_LAYERS + 1];
    int dim[NGCF_MAX_LAYERS + 1];
    int n;
    int64_t n_user;
    const int64_t* u_id;
    int64_t batch;
    const int64_t* excl_ptr;
    const int32_t* excl_idx;
    int n_items;
    int M;
    uint64_t seed;
    const uint64_t* seed_dev;
    int64_t* chosen;
    int64_t* cand;
    float* score;
    float inv_n;                                         // kMean: 1 / n (last, so the other fields keep their offsets)
};

// One warp per batch row.  The user's final row (gather_row's formula: E_0 raw, E_k / max(||E_k||, 1e-12)) stays in
// registers; M candidates are drawn with replacement, uniformly over the items outside the user's exclusion list (lane
// l draws j = l and l + 32), and scored HN_GROUP at a time against the candidates' final rows, whose layer blocks are
// normalised on the fly.  Only the B*M candidate rows of E_0..E_K are read.
// kSigned: the pick is the largest signed score instead (the hard negative of a softmax loss).
// kMean: the final rows are LightGCN's layer mean (E_0 + ... + E_K) * inv_n, summed in ngcf_layer_mean's order, instead
// of the normalised concat; every layer then has the width dim[0].  The user's mean row is kept in ur[0].
template <bool kSigned, bool kMean>
__global__ void __launch_bounds__(HN_WARPS * 32) hard_negatives_kernel(HardNegArgs a) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * HN_WARPS + warp;
    if (row >= a.batch) return;
    const int64_t usr = a.u_id[row];
    float ur[NGCF_MAX_LAYERS + 1][HN_Q];
    if constexpr (kMean) {
        const int d = a.dim[0];
        float acc[HN_Q] = {};
#pragma unroll
        for (int k = 0; k <= NGCF_MAX_LAYERS; ++k) {
            if (k < a.n) {
                const float* src = a.layer[k] + usr * (int64_t)d;
#pragma unroll
                for (int q = 0; q < HN_Q; ++q) {
                    const int c = lane + 32 * q;
                    if (c < d) acc[q] += src[c];
                }
            }
        }
#pragma unroll
        for (int q = 0; q < HN_Q; ++q) ur[0][q] = acc[q] * a.inv_n;
    } else {
#pragma unroll
        for (int k = 0; k <= NGCF_MAX_LAYERS; ++k) {
            if (k < a.n) {
                const int d = a.dim[k];
                const float* src = a.layer[k] + usr * (int64_t)d;
                float ss = 0.f;
#pragma unroll
                for (int q = 0; q < HN_Q; ++q) {
                    const int c = lane + 32 * q;
                    ur[k][q] = c < d ? src[c] : 0.f;
                    ss = fmaf(ur[k][q], ur[k][q], ss);
                }
                if (k > 0) {
                    const float scale = 1.f / fmaxf(sqrtf(warp_sum(ss)), 1e-12f);   // F.normalize, NGCF.py:144
#pragma unroll
                    for (int q = 0; q < HN_Q; ++q) ur[k][q] *= scale;
                }
            }
        }
    }
    const int64_t p0 = a.excl_ptr[usr];
    const int deg = (int)(a.excl_ptr[usr + 1] - p0);
    const int n_free = a.n_items - deg;                  // >= 1: checked by the caller (HardNegatives)
    const uint64_t seed = ngcf_seed(a.seed, a.seed_dev);
    int item[2] = {-1, -1};
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int j = lane + 32 * h;
        if (j < a.M && n_free > 0) {
            const uint2 x = ngcf_hash64(seed, (uint32_t)row, (uint32_t)(row >> 32), (uint32_t)j, NGCF_STREAM_HNEG);
            const int r = (int)(((uint64_t)x.x * (uint64_t)n_free) >> 32);              // uniform in [0, n_free)
            item[h] = nth_free(a.excl_idx + p0, deg, r);
        }
    }
    // The loss is logsigmoid(|u.p| - |u.n|) (bprloss.py:18, bpr_kernel): a negative is hardest when its score is
    // largest in ABSOLUTE value, so the pick is the candidate of largest |score|, ties to the lowest j.
    float best = kSigned ? -INFINITY : -1.f;
    int best_item = __shfl_sync(FULL_MASK, item[0], 0);
    for (int j0 = 0; j0 < a.M; j0 += HN_GROUP) {
        int it[HN_GROUP];
#pragma unroll
        for (int g = 0; g < HN_GROUP; ++g) {
            const int j = j0 + g < a.M ? j0 + g : j0;   // a short last group repeats its first candidate
            it[g] = __shfl_sync(FULL_MASK, j < 32 ? item[0] : item[1], j & 31);
        }
        float sc[HN_GROUP] = {};
        if constexpr (kMean) {
            const int d = a.dim[0];
            float acc[HN_GROUP][HN_Q] = {};
#pragma unroll
            for (int k = 0; k <= NGCF_MAX_LAYERS; ++k) {
                if (k < a.n) {
#pragma unroll
                    for (int g = 0; g < HN_GROUP; ++g) {
                        const float* src = a.layer[k] + (a.n_user + it[g]) * (int64_t)d;
#pragma unroll
                        for (int q = 0; q < HN_Q; ++q) {
                            const int c = lane + 32 * q;
                            if (c < d) acc[g][q] += src[c];
                        }
                    }
                }
            }
#pragma unroll
            for (int g = 0; g < HN_GROUP; ++g) {
                float dot = 0.f;
#pragma unroll
                for (int q = 0; q < HN_Q; ++q) dot = fmaf(ur[0][q], acc[g][q] * a.inv_n, dot);
                sc[g] = warp_sum(dot);
            }
        } else {
#pragma unroll
            for (int k = 0; k <= NGCF_MAX_LAYERS; ++k) {
                if (k < a.n) {
                    const int d = a.dim[k];
                    float v[HN_GROUP][HN_Q];
#pragma unroll
                    for (int g = 0; g < HN_GROUP; ++g) {
                        const float* src = a.layer[k] + (a.n_user + it[g]) * (int64_t)d;
#pragma unroll
                        for (int q = 0; q < HN_Q; ++q) {
                            const int c = lane + 32 * q;
                            v[g][q] = c < d ? src[c] : 0.f;
                        }
                    }
#pragma unroll
                    for (int g = 0; g < HN_GROUP; ++g) {
                        float dot = 0.f, ss = 0.f;
#pragma unroll
                        for (int q = 0; q < HN_Q; ++q) {
                            dot = fmaf(ur[k][q], v[g][q], dot);
                            ss = fmaf(v[g][q], v[g][q], ss);
                        }
                        dot = warp_sum(dot);
                        sc[g] += k > 0 ? dot / fmaxf(sqrtf(warp_sum(ss)), 1e-12f) : dot;
                    }
                }
            }
        }
#pragma unroll
        for (int g = 0; g < HN_GROUP; ++g) {
            const int j = j0 + g;
            if (j < a.M) {
                const float key = kSigned ? sc[g] : fabsf(sc[g]);
                if (key > best) { best = key; best_item = it[g]; }
                if (lane == 0 && a.cand) a.cand[row * a.M + j] = it[g];
                if (lane == 0 && a.score) a.score[row * a.M + j] = sc[g];
            }
        }
    }
    if (lane == 0) a.chosen[row] = best_item;
}

// ---- Laplacian entries from the rating pairs (matrix.py:41-62, restricted to the non-zeros) ------------------------
__global__ void lap_degree_kernel(const int64_t* __restrict__ user, const int64_t* __restrict__ item, int64_t n_pairs,
                                  int64_t n_user, int32_t* __restrict__ deg) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_pairs) return;
    atomicAdd(&deg[user[e]], 1);                     // np.count_nonzero(adj_mat, axis=1), matrix.py:55
    atomicAdd(&deg[n_user + item[e]], 1);
}

// d^-1/2 as float32 (np.power(diag, -0.5, dtype=np.float32), matrix.py:56; inf -> 0, :57): the correctly rounded
// float of the exact value (numpy's SIMD float32 power is within ~3e-7 relative of it, not bit-identical)
__device__ __forceinline__ double lap_dinv(int32_t d) { return d > 0 ? (double)(float)(1.0 / sqrt((double)d)) : 0.0; }

__global__ void lap_entries_kernel(const int64_t* __restrict__ user, const int64_t* __restrict__ item,
                                   const float* __restrict__ rating, int64_t n_pairs, int64_t n_user,
                                   const int32_t* __restrict__ deg, int64_t* __restrict__ row,
                                   int64_t* __restrict__ col, float* __restrict__ val) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_pairs) return;
    const int64_t u = user[e], i = n_user + item[e];
    const double a = (double)rating[e], du = lap_dinv(deg[u]), di = lap_dinv(deg[i]);
    row[e] = u; col[e] = i; val[e] = (float)(du * (a * di));                        // A = [[0, R], [R^T, 0]], :49-53
    row[n_pairs + e] = i; col[n_pairs + e] = u; val[n_pairs + e] = (float)(di * (a * du));   // D^-1/2 A D^-1/2, :62
}

}  // namespace

extern "C" int ngcf_laplacian_entries(const int64_t* user, const int64_t* item, const float* rating, int64_t n_pairs,
                                      int64_t n_user, int64_t n_item, int32_t* deg, int64_t* row, int64_t* col,
                                      float* val, void* stream) {
    NGCF_REQUIRE(n_pairs >= 0 && n_user > 0 && n_item > 0, "laplacian_entries: bad sizes");
    NGCF_REQUIRE(deg, "laplacian_entries: null degree buffer");
    cudaStream_t st = as_stream(stream);
    NGCF_CUDA(cudaMemsetAsync(deg, 0, sizeof(int32_t) * (size_t)(n_user + n_item), st));
    if (n_pairs == 0) return NGCF_OK;
    NGCF_REQUIRE(user && item && rating && row && col && val, "laplacian_entries: null pointer");
    const unsigned grid = (unsigned)ceil_div64(n_pairs, 256);
    lap_degree_kernel<<<grid, 256, 0, st>>>(user, item, n_pairs, n_user, deg);
    NGCF_LAUNCH_OK("lap_degree_kernel");
    lap_entries_kernel<<<grid, 256, 0, st>>>(user, item, rating, n_pairs, n_user, deg, row, col, val);
    NGCF_LAUNCH_OK("lap_entries_kernel");
    return NGCF_OK;
}

extern "C" int ngcf_eval_groups(const float* u, const float* items, const int64_t* item_ids, const float* rating,
                                const int64_t* group_ptr, int64_t n_groups, int group, int D, int k_hr, int k_ndcg,
                                float weight_decay, float batch_size_ctor, float* bpr, float* hit, float* ndcg,
                                float* rmse, float* scores, float* totals, void* stream) {
    NGCF_REQUIRE(u && items && item_ids && rating && bpr && hit && ndcg && rmse, "eval_groups: null pointer");
    NGCF_REQUIRE(n_groups >= 0 && D > 0, "eval_groups: bad sizes (n_groups %lld, D %d)", (long long)n_groups, D);
    NGCF_REQUIRE(group >= 2 && group <= EV_MAX_GROUP, "eval_groups: group size %d outside [2, %d]", group,
                 EV_MAX_GROUP);
    // torch.topk(pred_ratings[0], k) raises for k > group (experiment.py:104,109)
    NGCF_REQUIRE(k_hr >= 1 && k_hr <= group && k_ndcg >= 1 && k_ndcg <= group,
                 "selected index k out of range (k_hr %d, k_ndcg %d, group %d)", k_hr, k_ndcg, group);
    NGCF_REQUIRE(batch_size_ctor != 0.f, "eval_groups: batch_size is 0");
    if (n_groups == 0) return NGCF_OK;
    cudaStream_t st = as_stream(stream);
    const int64_t grid = n_groups < (int64_t)ngcf_num_sms() * 8 ? n_groups : (int64_t)ngcf_num_sms() * 8;
    const bool vec4 = (D % 4 == 0) && (((uintptr_t)u | (uintptr_t)items) % 16 == 0);
    if (vec4)
        eval_groups_kernel<true><<<(unsigned)grid, EV_THREADS, 0, st>>>(
            u, items, item_ids, rating, group_ptr, n_groups, group, D, k_hr, k_ndcg, weight_decay,
            1.f / batch_size_ctor, bpr, hit, ndcg, rmse, scores);
    else
        eval_groups_kernel<false><<<(unsigned)grid, EV_THREADS, 0, st>>>(
            u, items, item_ids, rating, group_ptr, n_groups, group, D, k_hr, k_ndcg, weight_decay,
            1.f / batch_size_ctor, bpr, hit, ndcg, rmse, scores);
    NGCF_LAUNCH_OK("eval_groups_kernel");
    if (totals) {
        eval_reduce_kernel<<<1, 256, 0, st>>>(bpr, hit, ndcg, rmse, n_groups, totals);
        NGCF_LAUNCH_OK("eval_reduce_kernel");
    }
    return NGCF_OK;
}

extern "C" int ngcf_sample_negatives(const int32_t* pos_ptr, const int32_t* pos_idx, const int64_t* row_user,
                                     int64_t n_rows, const int64_t* candidates, int n_candidates, int ng_ratio,
                                     uint64_t seed, int64_t* out, int32_t* n_short, void* stream) {
    NGCF_REQUIRE(pos_ptr && row_user && candidates && out && n_short, "sample_negatives: null pointer");
    NGCF_REQUIRE(n_rows >= 0 && n_candidates > 0, "sample_negatives: bad sizes");
    NGCF_REQUIRE(ng_ratio >= 1 && ng_ratio <= NS_MAX, "sample_negatives: ng_ratio %d outside [1, %d]", ng_ratio, NS_MAX);
    if (n_rows == 0) return NGCF_OK;
    sample_negatives_kernel<<<(unsigned)ceil_div64(n_rows, 128), 128, 0, as_stream(stream)>>>(
        pos_ptr, pos_idx, row_user, n_rows, candidates, n_candidates, ng_ratio, seed, out, n_short);
    NGCF_LAUNCH_OK("sample_negatives_kernel");
    return NGCF_OK;
}

static int hard_negatives(bool is_signed, bool mean, const float* const* layers_host, const int* dims_host,
                          int n_layers_plus1, int64_t n_user, const int64_t* u_id, int64_t batch, const int64_t* excl_ptr,
                          const int32_t* excl_idx, int64_t n_items, int M, uint64_t seed, const uint64_t* seed_dev,
                          int64_t* chosen, int64_t* cand, float* score, void* stream) {
    NGCF_REQUIRE(layers_host && dims_host, "hard_negatives: null layer array");
    NGCF_REQUIRE(n_layers_plus1 >= 1 && n_layers_plus1 <= NGCF_MAX_LAYERS + 1, "hard_negatives: %d blocks",
                 n_layers_plus1);
    HardNegArgs a{};
    for (int k = 0; k < n_layers_plus1; ++k) {
        NGCF_REQUIRE(layers_host[k] && dims_host[k] > 0 && dims_host[k] <= NGCF_MAX_WIDTH, "hard_negatives: bad block %d",
                     k);
        NGCF_REQUIRE(!mean || dims_host[k] == dims_host[0], "hard_negatives: layer %d is %d wide, layer 0 %d", k,
                     dims_host[k], dims_host[0]);
        a.layer[k] = layers_host[k];
        a.dim[k] = dims_host[k];
    }
    NGCF_REQUIRE(n_user > 0, "hard_negatives: n_user %lld", (long long)n_user);
    NGCF_REQUIRE(n_items >= 1 && n_items <= INT_MAX, "hard_negatives: n_items %lld not in [1, 2^31-1]",
                 (long long)n_items);
    NGCF_REQUIRE(M >= 1 && M <= HN_MAX_M, "hard_negatives: M %d outside [1, %d]", M, HN_MAX_M);
    NGCF_REQUIRE(batch >= 0, "hard_negatives: batch %lld", (long long)batch);
    NGCF_REQUIRE(batch == 0 || (u_id && excl_ptr && chosen), "hard_negatives: null pointer");
    a.n = n_layers_plus1; a.inv_n = 1.0f / (float)n_layers_plus1; a.n_user = n_user; a.u_id = u_id; a.batch = batch; a.excl_ptr = excl_ptr;
    a.excl_idx = excl_idx; a.n_items = (int)n_items; a.M = M; a.seed = seed; a.seed_dev = seed_dev;
    a.chosen = chosen; a.cand = cand; a.score = score;
    if (batch == 0) return NGCF_OK;
    const unsigned grid = (unsigned)ceil_div64(batch, HN_WARPS);
    if (mean && is_signed)
        hard_negatives_kernel<true, true><<<grid, HN_WARPS * 32, 0, as_stream(stream)>>>(a);
    else if (mean)
        hard_negatives_kernel<false, true><<<grid, HN_WARPS * 32, 0, as_stream(stream)>>>(a);
    else if (is_signed)
        hard_negatives_kernel<true, false><<<grid, HN_WARPS * 32, 0, as_stream(stream)>>>(a);
    else
        hard_negatives_kernel<false, false><<<grid, HN_WARPS * 32, 0, as_stream(stream)>>>(a);
    NGCF_LAUNCH_OK("hard_negatives_kernel");
    return NGCF_OK;
}

extern "C" int ngcf_hard_negatives(const float* const* layers_host, const int* dims_host, int n_layers_plus1,
                                   int64_t n_user, const int64_t* u_id, int64_t batch, const int64_t* excl_ptr,
                                   const int32_t* excl_idx, int64_t n_items, int M, uint64_t seed,
                                   const uint64_t* seed_dev, int64_t* chosen, int64_t* cand, float* score,
                                   void* stream) {
    return hard_negatives(false, false, layers_host, dims_host, n_layers_plus1, n_user, u_id, batch, excl_ptr, excl_idx,
                          n_items, M, seed, seed_dev, chosen, cand, score, stream);
}

extern "C" int ngcf_hard_negatives_signed(const float* const* layers_host, const int* dims_host, int n_layers_plus1,
                                          int64_t n_user, const int64_t* u_id, int64_t batch, const int64_t* excl_ptr,
                                          const int32_t* excl_idx, int64_t n_items, int M, uint64_t seed,
                                          const uint64_t* seed_dev, int64_t* chosen, int64_t* cand, float* score,
                                          void* stream) {
    return hard_negatives(true, false, layers_host, dims_host, n_layers_plus1, n_user, u_id, batch, excl_ptr, excl_idx,
                          n_items, M, seed, seed_dev, chosen, cand, score, stream);
}

extern "C" int ngcf_hard_negatives_mean(const float* const* layers_host, int d, int n_layers_plus1, int64_t n_user,
                                        const int64_t* u_id, int64_t batch, const int64_t* excl_ptr,
                                        const int32_t* excl_idx, int64_t n_items, int M, int signed_pick, uint64_t seed,
                                        const uint64_t* seed_dev, int64_t* chosen, int64_t* cand, float* score,
                                        void* stream) {
    NGCF_REQUIRE(n_layers_plus1 >= 1 && n_layers_plus1 <= NGCF_MAX_LAYERS + 1, "hard_negatives: %d blocks",
                 n_layers_plus1);
    int dims[NGCF_MAX_LAYERS + 1];
    for (int k = 0; k < n_layers_plus1; ++k) dims[k] = d;
    return hard_negatives(signed_pick != 0, true, layers_host, dims, n_layers_plus1, n_user, u_id, batch, excl_ptr,
                          excl_idx, n_items, M, seed, seed_dev, chosen, cand, score, stream);
}
