// Full-ranking evaluation metrics (the protocol of the NGCF paper's Gowalla / Yelp2018 / Amazon-Book results): per test
// user the top-k list that ngcf_score_topk_excluding returned (training items already removed) against the user's
// held-out items, Recall / Precision / NDCG / Hit at up to 8 cut-offs K, then the means over the users that have
// held-out items.  Tiny latency-bound integer kernels: k binary searches per user, no tensor cores.
#include <limits.h>

#include "common.cuh"

namespace {

constexpr int RK_MAXK = 128;
constexpr int RK_MAXNK = 8;
constexpr int RK_WARPS = 8;
constexpr int RK_REDUCE = 256;

struct RankArgs {
    const int64_t* topk_idx;   // [n_users, k]; -1 = empty slot
    int64_t n_users;
    int k, n_K;
    const int64_t* truth_ptr;  // [n_users + 1]
    const int32_t* truth_idx;  // per user ascending unique item ids
    int Ks[RK_MAXNK];
    float* per_user;           // [n_users, n_K, 4]: recall, precision, ndcg, hit
};

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
    return v;
}

// one warp per user: lane l looks up list positions l, l+32, l+64, l+96 in the user's truth list; the ballots give the
// hit positions, from which every K's counts and discounted gains follow
__global__ void __launch_bounds__(RK_WARPS * 32) rank_metrics_kernel(RankArgs a) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t user = (int64_t)blockIdx.x * RK_WARPS + warp;
    if (user >= a.n_users) return;                                        // warp-uniform
    const int nm = a.n_K * 4;
    float* out = a.per_user + user * nm;
    const int64_t tb = a.truth_ptr[user], te = a.truth_ptr[user + 1];
    const int64_t nt = te - tb;
    if (nt <= 0) {                                                        // no held-out items: not counted
        for (int m = lane; m < nm; m += 32) out[m] = 0.f;
        return;
    }
    uint32_t found[RK_MAXK / 32];
#pragma unroll
    for (int q = 0; q < RK_MAXK / 32; ++q) {
        const int p = q * 32 + lane;
        bool f = false;
        if (p < a.k) {
            const int64_t id = a.topk_idx[user * a.k + p];
            if (id >= 0 && id <= INT_MAX) {
                const int64_t pos = lower_bound_i32(a.truth_idx, tb, te, (int)id);
                f = pos < te && a.truth_idx[pos] == (int32_t)id;
            }
        }
        found[q] = __ballot_sync(FULL_MASK, f);
    }
#pragma unroll
    for (int kk = 0; kk < RK_MAXNK; ++kk) {                              // unrolled: Ks stays in the parameter bank
        if (kk >= a.n_K) break;
        const int K = a.Ks[kk];
        const int64_t ideal = nt < K ? nt : K;
        int hits = 0;
        double dcg = 0.0, idcg = 0.0;
#pragma unroll
        for (int q = 0; q < RK_MAXK / 32; ++q) {
            const int p = q * 32 + lane;
            const int below = K - q * 32;                                 // positions of this group that are < K
            hits += __popc(below >= 32 ? found[q] : below > 0 ? found[q] & ((1u << below) - 1u) : 0u);
            const double w = 1.0 / log2((double)(p + 2));
            if (p < K && (found[q] >> lane & 1u)) dcg += w;
            if (p < ideal) idcg += w;
        }
        dcg = warp_sum_d(dcg);
        idcg = warp_sum_d(idcg);
        if (lane == 0) {
            out[kk * 4 + 0] = (float)((double)hits / (double)nt);
            out[kk * 4 + 1] = (float)((double)hits / (double)K);
            out[kk * 4 + 2] = (float)(dcg / idcg);
            out[kk * 4 + 3] = hits > 0 ? 1.f : 0.f;
        }
    }
}

// block m < nm: mean of metric m over the users with held-out items; block nm: their number.  Double sums in a fixed
// order (per thread a strided run, then a fixed tree), so repeated calls give identical bits.
__global__ void __launch_bounds__(RK_REDUCE)
rank_reduce_kernel(const float* __restrict__ per_user, const int64_t* __restrict__ truth_ptr, int64_t n_users, int nm,
                   float* __restrict__ totals) {
    __shared__ double sh[RK_REDUCE];
    __shared__ int64_t shc[RK_REDUCE];
    const int m = blockIdx.x;
    double s = 0.0;
    int64_t c = 0;
    for (int64_t u = threadIdx.x; u < n_users; u += RK_REDUCE) {
        c += truth_ptr[u + 1] > truth_ptr[u];
        if (m < nm) s += (double)per_user[u * nm + m];
    }
    sh[threadIdx.x] = s;
    shc[threadIdx.x] = c;
    __syncthreads();
    for (int o = RK_REDUCE / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) { sh[threadIdx.x] += sh[threadIdx.x + o]; shc[threadIdx.x] += shc[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) totals[m] = m == nm ? (float)shc[0] : shc[0] ? (float)(sh[0] / (double)shc[0]) : 0.f;
}

}  // namespace

extern "C" int ngcf_rank_metrics(const int64_t* topk_idx, int64_t n_users, int k, const int64_t* truth_ptr,
                                 const int32_t* truth_idx, const int* Ks_host, int n_K, float* per_user, float* totals,
                                 void* stream) {
    NGCF_REQUIRE(topk_idx && truth_ptr && Ks_host && per_user && totals, "rank_metrics: null pointer");
    NGCF_REQUIRE(n_users >= 0 && n_users <= 0x7fffffffLL, "rank_metrics: bad number of users %lld", (long long)n_users);
    NGCF_REQUIRE(k >= 1 && k <= RK_MAXK, "rank_metrics: k %d not in [1,%d]", k, RK_MAXK);
    NGCF_REQUIRE(n_K >= 1 && n_K <= RK_MAXNK, "rank_metrics: %d cut-offs, 1 to %d allowed", n_K, RK_MAXNK);
    RankArgs a{topk_idx, n_users, k, n_K, truth_ptr, truth_idx, {}, per_user};
    for (int i = 0; i < n_K; ++i) {
        NGCF_REQUIRE(Ks_host[i] >= 1 && Ks_host[i] <= k, "rank_metrics: K %d not in [1, k = %d]", Ks_host[i], k);
        NGCF_REQUIRE(i == 0 || Ks_host[i] > Ks_host[i - 1], "rank_metrics: cut-offs must be strictly ascending");
        a.Ks[i] = Ks_host[i];
    }
    cudaStream_t st = as_stream(stream);
    if (n_users > 0) {
        rank_metrics_kernel<<<(unsigned)ceil_div64(n_users, RK_WARPS), RK_WARPS * 32, 0, st>>>(a);
        NGCF_LAUNCH_OK("rank_metrics_kernel");
    }
    rank_reduce_kernel<<<n_K * 4 + 1, RK_REDUCE, 0, st>>>(per_user, truth_ptr, n_users, n_K * 4, totals);
    NGCF_LAUNCH_OK("rank_reduce_kernel");
    return NGCF_OK;
}
