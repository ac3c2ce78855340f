// Fused scoring + top-k (demo.py:234-235: torch.mm(u_embeds, all_i_emb.T) then torch.topk;
// experiment.py:93,104,109).  The U x I score matrix is never written to HBM.
//
// v1: grid = (user, item split).  A CTA keeps its user row in shared memory, its warps stream item rows
// (coalesced, one dot product per warp via shuffle reduction) and keep a sorted per-warp top-k list in
// shared memory; the lists are merged per CTA, then per user by a second kernel.
#include <float.h>
#include <limits.h>

#include "common.cuh"

namespace {

constexpr int TK_WARPS = 4;
constexpr int TK_MAXK = 128;

__device__ __forceinline__ bool better(float v, int i, float v2, int i2) {
    return v > v2 || (v == v2 && i < i2);
}

// insert (s, id) into a descending list of length k held in shared memory; called by a whole warp with
// warp-uniform arguments
__device__ __forceinline__ void warp_insert(float* lv, int* li, int k, float s, int id, int lane) {
    if (!better(s, id, lv[k - 1], li[k - 1])) return;
    int cnt = 0;
    for (int j = lane; j < k; j += 32) cnt += better(lv[j], li[j], s, id) ? 1 : 0;
    const int pos = (int)warp_sum((float)cnt);
    float tv[TK_MAXK / 32];
    int ti[TK_MAXK / 32];
#pragma unroll
    for (int q = 0; q < TK_MAXK / 32; ++q) {
        const int j = lane + 32 * q;
        if (j >= pos && j < k - 1) { tv[q] = lv[j]; ti[q] = li[j]; }
    }
    __syncwarp();
#pragma unroll
    for (int q = 0; q < TK_MAXK / 32; ++q) {
        const int j = lane + 32 * q;
        if (j >= pos && j < k - 1) { lv[j + 1] = tv[q]; li[j + 1] = ti[q]; }
    }
    if (lane == 0) { lv[pos] = s; li[pos] = id; }
    __syncwarp();
}

// kExclude: the items of the user's ascending exclusion list [excl_ptr[user], excl_ptr[user+1]) of excl_idx are skipped
template <bool kExclude>
__global__ void __launch_bounds__(TK_WARPS * 32)
score_partial_kernel(const float* __restrict__ U, const float* __restrict__ I, int64_t n_items, int D, int k,
                     int n_split, float* __restrict__ pv, int* __restrict__ pi, const int64_t* __restrict__ excl_ptr,
                     const int32_t* __restrict__ excl_idx) {
    extern __shared__ __align__(16) float smem[];
    float* us = smem;                                  // [D]
    float* lv = us + ((D + 3) & ~3);                   // [TK_WARPS][k]
    int* li = reinterpret_cast<int*>(lv + TK_WARPS * k);
    const int user = blockIdx.x, split = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int c = threadIdx.x; c < D; c += blockDim.x) us[c] = U[(int64_t)user * D + c];
    for (int j = threadIdx.x; j < TK_WARPS * k; j += blockDim.x) { lv[j] = -FLT_MAX; li[j] = 0x7fffffff; }
    __syncthreads();
    const int64_t per = (n_items + n_split - 1) / n_split;
    const int64_t i0 = split * per, i1 = min(n_items, i0 + per);
    float* mylv = lv + warp * k;
    int* myli = li + warp * k;
    // exclusion cursor of the warp (warp-uniform): it visits its items in ascending order
    const int32_t *xp = nullptr, *xe = nullptr;
    int xnext = INT_MAX;
    if (kExclude) {
        const int64_t e = excl_ptr[user + 1];
        xp = excl_idx + lower_bound_i32(excl_idx, excl_ptr[user], e, (int)(i0 + warp));
        xe = excl_idx + e;
        xnext = xp < xe ? *xp : INT_MAX;
    }
    for (int64_t it = i0 + warp; it < i1; it += TK_WARPS) {
        if (kExclude) {
            while (xnext < it) xnext = ++xp < xe ? *xp : INT_MAX;
            if (xnext == it) continue;
        }
        const float* ir = I + it * D;
        float s = 0.f;
        for (int c = lane; c < D; c += 32) s = fmaf(us[c], ir[c], s);
        s = warp_sum(s);
        if (s == s) warp_insert(mylv, myli, k, s, (int)it, lane);      // NaN scores are never ranked
    }
    __syncthreads();
    // merge the per-warp lists: warp 0 inserts the others' entries into its own
    if (warp == 0) {
        for (int w = 1; w < TK_WARPS; ++w)
            for (int j = 0; j < k; ++j) {
                const float s = lv[w * k + j];
                const int id = li[w * k + j];
                if (id == 0x7fffffff) break;
                warp_insert(mylv, myli, k, s, id, lane);
            }
        float* ov = pv + ((int64_t)user * n_split + split) * k;
        int* oi = pi + ((int64_t)user * n_split + split) * k;
        for (int j = lane; j < k; j += 32) { ov[j] = lv[j]; oi[j] = li[j]; }
    }
}

// one warp per user: merge n_split sorted partial lists
__global__ void __launch_bounds__(32)
score_merge_kernel(const float* __restrict__ pv, const int* __restrict__ pi, int n_split, int k,
                   float* __restrict__ out_val, int64_t* __restrict__ out_idx) {
    extern __shared__ __align__(16) float smem[];
    float* lv = smem;
    int* li = reinterpret_cast<int*>(lv + k);
    const int user = blockIdx.x, lane = threadIdx.x;
    const float* v = pv + (int64_t)user * n_split * k;
    const int* ix = pi + (int64_t)user * n_split * k;
    for (int j = lane; j < k; j += 32) { lv[j] = -FLT_MAX; li[j] = 0x7fffffff; }
    __syncwarp();
    for (int sp = 0; sp < n_split; ++sp)                               // partial lists need not be sorted
        for (int j = 0; j < k; ++j) {
            const float s = v[sp * k + j];
            const int id = ix[sp * k + j];
            if (id == 0x7fffffff) continue;
            warp_insert(lv, li, k, s, id, lane);
        }
    for (int j = lane; j < k; j += 32) {
        out_val[(int64_t)user * k + j] = lv[j];
        out_idx[(int64_t)user * k + j] = li[j] == 0x7fffffff ? -1 : (int64_t)li[j];
    }
}

int pick_split(int64_t n_users, int64_t n_items) {
    const int64_t target = (int64_t)ngcf_num_sms() * 8;            // CTAs wanted in flight
    int64_t s = (target + n_users - 1) / n_users;
    const int64_t max_by_items = (n_items + 255) / 256;           // at least ~256 items per CTA
    if (s > max_by_items) s = max_by_items;
    if (s < 1) s = 1;
    if (s > 64) s = 64;
    return (int)s;
}

}  // namespace

bool ngcf_score_topk_tc_eligible(int64_t n_users, int64_t n_items, int D, int k);
int ngcf_score_topk_tc_splits(int64_t n_users, int64_t n_items);
size_t ngcf_score_topk_tc_pack_bytes(int64_t n_users, int64_t n_items, int D);
int ngcf_score_topk_tc(const float* U, int64_t n_users, const float* I, int64_t n_items, int D, int k, int n_split,
                       float* pv, int* pi, uint8_t* pack, const int64_t* excl_ptr, const int32_t* excl_idx,
                       cudaStream_t st);

extern "C" int ngcf_score_topk_workspace(int64_t n_users, int64_t n_items, int D, int k, size_t* bytes_host) {
    NGCF_REQUIRE(bytes_host, "score_topk_workspace: null pointer");
    NGCF_REQUIRE(n_users >= 0 && n_items >= 0 && k > 0 && k <= TK_MAXK, "score_topk_workspace: bad sizes");
    const int64_t nu = n_users > 0 ? n_users : 1;
    const int ns = max(pick_split(nu, n_items), ngcf_score_topk_tc_splits(nu, n_items));   // either kernel fits
    *bytes_host = (size_t)nu * ns * k * 8 + 256;
    if (D > 0 && ngcf_score_topk_tc_eligible(nu, n_items, D, k)) *bytes_host += ngcf_score_topk_tc_pack_bytes(nu, n_items, D);
    return NGCF_OK;
}

// ngcf_score_topk and ngcf_score_topk_excluding; excl_ptr == NULL: no exclusion (the kernels that read no list)
static int score_topk_impl(const float* U, int64_t n_users, const float* I, int64_t n_items, int D, int k,
                           const int64_t* excl_ptr, const int32_t* excl_idx, float* out_val, int64_t* out_idx,
                           void* workspace, size_t workspace_bytes, void* stream) {
    NGCF_REQUIRE(U && I && out_val && out_idx, "score_topk: null pointer");
    NGCF_REQUIRE(k > 0 && k <= TK_MAXK, "score_topk: k %d not in [1,%d]", k, TK_MAXK);
    NGCF_REQUIRE(k <= n_items, "score_topk: k %d > number of items %lld (torch.topk raises too)", k, (long long)n_items);
    NGCF_REQUIRE(D > 0 && n_users >= 0 && n_users < 65536 * 32768LL, "score_topk: bad sizes");
    if (n_users == 0) return NGCF_OK;
    size_t need = 0;
    int rc = ngcf_score_topk_workspace(n_users, n_items, D, k, &need);
    if (rc != NGCF_OK) return rc;
    if (!workspace || workspace_bytes < need) {
        ngcf_set_error("score_topk: workspace %zu bytes < required %zu", workspace_bytes, need);
        return NGCF_ERR_WORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    if (ngcf_score_topk_tc_eligible(n_users, n_items, D, k) &&
        (reinterpret_cast<uintptr_t>(U) & 15) == 0 && (reinterpret_cast<uintptr_t>(I) & 15) == 0) {
        // GEMM-shaped path on the tensor cores (topk_tc.cu); partial lists per item range, merged below
        const int ns = ngcf_score_topk_tc_splits(n_users, n_items);
        float* pv = reinterpret_cast<float*>(workspace);
        int* pi = reinterpret_cast<int*>(pv + (size_t)n_users * ns * k);
        uint8_t* pack = reinterpret_cast<uint8_t*>(pi + (size_t)n_users * ns * k);
        if ((rc = ngcf_score_topk_tc(U, n_users, I, n_items, D, k, ns, pv, pi, pack, excl_ptr, excl_idx, st)) != NGCF_OK)
            return rc;
        score_merge_kernel<<<(unsigned)n_users, 32, sizeof(float) * 2 * k, st>>>(pv, pi, ns, k, out_val, out_idx);
        NGCF_LAUNCH_OK("score_merge_kernel");
        return NGCF_OK;
    }
    const int ns = pick_split(n_users, n_items);
    float* pv = reinterpret_cast<float*>(workspace);
    int* pi = reinterpret_cast<int*>(pv + (size_t)n_users * ns * k);
    const size_t smem1 = sizeof(float) * (((D + 3) & ~3) + 2 * TK_WARPS * k);
    NGCF_REQUIRE(smem1 <= 48 * 1024, "score_topk: D %d too wide for the v1 kernel", D);
    NGCF_REQUIRE(n_users <= 0x7fffffffLL, "score_topk: too many users");
    dim3 grid((unsigned)n_users, (unsigned)ns);
    if (excl_ptr)
        score_partial_kernel<true><<<grid, TK_WARPS * 32, smem1, st>>>(U, I, n_items, D, k, ns, pv, pi, excl_ptr, excl_idx);
    else
        score_partial_kernel<false><<<grid, TK_WARPS * 32, smem1, st>>>(U, I, n_items, D, k, ns, pv, pi, nullptr, nullptr);
    NGCF_LAUNCH_OK("score_partial_kernel");
    score_merge_kernel<<<(unsigned)n_users, 32, sizeof(float) * 2 * k, st>>>(pv, pi, ns, k, out_val, out_idx);
    NGCF_LAUNCH_OK("score_merge_kernel");
    return NGCF_OK;
}

extern "C" int ngcf_score_topk(const float* U, int64_t n_users, const float* I, int64_t n_items, int D, int k,
                               float* out_val, int64_t* out_idx, void* workspace, size_t workspace_bytes,
                               void* stream) {
    return score_topk_impl(U, n_users, I, n_items, D, k, nullptr, nullptr, out_val, out_idx, workspace, workspace_bytes,
                           stream);
}

extern "C" int ngcf_score_topk_excluding(const float* U, int64_t n_users, const float* I, int64_t n_items, int D, int k,
                                         const int64_t* excl_ptr, const int32_t* excl_idx, float* out_val,
                                         int64_t* out_idx, void* workspace, size_t workspace_bytes, void* stream) {
    NGCF_REQUIRE(excl_ptr, "score_topk_excluding: null exclusion row pointer");
    NGCF_REQUIRE(n_items <= 0x7fffffffLL, "score_topk_excluding: more than 2^31-1 items");
    return score_topk_impl(U, n_users, I, n_items, D, k, excl_ptr, excl_idx, out_val, out_idx, workspace,
                           workspace_bytes, stream);
}
