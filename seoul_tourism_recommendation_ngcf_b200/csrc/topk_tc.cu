// Fused scoring + top-k on the tensor cores (demo.py:234-235, experiment.py:93,104,109: scores = U·I^T, torch.topk).
//
// The first kernel (topk.cu) is one matrix-vector product per user: every user re-reads all item rows (43 GB out of L2
// for 1 024 users x 40 981 items x 256: 8.5 ms, eight times slower than torch's SGEMM + topk).  This one is a GEMM:
// a persistent CTA owns a 128-user tile and a range of 128-item tiles.  A pre-pass (score_pack_kernel) splits U and I
// once into TF32 hi / lo planes stored as ready-made operand blocks — per (128-row tile, 32-column K block) one
// 32-KB image of the 128-byte-swizzled K-major UMMA layout — so the GEMM's producer is ONE thread issuing two 32-KB
// cp.async.bulk (TMA) copies per K step into a 2-stage ring (first version: 8 loader warps re-split both operands for
// every tile pair and bounded the kernel at ~26 us per tile against 3.4 us of tensor work); one thread issues the 3xTF32
// tcgen05.mma chain into a double-buffered 128 x 128 fp32 accumulator in TMEM, and the epilogue threads (TMEM lane = user) filter the 128 scores of their user
// against that user's current k-th best and put the few survivors into that user's list in shared memory.  The score
// matrix never exists; partial lists per (user, item range) are merged by score_merge_kernel (topk.cu).
// Full-ranking evaluation drops each user's training items (kExclude): an epilogue thread visits its user's items in
// ascending order, so a cursor into the user's ascending exclusion list plus the next excluded id in a register turn
// each 32-item chunk into one compare (a 32-bit mask is built only when that id falls inside the chunk); no shared
// memory is added.
#include <float.h>
#include <limits.h>

#include "tc_gemm.cuh"

namespace {

constexpr int ST_EXTRA = 64;                    // appended-but-not-yet-merged entries a user's list can hold
constexpr int ST_MAXK = 32;

struct ScoreTcArgs {
    const uint8_t* Up;         // packed operand blocks of U: [user tile][K block][hi | lo][16 KB image]
    const uint8_t* Ip;         // ... of I
    int64_t n_users, n_items;
    int D, k, n_split;
    int tiles_per_split;       // item tiles per split
    float* pv;                 // [n_users][n_split][k]
    int* pi;
    const int64_t* excl_ptr;   // kExclude: per user [excl_ptr[u], excl_ptr[u+1]) of excl_idx, ascending unique item ids
    const int32_t* excl_idx;
};

// kExclude: items on the user's exclusion list never enter its lists (the false instantiation reads no list at all)
template <bool kExclude>
__global__ void __launch_bounds__(ST_THREADS, 1) score_topk_tc_kernel(ScoreTcArgs a) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
    uint8_t* ring = smem;                                                 // [ST_STAGES][A hi | A lo | B hi | B lo]
    float* lv = reinterpret_cast<float*>(ring + ST_STAGES * ST_STAGE_BYTES);   // [k + ST_EXTRA][128]: user lists, slot-major
    const int cap = a.k + ST_EXTRA;
    int* li = reinterpret_cast<int*>(lv + cap * ST_ROWS);
    GemmBars* bars = reinterpret_cast<GemmBars*>(li + cap * ST_ROWS);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ut = blockIdx.x, sp = blockIdx.y;
    const int64_t u0 = (int64_t)ut * ST_ROWS;
    const int n_item_tiles = (int)((a.n_items + ST_ROWS - 1) / ST_ROWS);
    const int t0 = sp * a.tiles_per_split, t1 = min(n_item_tiles, t0 + a.tiles_per_split);
    const int n_t = max(0, t1 - t0);
    const int KB = (a.D + 31) / 32;

    for (int i = tid; i < a.k * ST_ROWS; i += ST_THREADS) { lv[i] = -FLT_MAX; li[i] = 0x7fffffff; }   // the k kept slots
    const uint32_t tmem_base = gemm_setup(bars, warp);

    if (warp < ST_EPI_WARPS) {
        // ======================= epilogue: per-user top-k ==========================================================
        // Slots [0, k) hold the user's k best so far (unsorted), slots [k, k + ST_EXTRA) collect survivors of the filter
        // "score > k-th best as of the last merge" with two stores each.  When any user of the warp runs short of room
        // all 32 merge together (per extra entry: scan the k kept slots for the weakest, replace it if beaten), so the
        // cost of a merge is paid once per warp, not once per user.  (First version: every survivor was merged at once —
        // 32 independent users per warp made nearly every score column an event: 11 of the kernel's 14 ms.)
        const int row = warp * 32 + lane;                                 // TMEM lane = user row of the tile
        const bool live = u0 + row < a.n_users;
        const int k = a.k;
        float thr = -FLT_MAX;                                             // k-th best as of the last merge
        int cnt = k;                                                      // next free slot
        // exclusion cursor: the thread walks its items in ascending order, so one pointer into the user's ascending
        // list suffices; xnext is the next excluded id at or after the current chunk (INT_MAX: none left)
        int64_t xp = 0, xe = 0;
        int xnext = INT_MAX;
        if (kExclude && live) {
            xe = a.excl_ptr[u0 + row + 1];
            xp = lower_bound_i32(a.excl_idx, a.excl_ptr[u0 + row], xe, t0 * ST_ROWS);
            xnext = xp < xe ? a.excl_idx[xp] : INT_MAX;
        }
        auto merge = [&]() {
            const int extras = __reduce_max_sync(FULL_MASK, cnt) - k;
            for (int x = 0; x < extras; ++x) {
                const bool has = k + x < cnt;
                const float s = has ? lv[(k + x) * ST_ROWS + row] : -FLT_MAX;
                const int id = has ? li[(k + x) * ST_ROWS + row] : 0x7fffffff;
                float mv = lv[row];
                int mi = li[row], mp = 0;
#pragma unroll 4
                for (int p = 1; p < k; ++p) {                             // weakest kept entry: lowest score, then highest id
                    const float pv_ = lv[p * ST_ROWS + row];
                    const int pi_ = li[p * ST_ROWS + row];
                    if (pv_ < mv || (pv_ == mv && pi_ > mi)) { mv = pv_; mi = pi_; mp = p; }
                }
                if (has && s > mv) {                                      // (an equal score keeps the earlier item)
                    lv[mp * ST_ROWS + row] = s;
                    li[mp * ST_ROWS + row] = id;
                }
            }
            float mv = lv[row];
            for (int p = 1; p < k; ++p) mv = fminf(mv, lv[p * ST_ROWS + row]);
            thr = mv;
            cnt = k;
        };
        for (int it = 0; it < n_t; ++it) {
            const int buf = it & 1;
            const int64_t i0 = (int64_t)(t0 + it) * ST_ROWS;
            mbar_wait(&bars->tmem_full[buf], (it >> 1) & 1);
            tc_fence_after_sync();
#pragma unroll 1
            for (int c = 0; c < ST_ROWS / 32; ++c) {
                float v[32];
                tmem_ld_32x32(tmem_base + ((uint32_t)(warp * 32) << 16) + buf * ST_ROWS + c * 32, v);
                if (c == ST_ROWS / 32 - 1) {                              // accumulator fully read
                    tc_fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars->tmem_empty[buf]);
                }
                if (__any_sync(FULL_MASK, cnt > k + ST_EXTRA - 32)) merge();   // room for a whole chunk of survivors
                if (!live) continue;
                uint32_t xmask = 0;                                       // bit j: item i0 + c*32 + j is excluded
                if (kExclude) {
                    const int cb = (int)(i0 + c * 32);
                    while (xnext < cb + 32) {                             // usually one compare per chunk
                        xmask |= 1u << (xnext - cb);
                        xnext = ++xp < xe ? a.excl_idx[xp] : INT_MAX;
                    }
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float s = v[j];
                    const int64_t item = i0 + c * 32 + j;
                    // NaN fails the comparison and is never ranked
                    if (s > thr && item < a.n_items && !(xmask >> j & 1u)) {
                        lv[cnt * ST_ROWS + row] = s;
                        li[cnt * ST_ROWS + row] = (int)item;
                        ++cnt;
                    }
                }
            }
        }
        merge();
        if (live) {
            float* ov = a.pv + ((u0 + row) * a.n_split + sp) * k;
            int* oi = a.pi + ((u0 + row) * a.n_split + sp) * k;
            for (int j = 0; j < k; ++j) { ov[j] = lv[j * ST_ROWS + row]; oi[j] = li[j * ST_ROWS + row]; }
        }
    } else if (warp == ST_EPI_WARPS) {
        gemm_issue(n_t, KB, ring, bars, tmem_base, lane);
    } else if (lane == 0) {
        gemm_produce(a.Up, a.Ip, ut, t0, n_t, KB, ring, bars);
    }
    gemm_teardown(tmem_base, warp);
}

}  // namespace

bool ngcf_score_topk_tc_eligible(int64_t n_users, int64_t n_items, int D, int k) {
    return n_users >= 1 && n_items >= 1024 && D % 4 == 0 && D >= 32 && k <= ST_MAXK;
}

// item splits so that user tiles x splits covers the SMs a few times over
int ngcf_score_topk_tc_splits(int64_t n_users, int64_t n_items) {
    const int64_t ut = (n_users + ST_ROWS - 1) / ST_ROWS, itiles = (n_items + ST_ROWS - 1) / ST_ROWS;
    int64_t s = (int64_t)ngcf_num_sms() / ut;                            // one wave of CTAs; long item ranges amortise
    if (s > itiles) s = itiles;                                           // the warm-up of the per-user lists
    if (s > 32) s = 32;                                                   // the per-user merge of the partial lists is serial
    if (s < 1) s = 1;
    return (int)s;
}

// bytes of the packed copies of U and I that ngcf_score_topk_tc needs behind the partial lists
size_t ngcf_score_topk_tc_pack_bytes(int64_t n_users, int64_t n_items, int D) {
    const size_t KB = (size_t)(D + 31) / 32;
    const size_t ut = (size_t)(n_users + ST_ROWS - 1) / ST_ROWS, it = (size_t)(n_items + ST_ROWS - 1) / ST_ROWS;
    return (ut + it) * KB * 2 * ST_BLOCK + 1024;
}

// excl_ptr / excl_idx: NULL for plain ranking, else per user the ascending unique item ids that are never ranked
int ngcf_score_topk_tc(const float* U, int64_t n_users, const float* I, int64_t n_items, int D, int k, int n_split,
                       float* pv, int* pi, uint8_t* pack, const int64_t* excl_ptr, const int32_t* excl_idx,
                       cudaStream_t st) {
    const int KB = (D + 31) / 32;
    const int64_t ut = (n_users + ST_ROWS - 1) / ST_ROWS, itiles = (n_items + ST_ROWS - 1) / ST_ROWS;
    uint8_t* Up = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(pack) + 1023) & ~(uintptr_t)1023);
    uint8_t* Ip = Up + (size_t)ut * KB * 2 * ST_BLOCK;
    int rc = gemm_pack<false>(false, U, n_users, D, D, KB, 0, KB, Up, st);
    if (rc == NGCF_OK) rc = gemm_pack<false>(false, I, n_items, D, D, KB, 0, KB, Ip, st);
    if (rc != NGCF_OK) return rc;
    ScoreTcArgs a{Up, Ip, n_users, n_items, D, k, n_split, (int)((itiles + n_split - 1) / n_split), pv, pi, excl_ptr,
                  excl_idx};
    const size_t smem = 1024 + (size_t)ST_STAGES * ST_STAGE_BYTES + (size_t)(k + ST_EXTRA) * ST_ROWS * 8 + sizeof(GemmBars);
    auto kern = excl_ptr ? score_topk_tc_kernel<true> : score_topk_tc_kernel<false>;
    NGCF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));   // per device
    dim3 grid((unsigned)ut, (unsigned)n_split);
    kern<<<grid, ST_THREADS, smem, st>>>(a);
    NGCF_LAUNCH_OK("score_topk_tc_kernel");
    return NGCF_OK;
}
