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

#include "tc.cuh"

namespace {

using namespace tc;

constexpr int ST_ROWS = 128;                   // users per tile (UMMA M) and items per tile (UMMA N)
constexpr int ST_EPI_WARPS = 4;
constexpr int ST_THREADS = (ST_EPI_WARPS + 2) * 32;                       // + MMA warp + producer warp
constexpr int ST_STAGES = 2;
constexpr int ST_EXTRA = 64;                    // appended-but-not-yet-merged entries a user's list can hold
constexpr int ST_BLOCK = ST_ROWS * 128;        // bytes of one 32-column K block of A or B (hi or lo)
constexpr int ST_STAGE_BYTES = 4 * ST_BLOCK;   // A hi, A lo, B hi, B lo
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

struct ScoreBars {
    uint64_t full[ST_STAGES], empty[ST_STAGES], tmem_full[2], tmem_empty[2];
    uint32_t tmem_base;
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
    ScoreBars* bars = reinterpret_cast<ScoreBars*>(li + cap * ST_ROWS);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ut = blockIdx.x, sp = blockIdx.y;
    const int64_t u0 = (int64_t)ut * ST_ROWS;
    const int n_item_tiles = (int)((a.n_items + ST_ROWS - 1) / ST_ROWS);
    const int t0 = sp * a.tiles_per_split, t1 = min(n_item_tiles, t0 + a.tiles_per_split);
    const int n_t = max(0, t1 - t0);
    const int KB = (a.D + 31) / 32;

    if (tid == 0) {
        for (int i = 0; i < ST_STAGES; ++i) {
            mbar_init(&bars->full[i], 1);                               // the producer's arrive.expect_tx; TMA completes the bytes
            mbar_init(&bars->empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bars->tmem_full[i], 1);
            mbar_init(&bars->tmem_empty[i], ST_EPI_WARPS);
        }
        fence_mbar_init();
    }
    if (warp == ST_EPI_WARPS) tmem_alloc(&bars->tmem_base, 256);          // 2 accumulators x 128 fp32 columns
    for (int i = tid; i < a.k * ST_ROWS; i += ST_THREADS) { lv[i] = -FLT_MAX; li[i] = 0x7fffffff; }   // the k kept slots
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = bars->tmem_base;

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
        // ======================= MMA issuer =====================================================================
        const uint32_t idesc = umma_idesc_tf32(ST_ROWS, ST_ROWS, 0, 0);
        int step = 0;
        for (int it = 0; it < n_t; ++it) {
            const int buf = it & 1;
            mbar_wait(&bars->tmem_empty[buf], ((it >> 1) & 1) ^ 1);
            tc_fence_after_sync();
            const uint32_t tmem_d = tmem_base + buf * ST_ROWS;
            for (int kb = 0; kb < KB; ++kb, ++step) {
                const int stg = step % ST_STAGES;
                mbar_wait(&bars->full[stg], (step / ST_STAGES) & 1);
                tc_fence_after_sync();
                if (lane == 0) {
                    const uint32_t a_hi = smem_u32(ring + stg * ST_STAGE_BYTES), a_lo = a_hi + ST_BLOCK;
                    const uint32_t b_hi = a_lo + ST_BLOCK, b_lo = b_hi + ST_BLOCK;
#pragma unroll
                    for (int k8 = 0; k8 < 4; ++k8) {                      // 4 x (K = 8 TF32 = 32 bytes) per block
                        const uint64_t dah = umma_desc_sw128(a_hi + k8 * 32, 16, 1024);
                        const uint64_t dal = umma_desc_sw128(a_lo + k8 * 32, 16, 1024);
                        const uint64_t dbh = umma_desc_sw128(b_hi + k8 * 32, 16, 1024);
                        const uint64_t dbl = umma_desc_sw128(b_lo + k8 * 32, 16, 1024);
                        umma_tf32(tmem_d, dah, dbh, idesc, (kb | k8) ? 1u : 0u);
                        umma_tf32(tmem_d, dal, dbh, idesc, 1);
                        umma_tf32(tmem_d, dah, dbl, idesc, 1);
                    }
                    umma_commit(&bars->empty[stg]);                       // the stage may be refilled
                }
                __syncwarp();
            }
            if (lane == 0) umma_commit(&bars->tmem_full[buf]);            // accumulator complete
            __syncwarp();
        }
    } else {
        // ======================= producer: two 32-KB bulk copies per K step ========================================
        if (lane == 0) {
            const int total = n_t * KB;
            for (int s = 0; s < total; ++s) {
                const int it = s / KB, kb = s - it * KB, stg = s % ST_STAGES;
                mbar_wait(&bars->empty[stg], ((s / ST_STAGES) & 1) ^ 1);  // the MMAs that read this stage are done
                const uint32_t dst = smem_u32(ring + stg * ST_STAGE_BYTES), bar = smem_u32(&bars->full[stg]);
                const uint8_t* srcA = a.Up + ((size_t)ut * KB + kb) * (2 * ST_BLOCK);
                const uint8_t* srcB = a.Ip + ((size_t)(t0 + it) * KB + kb) * (2 * ST_BLOCK);
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(ST_STAGE_BYTES) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(dst), "l"(srcA), "r"(2 * ST_BLOCK), "r"(bar) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(dst + 2 * ST_BLOCK), "l"(srcB), "r"(2 * ST_BLOCK), "r"(bar) : "memory");
            }
        }
    }

    tc_fence_before_sync();
    __syncthreads();
    if (warp == ST_EPI_WARPS) {
        tc_fence_after_sync();
        tmem_dealloc(tmem_base, 256);
    }
}

// X [n, D] row-major fp32 -> operand blocks: for row tile t and K block kb, a 16-KB hi image followed by a 16-KB lo image
// of the 128-byte-swizzled K-major layout (rows / columns past the end are zero).  hi = x (the tensor core truncates to
// TF32), lo = x - trunc(x).
__global__ void __launch_bounds__(256) score_pack_kernel(const float* __restrict__ X, int64_t n, int D, int KB,
                                                         uint8_t* __restrict__ out, int64_t n_chunks) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;     // one 16-byte chunk each
    if (i >= n_chunks) return;
    const int c = (int)(i & 7);
    const int64_t rk = i >> 3;                                            // (tile, kb, row) with row fastest ... no: row-major source
    const int kb = (int)(rk % KB);
    const int64_t row = rk / KB;
    const int col = kb * 32 + c * 4;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < n && col < D) x = ld_f4(X + row * D + col);
    float4 hi, lo;
    split_tf32_trunc(x, hi, lo);
    const int64_t t = row / ST_ROWS;
    const uint32_t off = sw128_offset((uint32_t)(row % ST_ROWS), (uint32_t)c);
    uint8_t* blk = out + ((size_t)t * KB + kb) * (2 * ST_BLOCK);
    *reinterpret_cast<float4*>(blk + off) = hi;
    *reinterpret_cast<float4*>(blk + ST_BLOCK + off) = lo;
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
    {
        const int64_t cu = ut * ST_ROWS * KB * 8, ci = itiles * ST_ROWS * KB * 8;
        score_pack_kernel<<<(unsigned)ceil_div64(cu, 256), 256, 0, st>>>(U, n_users, D, KB, Up, cu);
        NGCF_LAUNCH_OK("score_pack_kernel(U)");
        score_pack_kernel<<<(unsigned)ceil_div64(ci, 256), 256, 0, st>>>(I, n_items, D, KB, Ip, ci);
        NGCF_LAUNCH_OK("score_pack_kernel(I)");
    }
    ScoreTcArgs a{Up, Ip, n_users, n_items, D, k, n_split, (int)((itiles + n_split - 1) / n_split), pv, pi, excl_ptr,
                  excl_idx};
    const size_t smem = 1024 + (size_t)ST_STAGES * ST_STAGE_BYTES + (size_t)(k + ST_EXTRA) * ST_ROWS * 8 + sizeof(ScoreBars);
    auto kern = excl_ptr ? score_topk_tc_kernel<true> : score_topk_tc_kernel<false>;
    NGCF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));   // per device
    dim3 grid((unsigned)ut, (unsigned)n_split);
    kern<<<grid, ST_THREADS, smem, st>>>(a);
    NGCF_LAUNCH_OK("score_topk_tc_kernel");
    return NGCF_OK;
}
