// 3xTF32 GEMM main loop over packed operand images, shared by the fused scoring + top-k (topk_tc.cu) and the
// sampled-softmax loss (softmax_loss.cu).
//
// A pre-pass (score_pack_kernel) splits an fp32 operand once into TF32 hi / lo planes stored as ready-made operand
// blocks: per (128-row tile, 32-column K block) one 32-KB image (16-KB hi, 16-KB lo) of the 128-byte-swizzled K-major
// UMMA layout.  A CTA owns one 128-row tile of A and a range of 128-row tiles of B; one producer thread issues two
// 32-KB cp.async.bulk copies per K step into a 2-stage ring, and one thread issues the 3xTF32 tcgen05.mma chain into a
// double-buffered 128 x 128 fp32 accumulator in TMEM.  The kernels around it own the epilogue (TMEM lane = row of A).
#pragma once
#include "tc.cuh"

namespace {

using namespace tc;

constexpr int ST_ROWS = 128;                   // rows per tile of A (UMMA M) and of B (UMMA N)
constexpr int ST_EPI_WARPS = 4;
constexpr int ST_THREADS = (ST_EPI_WARPS + 2) * 32;                       // + MMA warp + producer warp
constexpr int ST_STAGES = 2;
constexpr int ST_BLOCK = ST_ROWS * 128;        // bytes of one 32-column K block of A or B (hi or lo)
constexpr int ST_STAGE_BYTES = 4 * ST_BLOCK;   // A hi, A lo, B hi, B lo

struct GemmBars {
    uint64_t full[ST_STAGES], empty[ST_STAGES], tmem_full[2], tmem_empty[2];
    uint32_t tmem_base;
};

// barriers and the 256 TMEM columns (2 accumulators x 128 fp32); ends in the block barrier that publishes them
__device__ __forceinline__ uint32_t gemm_setup(GemmBars* bars, int warp) {
    if (threadIdx.x == 0) {
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
    if (warp == ST_EPI_WARPS) tmem_alloc(&bars->tmem_base, 256);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    return bars->tmem_base;
}

__device__ __forceinline__ void gemm_teardown(uint32_t tmem_base, int warp) {
    tc_fence_before_sync();
    __syncthreads();
    if (warp == ST_EPI_WARPS) {
        tc_fence_after_sync();
        tmem_dealloc(tmem_base, 256);
    }
}

// MMA warp: for each of the n_t tiles of B, accumulator it & 1 = A tile · B tile over KB K blocks
__device__ __forceinline__ void gemm_issue(int n_t, int KB, uint8_t* ring, GemmBars* bars, uint32_t tmem_base, int lane) {
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
}

// producer (one thread): two 32-KB bulk copies per K step, A tile a_tile and B tiles b_tile0 .. b_tile0 + n_t - 1
__device__ __forceinline__ void gemm_produce(const uint8_t* Ap, const uint8_t* Bp, int64_t a_tile, int64_t b_tile0, int n_t,
                                             int KB, uint8_t* ring, GemmBars* bars) {
    const int total = n_t * KB;
    for (int s = 0; s < total; ++s) {
        const int it = s / KB, kb = s - it * KB, stg = s % ST_STAGES;
        mbar_wait(&bars->empty[stg], ((s / ST_STAGES) & 1) ^ 1);  // the MMAs that read this stage are done
        const uint32_t dst = smem_u32(ring + stg * ST_STAGE_BYTES), bar = smem_u32(&bars->full[stg]);
        const uint8_t* srcA = Ap + ((size_t)a_tile * KB + kb) * (2 * ST_BLOCK);
        const uint8_t* srcB = Bp + ((size_t)(b_tile0 + it) * KB + kb) * (2 * ST_BLOCK);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(ST_STAGE_BYTES) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(dst), "l"(srcA), "r"(2 * ST_BLOCK), "r"(bar) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(dst + 2 * ST_BLOCK), "l"(srcB), "r"(2 * ST_BLOCK), "r"(bar) : "memory");
    }
}

// Operand images: for row tile t and K block kb, a 16-KB hi image followed by a 16-KB lo image of the
// 128-byte-swizzled K-major layout; hi = x (the tensor core truncates to TF32), lo = x - trunc(x), or with kRna the
// round-to-nearest split of tc.cuh (split_tf32), whose errors do not share the sign of x: the choice for contractions
// over thousands of terms, where the truncating split's errors add up coherently.  The image holds
// KB_img K blocks per row tile and this call fills blocks kb0 .. kb0 + KB - 1.  Element (row r, k) is
//   X[r * ld + k]  (kT = false; rows r < n, k < D; rows / columns past the end are zero), or
//   X[k * ld + r]  (kT = true: the image of X^T; r < n, k < D; threads walk r fastest so the loads coalesce).
template <bool kT, bool kRna>
__global__ void __launch_bounds__(256) score_pack_kernel(const float* __restrict__ X, int64_t n, int D, int64_t ld,
                                                         int KB, int kb0, int KB_img, uint8_t* __restrict__ out,
                                                         int64_t n_chunks) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;     // one 16-byte chunk each
    if (i >= n_chunks) return;
    int c, kb;
    int64_t row;
    if (kT) {                                                             // (tile, kb, chunk, row in tile)
        const int64_t q = i >> 7;
        c = (int)(q & 7);
        kb = (int)((q >> 3) % KB);
        row = (q >> 3) / KB * ST_ROWS + (i & 127);
    } else {                                                              // (row, kb, chunk): row-major source
        c = (int)(i & 7);
        const int64_t rk = i >> 3;
        kb = (int)(rk % KB);
        row = rk / KB;
    }
    const int col = kb * 32 + c * 4;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < n) {
        if (!kT && col + 3 < D && (ld & 3) == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0) {
            x = ld_f4(X + row * ld + col);
        } else {
            float e[4];
#pragma unroll
            for (int q = 0; q < 4; ++q)
                e[q] = col + q < D ? X[kT ? (int64_t)(col + q) * ld + row : row * ld + col + q] : 0.f;
            x = make_float4(e[0], e[1], e[2], e[3]);
        }
    }
    float4 hi, lo;
    if (kRna)
        split_tf32(x, hi, lo);
    else
        split_tf32_trunc(x, hi, lo);
    const int64_t t = row / ST_ROWS;
    const uint32_t off = sw128_offset((uint32_t)(row % ST_ROWS), (uint32_t)c);
    uint8_t* blk = out + ((size_t)t * KB_img + kb0 + kb) * (2 * ST_BLOCK);
    *reinterpret_cast<float4*>(blk + off) = hi;
    *reinterpret_cast<float4*>(blk + ST_BLOCK + off) = lo;
}

// launches score_pack_kernel over every (row tile of n rows, K block) chunk: KB >= ceil(D / 32) blocks are filled, the
// columns past D with zeros
template <bool kRna>
int gemm_pack(bool transposed, const float* X, int64_t n, int D, int64_t ld, int KB, int kb0, int KB_img, uint8_t* out,
              cudaStream_t st) {
    const int64_t chunks = ceil_div64(n, ST_ROWS) * ST_ROWS * KB * 8;
    if (transposed)
        score_pack_kernel<true, kRna><<<(unsigned)ceil_div64(chunks, 256), 256, 0, st>>>(X, n, D, ld, KB, kb0, KB_img, out, chunks);
    else
        score_pack_kernel<false, kRna><<<(unsigned)ceil_div64(chunks, 256), 256, 0, st>>>(X, n, D, ld, KB, kb0, KB_img, out, chunks);
    NGCF_LAUNCH_OK(transposed ? "score_pack_kernel<T>" : "score_pack_kernel");
    return NGCF_OK;
}

}  // namespace
