// Tensor-core (tcgen05 / TMEM) version of the per-layer forward epilogue, NGCF.py:131-142:
//     E_out = Dropout(LeakyReLU((S+E)·W1^T + (S*E)·W2^T + 2 b1 + b2))
// as ONE GEMM per 128-row tile:  [128 x 2d] · [2d x d_out], A = [S+E | S*E] built on the fly, B = [W1 | W2]
// resident in shared memory for the whole (persistent) kernel, fp32 accumulator in TMEM, 3xTF32 (tc.cuh).
// The accumulator is double buffered in TMEM so the epilogue of tile t overlaps the loads and MMAs of tile t+1
// (warp roles: dense_fwd_tma_kernel).
#include <stdlib.h>

#include "tc.cuh"
#include "tmap.h"

namespace {

using namespace tc;

// optional per-role timeline of CTA 0 (tools/bwd_timeline.py): SM clock at the protocol points of each tile
__device__ long long g_bwd_dbg[4][8][8];   // [3][tile][k] = loader warp 0 inside its tile: first half computed, next loads issued, second half, fence
__device__ int g_bwd_dbg_on = 0;
#define BWD_STAMP(role, it, k)                                                   \
    do {                                                                         \
        if (dbg && lane == 0 && (it) < 8) g_bwd_dbg[role][it][k] = clock64();    \
    } while (0)

constexpr int TC_ROWS = 128;                 // UMMA M
constexpr int TC_EPI_WARPS = 4;
constexpr int TC_LOAD_WARPS = 8;
constexpr int TC_THREADS = (TC_EPI_WARPS + 1 + TC_LOAD_WARPS) * 32;
constexpr int TC_MAX_KB = 4;                 // K blocks of 32 TF32 (128 bytes): 2*d_in/32 <= 4  ->  d_in <= 64
constexpr int TC_A_BLOCK = TC_ROWS * 128;    // bytes of one K block of A (hi or lo)

struct FwdTcArgs {
    const float* S;
    const float* E;
    int64_t n_rows;
    int d_in, d_out;
    const float* wcat;        // [2*d_in, d_out]: wcat[k][o] = W1[o][k] (k < d_in), W2[o][k-d_in]
    const float* bias_eff;    // [d_out]
    float slope;
    const float* mess_mult;
    const uint32_t* mess_bits;
    float mess_p;
    uint64_t seed;
    const uint64_t* seed_dev;
    int layer;
    float* E_out;
    int n_tiles;
    int64_t row_off;          // global index of local row 0 (RNG keys only)
    // block decomposition of layers wider than 64 (d_in / d_out above are the BLOCK's widths): this launch contracts
    // columns [in_off, in_off + d_in) of S / E (row stride ld_in) against rows w_row1.. (W1 part) and w_row2.. (W2 part),
    // columns [out_off, out_off + d_out) of wcat (row stride d_out_full) into columns [out_off, ..) of E_out (row
    // stride d_out_full).  mode: FW_SINGLE = bias + activation; FW_PARTIAL = store the raw partial sums;
    // FW_FINAL = add the partial sums found in E_out, then bias + activation.
    int64_t ld_in;
    int in_off, w_row1, w_row2, out_off, d_out_full, mode;
};
enum { FW_SINGLE = 0, FW_PARTIAL = 1, FW_FINAL = 2 };

// Forward roles: warps 0-7 epilogue (warp w: TMEM lane quarter w & 3, 32-column chunk w >> 2), warp 8 MMA issuer.
// (ncu, first version with 4 epilogue + 8 loader warps: the loaders sat idle 59 % of the time waiting for the
// epilogue — bias/LeakyReLU/dropout RNG for 128 x 64 outputs per tile in 4 warps was the critical path.)
constexpr int FW_EPI_WARPS = 8;
constexpr int FW_MMA_WARP = FW_EPI_WARPS;

// 32 x 32 fp32 transposition buffer without padding: 16-byte chunk c of row r lives at chunk position c ^ (r & 7)
__device__ __forceinline__ int stage_off(int r, int c) { return r * 32 + ((c ^ (r & 7)) << 2); }

// message-dropout source, a compile-time mode so the per-element code is branch-free and the unrolled chains interleave
// (with run-time tests inside the loops the compiler kept every iteration a separate basic block: no overlap of
// the ~45-deep integer hash chains, measured 1200 cycles per 4-element step in the backward's loader)
enum { MM_NONE = 0, MM_MULT = 1, MM_BITS = 2, MM_HASH = 3 };
static inline int mess_mode(const float* mess_mult, const uint32_t* mess_bits, float mess_p) {
    return mess_mult ? MM_MULT : (mess_p > 0.f ? (mess_bits ? MM_BITS : MM_HASH) : MM_NONE);
}

// ======================= forward epilogue role (8 warps) =================================================================
// TMEM lane = tile row, so a thread holds one row of its chunk; the 32x32 block goes through a per-warp transposition
// buffer so that bias + LeakyReLU + dropout run, and the stores are issued, in a coalesced layout.
template <int MM>
__device__ __forceinline__ void fwd_epilogue_role(const FwdTcArgs& a, float* stage, const float* bias_s, uint64_t* tmem_full,
                                                  uint64_t* tmem_empty, uint32_t tmem_base, int n_my, int warp, int lane,
                                                  bool dbg) {
    const int d_out = a.d_out;
    // ======================= epilogue =======================================================================
    // TMEM lane = tile row, so a thread holds one row of its chunk; bias + LeakyReLU + dropout are applied in that
    // layout, then the 32x32 block goes through a per-warp transposition buffer so the stores are coalesced.
    const uint64_t seed = MM == MM_HASH ? ngcf_seed(a.seed, a.seed_dev) : 0ull;
    const uint32_t thr = ngcf_threshold16(a.mess_p);
    float* st = stage + warp * 32 * 32;
    const int quarter = warp & 3, c = warp >> 2;                      // TMEM lanes 32*quarter.., columns 32*c..
    const int rr = lane >> 3, c4 = lane & 7;                          // read-back mapping: 4 rows x 8 float4
    const bool has_chunk = c * 32 < d_out;
    const float inv_keep = 1.0f / (1.0f - a.mess_p);
    for (int it = 0; it < n_my; ++it) {
        const int tile = blockIdx.x + it * gridDim.x;
        const int buf = it & 1;
        BWD_STAMP(0, it, 0);
        mbar_wait(&tmem_full[buf], (it >> 1) & 1);
        BWD_STAMP(0, it, 1);
        tc_fence_after_sync();
        float v[32];
        if (has_chunk) tmem_ld_32x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * 64 + c * 32, v);
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tmem_empty[buf]);           // accumulator drained: next tile may reuse it
        BWD_STAMP(0, it, 3);
        if (!has_chunk) continue;
        const int64_t row_base = (int64_t)tile * TC_ROWS + quarter * 32;
        // raw accumulators through the per-warp transposition buffer; everything else happens in the coalesced
        // layout (thread = 4 consecutive columns of rows i * 4 + rr): partial sums of an earlier K block, bias,
        // LeakyReLU, dropout (one RNG call = exactly the thread's four columns), store
#pragma unroll
        for (int j = 0; j < 32; j += 4)
            st_f4(st + stage_off(lane, j >> 2), make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
        __syncwarp();
        float4 r4[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) r4[i] = ld_f4(st + stage_off(i * 4 + rr, c4));
        __syncwarp();
        BWD_STAMP(0, it, 4);
        const int col = c * 32 + c4 * 4;                              // within the block's d_out columns
        if (col < d_out) {
            const int gcol = a.out_off + col;                         // within the layer's d_out_full columns
            const float4 b4 = *reinterpret_cast<const float4*>(bias_s + col);
            const int words = (a.d_out_full + 31) >> 5;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int64_t row = row_base + i * 4 + rr;
                if (row >= a.n_rows) continue;
                float* dst = a.E_out + row * a.d_out_full + gcol;
                float4 x = r4[i];
                if (a.mode == FW_PARTIAL) {
                    st_f4(dst, x);
                    continue;
                }
                if (a.mode == FW_FINAL) {
                    const float4 prev = ld_f4(dst);
                    x.x += prev.x; x.y += prev.y; x.z += prev.z; x.w += prev.w;
                }
                x.x += b4.x; x.y += b4.y; x.z += b4.z; x.w += b4.w;
                x.x = x.x > 0.f ? x.x : a.slope * x.x;                // LeakyReLU, NGCF.py:140
                x.y = x.y > 0.f ? x.y : a.slope * x.y;
                x.z = x.z > 0.f ? x.z : a.slope * x.z;
                x.w = x.w > 0.f ? x.w : a.slope * x.w;
                if (MM == MM_BITS) {
                    const uint32_t w = a.mess_bits[row * words + (gcol >> 5)] >> (gcol & 31);
                    x.x = w & 1u ? x.x * inv_keep : 0.f; x.y = w & 2u ? x.y * inv_keep : 0.f;
                    x.z = w & 4u ? x.z * inv_keep : 0.f; x.w = w & 8u ? x.w * inv_keep : 0.f;
                } else if (MM == MM_HASH) {
                    const float4 mm = mess_multiplier4_pre(thr, inv_keep, seed, a.layer,
                                                           (uint64_t)((row + a.row_off) * a.d_out_full + gcol) >> 2);
                    x.x *= mm.x; x.y *= mm.y; x.z *= mm.z; x.w *= mm.w;
                } else if (MM == MM_MULT) {
                    const float4 mm = ld_f4(a.mess_mult + row * a.d_out_full + gcol);
                    x.x *= mm.x; x.y *= mm.y; x.z *= mm.z; x.w *= mm.w;
                }
                st_f4(dst, x);
            }
        }
        BWD_STAMP(0, it, 2);
    }
}

// ====================================================================================================================
// The forward with its S / E traffic on TMA.  ncu on round 1's version, whose four loader warps held their loads in
// registers: 30 % of the HBM peak with nothing saturated — ~16 KB in flight per SM, a third of what Little's law asks
// for.  Here ONE thread streams the tile's S and E blocks (128 rows x 32 columns, 16 KB each, 128-byte swizzled by the
// tensor map = already in the UMMA K-major operand layout) into a raw shared-memory ring with cp.async.bulk.tensor;
// four converter warps read a raw stage at the very byte offsets they then write (S+E and S*E, split into TF32 hi / lo)
// in a two-slot operand ring.  Up to 64 KB of loads are in flight per SM whatever the converters do.
//
// Warp roles (448 threads): 0-7 epilogue, 8 MMA issuer + TMEM, 9 TMA producer (one lane), 10-13 converters.
// ====================================================================================================================
constexpr int F2_CONV_WARPS = 4;
constexpr int F2_TMA_WARP = FW_EPI_WARPS + 1;
constexpr int F2_THREADS = (FW_EPI_WARPS + 2 + F2_CONV_WARPS) * 32;
constexpr int F2_RAW_STAGES = 2;             // raw ring: stage = S block + E block = 32 KB
constexpr int F2_A_SLOTS = 2;                // operand ring: slot = one K block, hi + lo = 32 KB
constexpr int F2_RAW_BYTES = 2 * TC_A_BLOCK;

struct FwdTmaArgs {
    FwdTcArgs b;
    alignas(64) CUtensorMap tmS;
    alignas(64) CUtensorMap tmE;
};

struct Bars2 {
    uint64_t raw_full[F2_RAW_STAGES], raw_empty[F2_RAW_STAGES];
    uint64_t a_full[F2_A_SLOTS], a_empty[F2_A_SLOTS];
    uint64_t tmem_full[2], tmem_empty[2];
    uint64_t b_ready;
    uint32_t tmem_base;
};

template <int MM>
__global__ void __launch_bounds__(F2_THREADS, 1) dense_fwd_tma_kernel(const __grid_constant__ FwdTmaArgs p) {
    extern __shared__ uint8_t smem_raw[];
    const FwdTcArgs& a = p.b;
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;          // TMA / UMMA tiles need 1024-byte alignment
    uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
    const int d_in = a.d_in, d_out = a.d_out;
    const int KBH = d_in / 32, KB = 2 * KBH;
    const int b_block = d_out * 128;
    uint8_t* RAW = smem;                                                  // [stage][S block | E block]
    uint8_t* AOP = RAW + F2_RAW_STAGES * F2_RAW_BYTES;                    // [slot][hi | lo]
    uint8_t* B_hi = AOP + F2_A_SLOTS * 2 * TC_A_BLOCK;
    uint8_t* B_lo = B_hi + KB * b_block;
    float* bias_s = reinterpret_cast<float*>(B_lo + KB * b_block);
    float* stage = bias_s + 64;
    Bars2* bars = reinterpret_cast<Bars2*>(stage + FW_EPI_WARPS * 32 * 32);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    pdl_launch_dependents();
    if (tid == 0) {
        for (int i = 0; i < F2_RAW_STAGES; ++i) {
            mbar_init(&bars->raw_full[i], 1);
            mbar_init(&bars->raw_empty[i], F2_CONV_WARPS);
        }
        for (int i = 0; i < F2_A_SLOTS; ++i) {
            mbar_init(&bars->a_full[i], F2_CONV_WARPS);
            mbar_init(&bars->a_empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bars->tmem_full[i], 1);
            mbar_init(&bars->tmem_empty[i], FW_EPI_WARPS);
        }
        mbar_init(&bars->b_ready, FW_EPI_WARPS);
        fence_mbar_init();
        tma_prefetch_desc(&p.tmS);
        tma_prefetch_desc(&p.tmE);
    }
    if (warp == FW_MMA_WARP) tmem_alloc(&bars->tmem_base, 128);
    tc_fence_before_sync();
    __syncthreads();                                                      // barriers + TMEM address visible to every role
    tc_fence_after_sync();
    const uint32_t tmem_base = bars->tmem_base;
    const int n_my = (a.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int n_q = n_my * KBH;                                           // raw stages this CTA consumes
    const bool dbg = g_bwd_dbg_on == 1 && blockIdx.x == 0 && (warp == 0 || warp >= FW_MMA_WARP);
    if (dbg && lane == 0 && warp == 0) g_bwd_dbg[0][7][7] = clock64();
    pdl_wait();      // wcat / bias_eff come from ngcf_pack_weights, S from the SpMM right before this launch
    if (dbg && lane == 0 && warp == 0) g_bwd_dbg[0][7][6] = clock64();

    if (warp < FW_EPI_WARPS) {
        // the epilogue warps have nothing to do until the first accumulator is complete: they stage [W1 | W2] (split and
        // swizzled: B[n][k] = wcat[k][n]) and the bias while the first S / E tiles are already in flight
        constexpr int ET = FW_EPI_WARPS * 32;
        constexpr int WMAX = 64 * TC_MAX_KB * 8 / ET;                     // items (float4 of 4 consecutive k) per thread
        float4 wv[WMAX];
        const int n_items = d_out * KB * 8;
#pragma unroll
        for (int q = 0; q < WMAX; ++q) {                                  // every load in flight before the first use
            const int i = q * ET + tid;
            wv[q] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < n_items) {
                const int n = i % d_out, c = (i / d_out) & 7, kb = i / (d_out * 8);
                const int k = kb * 32 + c * 4;
                const int wrow = k < d_in ? a.w_row1 + k : a.w_row2 + (k - d_in);
                const float* src = a.wcat + (int64_t)wrow * a.d_out_full + a.out_off + n;
                wv[q] = make_float4(src[0], src[a.d_out_full], src[2 * a.d_out_full], src[3 * a.d_out_full]);
            }
        }
#pragma unroll
        for (int q = 0; q < WMAX; ++q) {
            const int i = q * ET + tid;
            if (i < n_items) {
                const int n = i % d_out, c = (i / d_out) & 7, kb = i / (d_out * 8);
                float4 hi, lo;
                split_tf32(wv[q], hi, lo);
                const uint32_t off = kb * b_block + sw128_offset(n, c);
                *reinterpret_cast<float4*>(B_hi + off) = hi;
                *reinterpret_cast<float4*>(B_lo + off) = lo;
            }
        }
        for (int i = tid; i < 64; i += ET) bias_s[i] = i < d_out ? a.bias_eff[a.out_off + i] : 0.f;
        fence_proxy_async_smem();
        asm volatile("bar.sync 1, %0;" ::"n"(ET) : "memory");             // bias visible to all epilogue warps
        if (lane == 0) mbar_arrive(&bars->b_ready);
        if (dbg && lane == 0) g_bwd_dbg[0][7][5] = clock64();
        fwd_epilogue_role<MM>(a, stage, bias_s, bars->tmem_full, bars->tmem_empty, tmem_base, n_my, warp, lane, dbg);
    } else if (warp == FW_MMA_WARP) {
        // ======================= MMA issuer: one operand slot = one K block ========================================
        const uint32_t idesc = umma_idesc_tf32(TC_ROWS, d_out, 0, 0);
        int j = 0;                                                        // running index of the operand slot in use
        mbar_wait(&bars->b_ready, 0);                                     // [W1 | W2] tiles staged
        for (int it = 0; it < n_my; ++it) {
            const int buf = it & 1;
            mbar_wait(&bars->tmem_empty[buf], ((it >> 1) & 1) ^ 1);
            BWD_STAMP(1, it, 0);
            tc_fence_after_sync();
            const uint32_t tmem_d = tmem_base + buf * 64;
            uint32_t accumulate = 0;
            for (int hh = 0; hh < KBH; ++hh)
                for (int part = 0; part < 2; ++part, ++j) {
                    const int slot = j % F2_A_SLOTS;
                    mbar_wait(&bars->a_full[slot], (j / F2_A_SLOTS) & 1);
                    BWD_STAMP(1, it, 1 + hh * 2 + part);
                    tc_fence_after_sync();
                    if (lane == 0) {
                        const int kb = part * KBH + hh;                   // K block of [W1 | W2] this slot multiplies
                        const uint32_t a_hi = smem_u32(AOP + slot * 2 * TC_A_BLOCK), a_lo = a_hi + TC_A_BLOCK;
                        const uint32_t b_hi = smem_u32(B_hi + kb * b_block), b_lo = smem_u32(B_lo + kb * b_block);
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const uint64_t dah = umma_desc_sw128(a_hi + k * 32, 16, 1024);
                            const uint64_t dal = umma_desc_sw128(a_lo + k * 32, 16, 1024);
                            const uint64_t dbh = umma_desc_sw128(b_hi + k * 32, 16, 1024);
                            const uint64_t dbl = umma_desc_sw128(b_lo + k * 32, 16, 1024);
                            umma_tf32(tmem_d, dah, dbh, idesc, accumulate);
                            umma_tf32(tmem_d, dal, dbh, idesc, 1);
                            umma_tf32(tmem_d, dah, dbl, idesc, 1);
                            accumulate = 1;
                        }
                        umma_commit(&bars->a_empty[slot]);
                    }
                    __syncwarp();
                }
            if (lane == 0) umma_commit(&bars->tmem_full[buf]);
            __syncwarp();
        }
    } else if (warp == F2_TMA_WARP) {
        // ======================= TMA producer ======================================================================
        if (lane == 0) {
            for (int q = 0; q < n_q; ++q) {
                const int it = q / KBH, hh = q % KBH, s = q % F2_RAW_STAGES;
                const int tile = blockIdx.x + it * gridDim.x;
                mbar_wait(&bars->raw_empty[s], ((q / F2_RAW_STAGES) & 1) ^ 1);
                BWD_STAMP(3, it, hh);
                mbar_expect_tx(&bars->raw_full[s], F2_RAW_BYTES);
                const uint32_t dst = smem_u32(RAW + s * F2_RAW_BYTES);
                tma_load_2d(dst, &p.tmS, a.in_off + hh * 32, tile * TC_ROWS, &bars->raw_full[s]);
                tma_load_2d(dst + TC_A_BLOCK, &p.tmE, a.in_off + hh * 32, tile * TC_ROWS, &bars->raw_full[s]);
            }
        }
    } else {
        // ======================= converters ========================================================================
        // raw S / E blocks arrive in the operand layout, so a thread reads and writes the same byte offsets
        const int lt = tid - (FW_EPI_WARPS + 2) * 32;                     // 0 .. 127
        constexpr int LT = F2_CONV_WARPS * 32;
        constexpr int NQ = TC_A_BLOCK / 16 / LT;                          // float4 per thread per block = 8
        int j = 0;
        for (int q = 0; q < n_q; ++q, j += 2) {
            const int s = q % F2_RAW_STAGES;
            mbar_wait(&bars->raw_full[s], (q / F2_RAW_STAGES) & 1);
            if (dbg && lane == 0 && warp == F2_TMA_WARP + 1 && q / KBH < 8) g_bwd_dbg[2][q / KBH][(q % KBH) * 3] = clock64();
            const uint8_t* rs = RAW + s * F2_RAW_BYTES;
            float4 sv[NQ], ev[NQ];
#pragma unroll
            for (int i = 0; i < NQ; ++i) {
                const uint32_t off = (uint32_t)(i * LT + lt) * 16u;
                sv[i] = *reinterpret_cast<const float4*>(rs + off);
                ev[i] = *reinterpret_cast<const float4*>(rs + TC_A_BLOCK + off);
            }
            // first operand slot: S + E
            {
                const int slot = j % F2_A_SLOTS;
                mbar_wait(&bars->a_empty[slot], ((j / F2_A_SLOTS) & 1) ^ 1);
                if (dbg && lane == 0 && warp == F2_TMA_WARP + 1 && q / KBH < 8) g_bwd_dbg[2][q / KBH][(q % KBH) * 3 + 1] = clock64();
                uint8_t* hi_p = AOP + slot * 2 * TC_A_BLOCK;
#pragma unroll
                for (int i = 0; i < NQ; ++i) {
                    const uint32_t off = (uint32_t)(i * LT + lt) * 16u;
                    const float4 x = make_float4(sv[i].x + ev[i].x, sv[i].y + ev[i].y, sv[i].z + ev[i].z, sv[i].w + ev[i].w);
                    float4 hi, lo;
                    split_tf32_trunc(x, hi, lo);
                    *reinterpret_cast<float4*>(hi_p + off) = hi;
                    *reinterpret_cast<float4*>(hi_p + TC_A_BLOCK + off) = lo;
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(&bars->raw_empty[s]);                     // the raw stage now lives in registers
                    mbar_arrive(&bars->a_full[slot]);
                }
            }
            // second operand slot: S * E
            {
                const int slot = (j + 1) % F2_A_SLOTS;
                mbar_wait(&bars->a_empty[slot], (((j + 1) / F2_A_SLOTS) & 1) ^ 1);
                uint8_t* hi_p = AOP + slot * 2 * TC_A_BLOCK;
#pragma unroll
                for (int i = 0; i < NQ; ++i) {
                    const uint32_t off = (uint32_t)(i * LT + lt) * 16u;
                    const float4 x = make_float4(sv[i].x * ev[i].x, sv[i].y * ev[i].y, sv[i].z * ev[i].z, sv[i].w * ev[i].w);
                    float4 hi, lo;
                    split_tf32_trunc(x, hi, lo);
                    *reinterpret_cast<float4*>(hi_p + off) = hi;
                    *reinterpret_cast<float4*>(hi_p + TC_A_BLOCK + off) = lo;
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->a_full[slot]);
                if (dbg && lane == 0 && warp == F2_TMA_WARP + 1 && q / KBH < 8) g_bwd_dbg[2][q / KBH][(q % KBH) * 3 + 2] = clock64();
            }
        }
    }

    tc_fence_before_sync();
    __syncthreads();
    if (dbg && lane == 0 && warp == 0) g_bwd_dbg[1][7][7] = clock64();
    if (warp == FW_MMA_WARP) {
        tc_fence_after_sync();
        tmem_dealloc(tmem_base, 128);
    }
}

}  // namespace
namespace {

// ====================================================================================================================
// Backward of the same layer (row-local part; SURVEY.md section 3.4), d_in = 64, as two kernels:
//
// dense_bwd_tc_kernel (per 128-row tile, persistent)
//   gM   = (gE_next + normalize-backward(gH)) * dropout * LeakyReLU'       loader warps, CUDA cores; also -> global
//   T    = gM · [W1 | W2]            [128 x 128], K = d_out                GEMM 1, K-major operands, 3xTF32
//   gS   = T1 + T2*E,  gEl = T1 + T2*S                                      epilogue warps (TMEM -> per-warp
//                                                                           transposition buffer -> coalesced I/O)
//   gb2 += colsum(gM), gb1 += 2 colsum(gM)
//
// wgrad_tc_kernel (split over rows, 64 rows per pipeline stage, persistent)
//   [gW1 | gW2]^T = [S+E | S*E]^T · gM   [128 x d_out], K = rows           GEMM 2, both operands MN-major
//   (SWIZZLE_128B_BASE32B), accumulator resident in TMEM across the CTA's whole row range, flushed once with
//   coalesced atomics.
// gM is kept in two shared-memory buffers in the first kernel so the loaders run one tile ahead of the MMAs.
// ====================================================================================================================
struct BwdTcArgs {
    const float* gE_next;
    const int32_t* slot;
    const float* gsum;
    int64_t ld_gsum;
    int col_off;
    const float* E_out;
    const float* S;
    const float* E;
    int64_t n_rows;
    int d_in, d_out;
    const float* W1;
    const float* W2;
    float slope;
    const float* mess_mult;
    const uint32_t* mess_bits;
    float mess_p;
    uint64_t seed;
    const uint64_t* seed_dev;
    int layer;
    float* gS;
    float* gEl;
    float* gM;                // [n_rows, d_out] scratch, consumed by wgrad_tc_kernel
    float* gb1;
    float* gb2;
    int n_tiles;
    int64_t row_off;
    // block decomposition of layers wider than 64 (d_in = 64 and d_out above are the BLOCK's widths): this launch takes
    // columns [out_off, out_off + d_out) of E_out / gE_next / gM / the dropout source (row stride d_out_full) and
    // rows out_off.. of W1 / W2, and produces columns [in_off, in_off + 64) of gS / gEl from the same columns of E / S
    // (row stride d_in_full) and of W1 / W2.  accumulate: add to the gS / gEl already there (an earlier d_out block);
    // first_in: this launch also writes gM and the bias gradients (once per d_out block).
    int d_out_full, out_off, d_in_full, in_off, accumulate, first_in;
    // L2 prefetch distance in tiles (0 = off): the MMA warp's elected thread asks for the E_out / gE_next / S / E rows of
    // tile it + pf while tile it is in progress.  The kernel's loads are in-flight-limited (32 KB per SM in the loaders'
    // registers, 64 KB of cp.async in the epilogue) against DRAM latency; against L2 latency the same window is enough.
    int pf;
};

struct BwdBars {
    uint64_t full_gm, empty_gm, tmem_full[2], tmem_empty[2];
    uint32_t tmem_base;
    float colsum[64];         // CTA-level column sums of gM (bias gradients): one global atomic per column per CTA
};

// E / S tile of the epilogue in shared memory: 128 rows of 256 bytes (d_in = 64), the 16-byte chunk c of row r at
// chunk position c ^ (r & 15): conflict-free both for "lane = row" accesses (the TMEM layout) and for row-contiguous
// ones (coalesced global traffic)
__device__ __forceinline__ uint32_t es_off(int r, int c) { return (uint32_t)r * 256u + (uint32_t)((c ^ (r & 15)) << 4); }

// Roles (416 threads): warps 0-3 epilogue, warp 4 MMA issuer, warps 5-12 loaders.
// The first version's epilogue fetched E and S from global memory after every TMEM read: ncu showed the four epilogue
// warps as the critical path (60 % of their time waiting on those loads) and the loaders idle 74 % of the time.  Now
// the loaders also bring the tile's E and S rows into shared memory (registers as the second pipeline stage, so the
// global latency overlaps the previous tile's epilogue); the epilogue combines them with T in TMEM layout IN PLACE
// (gS over E, gEl over S), then each warp streams its 32 rows out with coalesced 128-bit stores.
// PRE: gsum went through ngcf_rowgrad_normalize, the loader adds its slice as it is (no reductions, no divisions)
template <int MM, bool PRE>
__global__ void __launch_bounds__(TC_THREADS, 1) dense_bwd_tc_kernel(BwdTcArgs a) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
    constexpr int d_in = 64;
    const int d_out = a.d_out;
    const int KBo = d_out / 32;                                           // 32-column blocks of gM
    uint8_t* GM_hi = smem;                                                // [hi | lo][KBo blocks]
    uint8_t* GM_lo = GM_hi + KBo * TC_A_BLOCK;
    uint8_t* BT_hi = GM_lo + KBo * TC_A_BLOCK;                            // [n = 0..127][k = o], K blocks of 32 o
    uint8_t* BT_lo = BT_hi + KBo * TC_A_BLOCK;
    uint8_t* E_s = BT_lo + KBo * TC_A_BLOCK;                              // [128][64] fp32, es_off layout
    uint8_t* S_s = E_s + TC_ROWS * 256;
    BwdBars* bars = reinterpret_cast<BwdBars*>(S_s + TC_ROWS * 256);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    pdl_launch_dependents();

    if (tid == 0) {
        mbar_init(&bars->full_gm, TC_LOAD_WARPS);
        mbar_init(&bars->empty_gm, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bars->tmem_full[i], 1);
            mbar_init(&bars->tmem_empty[i], TC_EPI_WARPS);
        }
        fence_mbar_init();
    }
    if (warp == TC_EPI_WARPS) tmem_alloc(&bars->tmem_base, 256);          // T x2 (128 columns each)
    if (tid < 64) bars->colsum[tid] = 0.f;
    // rows of tile t in the three forward-pass tensors this kernel reads (contiguous: full-width launches only)
    auto prefetch_tile = [&](int tile, bool fwd_tensors, bool grad) {
        const int64_t row0 = (int64_t)tile * TC_ROWS;
        if (row0 >= a.n_rows) return;
        const int64_t nr = a.n_rows - row0 < TC_ROWS ? a.n_rows - row0 : TC_ROWS;
        if (fwd_tensors) {
            l2_prefetch_bulk(a.E_out + row0 * a.d_out_full, (uint32_t)(nr * a.d_out_full * 4));
            l2_prefetch_bulk(a.S + row0 * a.d_in_full, (uint32_t)(nr * a.d_in_full * 4));
            l2_prefetch_bulk(a.E + row0 * a.d_in_full, (uint32_t)(nr * a.d_in_full * 4));
        }
        if (grad && a.gE_next) l2_prefetch_bulk(a.gE_next + row0 * a.d_out_full, (uint32_t)(nr * a.d_out_full * 4));
    };
    if (a.pf > 0 && warp == TC_EPI_WARPS + 1 && lane == 0) {
        // the first tiles' forward-pass tensors (E_out, S, E: nothing between the forward and here writes them) are asked
        // for while the previous kernel still drains
        for (int i = 0; i < a.pf; ++i) {
            const int tile = blockIdx.x + i * gridDim.x;
            if (tile < a.n_tiles) prefetch_tile(tile, true, false);
        }
    }
    // BT[n][o] = W1[o][n] (n < 64), W2[o][n-64]; W1/W2 are [d_out, d_in] row-major
    // W1 / W2 are the layer's parameters: nothing inside a step writes them, so their tile is built BEFORE pdl_wait()
    // (consecutive threads take consecutive n = consecutive addresses of W1 / W2: coalesced)
    for (int i = tid; i < 128 * KBo * 8; i += TC_THREADS) {
        const int n = i & 127, c = (i >> 7) & 7, kb = i >> 10;
        const float* W = (n < d_in ? a.W1 : a.W2) + a.in_off + (n & 63);
        const int o0 = a.out_off + kb * 32 + c * 4;
        const int64_t ldw = a.d_in_full;
        float4 w = make_float4(W[(int64_t)o0 * ldw], W[(int64_t)(o0 + 1) * ldw], W[(int64_t)(o0 + 2) * ldw],
                               W[(int64_t)(o0 + 3) * ldw]);
        float4 hi, lo;
        split_tf32(w, hi, lo);
        const uint32_t off = kb * TC_A_BLOCK + sw128_offset(n, c);
        *reinterpret_cast<float4*>(BT_hi + off) = hi;
        *reinterpret_cast<float4*>(BT_lo + off) = lo;
    }
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    pdl_wait();      // gE_next, gsum, E_out, S, E and every output belong to the stream order
    const uint32_t tmem_base = bars->tmem_base;
    const int n_my = (a.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const bool dbg = g_bwd_dbg_on == 1 && blockIdx.x == 0 && (warp == 0 || warp == TC_EPI_WARPS || warp == TC_EPI_WARPS + 1);
    if (dbg && lane == 0 && warp == 0) g_bwd_dbg[0][7][7] = clock64();   // start of the steady state

    if (warp < TC_EPI_WARPS) {
        // ======================= epilogue: gS / gEl ==============================================================
        // Each warp owns tile rows [32 warp, 32 warp + 32): it brings their E and S into shared memory itself (two
        // rounds of 8 row pairs; the first round of the NEXT tile is in flight while this tile streams out), combines
        // them with T in TMEM layout in place, and streams the 32 rows out — warp-local, no CTA-level barrier.
        const int r = warp * 32 + lane;                                   // TMEM lane = tile row
        uint8_t* e_row = E_s + r * 256;
        uint8_t* s_row = S_s + r * 256;
        const int sw = r & 15;
        const int c = lane & 15, hsel = lane >> 4;
        // fill: this warp's 32 rows of E and S of a tile -> shared memory with cp.async (no registers held; rows past
        // the end are zero-filled), issued right after the previous tile streamed out
        const uint32_t e_s32 = smem_u32(E_s), s_s32 = smem_u32(S_s);
        auto fill = [&](int tile) {
            const int64_t row0 = (int64_t)tile * TC_ROWS;
#pragma unroll 4
            for (int i = 0; i < 16; ++i) {
                const int rl = warp * 32 + 2 * i + hsel;
                const int64_t row = row0 + rl;
                const bool ok = row < a.n_rows;
                const int64_t src = (ok ? row : 0) * a.d_in_full + a.in_off + c * 4;
                const uint32_t off = es_off(rl, c);
                cp_async16(e_s32 + off, a.E + src, ok ? 16u : 0u);
                cp_async16(s_s32 + off, a.S + src, ok ? 16u : 0u);
            }
        };
        if (n_my > 0) fill(blockIdx.x);
        for (int it = 0; it < n_my; ++it) {
            const int tile = blockIdx.x + it * gridDim.x;
            const int buf = it & 1;
            BWD_STAMP(0, it, 0);
            cp_async_wait_all();
            __syncwarp();
            BWD_STAMP(0, it, 1);
            mbar_wait(&bars->tmem_full[buf], (it >> 1) & 1);
            BWD_STAMP(0, it, 2);
            tc_fence_after_sync();
            const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + buf * 128;
#pragma unroll 1
            for (int half = 0; half < d_in / 32; ++half) {
                float v1[32], v2[32];
                tmem_ld_32x32(taddr + half * 32, v1);                     // T1[row][32 half .. +32)
                tmem_ld_32x32(taddr + d_in + half * 32, v2);              // T2
                if (half == d_in / 32 - 1) {                              // accumulator fully read
                    tc_fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars->tmem_empty[buf]);
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const uint32_t off = (uint32_t)(((half * 8 + j) ^ sw) << 4);
                    const float4 e = *reinterpret_cast<const float4*>(e_row + off);
                    const float4 s = *reinterpret_cast<const float4*>(s_row + off);
                    *reinterpret_cast<float4*>(e_row + off) =              // gS = T1 + T2 * E
                        make_float4(fmaf(v2[4 * j], e.x, v1[4 * j]), fmaf(v2[4 * j + 1], e.y, v1[4 * j + 1]),
                                    fmaf(v2[4 * j + 2], e.z, v1[4 * j + 2]), fmaf(v2[4 * j + 3], e.w, v1[4 * j + 3]));
                    *reinterpret_cast<float4*>(s_row + off) =              // gEl = T1 + T2 * S
                        make_float4(fmaf(v2[4 * j], s.x, v1[4 * j]), fmaf(v2[4 * j + 1], s.y, v1[4 * j + 1]),
                                    fmaf(v2[4 * j + 2], s.z, v1[4 * j + 2]), fmaf(v2[4 * j + 3], s.w, v1[4 * j + 3]));
                }
            }
            __syncwarp();
            BWD_STAMP(0, it, 3);
            // this warp's 32 rows, two rows per instruction: coalesced 128-bit stores
            const int64_t row0 = (int64_t)tile * TC_ROWS;
#pragma unroll 4
            for (int i = 0; i < 16; ++i) {
                const int rl = warp * 32 + 2 * i + hsel;
                const int64_t row = row0 + rl;
                const uint32_t off = es_off(rl, c);
                float4 x = *reinterpret_cast<const float4*>(E_s + off);
                float4 y = *reinterpret_cast<const float4*>(S_s + off);
                if (row < a.n_rows) {
                    float* ps = a.gS + row * a.d_in_full + a.in_off + c * 4;
                    float* pe = a.gEl + row * a.d_in_full + a.in_off + c * 4;
                    if (a.accumulate) {                                   // an earlier d_out block left its share there
                        const float4 x0 = ld_f4(ps), y0 = ld_f4(pe);
                        x.x += x0.x; x.y += x0.y; x.z += x0.z; x.w += x0.w;
                        y.x += y0.x; y.y += y0.y; y.z += y0.z; y.w += y0.w;
                    }
                    st_f4(ps, x);
                    st_f4(pe, y);
                }
            }
            __syncwarp();
            BWD_STAMP(0, it, 4);
            if (it + 1 < n_my) fill(tile + gridDim.x);
        }
    } else if (warp == TC_EPI_WARPS) {
        // ======================= MMA issuer =====================================================================
        const uint32_t idesc1 = umma_idesc_tf32(TC_ROWS, 2 * d_in, 0, 0);
        if (a.pf > 0 && lane == 0)                                        // gE_next comes from the kernel right before
            for (int i = 0; i < a.pf && i < n_my; ++i) prefetch_tile(blockIdx.x + i * gridDim.x, false, true);
        for (int it = 0; it < n_my; ++it) {
            const int buf = it & 1;
            BWD_STAMP(1, it, 0);
            if (a.pf > 0 && lane == 0 && it + a.pf < n_my) prefetch_tile(blockIdx.x + (it + a.pf) * gridDim.x, true, true);
            mbar_wait(&bars->full_gm, it & 1);
            BWD_STAMP(1, it, 1);
            mbar_wait(&bars->tmem_empty[buf], ((it >> 1) & 1) ^ 1);
            BWD_STAMP(1, it, 2);
            tc_fence_after_sync();
            if (lane == 0) {
                const uint32_t tmem_t = tmem_base + buf * 128;
                const uint32_t gm_hi = smem_u32(GM_hi), gm_lo = smem_u32(GM_lo);
                uint32_t acc1 = 0;
                for (int kb = 0; kb < KBo; ++kb) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint32_t off = kb * TC_A_BLOCK + k * 32;
                        const uint64_t dah = umma_desc_sw128(gm_hi + off, 16, 1024);
                        const uint64_t dal = umma_desc_sw128(gm_lo + off, 16, 1024);
                        const uint64_t dbh = umma_desc_sw128(smem_u32(BT_hi) + off, 16, 1024);
                        const uint64_t dbl = umma_desc_sw128(smem_u32(BT_lo) + off, 16, 1024);
                        umma_tf32(tmem_t, dah, dbh, idesc1, acc1);
                        umma_tf32(tmem_t, dal, dbh, idesc1, 1);
                        umma_tf32(tmem_t, dah, dbl, idesc1, 1);
                        acc1 = 1;
                    }
                }
                umma_commit(&bars->tmem_full[buf]);
                umma_commit(&bars->empty_gm);
            }
            __syncwarp();
            BWD_STAMP(1, it, 3);
        }
    } else {
        // ======================= loaders: gM rows =================================================================
        // half a warp per row: lane owns the four columns 4*(lane & 15) .. +3 (one RNG call = exactly its four
        // dropout decisions, 128-bit loads and shared-memory stores).  Software-pipelined by half tiles (4 row pairs
        // per warp): the loads of the next half are in flight while this half is computed, across tiles too.
        const int lw = warp - (TC_EPI_WARPS + 1);                         // 0 .. 7
        const int hl = lane & 15, hsel = lane >> 4;
        const int c0 = hl * 4;
        const bool col_ok = c0 < d_out;
        const uint64_t seed = MM == MM_HASH ? ngcf_seed(a.seed, a.seed_dev) : 0ull;
        const uint32_t thr = ngcf_threshold16(a.mess_p);
        const float inv_keep = 1.0f / (1.0f - a.mess_p);
        float4 colsum = make_float4(0.f, 0.f, 0.f, 0.f);
        constexpr int HP = TC_ROWS / (4 * TC_LOAD_WARPS);                 // row pairs per warp per half tile
        struct Half {
            float4 e[HP], gn[HP];
            int sl[HP];
        };
        auto issue = [&](Half& h, int tile, int half) {
            const int64_t row0 = (int64_t)tile * TC_ROWS;
#pragma unroll
            for (int j = 0; j < HP; ++j) {
                const int64_t row = row0 + 2 * (lw + TC_LOAD_WARPS * (half * HP + j)) + hsel;
                const bool ok = row < a.n_rows && col_ok;
                h.e[j] = h.gn[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                h.sl[j] = -1;
                if (ok) {
                    h.e[j] = ld_stream_f4(a.E_out + row * a.d_out_full + a.out_off + c0);
                    if (a.gE_next) h.gn[j] = ld_stream_f4(a.gE_next + row * a.d_out_full + a.out_off + c0);
                    if (a.slot) h.sl[j] = a.slot[row];
                }
            }
        };
        auto compute = [&](Half& h, int tile, int half) {
            const int64_t row0 = (int64_t)tile * TC_ROWS;
            // (1) rows of the batch only (~4 % of all rows): their output-row gradient
            if (PRE) {                                                    // already normalize-backwarded: predicated add
#pragma unroll
                for (int j = 0; j < HP; ++j) {
                    const int s = h.sl[j];
                    if (s >= 0) {                                         // col_off need not be a multiple of 4 (width 65 first)
                        const float* gp = a.gsum + (int64_t)s * a.ld_gsum + a.col_off + a.out_off + c0;
                        h.gn[j].x += gp[0]; h.gn[j].y += gp[1]; h.gn[j].z += gp[2]; h.gn[j].w += gp[3];
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < HP; ++j) {
                    const int s = h.sl[j];
                    if (__any_sync(FULL_MASK, s >= 0)) {
                        float4 gh = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (s >= 0) {                                         // col_off need not be a multiple of 4 (width 65 first)
                            const float* gp = a.gsum + (int64_t)s * a.ld_gsum + a.col_off + a.out_off + c0;
                            gh = make_float4(gp[0], gp[1], gp[2], gp[3]);
                        }
                        const float4 e = h.e[j];
                        float nrm2 = e.x * e.x + e.y * e.y + e.z * e.z + e.w * e.w;
                        float dot = e.x * gh.x + e.y * gh.y + e.z * gh.z + e.w * gh.w;
#pragma unroll
                        for (int o = 8; o > 0; o >>= 1) {                     // reduce over the 16 lanes of the row
                            nrm2 += __shfl_xor_sync(FULL_MASK, nrm2, o);
                            dot += __shfl_xor_sync(FULL_MASK, dot, o);
                        }
                        if (s >= 0) {
                            const float rn = 1.0f / fmaxf(sqrtf(nrm2), 1e-12f);   // F.normalize eps, NGCF.py:144
                            const float hd = dot * rn;                        // H . gH
                            h.gn[j].x += (gh.x - (e.x * rn) * hd) * rn;       // normalize backward
                            h.gn[j].y += (gh.y - (e.y * rn) * hd) * rn;
                            h.gn[j].z += (gh.z - (e.z * rn) * hd) * rn;
                            h.gn[j].w += (gh.w - (e.w * rn) * hd) * rn;
                        }
                    }
                }
            }
            // (2) every row, branch-free: dropout + LeakyReLU backward, gM out, TF32 split into the operand tile
#pragma unroll
            for (int j = 0; j < HP; ++j) {
                const int r = 2 * (lw + TC_LOAD_WARPS * (half * HP + j)) + hsel;
                const int64_t row = row0 + r;
                const bool in = row < a.n_rows && col_ok;
                const float4 e = h.e[j];
                float4 g = h.gn[j];
                float4 mult = make_float4(1.f, 1.f, 1.f, 1.f);
                if (MM == MM_MULT) {
                    if (in) mult = ld_f4(a.mess_mult + row * a.d_out_full + a.out_off + c0);
                } else if (MM == MM_BITS) {
                    uint32_t w = 0;
                    if (in) w = a.mess_bits[row * ((a.d_out_full + 31) >> 5) + ((a.out_off + c0) >> 5)] >> ((a.out_off + c0) & 31);
                    mult = make_float4(w & 1u ? inv_keep : 0.f, w & 2u ? inv_keep : 0.f, w & 4u ? inv_keep : 0.f,
                                       w & 8u ? inv_keep : 0.f);
                } else if (MM == MM_HASH) {
                    mult = mess_multiplier4_pre(thr, inv_keep, seed, a.layer,
                                                (uint64_t)((row + a.row_off) * a.d_out_full + a.out_off + c0) >> 2);
                }
                g.x *= mult.x * (e.x > 0.f ? 1.f : a.slope);              // dropout + LeakyReLU backward
                g.y *= mult.y * (e.y > 0.f ? 1.f : a.slope);
                g.z *= mult.z * (e.z > 0.f ? 1.f : a.slope);
                g.w *= mult.w * (e.w > 0.f ? 1.f : a.slope);
                if (!in) g = make_float4(0.f, 0.f, 0.f, 0.f);             // rows past the end / unused columns
                if (in && a.first_in) st_f4(a.gM + row * a.d_out_full + a.out_off + c0, g);
                colsum.x += g.x; colsum.y += g.y; colsum.z += g.z; colsum.w += g.w;
                if (col_ok) {
                    float4 hi, lo;
                    split_tf32_trunc(g, hi, lo);
                    const uint32_t off = (hl >> 3) * TC_A_BLOCK + sw128_offset(r, hl & 7);
                    *reinterpret_cast<float4*>(GM_hi + off) = hi;
                    *reinterpret_cast<float4*>(GM_lo + off) = lo;
                }
            }
        };
        Half h0, h1;
        if (n_my > 0) issue(h0, blockIdx.x, 0);
        for (int it = 0; it < n_my; ++it) {
            const int tile = blockIdx.x + it * gridDim.x;
            BWD_STAMP(2, it, 0);
            issue(h1, tile, 1);
            BWD_STAMP(2, it, 1);
            mbar_wait(&bars->empty_gm, (it & 1) ^ 1);                     // the MMAs of the previous tile have read gM
            BWD_STAMP(2, it, 2);
            compute(h0, tile, 0);
            BWD_STAMP(3, it, 0);
            if (it + 1 < n_my) issue(h0, tile + gridDim.x, 0);
            BWD_STAMP(3, it, 1);
            compute(h1, tile, 1);
            BWD_STAMP(3, it, 2);
            fence_proxy_async_smem();
            BWD_STAMP(3, it, 3);
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->full_gm);
            BWD_STAMP(2, it, 3);
        }
        colsum.x += __shfl_xor_sync(FULL_MASK, colsum.x, 16);
        colsum.y += __shfl_xor_sync(FULL_MASK, colsum.y, 16);
        colsum.z += __shfl_xor_sync(FULL_MASK, colsum.z, 16);
        colsum.w += __shfl_xor_sync(FULL_MASK, colsum.w, 16);
        // the 8 loader warps first reduce in shared memory: 148 x 8 warps hammering the same 128 global addresses
        // with atomics (150 k of them on four cache lines) jammed the L2 slices behind them for tens of microseconds
        if (hsel == 0 && col_ok) {
            atomicAdd(&bars->colsum[c0 + 0], colsum.x);
            atomicAdd(&bars->colsum[c0 + 1], colsum.y);
            atomicAdd(&bars->colsum[c0 + 2], colsum.z);
            atomicAdd(&bars->colsum[c0 + 3], colsum.w);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(TC_LOAD_WARPS * 32) : "memory");   // loader warps only
        const int lt = tid - (TC_EPI_WARPS + 1) * 32;
        if (lt < d_out && a.first_in) {
            const float cs = bars->colsum[lt];
            atomicAdd(a.gb2 + a.out_off + lt, cs);
            atomicAdd(a.gb1 + a.out_off + lt, 2.0f * cs);                 // w1_list[i] is applied twice (NGCF.py:131,133)
        }
    }

    tc_fence_before_sync();
    __syncthreads();
    if (dbg && lane == 0 && warp == 0) g_bwd_dbg[1][7][7] = clock64();   // every role done
    if (warp == TC_EPI_WARPS) {
        tc_fence_after_sync();
        tmem_dealloc(tmem_base, 256);
    }
}

// --------------------------------------------------------------------------------------------------------------------
// weight gradients: D[j][o] = sum_rows X[row][j] * gM[row][o],  X = [S+E | S*E]  (gW1[o][j] = D[j][o], gW2[o][j] = D[64+j][o])
// --------------------------------------------------------------------------------------------------------------------
constexpr int WG_ROWS = 64;                   // rows (= GEMM K) per pipeline stage
constexpr int WG_BLOCK = WG_ROWS * 128;       // bytes of one 32-wide M/N group of a stage (hi or lo)

struct WgradArgs {
    const float* S;
    const float* E;
    const float* gM;
    int64_t n_rows;
    int d_out;
    float* gW1;
    float* gW2;
    int n_chunks;
    // block decomposition: columns [in_off, in_off + 64) of S / E (row stride d_in_full) against columns
    // [out_off, out_off + d_out) of gM (row stride d_out_full) -> rows out_off.., columns in_off.. of gW1 / gW2
    int d_in_full, in_off, d_out_full, out_off;
    int pf;                       // != 0: an idle epilogue thread asks for the CTA's S / E / gM rows in L2 up front
};

struct WgBars {
    uint64_t full[2], empty[2], d_full;
    uint32_t tmem_base;
};

__global__ void __launch_bounds__(TC_THREADS, 1) wgrad_tc_kernel(WgradArgs a) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
    constexpr int d_in = 64;
    const int d_out = a.d_out;
    const int KBo = d_out / 32;
    const int stage_bytes = (8 + 2 * KBo) * WG_BLOCK;                     // X hi (4) + X lo (4) + gM hi + gM lo
    WgBars* bars = reinterpret_cast<WgBars*>(smem + 2 * stage_bytes);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    pdl_launch_dependents();

    if (tid == 0) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bars->full[i], TC_LOAD_WARPS);
            mbar_init(&bars->empty[i], 1);
        }
        mbar_init(&bars->d_full, 1);
        fence_mbar_init();
    }
    if (warp == TC_EPI_WARPS) tmem_alloc(&bars->tmem_base, 64);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    pdl_wait();
    const uint32_t tmem_d = bars->tmem_base;
    const int n_my = (a.n_chunks - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const bool dbg = g_bwd_dbg_on == 2 && blockIdx.x == 0 && (warp == 0 || warp == TC_EPI_WARPS || warp == TC_EPI_WARPS + 1);
    if (dbg && lane == 0 && warp == 0) g_bwd_dbg[0][7][7] = clock64();

    if (warp < TC_EPI_WARPS) {
        // ======================= final flush =====================================================================
        // until then these warps are idle: one thread asks for every chunk of this CTA in L2 (the whole input of the
        // launch, 12 * d bytes per row, fits L2 many times over), so the loaders' register-staged loads - 48 KB in flight
        // per SM - meet L2 latency instead of DRAM latency
        if (a.pf && warp == 0 && lane == 0) {
            for (int it = 0; it < n_my; ++it) {
                const int64_t row0 = (int64_t)(blockIdx.x + it * gridDim.x) * WG_ROWS;
                if (row0 >= a.n_rows) break;
                const int64_t nr = a.n_rows - row0 < WG_ROWS ? a.n_rows - row0 : WG_ROWS;
                l2_prefetch_bulk(a.gM + row0 * a.d_out_full, (uint32_t)(nr * a.d_out_full * 4));
                l2_prefetch_bulk(a.S + row0 * a.d_in_full, (uint32_t)(nr * a.d_in_full * 4));
                l2_prefetch_bulk(a.E + row0 * a.d_in_full, (uint32_t)(nr * a.d_in_full * 4));
            }
        }
        mbar_wait(&bars->d_full, 0);
        BWD_STAMP(0, 0, 0);
        tc_fence_after_sync();
        const int m = warp * 32 + lane;                                   // TMEM lane = column j of [W1 | W2]
        float* gw = (m < d_in ? a.gW1 : a.gW2) + (int64_t)a.out_off * a.d_in_full + a.in_off + (m & 63);
        for (int c = 0; c < KBo; ++c) {
            float v[32];
            tmem_ld_32x32(tmem_d + ((uint32_t)(warp * 32) << 16) + c * 32, v);
#pragma unroll
            for (int j = 0; j < 32; ++j) atomicAdd(gw + (int64_t)(c * 32 + j) * a.d_in_full, v[j]);
        }
        BWD_STAMP(0, 0, 1);
    } else if (warp == TC_EPI_WARPS) {
        // ======================= MMA issuer =====================================================================
        const uint32_t idesc = umma_idesc_tf32(TC_ROWS, d_out, 1, 1);
        constexpr uint32_t layout = UMMA_SW128_BASE32B, sbo = 512;       // 4-row K atoms of 512 bytes
        uint32_t acc = 0;
        for (int it = 0; it < n_my; ++it) {
            const int sgi = it & 1;
            mbar_wait(&bars->full[sgi], (it >> 1) & 1);
            tc_fence_after_sync();
            if (lane == 0) {
                const uint32_t x_hi = smem_u32(smem + sgi * stage_bytes), x_lo = x_hi + 4 * WG_BLOCK;
                const uint32_t g_hi = x_lo + 4 * WG_BLOCK, g_lo = g_hi + KBo * WG_BLOCK;
#pragma unroll
                for (int kk = 0; kk < WG_ROWS / 8; ++kk) {                // K = 8 rows per MMA = two 4-row atoms
                    const uint32_t off = kk * 1024;
                    const uint64_t dah = umma_desc(x_hi + off, WG_BLOCK, sbo, layout);
                    const uint64_t dal = umma_desc(x_lo + off, WG_BLOCK, sbo, layout);
                    const uint64_t dbh = umma_desc(g_hi + off, WG_BLOCK, sbo, layout);
                    const uint64_t dbl = umma_desc(g_lo + off, WG_BLOCK, sbo, layout);
                    umma_tf32(tmem_d, dah, dbh, idesc, acc);
                    umma_tf32(tmem_d, dal, dbh, idesc, 1);
                    umma_tf32(tmem_d, dah, dbl, idesc, 1);
                    acc = 1;
                }
                umma_commit(&bars->empty[sgi]);
            }
            __syncwarp();
        }
        if (lane == 0) umma_commit(&bars->d_full);
        __syncwarp();
    } else {
        // ======================= loaders =========================================================================
        // software-pipelined by half stages (32 rows: 2 + 2 + 2 float4 per thread): the loads of the next half are in
        // flight while this one is split and stored (first version: load a 64-row stage, wait, convert — one exposed
        // round trip per stage, ~7.5 stages per CTA)
        const int lt = tid - (TC_EPI_WARPS + 1) * 32;                     // 0 .. 255
        constexpr int LT = TC_LOAD_WARPS * 32;
        const int gq = d_out / 4;                                         // float4 per gM row
        struct Half {
            float4 s[2], e[2], g[2];
        };
        const int total = 2 * n_my;
        auto issue = [&](Half& h, int i) {
            const int64_t row0 = (int64_t)(blockIdx.x + (i >> 1) * gridDim.x) * WG_ROWS;
#pragma unroll
            for (int q2 = 0; q2 < 2; ++q2) {                              // 64 rows x 16 float4 = 4 per thread per stage
                const int idx = ((i & 1) * 2 + q2) * LT + lt, r = idx >> 4, c = idx & 15;
                const int64_t row = row0 + r;
                h.s[q2] = h.e[q2] = h.g[q2] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (row < a.n_rows) {
                    h.s[q2] = ld_stream_f4(a.S + row * a.d_in_full + a.in_off + c * 4);
                    h.e[q2] = ld_stream_f4(a.E + row * a.d_in_full + a.in_off + c * 4);
                    if (c < gq) h.g[q2] = ld_stream_f4(a.gM + row * a.d_out_full + a.out_off + c * 4);
                }
            }
        };
        auto convert = [&](const Half& h, int i) {
            const int sgi = (i >> 1) & 1;
            uint8_t* x_hi = smem + sgi * stage_bytes;
            uint8_t* x_lo = x_hi + 4 * WG_BLOCK;
            uint8_t* g_hi = x_lo + 4 * WG_BLOCK;
            uint8_t* g_lo = g_hi + KBo * WG_BLOCK;
#pragma unroll
            for (int q2 = 0; q2 < 2; ++q2) {
                const int idx = ((i & 1) * 2 + q2) * LT + lt, r = idx >> 4, c = idx & 15;
                const uint32_t off = (c >> 3) * WG_BLOCK + sw128b32_offset(r, c & 7);
                const float4 sv = h.s[q2], ev = h.e[q2];
                const float4 x1 = make_float4(sv.x + ev.x, sv.y + ev.y, sv.z + ev.z, sv.w + ev.w);
                const float4 x2 = make_float4(sv.x * ev.x, sv.y * ev.y, sv.z * ev.z, sv.w * ev.w);
                float4 hi, lo;
                split_tf32(x1, hi, lo);
                *reinterpret_cast<float4*>(x_hi + off) = hi;
                *reinterpret_cast<float4*>(x_lo + off) = lo;
                split_tf32(x2, hi, lo);
                *reinterpret_cast<float4*>(x_hi + 2 * WG_BLOCK + off) = hi;
                *reinterpret_cast<float4*>(x_lo + 2 * WG_BLOCK + off) = lo;
                if (c < gq) {
                    split_tf32(h.g[q2], hi, lo);
                    *reinterpret_cast<float4*>(g_hi + off) = hi;
                    *reinterpret_cast<float4*>(g_lo + off) = lo;
                }
            }
        };
        Half h0, h1;
        if (total > 0) issue(h0, 0);
        for (int i = 0; i < total; i += 2) {                              // half i: rows 0..31 of its stage, i + 1: rows 32..63
            const int it = i >> 1, sgi = it & 1;
            issue(h1, i + 1);
            mbar_wait(&bars->empty[sgi], ((it >> 1) & 1) ^ 1);
            convert(h0, i);
            if (i + 2 < total) issue(h0, i + 2);
            convert(h1, i + 1);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->full[sgi]);
            BWD_STAMP(2, it, 0);
        }
    }

    tc_fence_before_sync();
    __syncthreads();
    if (dbg && lane == 0 && warp == 0) g_bwd_dbg[1][7][7] = clock64();
    if (warp == TC_EPI_WARPS) {
        tc_fence_after_sync();
        tmem_dealloc(tmem_d, 64);
    }
}

}  // namespace

// widths up to 64 are one block; 128 is decomposed into 64-wide blocks of the same kernel (K halves accumulate through
// the partial sums parked in E_out, N halves are independent)
bool ngcf_dense_fwd_tc_eligible(int d_in, int d_out) {
    const bool in_ok = d_in == 32 || d_in == 64 || d_in == 128;
    const bool out_ok = (d_out >= 16 && d_out <= 64 && d_out % 16 == 0) || d_out == 128;
    return in_ok && out_ok;
}

int ngcf_dense_fwd_tc(const float* S, const float* E, int64_t n_rows, int d_in, int d_out, const float* wcat,
                      const float* bias_eff, float slope, const float* mess_mult, const uint32_t* mess_bits, float mess_p,
                      uint64_t seed, const uint64_t* seed_dev, int layer, int64_t row_offset, float* E_out,
                      cudaStream_t st) {
    // (function attributes are per device: a module on cuda:1 needs them set there too)
    static bool attr_set_dev[64] = {};
    int cur_dev = 0;
    NGCF_CUDA(cudaGetDevice(&cur_dev));
    bool& attr_set = attr_set_dev[cur_dev & 63];
    if (!attr_set) {
        NGCF_CUDA(cudaFuncSetAttribute(dense_fwd_tma_kernel<MM_NONE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        NGCF_CUDA(cudaFuncSetAttribute(dense_fwd_tma_kernel<MM_MULT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        NGCF_CUDA(cudaFuncSetAttribute(dense_fwd_tma_kernel<MM_BITS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        NGCF_CUDA(cudaFuncSetAttribute(dense_fwd_tma_kernel<MM_HASH>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        attr_set = true;
    }
    const int bk = d_in > 64 ? 64 : d_in, bn = d_out > 64 ? 64 : d_out;   // block widths
    const int KH = d_in / bk, NH = d_out / bn;
    const int n_tiles = (int)ceil_div64(n_rows, TC_ROWS);
    const int grid = (int)min((int64_t)n_tiles, (int64_t)ngcf_num_sms());
    const int KB = 2 * bk / 32;
    const size_t smem = 1024 + (size_t)F2_RAW_STAGES * F2_RAW_BYTES + (size_t)F2_A_SLOTS * 2 * TC_A_BLOCK +
                        (size_t)KB * 2 * bn * 128 + 64 * sizeof(float) + FW_EPI_WARPS * 32 * 32 * sizeof(float) +
                        sizeof(Bars2);
    FwdTmaArgs p{};
    // S / E as [n_rows, d_in] fp32 with boxes of 128 rows x 32 columns, 128-byte swizzle; rows past the end read as 0
    int rc = ngcf_encode_tmap_2d(&p.tmS, S, (uint64_t)n_rows, (uint64_t)d_in, (uint64_t)d_in, 32, TC_ROWS,
                                 CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc == 0)
        rc = ngcf_encode_tmap_2d(&p.tmE, E, (uint64_t)n_rows, (uint64_t)d_in, (uint64_t)d_in, 32, TC_ROWS,
                                 CU_TENSOR_MAP_SWIZZLE_128B);
    NGCF_REQUIRE(rc == 0, "dense_fwd: cuTensorMapEncodeTiled failed (%d)", rc);
    for (int nh = 0; nh < NH; ++nh)
        for (int kh = 0; kh < KH; ++kh) {
            FwdTcArgs a{S, E, n_rows, bk, bn, wcat, bias_eff, slope, mess_mult, mess_bits, mess_p, seed, seed_dev, layer,
                        E_out, n_tiles, row_offset};
            a.ld_in = d_in; a.in_off = kh * bk;
            a.w_row1 = kh * bk; a.w_row2 = d_in + kh * bk;
            a.out_off = nh * bn; a.d_out_full = d_out;
            a.mode = KH == 1 ? FW_SINGLE : (kh == 0 ? FW_PARTIAL : FW_FINAL);
            const int mm = a.mode == FW_PARTIAL ? MM_NONE : mess_mode(mess_mult, mess_bits, mess_p);
            p.b = a;
            switch (mm) {
                case MM_NONE: NGCF_CUDA(ngcf_launch_pdl(dense_fwd_tma_kernel<MM_NONE>, dim3(grid), dim3(F2_THREADS), smem, st, p)); break;
                case MM_MULT: NGCF_CUDA(ngcf_launch_pdl(dense_fwd_tma_kernel<MM_MULT>, dim3(grid), dim3(F2_THREADS), smem, st, p)); break;
                case MM_BITS: NGCF_CUDA(ngcf_launch_pdl(dense_fwd_tma_kernel<MM_BITS>, dim3(grid), dim3(F2_THREADS), smem, st, p)); break;
                default: NGCF_CUDA(ngcf_launch_pdl(dense_fwd_tma_kernel<MM_HASH>, dim3(grid), dim3(F2_THREADS), smem, st, p)); break;
            }
            NGCF_LAUNCH_OK("dense_fwd_tma_kernel");
        }
    return NGCF_OK;
}

// Optional second stream for the weight-gradient launches (ngcf_set_wgrad_stream): they depend on the backward kernel's
// gM only, so a caller with other work queued behind the backward kernel (the row-sharded step: the gS exchange and the
// transposed product) can let them run beside it.  Thread-local; the caller joins the stream.
static thread_local cudaStream_t g_wgrad_stream = nullptr;
static thread_local int g_wgrad_forked = 0;      // a launch went to the second stream since the last query
extern "C" int ngcf_set_wgrad_stream(void* stream_or_null) {
    g_wgrad_stream = as_stream(stream_or_null);
    return NGCF_OK;
}
// 1 if any weight-gradient launch since the last call went to the second stream (the caller then has to join it; a
// layer on the FFMA kernels never forks, and waiting on a stream without captured work breaks a graph capture)
extern "C" int ngcf_wgrad_stream_forked(void) {
    const int v = g_wgrad_forked;
    g_wgrad_forked = 0;
    return v;
}

// NGCF_B200_PREFETCH = L2 prefetch distance of the backward kernel in tiles; != 0 also switches the weight-gradient
// kernel's up-front prefetch on.  Default 0 = off: measured on a B200 (profiles/r02_prefetch_experiment.txt) the step is
// not faster with it (0.505 ms off, 0.513 ms at distance 2 or 4) - the in-kernel timelines show both kernels' steady
// state already near the DRAM rate (backward ~15 k cycles per 224-KB tile, weight gradients ~2.4 k cycles per 48-KB
// stage = 5.8 TB/s), what separates them from the roofline is per-launch fixed cost, not load latency.
static int dense_prefetch_tiles() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("NGCF_B200_PREFETCH");
        v = e ? atoi(e) : 0;
        if (v < 0) v = 0;
        if (v > 8) v = 8;
    }
    return v;
}

// d_in = 64 with d_out in {32, 64} is one block; 128-wide sides are decomposed into 64-wide blocks of the same kernels:
// T = gM·[W1|W2] is linear in gM, so the d_out halves accumulate into gS / gEl in place; the weight-gradient blocks are
// independent.  A blocked d_out needs the output-row gradients already normalize-backwarded (gh_normalized): the
// in-kernel version needs the norm of the whole E_out row.
bool ngcf_dense_bwd_tc_eligible(int d_in, int d_out, int gh_normalized) {
    if (d_in == 64 && (d_out == 32 || d_out == 64)) return true;
    return (d_in == 64 || d_in == 128) && (d_out == 64 || d_out == 128) && (d_out <= 64 || gh_normalized);
}

int ngcf_dense_bwd_tc(const float* gE_next, const int32_t* slot, const float* gsum, int64_t ld_gsum, int col_off,
                      const float* E_out, const float* S, const float* E, int64_t n_rows, int d_in, int d_out,
                      const float* W1, const float* W2, float slope, const float* mess_mult, const uint32_t* mess_bits,
                      float mess_p, uint64_t seed, const uint64_t* seed_dev, int layer, int64_t row_offset,
                      int gh_normalized, float* gS, float* gEl, float* gW1, float* gb1, float* gW2, float* gb2,
                      float* gM_scratch, cudaStream_t st) {
    const int bn = d_out > 64 ? 64 : d_out;                               // block width on the d_out side
    const int IH = d_in / 64, OH = d_out / bn;
    const int KBo = bn / 32;
    const int n_tiles = (int)ceil_div64(n_rows, TC_ROWS);
    const size_t smem = 1024 + (size_t)4 * KBo * TC_A_BLOCK + 2 * TC_ROWS * 256 + sizeof(BwdBars);
    const int grid = (int)min((int64_t)n_tiles, (int64_t)ngcf_num_sms());
    void (*kern)(BwdTcArgs) = nullptr;
    const bool pre = gh_normalized != 0;
    switch (mess_mode(mess_mult, mess_bits, mess_p)) {
        case MM_NONE: kern = pre ? dense_bwd_tc_kernel<MM_NONE, true> : dense_bwd_tc_kernel<MM_NONE, false>; break;
        case MM_MULT: kern = pre ? dense_bwd_tc_kernel<MM_MULT, true> : dense_bwd_tc_kernel<MM_MULT, false>; break;
        case MM_BITS: kern = pre ? dense_bwd_tc_kernel<MM_BITS, true> : dense_bwd_tc_kernel<MM_BITS, false>; break;
        default: kern = pre ? dense_bwd_tc_kernel<MM_HASH, true> : dense_bwd_tc_kernel<MM_HASH, false>; break;
    }
    NGCF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    NGCF_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    for (int ih = 0; ih < IH; ++ih)
        for (int oh = 0; oh < OH; ++oh) {
            BwdTcArgs a{gE_next, slot, gsum, ld_gsum, col_off, E_out, S, E, n_rows, 64, bn, W1, W2, slope, mess_mult,
                        mess_bits, mess_p, seed, seed_dev, layer, gS, gEl, gM_scratch, gb1, gb2, n_tiles, row_offset};
            a.d_out_full = d_out; a.out_off = oh * bn; a.d_in_full = d_in; a.in_off = ih * 64;
            a.accumulate = oh > 0; a.first_in = ih == 0;
            // whole-row prefetches: full-width launches on 16-byte aligned tensors only
            const bool contiguous = d_out == bn && d_in == 64 && ((uintptr_t)E_out & 15) == 0 && ((uintptr_t)S & 15) == 0 &&
                                    ((uintptr_t)E & 15) == 0 && ((uintptr_t)gE_next & 15) == 0 && bn % 4 == 0;
            a.pf = contiguous ? dense_prefetch_tiles() : 0;
            NGCF_CUDA(ngcf_launch_pdl(kern, dim3(grid), dim3(TC_THREADS), smem, st, a));
            NGCF_LAUNCH_OK("dense_bwd_tc_kernel");
        }
    const int n_chunks = (int)ceil_div64(n_rows, WG_ROWS);
    const size_t smem2 = 1024 + (size_t)2 * (8 + 2 * KBo) * WG_BLOCK + sizeof(WgBars);
    const int grid2 = (int)min((int64_t)n_chunks, (int64_t)ngcf_num_sms());
    cudaStream_t ws = st;
    if (g_wgrad_stream && g_wgrad_stream != st) {                        // fork: the weight gradients wait for gM only
        static cudaEvent_t ev[64] = {};
        int dev = 0;
        NGCF_CUDA(cudaGetDevice(&dev));
        if (!ev[dev & 63]) NGCF_CUDA(cudaEventCreateWithFlags(&ev[dev & 63], cudaEventDisableTiming));
        NGCF_CUDA(cudaEventRecord(ev[dev & 63], st));
        NGCF_CUDA(cudaStreamWaitEvent(g_wgrad_stream, ev[dev & 63], 0));
        ws = g_wgrad_stream;
        g_wgrad_forked = 1;
    }
    for (int ih = 0; ih < IH; ++ih)
        for (int oh = 0; oh < OH; ++oh) {
            WgradArgs w{S, E, gM_scratch, n_rows, bn, gW1, gW2, n_chunks, d_in, ih * 64, d_out, oh * bn, 0};
            w.pf = (d_out == bn && d_in == 64 && ((uintptr_t)S & 15) == 0 && ((uintptr_t)E & 15) == 0 &&
                    ((uintptr_t)gM_scratch & 15) == 0 && bn % 4 == 0) ? dense_prefetch_tiles() : 0;
            NGCF_CUDA(ngcf_launch_pdl(wgrad_tc_kernel, dim3(grid2), dim3(TC_THREADS), smem2, ws, w));
            NGCF_LAUNCH_OK("wgrad_tc_kernel");
        }
    return NGCF_OK;
}

// debugging aid (tools/bwd_timeline.py): switch the CTA-0 timeline of dense_bwd_tc_kernel on/off and read it back
extern "C" int ngcf_debug_bwd_timeline(int enable, long long* out_host /*[4*8*8] or NULL*/) {
    NGCF_CUDA(cudaMemcpyToSymbol(g_bwd_dbg_on, &enable, sizeof(int)));
    if (out_host) NGCF_CUDA(cudaMemcpyFromSymbol(out_host, g_bwd_dbg, sizeof(long long) * 4 * 8 * 8));
    return NGCF_OK;
}
