// Tiled CSR SpMM  Y = L·X (+ addend) (+ sparse row-gradient rows).
// Replaces torch.mm(L, E) (NGCF.py:130: coalesce -> COO->CSR -> cusparseSpMM on CUDA) and the transposed
// product of its backward (MmBackward0).  See spmm_core.cuh for the data layout and the mapping.
//
// spmm_stream_kernel (widths that are multiples of 4): ONE launch covers the hub-chunk tiles (first: they are the
// longest) and the ordinary-row tiles, one 64-thread CTA per tile, the hardware block scheduler balances them;
// hub_finish_kernel behind it sums the chunk partials of every hub row in a fixed order.  spmm_tile_kernel (any width
// <= 128, e.g. the reference's 65): one row per warp; the warp that stores the last chunk partial of a hub row completes
// that row (fence + counter).  (First version: hub pass and row pass as two launches, the row pass reading
// hub_of_row[row] before every row - tools/spmm_timeline.py showed that dependent load plus the narrow tail batches as
// 4-8 exposed round trips per 16-row tile, and the two launches each paid their own tail.)
#include "spmm_core.cuh"

namespace {

using namespace ngcf;

#ifndef NGCF_SPMM_THREADS
#define NGCF_SPMM_THREADS 64
#endif
constexpr int SP_THREADS = NGCF_SPMM_THREADS;
constexpr int SP_WARPS = SP_THREADS / 32;

struct TileSide {                   // one tile list: the ordinary rows, or the hub chunks
    const TileInfo* tiles;
    const int32_t* rowptr;
    const int2* ent;
    const int32_t* row_key;         // chunk side: row of each chunk (dropout key); row side: NULL
    const uint8_t* bits;            // optional decision bytes (ngcf_node_dropout_bits), indexed like `ent`
    const int2* cent;               // optional: this layer's compacted entries (ngcf_node_dropout_compact), tile t at e0
    const int32_t* ccnt;            // ... and the number of survivors of each tile [n_tiles]
    float* Y;                       // output rows (chunk side: hub_partial, one row per chunk)
    int64_t ldy;
};

struct SpmmArgs {
    TileSide rows, chunks;
    int n_chunk_tiles;              // CTAs [0, n_chunk_tiles) take chunk tiles, the rest row tiles
    const float* X;
    uint32_t ldx;
    int d;
    const float* addend;            // row side only
    int64_t ld_add;
    const int32_t* slot;
    const float* gsum;
    int64_t ld_gsum;
    // hub rows: the warp that stores the LAST chunk partial of a hub (counted in hub_done) sums the hub's partials in
    // chunk order and writes the row; the counter is left at zero again
    const int32_t* hub_of_row;      // [n_rows] hub id or -1 (NULL: no hubs)
    const int32_t* hub_chunk_ptr;   // [n_hub + 1]
    int32_t* hub_done;              // [n_hub], all zero between calls
    float* Yrows;                   // the product's output (chunk side writes its own hub rows there)
    int64_t ld_yrows;
    float drop_p;
    uint64_t seed;
    const uint64_t* seed_dev;
    int layer;
    int transposed;
    uint32_t row_off;
    unsigned long long* dbg;        // optional [n_ctas][4] = {start, staged, done, smid} in globaltimer ns (tools/spmm_timeline.py)
    // streaming kernel
    const uint32_t* tile_hubmask;   // [n_row_tiles] bit i = row i of the tile is a hub (written by hub_finish_kernel); NULL: no hubs
    int n_row_tiles;
    int add_mode;                   // Y already holds the addend: row sums are ADDED to it (red.global.add)
    const int32_t* hub_rows;        // [n_hub]
    int n_hub;
};

__device__ __forceinline__ unsigned long long gtime_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void stamp_done(unsigned long long* dbg) {
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        dbg[blockIdx.x * 4 + 2] = gtime_ns();
        dbg[blockIdx.x * 4 + 3] = smid;
    }
}

struct CtaSync {
    __device__ __forceinline__ void operator()() const { __syncthreads(); }
};

// G > 0: vector path with G lanes per gathered row; G == 0: scalar path
#ifndef NGCF_SPMM_CTAS
#define NGCF_SPMM_CTAS 20
#endif
template <int G>
__global__ void __launch_bounds__(SP_THREADS, NGCF_SPMM_CTAS) spmm_tile_kernel(SpmmArgs a) {
    __shared__ __align__(16) int2 ent_s[SP_TILE_ENT];
    __shared__ int rp_s[SP_TILE_ROWS + 1];
    __shared__ int hub_s[SP_TILE_ROWS];                               // row side: hub id of each tile row, or -1
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    pdl_launch_dependents();
    if (a.dbg && tid == 0) a.dbg[blockIdx.x * 4 + 0] = gtime_ns();
    const bool chunk_side = (int)blockIdx.x < a.n_chunk_tiles;
    const TileSide& sd = chunk_side ? a.chunks : a.rows;
    const int t = chunk_side ? (int)blockIdx.x : (int)blockIdx.x - a.n_chunk_tiles;
    const int4 raw = *reinterpret_cast<const int4*>(sd.tiles + t);
    const TileInfo ti{raw.x, raw.y, raw.z, raw.w};
    const int nr = ti.r1 - ti.r0;
    if (tid < nr)      // chunk side: the chunk's row; row side: is the row a hub (then it is not written here)
        hub_s[tid] = chunk_side ? a.hub_of_row[sd.row_key[ti.r0 + tid]] : (a.hub_of_row ? a.hub_of_row[ti.r0 + tid] : -1);
    // everything above is the plan's static layout; entries (possibly this step's compacted survivors), X, addend and
    // the outputs belong to the stream order
    pdl_wait();
    {
        DropArgs dr{a.drop_p, a.drop_p > 0.f ? ngcf_seed(a.seed, a.seed_dev) : 0ull, a.layer, a.transposed,
                    a.row_off, sd.bits};
        stage_tile<SP_THREADS>(ti, sd.rowptr, sd.ent, sd.row_key, dr, rp_s, ent_s, tid, CtaSync());
    }
    if (a.dbg && tid == 0) a.dbg[blockIdx.x * 4 + 1] = gtime_ns();

    if (chunk_side) {
        // a chunk = up to SPLIT entries of one hub row: the whole warp gathers it (lane groups split the entries)
        for (int i = warp; i < nr; i += SP_WARPS) {
            const int64_t chunk = ti.r0 + i;
            const int h = hub_s[i];
            if constexpr (G > 0) {
                const float4 acc = gather_row_vec<G>(ent_s, rp_s[i], rp_s[i + 1], a.X, a.ldx, a.d, lane);
                if (lane < G && lane * 4 < a.d) st_f4(sd.Y + chunk * sd.ldy + lane * 4, acc);
            } else {
                float acc[SC_MAXQ];
                gather_row_sc(ent_s, rp_s[i], rp_s[i + 1], a.X, a.ldx, a.d, lane, acc);
#pragma unroll
                for (int q = 0; q < SC_MAXQ; ++q)
                    if (lane + 32 * q < a.d) sd.Y[chunk * sd.ldy + lane + 32 * q] = acc[q];
            }
            // completion count of the hub; the last arriving warp finishes the row
            __threadfence();
            __syncwarp();
            const int c0 = a.hub_chunk_ptr[h], c1 = a.hub_chunk_ptr[h + 1];
            int last = 0;
            if (lane == 0) last = (atomicAdd(a.hub_done + h, 1) + 1 == c1 - c0);
            last = __shfl_sync(FULL_MASK, last, 0);
            if (!last) continue;
            __threadfence();
            if (lane == 0) a.hub_done[h] = 0;                         // ready for the next product
            const int64_t row = sd.row_key[chunk] ;
            const int s = a.slot ? a.slot[row] : -1;
            if constexpr (G > 0) {
                float4 sum = sum_partials_split<G>(sd.Y, c0, c1, a.d, lane);
                if (lane < G && lane * 4 < a.d) {
                    const int c = lane * 4;
                    if (a.addend) {
                        const float4 ad = ld_f4(a.addend + row * a.ld_add + c);
                        sum.x += ad.x; sum.y += ad.y; sum.z += ad.z; sum.w += ad.w;
                    }
                    if (s >= 0) {
                        const float4 gs = ld_f4(a.gsum + (int64_t)s * a.ld_gsum + c);
                        sum.x += gs.x; sum.y += gs.y; sum.z += gs.z; sum.w += gs.w;
                    }
                    st_f4(a.Yrows + row * a.ld_yrows + c, sum);
                }
            } else {
                float sum[SC_MAXQ];
                sum_partials_sc(sd.Y, c0, c1, a.d, lane, sum);
#pragma unroll
                for (int q = 0; q < SC_MAXQ; ++q) {
                    const int col = lane + 32 * q;
                    if (col < a.d) {
                        float r = sum[q];
                        if (a.addend) r += a.addend[row * a.ld_add + col];
                        if (s >= 0) r += a.gsum[(int64_t)s * a.ld_gsum + col];
                        a.Yrows[row * a.ld_yrows + col] = r;
                    }
                }
            }
        }
        if (a.dbg) stamp_done(a.dbg);
        return;
    }

    // ordinary rows (hub rows are written by the chunk side)
    if constexpr (G > 0) {
        // the warp's lane groups split one row's entries (measured faster than one row per group: 43.9 vs 47.3 us for
        // the launch at Gowalla shape — short rows leave fewer lanes idle this way)
        for (int i = warp; i < nr; i += SP_WARPS) {
            if (hub_s[i] >= 0) continue;
            const int64_t row = ti.r0 + i;
            const bool ok = lane < G && lane * 4 < a.d;
            float4 ad = make_float4(0.f, 0.f, 0.f, 0.f);                // requested before the gathers, not after them
            int s = -1;
            if (ok && a.addend) ad = ld_f4(a.addend + row * a.ld_add + lane * 4);
            if (ok && a.slot) s = a.slot[row];
            float4 acc = gather_row_vec<G>(ent_s, rp_s[i], rp_s[i + 1], a.X, a.ldx, a.d, lane);
            if (ok) {
                acc.x += ad.x; acc.y += ad.y; acc.z += ad.z; acc.w += ad.w;
                if (s >= 0) {
                    const float4 gs = ld_f4(a.gsum + (int64_t)s * a.ld_gsum + lane * 4);
                    acc.x += gs.x; acc.y += gs.y; acc.z += gs.z; acc.w += gs.w;
                }
                st_f4(sd.Y + row * sd.ldy + lane * 4, acc);
            }
        }
    } else {
        for (int i = warp; i < nr; i += SP_WARPS) {
            if (hub_s[i] >= 0) continue;
            const int64_t row = ti.r0 + i;
            float acc[SC_MAXQ];
            gather_row_sc(ent_s, rp_s[i], rp_s[i + 1], a.X, a.ldx, a.d, lane, acc);
            const int s = a.slot ? a.slot[row] : -1;
#pragma unroll
            for (int q = 0; q < SC_MAXQ; ++q) {
                const int col = lane + 32 * q;
                if (col < a.d) {
                    float r = acc[q];
                    if (a.addend) r += a.addend[row * a.ld_add + col];
                    if (s >= 0) r += a.gsum[(int64_t)s * a.ld_gsum + col];
                    sd.Y[row * sd.ldy + col] = r;
                }
            }
        }
    }
    if (a.dbg) stamp_done(a.dbg);
}

__device__ __forceinline__ void red_add_f4(float* p, float4 v) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// ---- streaming version (round 2) -------------------------------------------------------------------------------------
// tools/l2_gather_bench.cu: 40 resident warps that do nothing but gather the real column stream of the Gowalla-shaped
// product, 4 rows in flight per lane group, move 19.6 TB/s out of L2 on a B200 (27 us per product; 32 us with one
// short-lived CTA per 512-entry tile); the row-per-warp kernel above takes 48-53 us.  An ablation (profiles/
// r02_spmm_experiments.txt) located the difference in what every short-lived CTA does SERIALLY around its gathers:
// tile record -> hub flags (a dependent global load) -> entries, the write-out, and the hub completion protocol with
// its two __threadfence() (each one also invalidates the SM's L1).  This kernel keeps the CTA-per-tile shape but
// removes those: hub flags are a bit mask in a per-tile word read next to the tile record, hub rows are finished by
// hub_finish_kernel behind it (no fences or counters here), an addend is not re-read (Y already holds it and the row
// sums are ADDED with red.global.add.v4), and the tile's entries are ONE stream, cut into equal contiguous ranges for the CTA's lane groups; a group runs full
// batches over its range whatever the row lengths are, and every entry names its row (top bits of the column word, see
// spmm_core.cuh), so a change of row just parks the running sum in a shared-memory row buffer.  A row that straddles two
// ranges is completed in fixed order afterwards (no float atomics: results stay bit-reproducible): each group parks
// the sum of the FIRST row it meets in its own slot `pf` (that row may have started in an earlier range), every later
// row of its range starts inside the range, is therefore owned by this group alone and goes to `ysum`; the write-out
// adds, per row, ysum and the pf slots that name the row, in group order.
template <int G>
__global__ void __launch_bounds__(SP_THREADS, NGCF_SPMM_CTAS) spmm_stream_kernel(SpmmArgs a) {
    constexpr int NGRP = SP_THREADS / G;                              // lane groups of the CTA
    __shared__ __align__(16) int2 ent_s[SP_TILE_ENT];
    __shared__ __align__(16) float ysum[SP_TILE_ROWS * G * 4];
    __shared__ __align__(16) float pf[SP_THREADS * 4];                // [NGRP][G * 4]
    __shared__ int rp_s[SP_TILE_ROWS + 1];
    __shared__ int first_row[NGRP];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int grp = tid / G, l = tid % G;
    pdl_launch_dependents();
    if (a.dbg && tid == 0) a.dbg[blockIdx.x * 4 + 0] = gtime_ns();
    const bool chunk_side = (int)blockIdx.x < a.n_chunk_tiles;
    const TileSide& sd = chunk_side ? a.chunks : a.rows;
    const int t = chunk_side ? (int)blockIdx.x : (int)blockIdx.x - a.n_chunk_tiles;
    const int4 raw = *reinterpret_cast<const int4*>(sd.tiles + t);
    const TileInfo ti{raw.x, raw.y, raw.z, raw.w};
    const int nr = ti.r1 - ti.r0;
    // rows of this tile that are hubs (their entries live in the chunk tiles; hub_finish_kernel writes them)
    const uint32_t hubmask = (!chunk_side && a.tile_hubmask) ? a.tile_hubmask[t] : 0u;
    // every row slot is cleared, not just the tile's nr: the loop then does not wait for the tile record, whose round
    // trip overlaps the survivor count's below instead of preceding it (one L2 round trip less in every CTA's serial
    // chain record -> count -> entries -> gathers)
#pragma unroll
    for (int i = tid; i < SP_TILE_ROWS * G; i += SP_THREADS) reinterpret_cast<float4*>(ysum)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    pdl_wait();
    int cnt;
    if (sd.ccnt) {
        cnt = sd.ccnt[t];                                             // this step's survivors of the tile, compacted at e0
        for (int i = tid; i < cnt; i += SP_THREADS) ent_s[i] = ld_stream_i2(sd.cent + ti.e0 + i);
        __syncthreads();
    } else {
        cnt = ti.e1 - ti.e0;
        DropArgs dr{a.drop_p, a.drop_p > 0.f ? ngcf_seed(a.seed, a.seed_dev) : 0ull, a.layer, a.transposed,
                    a.row_off, sd.bits};
        stage_tile<SP_THREADS>(ti, sd.rowptr, sd.ent, sd.row_key, dr, rp_s, ent_s, tid, CtaSync());
    }
    if (a.dbg && tid == 0) a.dbg[blockIdx.x * 4 + 1] = gtime_ns();

    {
        const int per = (cnt + NGRP - 1) / NGRP;
        int j = min(grp * per, cnt);
        const int end = min(j + per, cnt);
        const char* xl = reinterpret_cast<const char*>(a.X + ((l * 4) < a.d ? l * 4 : 0));
        const uint32_t row_bytes = a.ldx * 4u;
        float* const pf_l = pf + grp * (G * 4) + l * 4;
        float* const ys_l = ysum + l * 4;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        int cur = -1, frow = -1;
        bool isfirst = true;
        auto step = [&](const int2 e, const float4 x) {
            const int lr = ent_lrow(e.x);
            if (lr != cur) {                                          // the previous row of this range is complete
                if (cur >= 0) {
                    st_f4(isfirst ? pf_l : ys_l + cur * (G * 4), acc);
                    if (isfirst) frow = cur;
                    isfirst = false;
                }
                acc = make_float4(0.f, 0.f, 0.f, 0.f);
                cur = lr;
            }
            const float w = __int_as_float(e.y);
            acc.x = fmaf(w, x.x, acc.x);
            acc.y = fmaf(w, x.y, acc.y);
            acc.z = fmaf(w, x.z, acc.z);
            acc.w = fmaf(w, x.w, acc.w);
        };
        for (; j + UNROLL <= end; j += UNROLL) {
            int2 e[UNROLL];
            float4 x[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) e[u] = ent_s[j + u];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u)
                x[u] = ld_f4(reinterpret_cast<const float*>(xl + (uint64_t)ent_col(e[u].x) * row_bytes));
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) step(e[u], x[u]);
        }
        if (j < end) {                                                // one predicated batch per range
            int2 e[UNROLL];
            float4 x[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                e[u] = make_int2(0, 0);
                x[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (j + u < end) {
                    e[u] = ent_s[j + u];
                    x[u] = ld_f4(reinterpret_cast<const float*>(xl + (uint64_t)ent_col(e[u].x) * row_bytes));
                }
            }
#pragma unroll
            for (int u = 0; u < UNROLL; ++u)
                if (j + u < end) step(e[u], x[u]);
        }
        if (cur >= 0) {
            st_f4(isfirst ? pf_l : ys_l + cur * (G * 4), acc);
            if (isfirst) frow = cur;
        }
        if (l == 0) first_row[grp] = frow;
    }
    __syncthreads();

    // the completed sum of tile row i for this lane's four columns
    auto row_sum = [&](int i, int ll) {
        float4 y = ld_f4(ysum + i * (G * 4) + ll * 4);
#pragma unroll
        for (int q = 0; q < NGRP; ++q)
            if (first_row[q] == i) {
                const float4 p = ld_f4(pf + q * (G * 4) + ll * 4);
                y.x += p.x; y.y += p.y; y.z += p.z; y.w += p.w;
            }
        return y;
    };

    if (chunk_side) {
        // a "row" here is a chunk of a hub row: its sum goes to hub_partial; hub_finish_kernel adds the partials up
        const bool okc = l * 4 < a.d;
        for (int i = grp; i < nr; i += NGRP)
            if (okc) st_f4(sd.Y + (int64_t)(ti.r0 + i) * sd.ldy + l * 4, row_sum(i, l));
        if (a.dbg) stamp_done(a.dbg);
        return;
    }

    // ordinary rows; a lane group writes one row: coalesced 16 * G bytes.  add_mode: Y already holds the addend
    const bool ok = l * 4 < a.d;
    for (int i = grp; i < nr; i += NGRP) {
        if (((hubmask >> i) & 1u) || !ok) continue;
        const int64_t row = ti.r0 + i;
        float4 y = row_sum(i, l);
        const int s = a.slot ? a.slot[row] : -1;
        if (s >= 0) {
            const float4 gs = ld_f4(a.gsum + (int64_t)s * a.ld_gsum + l * 4);
            y.x += gs.x; y.y += gs.y; y.z += gs.z; y.w += gs.w;
        }
        float* dst = sd.Y + row * sd.ldy + l * 4;
        if (a.add_mode) red_add_f4(dst, y); else st_f4(dst, y);
    }
    if (a.dbg) stamp_done(a.dbg);
}

// One CTA per hub row: the chunk partials (written by spmm_stream_kernel right before) summed in a fixed order - lane
// group g adds chunks g, g + NGRP, ... (4 loads in flight), group 0 then adds the group sums in group order.  (First
// version: one warp per hub; the widest hub of the Gowalla-shaped graph has 107 chunks = 14 dependent round trips for
// one warp, an 11-us launch for 2 MB of data.)
constexpr int HF_THREADS = 128;
template <int G>
__global__ void __launch_bounds__(HF_THREADS) hub_finish_kernel(SpmmArgs a) {
    constexpr int NGRP = HF_THREADS / G;
    __shared__ __align__(16) float gs[HF_THREADS * 4];                   // [NGRP][G * 4]
    pdl_launch_dependents();
    const int tid = threadIdx.x, g = tid / G, l = tid % G;
    const int h = blockIdx.x;
    const int c0 = a.hub_chunk_ptr[h], c1 = a.hub_chunk_ptr[h + 1];      // static plan data
    const int64_t row = a.hub_rows[h];
    pdl_wait();
    const bool ok = l * 4 < a.d;
    // the row's addend and batch-row gradient slot are requested before the partial sums, not after them
    float* const dst = a.Yrows + row * a.ld_yrows + l * 4;
    float4 ad = make_float4(0.f, 0.f, 0.f, 0.f);
    int s = -1;
    if (g == 0 && ok) {
        if (a.add_mode) ad = ld_f4(dst);
        if (a.slot) s = a.slot[row];
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ok) {
        const float* p = a.chunks.Y + l * 4;
        int c = c0 + g;
        for (; c + 3 * NGRP < c1; c += 4 * NGRP) {
            float4 x[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) x[u] = __ldcg(reinterpret_cast<const float4*>(p + (int64_t)(c + u * NGRP) * a.d));
#pragma unroll
            for (int u = 0; u < 4; ++u) { acc.x += x[u].x; acc.y += x[u].y; acc.z += x[u].z; acc.w += x[u].w; }
        }
        for (; c < c1; c += NGRP) {
            const float4 x = __ldcg(reinterpret_cast<const float4*>(p + (int64_t)c * a.d));
            acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
        }
    }
    st_f4(gs + g * (G * 4) + l * 4, acc);
    __syncthreads();
    if (g == 0 && ok) {
        float4 sum = acc;
#pragma unroll
        for (int q = 1; q < NGRP; ++q) {
            const float4 v = ld_f4(gs + q * (G * 4) + l * 4);
            sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
        }
        if (a.add_mode) {                                             // Y holds the addend; this CTA owns the row
            sum.x += ad.x; sum.y += ad.y; sum.z += ad.z; sum.w += ad.w;
        }
        if (s >= 0) {
            const float4 gsv = ld_f4(a.gsum + (int64_t)s * a.ld_gsum + l * 4);
            sum.x += gsv.x; sum.y += gsv.y; sum.z += gsv.z; sum.w += gsv.w;
        }
        st_f4(dst, sum);
    }
}

// Node-dropout decisions of one step for every entry of a tile list, all layers at once (bit k = survives layer k).
// out_f: keyed on (row, col) = this CSR read as L; out_t: keyed on (col, row) = the same CSR read as L^T (a
// symmetric L shares one CSR for both directions).  Either may be NULL.
struct BitsArgs {
    const TileInfo* tiles;
    const int32_t* rowptr;
    const int2* ent;
    const int32_t* row_key;
    float p;
    uint64_t seed;
    const uint64_t* seed_dev;
    int n_layers;
    uint32_t row_off;
    uint8_t* out_f;
    uint8_t* out_t;
};

// One CTA covers BITS_TILES consecutive tiles (= one contiguous row range and one contiguous entry range): with a
// CTA per 512-entry tile the pass was bound by the tile-info -> rowptr -> entries latency chain of ~6000 tiny CTAs.
constexpr int BITS_THREADS = 256;
constexpr int BITS_TILES = 8;
__global__ void __launch_bounds__(BITS_THREADS) dropout_bits_kernel(BitsArgs a, int n_tiles) {
    __shared__ int rp_s[BITS_TILES * SP_TILE_ROWS + 1];
    const int tid = threadIdx.x;
    const int t0 = blockIdx.x * BITS_TILES, t1 = min(t0 + BITS_TILES, n_tiles) - 1;
    const int4 first = *reinterpret_cast<const int4*>(a.tiles + t0);
    const int4 last = *reinterpret_cast<const int4*>(a.tiles + t1);
    const int r0 = first.x, nr = last.y - first.x, e0 = first.z, cnt = last.w - first.z;
    for (int i = tid; i <= nr; i += BITS_THREADS) rp_s[i] = a.rowptr[r0 + i] - e0;
    __syncthreads();
    const uint64_t seed = ngcf_seed(a.seed, a.seed_dev);
    for (int i = tid; i < cnt; i += BITS_THREADS) {
        const uint32_t c = ent_col(ld_stream_i2(a.ent + e0 + i).x);
        int lo = 0, hi = nr - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (rp_s[mid] <= i) lo = mid; else hi = mid - 1;
        }
        const uint32_t r = (uint32_t)(a.row_key ? a.row_key[r0 + lo] : r0 + lo) + a.row_off;
        if (a.out_f) a.out_f[e0 + i] = (uint8_t)node_keep_bits(a.p, seed, a.n_layers, r, c);
        if (a.out_t) a.out_t[e0 + i] = (uint8_t)node_keep_bits(a.p, seed, a.n_layers, c, r);
    }
}

// Static node-dropout keys of every entry of a tile list (plan time, once): key_l = ngcf_node_key(row, col) for the
// CSR read as L, key_t = ngcf_node_key(col, row) for the same CSR read as L^T.
struct KeyArgs {
    const TileInfo* tiles;
    const int32_t* rowptr;
    const int2* ent;
    const int32_t* row_key;
    uint32_t row_off;
    uint32_t* key_l;
    uint32_t* key_t;
};
__global__ void __launch_bounds__(BITS_THREADS) entry_keys_kernel(KeyArgs a, int n_tiles) {
    __shared__ int rp_s[BITS_TILES * SP_TILE_ROWS + 1];
    const int tid = threadIdx.x;
    const int t0 = blockIdx.x * BITS_TILES, t1 = min(t0 + BITS_TILES, n_tiles) - 1;
    const int4 first = *reinterpret_cast<const int4*>(a.tiles + t0);
    const int4 last = *reinterpret_cast<const int4*>(a.tiles + t1);
    const int r0 = first.x, nr = last.y - first.x, e0 = first.z, cnt = last.w - first.z;
    for (int i = tid; i <= nr; i += BITS_THREADS) rp_s[i] = a.rowptr[r0 + i] - e0;
    __syncthreads();
    for (int i = tid; i < cnt; i += BITS_THREADS) {
        const uint32_t c = ent_col(ld_stream_i2(a.ent + e0 + i).x);
        int lo = 0, hi = nr - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (rp_s[mid] <= i) lo = mid; else hi = mid - 1;
        }
        const uint32_t r = (uint32_t)(a.row_key ? a.row_key[r0 + lo] : r0 + lo) + a.row_off;
        a.key_l[e0 + i] = ngcf_node_key(r, c);
        a.key_t[e0 + i] = ngcf_node_key(c, r);
    }
}

// ---- per-step node-dropout compaction -----------------------------------------------------------------------------
// The reference's sparse_dropout (NGCF.py:93-100) DELETES the dropped entries, cumulatively over the layers, so its
// layer-k product walks only (1-p)^(k+1) of the Laplacian.  One pass per step does the same for every layer and both
// directions at once: the surviving entries of tile t are written, in their original order, to the front of the
// tile's own slot range [e0, e1) of a per-(direction, layer) entry array, and their number to a per-tile count array.
// The products then stage and gather the survivors only (same sums: a dropped entry contributed +0.0), which at
// p = 0.3 halves the gathered bytes of a 3-layer step.  Entries carry their row (spmm_core.cuh), so no row pointers
// have to be rebuilt.
constexpr int WS_PER = SP_TILE_ENT / 32;     // entries of a tile per lane of the compaction warp
static_assert(WS_PER * 32 == SP_TILE_ENT, "tile entries must be a multiple of the warp size");

struct CompactArgs {
    const TileInfo* tiles;
    const int2* ent;
    const int32_t* row_key;
    float p;
    uint64_t seed;
    const uint64_t* seed_dev;
    int n_layers;
    uint32_t row_off;
    const uint32_t* key_l;                   // optional static per-entry keys (ngcf_entry_keys), indexed like `ent`:
    const uint32_t* key_t;                   //   ngcf_node_key(row, col) and ngcf_node_key(col, row)
    int2* out_ent[2][NGCF_MAX_LAYERS];       // [0] keyed (row, col) = this CSR read as L, [1] keyed (col, row) = as L^T
    int32_t* out_cnt[2][NGCF_MAX_LAYERS];    // NULL: direction/layer not wanted
};

// One WARP per tile (<= 128 entries: WS_PER per lane, entry q * 32 + lane), no barrier.  Order-preserving compaction by
// warp ballots: the position of an entry among a combo's survivors is the survivors of earlier 32-entry segments plus
// the survivors below its lane; consecutive lanes write consecutive survivors, so the stores are coalesced.
constexpr int CW_WARPS = 4;
__global__ void __launch_bounds__(CW_WARPS * 32) compact_kernel(CompactArgs a, int n_tiles) {
    const int lane = threadIdx.x & 31;
    const int t = blockIdx.x * CW_WARPS + (threadIdx.x >> 5);
    if (t >= n_tiles) return;
    const int4 raw = *reinterpret_cast<const int4*>(a.tiles + t);
    const TileInfo ti{raw.x, raw.y, raw.z, raw.w};
    const int cnt = ti.e1 - ti.e0;
    const int K = a.n_layers;
    const bool want_l = a.out_ent[0][0] != nullptr, want_t = a.out_ent[1][0] != nullptr;
    int2 e[WS_PER];
    uint32_t kl[WS_PER], kt[WS_PER];
#pragma unroll
    for (int q = 0; q < WS_PER; ++q) {
        const int p = q * 32 + lane;
        e[q] = make_int2(0, 0);
        kl[q] = kt[q] = 0;
        if (p < cnt) {
            e[q] = ld_stream_i2(a.ent + ti.e0 + p);
            if (a.key_l) {
                if (want_l) kl[q] = a.key_l[ti.e0 + p];
                if (want_t) kt[q] = a.key_t[ti.e0 + p];
            }
        }
    }
    const uint64_t seed = ngcf_seed(a.seed, a.seed_dev);
    const uint32_t thr = ngcf_threshold16(a.p);
    uint32_t keep[WS_PER];                            // bit c = the entry survives combo c = dir * K + layer
#pragma unroll
    for (int q = 0; q < WS_PER; ++q) {
        const int p = q * 32 + lane;
        keep[q] = 0;
        if (p < cnt) {
            if (!a.key_l) {                           // no static keys in the plan: derive them from the coordinates
                const int lr = ent_lrow(e[q].x);
                const uint32_t r = (uint32_t)(a.row_key ? a.row_key[ti.r0 + lr] : ti.r0 + lr) + a.row_off;
                kl[q] = ngcf_node_key(r, ent_col(e[q].x));
                kt[q] = ngcf_node_key(ent_col(e[q].x), r);
            }
            if (want_l) keep[q] = node_keep_bits_key(thr, seed, K, kl[q]);
            if (want_t) keep[q] |= node_keep_bits_key(thr, seed, K, kt[q]) << K;
        }
    }
    const uint32_t below = (1u << lane) - 1u;
    for (int c = 0; c < 2 * K; ++c) {
        const int dir = c >= K, layer = dir ? c - K : c;
        int2* out = a.out_ent[dir][layer];
        if (!out) continue;
        int base = 0;
#pragma unroll
        for (int q = 0; q < WS_PER; ++q) {
            const bool k = (keep[q] >> c) & 1u;
            const uint32_t m = __ballot_sync(FULL_MASK, k);
            if (k) out[ti.e0 + base + __popc(m & below)] = e[q];
            base += __popc(m);
        }
        if (lane == 0) a.out_cnt[dir][layer][t] = base;
    }
}

template <int G>
int launch(const SpmmArgs& a, int n_ctas, bool stream, cudaStream_t st) {
    if (n_ctas <= 0) return NGCF_OK;
    if constexpr (G > 0) {
        if (stream) {
            NGCF_CUDA(ngcf_launch_pdl(spmm_stream_kernel<G>, dim3((unsigned)n_ctas), dim3(SP_THREADS), 0, st, a));
            NGCF_LAUNCH_OK("spmm_stream_kernel");
            if (a.n_hub > 0) {
                NGCF_CUDA(ngcf_launch_pdl(hub_finish_kernel<G>, dim3((unsigned)a.n_hub), dim3(HF_THREADS), 0, st, a));
                NGCF_LAUNCH_OK("hub_finish_kernel");
            }
            return NGCF_OK;
        }
    }
    NGCF_CUDA(ngcf_launch_pdl(spmm_tile_kernel<G>, dim3((unsigned)n_ctas), dim3(SP_THREADS), 0, st, a));
    NGCF_LAUNCH_OK("spmm_tile_kernel");
    return NGCF_OK;
}

int launch_any(const SpmmArgs& a, int n_ctas, bool vec, bool stream, cudaStream_t st) {
    if (!vec) return launch<0>(a, n_ctas, false, st);
    const int d4 = a.d / 4;
    if (d4 <= 1) return launch<1>(a, n_ctas, stream, st);
    if (d4 <= 2) return launch<2>(a, n_ctas, stream, st);
    if (d4 <= 4) return launch<4>(a, n_ctas, stream, st);
    if (d4 <= 8) return launch<8>(a, n_ctas, stream, st);
    if (d4 <= 16) return launch<16>(a, n_ctas, stream, st);
    return launch<32>(a, n_ctas, stream, st);
}

unsigned long long* g_spmm_dbg = nullptr;    // host copy of the debug buffer pointer
unsigned long long* g_spmm_dbg_compact = nullptr;   // ... for the row launch of the compaction pass

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

extern "C" int ngcf_spmm_split_threshold(void) { return ngcf::SPLIT; }
extern "C" int ngcf_spmm_tile_rows(void) { return SP_TILE_ROWS; }
extern "C" int ngcf_spmm_tile_entries(void) { return SP_TILE_ENT; }

int ngcf_check_csr(const ngcf_csr* g, const char* who) {
    NGCF_REQUIRE(g != nullptr, "%s: csr descriptor is null", who);
    NGCF_REQUIRE(g->n_rows >= 0 && g->n_rows < ((int64_t)1 << 31), "%s: n_rows %lld", who, (long long)g->n_rows);
    NGCF_REQUIRE(g->n_rows == 0 || (g->rowptr && g->ent), "%s: rowptr/ent missing", who);
    NGCF_REQUIRE(g->n_hub >= 0 && g->n_chunks >= 0, "%s: negative hub counts", who);
    NGCF_REQUIRE(g->n_hub == 0 || (g->hub_of_row && g->hub_chunk_ptr && g->chunk_ptr && g->hub_ent && g->chunk_row),
                 "%s: hub arrays missing", who);
    return NGCF_OK;
}

extern "C" int ngcf_spmm(const ngcf_csr* g, const float* X, int64_t ldx, int d, const float* addend, int64_t ld_add,
                         const int32_t* slot, const float* gsum, int64_t ld_gsum, float* hub_partial, float drop_p,
                         uint64_t seed, const uint64_t* seed_dev, int layer, int transposed, int64_t row_offset,
                         const uint8_t* keep_bits, const int32_t* c_ent, const int32_t* c_cnt, float* Y, int64_t ldy,
                         void* stream) {
    int rc = ngcf_check_csr(g, "spmm");
    if (rc != NGCF_OK) return rc;
    NGCF_REQUIRE(X && Y, "spmm: null pointer");
    NGCF_REQUIRE(d > 0 && d <= NGCF_MAX_WIDTH, "spmm: width %d not in [1,%d]", d, NGCF_MAX_WIDTH);
    NGCF_REQUIRE(ldx >= d && ldy >= d, "spmm: leading dimension below the width %d (ldx %lld, ldy %lld)", d,
                 (long long)ldx, (long long)ldy);
    // the vector gathers address X rows with a 32-bit byte stride (one IMAD.WIDE.U32 per gathered row)
    NGCF_REQUIRE(ldx < ((int64_t)1 << 30), "spmm: ldx %lld must be below 2^30 (byte stride ldx * 4 < 2^32)",
                 (long long)ldx);
    NGCF_REQUIRE(addend != Y || ld_add == ldy, "spmm: an in-place addend (addend == Y) needs ld_add == ldy (%lld != %lld)",
                 (long long)ld_add, (long long)ldy);
    NGCF_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "spmm: drop_p %f not in [0,1)", drop_p);
    NGCF_REQUIRE(layer >= 0 && layer < NGCF_MAX_LAYERS, "spmm: layer %d", layer);
    NGCF_REQUIRE(row_offset >= 0 && row_offset < ((int64_t)1 << 31), "spmm: row_offset %lld", (long long)row_offset);
    NGCF_REQUIRE(!slot || gsum, "spmm: slot given without gsum");
    NGCF_REQUIRE((c_ent == nullptr) == (c_cnt == nullptr), "spmm: c_ent and c_cnt go together");
    NGCF_REQUIRE(g->n_hub == 0 || hub_partial, "spmm: hub_partial scratch missing");
    NGCF_REQUIRE(g->n_tiles == 0 || g->tiles, "spmm: SpMM tiles missing");
    NGCF_REQUIRE(g->n_chunk_tiles == 0 || g->chunk_tiles, "spmm: chunk tiles missing");
    if (g->n_rows == 0) return NGCF_OK;
    cudaStream_t st = as_stream(stream);
    const bool vec = (d % 4 == 0) && (ldx % 4 == 0) && (ldy % 4 == 0) && aligned16(X) && aligned16(Y) &&
                     (!addend || (aligned16(addend) && ld_add % 4 == 0)) &&
                     (!slot || (aligned16(gsum) && ld_gsum % 4 == 0)) && (g->n_hub == 0 || aligned16(hub_partial));
    const bool hubs = g->n_hub > 0 && g->n_chunks > 0;
    // vector widths: the streaming kernel; any other width: the row-per-warp kernel
    const bool stream_k = vec && (!hubs || (g->tile_hubmask && g->hub_rows));
    NGCF_REQUIRE(stream_k || !c_ent, "spmm: compacted survivor lists need the streaming kernel (width %% 4 == 0)");
    NGCF_REQUIRE(stream_k || !hubs || g->hub_done, "spmm: hub_done counters missing");
    SpmmArgs a{};
    a.rows = TileSide{reinterpret_cast<const TileInfo*>(g->tiles), g->rowptr, reinterpret_cast<const int2*>(g->ent), nullptr,
                      keep_bits, reinterpret_cast<const int2*>(c_ent), c_cnt, Y, ldy};
    a.n_chunk_tiles = hubs ? g->n_chunk_tiles : 0;
    if (hubs)
        a.chunks = TileSide{reinterpret_cast<const TileInfo*>(g->chunk_tiles), g->chunk_ptr,
                            reinterpret_cast<const int2*>(g->hub_ent), g->chunk_row,
                            keep_bits ? keep_bits + g->rowptr_nnz : nullptr,
                            c_ent ? reinterpret_cast<const int2*>(c_ent) + g->rowptr_nnz : nullptr,
                            c_cnt ? c_cnt + g->n_tiles : nullptr, hub_partial, d};
    a.X = X; a.ldx = (uint32_t)ldx; a.d = d;
    a.addend = addend; a.ld_add = ld_add; a.slot = slot; a.gsum = gsum; a.ld_gsum = ld_gsum;
    a.drop_p = drop_p; a.seed = seed; a.seed_dev = seed_dev; a.layer = layer; a.transposed = transposed;
    a.row_off = (uint32_t)row_offset;
    a.dbg = g_spmm_dbg;
    a.hub_of_row = hubs ? g->hub_of_row : nullptr;
    a.hub_chunk_ptr = g->hub_chunk_ptr;
    a.hub_done = g->hub_done;
    a.Yrows = Y;
    a.ld_yrows = ldy;
    a.tile_hubmask = hubs ? g->tile_hubmask : nullptr;
    a.n_row_tiles = g->n_tiles;
    a.hub_rows = g->hub_rows;
    a.n_hub = hubs ? g->n_hub : 0;
    if (stream_k && addend) {
        // the streaming kernel ADDS its row sums to a Y that already holds the addend (in place when addend == Y)
        if (addend != Y)
            NGCF_CUDA(cudaMemcpy2DAsync(Y, (size_t)ldy * sizeof(float), addend, (size_t)ld_add * sizeof(float),
                                        (size_t)d * sizeof(float), (size_t)g->n_rows, cudaMemcpyDeviceToDevice, st));
        a.add_mode = 1;
        a.addend = nullptr;
    }
    return launch_any(a, a.n_chunk_tiles + g->n_tiles, vec, stream_k, st);
}

extern "C" int ngcf_node_dropout_bits(const ngcf_csr* g, float drop_p, uint64_t seed, const uint64_t* seed_dev,
                                      int n_layers, int64_t row_offset, uint8_t* bits_as_L, uint8_t* bits_as_Lt,
                                      void* stream) {
    int rc = ngcf_check_csr(g, "node_dropout_bits");
    if (rc != NGCF_OK) return rc;
    NGCF_REQUIRE(drop_p > 0.f && drop_p < 1.f, "node_dropout_bits: drop_p %f not in (0,1)", drop_p);
    NGCF_REQUIRE(n_layers >= 1 && n_layers <= NGCF_MAX_LAYERS, "node_dropout_bits: n_layers %d", n_layers);
    NGCF_REQUIRE(bits_as_L || bits_as_Lt, "node_dropout_bits: no output");
    NGCF_REQUIRE(row_offset >= 0 && row_offset < ((int64_t)1 << 31), "node_dropout_bits: row_offset");
    cudaStream_t st = as_stream(stream);
    if (g->n_tiles > 0) {
        BitsArgs a{reinterpret_cast<const TileInfo*>(g->tiles), g->rowptr, reinterpret_cast<const int2*>(g->ent), nullptr,
                   drop_p, seed, seed_dev, n_layers, (uint32_t)row_offset, bits_as_L, bits_as_Lt};
        dropout_bits_kernel<<<(unsigned)ceil_div64(g->n_tiles, BITS_TILES), BITS_THREADS, 0, st>>>(a, g->n_tiles);
        NGCF_LAUNCH_OK("dropout_bits_kernel(rows)");
    }
    if (g->n_hub > 0 && g->n_chunk_tiles > 0) {
        BitsArgs a{reinterpret_cast<const TileInfo*>(g->chunk_tiles), g->chunk_ptr,
                   reinterpret_cast<const int2*>(g->hub_ent), g->chunk_row, drop_p, seed, seed_dev, n_layers,
                   (uint32_t)row_offset, bits_as_L ? bits_as_L + g->rowptr_nnz : nullptr,
                   bits_as_Lt ? bits_as_Lt + g->rowptr_nnz : nullptr};
        dropout_bits_kernel<<<(unsigned)ceil_div64(g->n_chunk_tiles, BITS_TILES), BITS_THREADS, 0, st>>>(a, g->n_chunk_tiles);
        NGCF_LAUNCH_OK("dropout_bits_kernel(hub chunks)");
    }
    return NGCF_OK;
}

extern "C" int ngcf_node_dropout_compact(const ngcf_csr* g, float drop_p, uint64_t seed, const uint64_t* seed_dev,
                                         int n_layers, int64_t row_offset, int32_t* const* ent_as_L_host,
                                         int32_t* const* cnt_as_L_host, int32_t* const* ent_as_Lt_host,
                                         int32_t* const* cnt_as_Lt_host, void* stream) {
    int rc = ngcf_check_csr(g, "node_dropout_compact");
    if (rc != NGCF_OK) return rc;
    NGCF_REQUIRE(drop_p > 0.f && drop_p < 1.f, "node_dropout_compact: drop_p %f not in (0,1)", drop_p);
    NGCF_REQUIRE(n_layers >= 1 && n_layers <= NGCF_MAX_LAYERS, "node_dropout_compact: n_layers %d", n_layers);
    NGCF_REQUIRE((ent_as_L_host && cnt_as_L_host) || (ent_as_Lt_host && cnt_as_Lt_host), "node_dropout_compact: no output");
    NGCF_REQUIRE((ent_as_L_host == nullptr) == (cnt_as_L_host == nullptr) &&
                 (ent_as_Lt_host == nullptr) == (cnt_as_Lt_host == nullptr), "node_dropout_compact: ent/cnt go together");
    NGCF_REQUIRE(row_offset >= 0 && row_offset < ((int64_t)1 << 31), "node_dropout_compact: row_offset");
    for (int k = 0; k < n_layers; ++k) {
        NGCF_REQUIRE(!ent_as_L_host || (ent_as_L_host[k] && cnt_as_L_host[k]), "node_dropout_compact: null L output %d", k);
        NGCF_REQUIRE(!ent_as_Lt_host || (ent_as_Lt_host[k] && cnt_as_Lt_host[k]), "node_dropout_compact: null L^T output %d", k);
    }
    cudaStream_t st = as_stream(stream);
    // pass 0: ordinary rows; pass 1: hub chunks (entry arrays continue after rowptr_nnz, tile arrays after n_tiles)
    for (int pass = 0; pass < 2; ++pass) {
        const int n_tiles = pass ? g->n_chunk_tiles : g->n_tiles;
        if (n_tiles <= 0 || (pass && g->n_hub == 0)) continue;
        CompactArgs a{};
        a.tiles = reinterpret_cast<const TileInfo*>(pass ? g->chunk_tiles : g->tiles);
        a.ent = reinterpret_cast<const int2*>(pass ? g->hub_ent : g->ent);
        a.row_key = pass ? g->chunk_row : nullptr;
        a.p = drop_p; a.seed = seed; a.seed_dev = seed_dev; a.n_layers = n_layers; a.row_off = (uint32_t)row_offset;
        const size_t e_off = pass ? (size_t)g->rowptr_nnz : 0, t_off = pass ? (size_t)g->n_tiles : 0;
        if (g->key_l && g->key_t && g->key_row_offset == row_offset) {
            a.key_l = g->key_l + e_off;
            a.key_t = g->key_t + e_off;
        }
        for (int k = 0; k < n_layers; ++k) {
            if (ent_as_L_host) {
                a.out_ent[0][k] = reinterpret_cast<int2*>(ent_as_L_host[k]) + e_off;
                a.out_cnt[0][k] = cnt_as_L_host[k] + t_off;
            }
            if (ent_as_Lt_host) {
                a.out_ent[1][k] = reinterpret_cast<int2*>(ent_as_Lt_host[k]) + e_off;
                a.out_cnt[1][k] = cnt_as_Lt_host[k] + t_off;
            }
        }
        compact_kernel<<<(unsigned)ceil_div64(n_tiles, CW_WARPS), CW_WARPS * 32, 0, st>>>(a, n_tiles);
        NGCF_LAUNCH_OK(pass ? "compact_kernel(hub chunks)" : "compact_kernel(rows)");
    }
    return NGCF_OK;
}

// debugging aid (tools/spmm_timeline.py): device buffer [n_ctas][4] of uint64 that every spmm_tile_kernel CTA stamps
extern "C" int ngcf_debug_spmm_timeline(unsigned long long* dev_buf_or_null) {
    g_spmm_dbg = dev_buf_or_null;
    return NGCF_OK;
}
extern "C" int ngcf_debug_compact_timeline(unsigned long long* dev_buf_or_null) {
    g_spmm_dbg_compact = dev_buf_or_null;
    return NGCF_OK;
}

extern "C" int ngcf_entry_keys(const ngcf_csr* g, int64_t row_offset, uint32_t* key_l, uint32_t* key_t, void* stream) {
    int rc = ngcf_check_csr(g, "entry_keys");
    if (rc != NGCF_OK) return rc;
    NGCF_REQUIRE(key_l && key_t, "entry_keys: null output");
    NGCF_REQUIRE(row_offset >= 0 && row_offset < ((int64_t)1 << 31), "entry_keys: row_offset");
    cudaStream_t st = as_stream(stream);
    if (g->n_tiles > 0) {
        KeyArgs a{reinterpret_cast<const TileInfo*>(g->tiles), g->rowptr, reinterpret_cast<const int2*>(g->ent), nullptr,
                  (uint32_t)row_offset, key_l, key_t};
        entry_keys_kernel<<<(unsigned)ceil_div64(g->n_tiles, BITS_TILES), BITS_THREADS, 0, st>>>(a, g->n_tiles);
        NGCF_LAUNCH_OK("entry_keys_kernel(rows)");
    }
    if (g->n_hub > 0 && g->n_chunk_tiles > 0) {
        KeyArgs a{reinterpret_cast<const TileInfo*>(g->chunk_tiles), g->chunk_ptr, reinterpret_cast<const int2*>(g->hub_ent),
                  g->chunk_row, (uint32_t)row_offset, key_l + g->rowptr_nnz, key_t + g->rowptr_nnz};
        entry_keys_kernel<<<(unsigned)ceil_div64(g->n_chunk_tiles, BITS_TILES), BITS_THREADS, 0, st>>>(a, g->n_chunk_tiles);
        NGCF_LAUNCH_OK("entry_keys_kernel(hub chunks)");
    }
    return NGCF_OK;
}
