// Row-local dense parts of one NGCF layer: the W1/W2 epilogue (NGCF.py:131-142) and its backward
// (AddmmBackward / LeakyReluBackward / the backward of F.normalize, SURVEY.md section 3.4).
//
// v1 arithmetic: exact fp32 FFMA register-tiled micro-kernels (4x4 per thread, operands in shared memory,
// LDS.128).  Every width 1..128 is accepted (the reference's own width is 65).
#include "common.cuh"

namespace {

// ------------------------------------------------------------------------------------------------
// pack: wcat = [W1^T ; W2^T]  ([2*d_in, d_out]),  bias_eff = 2*b1 + b2
// ------------------------------------------------------------------------------------------------
__global__ void pack_weights_kernel(const float* __restrict__ W1, const float* __restrict__ b1,
                                    const float* __restrict__ W2, const float* __restrict__ b2, int d_in, int d_out,
                                    float* __restrict__ wcat, float* __restrict__ bias_eff) {
    const int total = 2 * d_in * d_out;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int k = i / d_out, o = i % d_out;
        wcat[i] = k < d_in ? W1[o * d_in + k] : W2[o * d_in + (k - d_in)];
    }
    for (int o = blockIdx.x * blockDim.x + threadIdx.x; o < d_out; o += gridDim.x * blockDim.x)
        bias_eff[o] = 2.0f * b1[o] + b2[o];
}

struct PackAllArgs {
    const float* W1[NGCF_MAX_LAYERS];
    const float* b1[NGCF_MAX_LAYERS];
    const float* W2[NGCF_MAX_LAYERS];
    const float* b2[NGCF_MAX_LAYERS];
    float* wcat[NGCF_MAX_LAYERS];
    float* bias[NGCF_MAX_LAYERS];
    int d_in[NGCF_MAX_LAYERS], d_out[NGCF_MAX_LAYERS];
};
// every layer of a step in one launch: blockIdx.y = layer
__global__ void pack_weights_all_kernel(PackAllArgs a) {
    const int l = blockIdx.y, d_in = a.d_in[l], d_out = a.d_out[l];
    const float* __restrict__ W1 = a.W1[l];
    const float* __restrict__ W2 = a.W2[l];
    const int total = 2 * d_in * d_out;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int k = i / d_out, o = i % d_out;
        a.wcat[l][i] = k < d_in ? W1[o * d_in + k] : W2[o * d_in + (k - d_in)];
    }
    for (int o = blockIdx.x * blockDim.x + threadIdx.x; o < d_out; o += gridDim.x * blockDim.x)
        a.bias[l][o] = 2.0f * a.b1[l][o] + a.b2[l][o];
}

// ------------------------------------------------------------------------------------------------
// forward epilogue
// ------------------------------------------------------------------------------------------------
constexpr int FWD_R = 64;          // rows per tile
constexpr int FWD_THREADS = 256;   // 16 (ty) x 16 (tx); thread = 4 rows x 4 cols per 64-column group

struct FwdArgs {
    const float* S;
    const float* E;
    int64_t n_rows;
    int d_in, d_out;
    const float* wcat;
    const float* bias_eff;
    float slope;
    const float* mess_mult;
    const uint32_t* mess_bits;
    float mess_p;
    uint64_t seed;
    const uint64_t* seed_dev;
    int layer;
    float* E_out;
    int KP;        // padded K = round_up(2*d_in, 4)
    int n_tiles;
    int64_t row_off;   // global index of local row 0 (RNG keys only)
};

template <int NCG>
__global__ void __launch_bounds__(FWD_THREADS) dense_fwd_kernel(FwdArgs a) {
    extern __shared__ __align__(16) float smem[];
    constexpr int NP = 64 * NCG;
    const int KP = a.KP, XLD = KP + 4;
    float* Ws = smem;                       // [KP][NP]
    float* Xs = Ws + (size_t)KP * NP;       // [FWD_R][XLD]
    float* Bs = Xs + (size_t)FWD_R * XLD;   // [NP]
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int d_in = a.d_in, d_out = a.d_out, K = 2 * d_in;
    const uint64_t seed = a.mess_p > 0.f ? ngcf_seed(a.seed, a.seed_dev) : 0ull;

    for (int i = tid; i < KP * NP; i += FWD_THREADS) {
        const int k = i / NP, o = i % NP;
        Ws[i] = (k < K && o < d_out) ? a.wcat[k * d_out + o] : 0.f;
    }
    for (int o = tid; o < NP; o += FWD_THREADS) Bs[o] = o < d_out ? a.bias_eff[o] : 0.f;

    const bool vec_in = (d_in % 4 == 0);
    const bool vec_out = (d_out % 4 == 0);
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const int64_t row0 = (int64_t)tile * FWD_R;
        __syncthreads();                    // previous tile's Xs fully consumed (and Ws visible on first pass)
        if (vec_in) {
            const int d4 = d_in / 4;
            for (int i = tid; i < FWD_R * d4; i += FWD_THREADS) {
                const int r = i / d4, c = (i % d4) * 4;
                const int64_t row = row0 + r;
                float4 s = make_float4(0.f, 0.f, 0.f, 0.f), e = s;
                if (row < a.n_rows) {
                    s = ld_f4(a.S + row * d_in + c);
                    e = ld_f4(a.E + row * d_in + c);
                }
                st_f4(Xs + r * XLD + c, make_float4(s.x + e.x, s.y + e.y, s.z + e.z, s.w + e.w));
                st_f4(Xs + r * XLD + d_in + c, make_float4(s.x * e.x, s.y * e.y, s.z * e.z, s.w * e.w));
            }
        } else {
            for (int i = tid; i < FWD_R * d_in; i += FWD_THREADS) {
                const int r = i / d_in, c = i % d_in;
                const int64_t row = row0 + r;
                float s = 0.f, e = 0.f;
                if (row < a.n_rows) {
                    s = a.S[row * d_in + c];
                    e = a.E[row * d_in + c];
                }
                Xs[r * XLD + c] = s + e;
                Xs[r * XLD + d_in + c] = s * e;
            }
        }
        if (KP > K) {
            for (int i = tid; i < FWD_R * (KP - K); i += FWD_THREADS) {
                const int r = i / (KP - K), c = K + i % (KP - K);
                Xs[r * XLD + c] = 0.f;
            }
        }
        __syncthreads();

        float acc[NCG][4][4];
#pragma unroll
        for (int g = 0; g < NCG; ++g)
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[g][r][c] = 0.f;

        for (int k = 0; k < KP; k += 4) {
            float4 av[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) av[r] = ld_f4(Xs + (ty * 4 + r) * XLD + k);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
                for (int g = 0; g < NCG; ++g) {
                    const float4 b = ld_f4(Ws + (k + kk) * NP + g * 64 + tx * 4);
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const float x = kk == 0 ? av[r].x : kk == 1 ? av[r].y : kk == 2 ? av[r].z : av[r].w;
                        acc[g][r][0] = fmaf(x, b.x, acc[g][r][0]);
                        acc[g][r][1] = fmaf(x, b.y, acc[g][r][1]);
                        acc[g][r][2] = fmaf(x, b.z, acc[g][r][2]);
                        acc[g][r][3] = fmaf(x, b.w, acc[g][r][3]);
                    }
                }
            }
        }

#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int64_t row = row0 + ty * 4 + r;
            if (row >= a.n_rows) continue;
#pragma unroll
            for (int g = 0; g < NCG; ++g) {
                const int c0 = g * 64 + tx * 4;
                if (c0 >= d_out) continue;
                float o[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    float m = acc[g][r][c] + Bs[c0 + c];
                    float v = m > 0.f ? m : a.slope * m;                 // LeakyReLU, NGCF.py:140
                    const int col = c0 + c;
                    if (col < d_out) {
                        if (a.mess_mult) v *= a.mess_mult[row * d_out + col];
                        else if (a.mess_bits) v *= mess_multiplier_bits(a.mess_bits, a.mess_p, row, d_out, col);
                        else if (a.mess_p > 0.f) v *= mess_multiplier(a.mess_p, seed, a.layer, (uint64_t)((row + a.row_off) * d_out + col));
                    }
                    o[c] = v;
                }
                if (vec_out) {
                    st_f4(a.E_out + row * d_out + c0, make_float4(o[0], o[1], o[2], o[3]));
                } else {
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        if (c0 + c < d_out) a.E_out[row * d_out + c0 + c] = o[c];
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// backward (row-local part)
// ------------------------------------------------------------------------------------------------
struct BwdArgs {
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
    float* gW1;
    float* gb1;
    float* gW2;
    float* gb2;
    int n_tiles;
    int64_t row_off;
    int gh_normalized;        // gsum already went through ngcf_rowgrad_normalize: add its slice as it is
};

template <int DC, int R, int THREADS>
__global__ void __launch_bounds__(THREADS) dense_bwd_kernel(BwdArgs a) {
    constexpr int TX = DC / 4;            // threads across columns (4 columns each)
    constexpr int TY = THREADS / TX;      // threads across rows
    constexpr int RPT = R / TY;           // rows per thread in the T phase
    constexpr int OB = (DC / 4) / TY;     // 4-row blocks of gW per thread in the weight-gradient phase
    constexpr int LD = DC + 4;
    constexpr int NW = THREADS / 32;
    constexpr int QN = DC / 32;
    static_assert(R % TY == 0 && (DC / 4) % TY == 0 && R % NW == 0, "tile shape");

    extern __shared__ __align__(16) float smem[];
    float* W1s = smem;                    // [DC][DC]  (k = o rows, j cols), zero padded
    float* W2s = W1s + DC * DC;
    float* GM = W2s + DC * DC;            // [R][LD]
    float* Ss = GM + R * LD;              // [R][LD]
    float* Es = Ss + R * LD;              // [R][LD]
    float* CS = Es + R * LD;              // [NW][DC] column sums of gM

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tx = tid % TX, ty = tid / TX;
    const int d_in = a.d_in, d_out = a.d_out;
    const uint64_t seed = a.mess_p > 0.f ? ngcf_seed(a.seed, a.seed_dev) : 0ull;

    for (int i = tid; i < DC * DC; i += THREADS) {
        const int o = i / DC, j = i % DC;
        const bool in = (o < d_out && j < d_in);
        W1s[i] = in ? a.W1[o * d_in + j] : 0.f;
        W2s[i] = in ? a.W2[o * d_in + j] : 0.f;
    }

    float accW1[OB][4][4], accW2[OB][4][4];
#pragma unroll
    for (int q = 0; q < OB; ++q)
#pragma unroll
        for (int o = 0; o < 4; ++o)
#pragma unroll
            for (int j = 0; j < 4; ++j) accW1[q][o][j] = accW2[q][o][j] = 0.f;
    float colsum[QN];
#pragma unroll
    for (int q = 0; q < QN; ++q) colsum[q] = 0.f;

    const bool vec_in = (d_in % 4 == 0);
    const int KO = (d_out + 3) & ~3;      // padded reduction length of the T phase

    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const int64_t row0 = (int64_t)tile * R;
        __syncthreads();
        // ---- phase A: gM rows (one warp per row), S/E tiles ------------------------------------------
        for (int r = warp; r < R; r += NW) {
            const int64_t row = row0 + r;
            float e[QN], gm[QN];
            float nrm2 = 0.f;
#pragma unroll
            for (int q = 0; q < QN; ++q) {
                const int c = lane + 32 * q;
                e[q] = (row < a.n_rows && c < d_out) ? a.E_out[row * d_out + c] : 0.f;
                nrm2 = fmaf(e[q], e[q], nrm2);
            }
            nrm2 = warp_sum(nrm2);
            const float n = fmaxf(sqrtf(nrm2), 1e-12f);                  // F.normalize eps, NGCF.py:144
            const int s = (row < a.n_rows && a.slot) ? a.slot[row] : -1;
            float gh[QN];
            float dot = 0.f;
#pragma unroll
            for (int q = 0; q < QN; ++q) {
                const int c = lane + 32 * q;
                gh[q] = (s >= 0 && c < d_out) ? a.gsum[(int64_t)s * a.ld_gsum + a.col_off + c] : 0.f;
                dot = fmaf(e[q], gh[q], dot);
            }
            if (s >= 0) dot = warp_sum(dot) / n;                         // H . gH
#pragma unroll
            for (int q = 0; q < QN; ++q) {
                const int c = lane + 32 * q;
                float g = 0.f;
                if (row < a.n_rows && c < d_out) {
                    g = a.gE_next ? a.gE_next[row * d_out + c] : 0.f;
                    if (s >= 0) g += a.gh_normalized ? gh[q] : (gh[q] - (e[q] / n) * dot) / n;   // normalize backward
                    float mult = 1.f;
                    if (a.mess_mult) mult = a.mess_mult[row * d_out + c];
                    else if (a.mess_bits) mult = mess_multiplier_bits(a.mess_bits, a.mess_p, row, d_out, c);
                    else if (a.mess_p > 0.f) mult = mess_multiplier(a.mess_p, seed, a.layer, (uint64_t)((row + a.row_off) * d_out + c));
                    g *= mult * (e[q] > 0.f ? 1.f : a.slope);            // dropout + LeakyReLU backward
                }
                gm[q] = g;
                colsum[q] += g;
                if (c < DC) GM[r * LD + c] = g;
            }
        }
        if (vec_in) {
            const int d4 = d_in / 4;
            for (int i = tid; i < R * (DC / 4); i += THREADS) {
                const int r = i / (DC / 4), c4 = i % (DC / 4);
                const int64_t row = row0 + r;
                float4 s = make_float4(0.f, 0.f, 0.f, 0.f), e = s;
                if (row < a.n_rows && c4 < d4) {
                    s = ld_f4(a.S + row * d_in + c4 * 4);
                    e = ld_f4(a.E + row * d_in + c4 * 4);
                }
                st_f4(Ss + r * LD + c4 * 4, s);
                st_f4(Es + r * LD + c4 * 4, e);
            }
        } else {
            for (int i = tid; i < R * DC; i += THREADS) {
                const int r = i / DC, c = i % DC;
                const int64_t row = row0 + r;
                const bool in = (row < a.n_rows && c < d_in);
                Ss[r * LD + c] = in ? a.S[row * d_in + c] : 0.f;
                Es[r * LD + c] = in ? a.E[row * d_in + c] : 0.f;
            }
        }
        __syncthreads();

        // ---- phase B: T1 = gM·W1, T2 = gM·W2; gS = T1 + T2*E, gEl = T1 + T2*S ---------------------------
        {
            float t1[RPT][4], t2[RPT][4];
#pragma unroll
            for (int r = 0; r < RPT; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) t1[r][c] = t2[r][c] = 0.f;
            for (int k = 0; k < KO; k += 4) {
                float4 av[RPT];
#pragma unroll
                for (int r = 0; r < RPT; ++r) av[r] = ld_f4(GM + (ty * RPT + r) * LD + k);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const float4 b1 = ld_f4(W1s + (k + kk) * DC + tx * 4);
                    const float4 b2 = ld_f4(W2s + (k + kk) * DC + tx * 4);
#pragma unroll
                    for (int r = 0; r < RPT; ++r) {
                        const float x = kk == 0 ? av[r].x : kk == 1 ? av[r].y : kk == 2 ? av[r].z : av[r].w;
                        t1[r][0] = fmaf(x, b1.x, t1[r][0]); t1[r][1] = fmaf(x, b1.y, t1[r][1]);
                        t1[r][2] = fmaf(x, b1.z, t1[r][2]); t1[r][3] = fmaf(x, b1.w, t1[r][3]);
                        t2[r][0] = fmaf(x, b2.x, t2[r][0]); t2[r][1] = fmaf(x, b2.y, t2[r][1]);
                        t2[r][2] = fmaf(x, b2.z, t2[r][2]); t2[r][3] = fmaf(x, b2.w, t2[r][3]);
                    }
                }
            }
            const int j0 = tx * 4;
#pragma unroll
            for (int r = 0; r < RPT; ++r) {
                const int rr = ty * RPT + r;
                const int64_t row = row0 + rr;
                if (row >= a.n_rows || j0 >= d_in) continue;
                const float4 e4 = ld_f4(Es + rr * LD + j0), s4 = ld_f4(Ss + rr * LD + j0);
                float gs[4] = {fmaf(t2[r][0], e4.x, t1[r][0]), fmaf(t2[r][1], e4.y, t1[r][1]),
                               fmaf(t2[r][2], e4.z, t1[r][2]), fmaf(t2[r][3], e4.w, t1[r][3])};
                float ge[4] = {fmaf(t2[r][0], s4.x, t1[r][0]), fmaf(t2[r][1], s4.y, t1[r][1]),
                               fmaf(t2[r][2], s4.z, t1[r][2]), fmaf(t2[r][3], s4.w, t1[r][3])};
                if (vec_in) {
                    st_f4(a.gS + row * d_in + j0, make_float4(gs[0], gs[1], gs[2], gs[3]));
                    st_f4(a.gEl + row * d_in + j0, make_float4(ge[0], ge[1], ge[2], ge[3]));
                } else {
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        if (j0 + c < d_in) {
                            a.gS[row * d_in + j0 + c] = gs[c];
                            a.gEl[row * d_in + j0 + c] = ge[c];
                        }
                }
            }
        }

        // ---- phase C: gW1 += gM^T (S+E), gW2 += gM^T (S*E), accumulated in registers across tiles ----
        for (int r = 0; r < R; ++r) {
            const float4 s4 = ld_f4(Ss + r * LD + tx * 4), e4 = ld_f4(Es + r * LD + tx * 4);
            const float x1[4] = {s4.x + e4.x, s4.y + e4.y, s4.z + e4.z, s4.w + e4.w};
            const float x2[4] = {s4.x * e4.x, s4.y * e4.y, s4.z * e4.z, s4.w * e4.w};
#pragma unroll
            for (int q = 0; q < OB; ++q) {
                const float4 g4 = ld_f4(GM + r * LD + (ty + TY * q) * 4);
                const float g[4] = {g4.x, g4.y, g4.z, g4.w};
#pragma unroll
                for (int o = 0; o < 4; ++o)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        accW1[q][o][j] = fmaf(g[o], x1[j], accW1[q][o][j]);
                        accW2[q][o][j] = fmaf(g[o], x2[j], accW2[q][o][j]);
                    }
            }
        }
    }

    // ---- flush weight / bias gradients --------------------------------------------------------------
#pragma unroll
    for (int q = 0; q < OB; ++q)
#pragma unroll
        for (int o = 0; o < 4; ++o) {
            const int oo = (ty + TY * q) * 4 + o;
            if (oo >= d_out) continue;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int jj = tx * 4 + j;
                if (jj < d_in) {
                    atomicAdd(a.gW1 + oo * d_in + jj, accW1[q][o][j]);
                    atomicAdd(a.gW2 + oo * d_in + jj, accW2[q][o][j]);
                }
            }
        }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < QN; ++q) CS[warp * DC + lane + 32 * q] = colsum[q];
    __syncthreads();
    for (int c = tid; c < d_out; c += THREADS) {
        float s = 0.f;
        for (int w = 0; w < NW; ++w) s += CS[w * DC + c];
        atomicAdd(a.gb2 + c, s);
        atomicAdd(a.gb1 + c, 2.0f * s);          // w1_list[i] is applied twice (NGCF.py:131,133)
    }
}

template <typename K>
int set_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) {
            ngcf_set_error("cudaFuncSetAttribute(%zu bytes smem) failed: %s", bytes, cudaGetErrorString(e));
            return NGCF_ERR_CUDA;
        }
    }
    return NGCF_OK;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

// dense_tc.cu: tcgen05 / TMEM versions (3xTF32) of the dense parts, used whenever the widths allow
bool ngcf_dense_fwd_tc_eligible(int d_in, int d_out);
int ngcf_dense_fwd_tc(const float* S, const float* E, int64_t n_rows, int d_in, int d_out, const float* wcat,
                      const float* bias_eff, float slope, const float* mess_mult, const uint32_t* mess_bits, float mess_p,
                      uint64_t seed,
                      const uint64_t* seed_dev, int layer, int64_t row_offset, float* E_out, cudaStream_t st);

bool ngcf_dense_bwd_tc_eligible(int d_in, int d_out, int gh_normalized);
int ngcf_dense_bwd_tc(const float* gE_next, const int32_t* slot, const float* gsum, int64_t ld_gsum, int col_off,
                      const float* E_out, const float* S, const float* E, int64_t n_rows, int d_in, int d_out,
                      const float* W1, const float* W2, float slope, const float* mess_mult, const uint32_t* mess_bits,
                      float mess_p,
                      uint64_t seed, const uint64_t* seed_dev, int layer, int64_t row_offset, int gh_normalized, float* gS, float* gEl,
                      float* gW1, float* gb1, float* gW2, float* gb2, float* gM_scratch, cudaStream_t st);

extern "C" int ngcf_pack_weights(const float* W1, const float* b1, const float* W2, const float* b2, int d_in,
                                 int d_out, float* wcat, float* bias_eff, void* stream) {
    NGCF_REQUIRE(W1 && b1 && W2 && b2 && wcat && bias_eff, "pack_weights: null pointer");
    NGCF_REQUIRE(d_in > 0 && d_in <= NGCF_MAX_WIDTH && d_out > 0 && d_out <= NGCF_MAX_WIDTH,
                 "pack_weights: widths %d -> %d not in [1,%d]", d_in, d_out, NGCF_MAX_WIDTH);
    pack_weights_kernel<<<32, 256, 0, as_stream(stream)>>>(W1, b1, W2, b2, d_in, d_out, wcat, bias_eff);
    NGCF_LAUNCH_OK("pack_weights_kernel");
    return NGCF_OK;
}

extern "C" int ngcf_pack_weights_all(const float* const* W1_host, const float* const* b1_host, const float* const* W2_host,
                                     const float* const* b2_host, const int* d_in_host, const int* d_out_host, int n_layers,
                                     float* const* wcat_host, float* const* bias_host, void* stream) {
    NGCF_REQUIRE(W1_host && b1_host && W2_host && b2_host && d_in_host && d_out_host && wcat_host && bias_host,
                 "pack_weights_all: null pointer");
    NGCF_REQUIRE(n_layers >= 1 && n_layers <= NGCF_MAX_LAYERS, "pack_weights_all: %d layers", n_layers);
    PackAllArgs a{};
    for (int l = 0; l < n_layers; ++l) {
        NGCF_REQUIRE(W1_host[l] && b1_host[l] && W2_host[l] && b2_host[l] && wcat_host[l] && bias_host[l],
                     "pack_weights_all: null pointer (layer %d)", l);
        NGCF_REQUIRE(d_in_host[l] > 0 && d_in_host[l] <= NGCF_MAX_WIDTH && d_out_host[l] > 0 && d_out_host[l] <= NGCF_MAX_WIDTH,
                     "pack_weights_all: widths %d -> %d not in [1,%d]", d_in_host[l], d_out_host[l], NGCF_MAX_WIDTH);
        a.W1[l] = W1_host[l]; a.b1[l] = b1_host[l]; a.W2[l] = W2_host[l]; a.b2[l] = b2_host[l];
        a.wcat[l] = wcat_host[l]; a.bias[l] = bias_host[l]; a.d_in[l] = d_in_host[l]; a.d_out[l] = d_out_host[l];
    }
    pack_weights_all_kernel<<<dim3(32, (unsigned)n_layers), 256, 0, as_stream(stream)>>>(a);
    NGCF_LAUNCH_OK("pack_weights_all_kernel");
    return NGCF_OK;
}

extern "C" int ngcf_dense_fwd(const float* S, const float* E, int64_t n_rows, int d_in, int d_out, const float* wcat,
                              const float* bias_eff, float slope, const float* mess_mult, const uint32_t* mess_bits, float mess_p,
                      uint64_t seed,
                              const uint64_t* seed_dev, int layer, int64_t row_offset, float* E_out, void* stream) {
    NGCF_REQUIRE(S && E && wcat && bias_eff && E_out, "dense_fwd: null pointer");
    NGCF_REQUIRE(d_in > 0 && d_in <= NGCF_MAX_WIDTH && d_out > 0 && d_out <= NGCF_MAX_WIDTH,
                 "dense_fwd: widths %d -> %d not in [1,%d]", d_in, d_out, NGCF_MAX_WIDTH);
    NGCF_REQUIRE(mess_p >= 0.f && mess_p < 1.f, "dense_fwd: mess_p %f not in [0,1)", mess_p);
    NGCF_REQUIRE(n_rows >= 0 && n_rows < ((int64_t)1 << 31), "dense_fwd: n_rows %lld", (long long)n_rows);
    if (n_rows == 0) return NGCF_OK;
    if (ngcf_dense_fwd_tc_eligible(d_in, d_out) && aligned16(S) && aligned16(E) &&
        aligned16(E_out) && (!mess_mult || aligned16(mess_mult)))
        return ngcf_dense_fwd_tc(S, E, n_rows, d_in, d_out, wcat, bias_eff, slope, mess_mult, mess_bits, mess_p, seed, seed_dev,
                                 layer, row_offset, E_out, as_stream(stream));
    FwdArgs a{S, E, n_rows, d_in, d_out, wcat, bias_eff, slope, mess_mult, mess_bits, mess_p, seed, seed_dev, layer, E_out,
              (2 * d_in + 3) & ~3, (int)ceil_div64(n_rows, FWD_R), row_offset};
    const int ncg = d_out <= 64 ? 1 : 2;
    const size_t smem = sizeof(float) * ((size_t)a.KP * 64 * ncg + (size_t)FWD_R * (a.KP + 4) + 64 * ncg);
    const int per_sm = smem > 110 * 1024 ? 1 : (smem > 72 * 1024 ? 2 : 3);
    const int grid = (int)min((int64_t)a.n_tiles, (int64_t)ngcf_num_sms() * per_sm);
    int rc;
    if (ncg == 1) {
        if ((rc = set_smem(dense_fwd_kernel<1>, smem)) != NGCF_OK) return rc;
        dense_fwd_kernel<1><<<grid, FWD_THREADS, smem, as_stream(stream)>>>(a);
    } else {
        if ((rc = set_smem(dense_fwd_kernel<2>, smem)) != NGCF_OK) return rc;
        dense_fwd_kernel<2><<<grid, FWD_THREADS, smem, as_stream(stream)>>>(a);
    }
    NGCF_LAUNCH_OK("dense_fwd_kernel");
    return NGCF_OK;
}

extern "C" int ngcf_dense_bwd(const float* gE_next, const int32_t* slot, const float* gsum, int64_t ld_gsum,
                              int col_off, const float* E_out, const float* S, const float* E, int64_t n_rows,
                              int d_in, int d_out, const float* W1, const float* W2, float slope,
                              const float* mess_mult, const uint32_t* mess_bits, float mess_p, uint64_t seed,
                              const uint64_t* seed_dev, int layer, int64_t row_offset, int gh_normalized, float* gS,
                              float* gEl, float* gW1, float* gb1, float* gW2, float* gb2, float* gM_scratch, void* stream) {
    NGCF_REQUIRE(E_out && S && E && W1 && W2 && gS && gEl && gW1 && gb1 && gW2 && gb2, "dense_bwd: null pointer");
    NGCF_REQUIRE(!slot || gsum, "dense_bwd: slot given without gsum");
    NGCF_REQUIRE(d_in > 0 && d_in <= NGCF_MAX_WIDTH && d_out > 0 && d_out <= NGCF_MAX_WIDTH,
                 "dense_bwd: widths %d -> %d not in [1,%d]", d_in, d_out, NGCF_MAX_WIDTH);
    NGCF_REQUIRE(mess_p >= 0.f && mess_p < 1.f, "dense_bwd: mess_p %f not in [0,1)", mess_p);
    NGCF_REQUIRE(n_rows >= 0 && n_rows < ((int64_t)1 << 31), "dense_bwd: n_rows %lld", (long long)n_rows);
    if (n_rows == 0) return NGCF_OK;
    if (gM_scratch && ngcf_dense_bwd_tc_eligible(d_in, d_out, gh_normalized) && aligned16(S) &&
        aligned16(E) && aligned16(gS) && aligned16(gEl) && aligned16(gM_scratch))
        return ngcf_dense_bwd_tc(gE_next, slot, gsum, ld_gsum, col_off, E_out, S, E, n_rows, d_in, d_out, W1, W2,
                                 slope, mess_mult, mess_bits, mess_p, seed, seed_dev, layer, row_offset, gh_normalized, gS,
                                 gEl, gW1, gb1, gW2, gb2, gM_scratch, as_stream(stream));
    BwdArgs a{gE_next, slot, gsum, ld_gsum, col_off, E_out, S, E, n_rows, d_in, d_out, W1, W2, slope, mess_mult,
              mess_bits, mess_p, seed, seed_dev, layer, gS, gEl, gW1, gb1, gW2, gb2, 0, row_offset, gh_normalized};
    int rc;
    if (d_in <= 64 && d_out <= 64) {
        constexpr int DC = 64, R = 64, T = 256;
        a.n_tiles = (int)ceil_div64(n_rows, R);
        const size_t smem = sizeof(float) * (2 * DC * DC + 3 * R * (DC + 4) + (T / 32) * DC);
        const int grid = (int)min((int64_t)a.n_tiles, (int64_t)ngcf_num_sms() * 2);
        if ((rc = set_smem(dense_bwd_kernel<DC, R, T>, smem)) != NGCF_OK) return rc;
        dense_bwd_kernel<DC, R, T><<<grid, T, smem, as_stream(stream)>>>(a);
    } else {
        constexpr int DC = 128, R = 32, T = 512;
        a.n_tiles = (int)ceil_div64(n_rows, R);
        const size_t smem = sizeof(float) * (2 * DC * DC + 3 * R * (DC + 4) + (T / 32) * DC);
        const int grid = (int)min((int64_t)a.n_tiles, (int64_t)ngcf_num_sms());
        if ((rc = set_smem(dense_bwd_kernel<DC, R, T>, smem)) != NGCF_OK) return rc;
        dense_bwd_kernel<DC, R, T><<<grid, T, smem, as_stream(stream)>>>(a);
    }
    NGCF_LAUNCH_OK("dense_bwd_kernel");
    return NGCF_OK;
}

// ------------------------------------------------------------------------------------------------
// message-dropout decisions for a whole layer, one 32-column word per thread
// ------------------------------------------------------------------------------------------------
namespace {
__global__ void mess_bits_kernel(int64_t n_rows, int d_out, int words, float p, uint64_t seed0, const uint64_t* seed_dev,
                                 int layer, int64_t row_off, uint32_t* __restrict__ bits) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_rows * words) return;
    const int64_t row = i / words;
    const int w = (int)(i % words);
    const uint64_t seed = ngcf_seed(seed0, seed_dev);
    uint32_t out = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int col = w * 32 + q * 4;
        if (col < d_out) {
            const float4 m = mess_multiplier4(p, seed, layer, (uint64_t)((row + row_off) * d_out + col) >> 2);
            out |= (m.x != 0.f ? 1u : 0u) << (q * 4) | (m.y != 0.f ? 2u : 0u) << (q * 4) | (m.z != 0.f ? 4u : 0u) << (q * 4) |
                   (m.w != 0.f ? 8u : 0u) << (q * 4);
        }
    }
    bits[i] = out;
}
}  // namespace

extern "C" int ngcf_mess_dropout_bits(int64_t n_rows, int d_out, float mess_p, uint64_t seed, const uint64_t* seed_dev,
                                      int layer, int64_t row_offset, uint32_t* bits, void* stream) {
    NGCF_REQUIRE(bits && n_rows >= 0, "mess_dropout_bits: null pointer");
    NGCF_REQUIRE(d_out > 0 && d_out <= NGCF_MAX_WIDTH && d_out % 4 == 0, "mess_dropout_bits: width %d", d_out);
    NGCF_REQUIRE(mess_p > 0.f && mess_p < 1.f, "mess_dropout_bits: mess_p %f not in (0,1)", mess_p);
    if (n_rows == 0) return NGCF_OK;
    const int words = (d_out + 31) / 32;
    mess_bits_kernel<<<(unsigned)ceil_div64(n_rows * words, 256), 256, 0, as_stream(stream)>>>(
        n_rows, d_out, words, mess_p, seed, seed_dev, layer, row_offset, bits);
    NGCF_LAUNCH_OK("mess_bits_kernel");
    return NGCF_OK;
}
