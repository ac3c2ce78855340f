// LightGCN's two kernels of its own (the propagation itself is ngcf_spmm):
//   * the layer-mean readout (1/(K+1)) sum_k E_k[row] for the batch's row sets or for every row, the mean-readout
//     counterpart of ngcf_gather_concat(_sets);
//   * the dense last-layer gradient s * gsum[slot[i]] from the row-gradient slot map, which also scales gsum in place
//     so that the transposed products' slot/gsum addend adds the same scaled rows.
#include "common.cuh"

namespace {

constexpr int LM_Q = NGCF_MAX_WIDTH / 32;               // columns per lane

struct MeanArgs {
    const float* layer[NGCF_MAX_LAYERS + 1];
    int n;               // number of layers summed (K+1)
    int d;
    float inv_n;         // 1 / n
    const int64_t* rows[4];
    int64_t row_offset[4];
    int64_t base[5];     // first global output index of set j; base[n_sets] = total
    float* out[4];
    int n_sets;
    int64_t ld_out;
};

// one warp per output row: E_0 + E_1 + ... + E_K in that order, then times 1/(K+1); every load of the row is issued
// before the first add (LM_Q columns per lane and layer)
__device__ __forceinline__ void mean_row(const MeanArgs& a, int64_t r, float* o, int lane) {
    float acc[LM_Q] = {};
#pragma unroll
    for (int k = 0; k <= NGCF_MAX_LAYERS; ++k) {
        if (k < a.n) {
            const float* src = a.layer[k] + r * (int64_t)a.d;
#pragma unroll
            for (int q = 0; q < LM_Q; ++q) {
                const int c = lane + 32 * q;
                if (c < a.d) acc[q] += src[c];
            }
        }
    }
#pragma unroll
    for (int q = 0; q < LM_Q; ++q) {
        const int c = lane + 32 * q;
        if (c < a.d) o[c] = acc[q] * a.inv_n;
    }
}

__global__ void __launch_bounds__(256) layer_mean_sets_kernel(MeanArgs a) {
    const int64_t b = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (b >= a.base[a.n_sets]) return;
    int j = 0;
    while (b >= a.base[j + 1]) ++j;
    const int64_t i = b - a.base[j];
    mean_row(a, (a.rows[j] ? a.rows[j][i] : i) + a.row_offset[j], a.out[j] + i * a.ld_out, lane);
}

// out[i, :] = slot[i] >= 0 ? s * gsum[slot[i], :] : 0, and gsum[slot[i], :] *= s.  A slot belongs to one row only
// (ngcf_rowgrad_scatter), so each gsum element is read and rewritten by the one thread that owns it.
template <bool VEC4>
__global__ void __launch_bounds__(256) rowgrad_expand_kernel(const int32_t* __restrict__ slot, int64_t n_rows,
                                                             float* __restrict__ gsum, int64_t ld_gsum, int d,
                                                             float s, float* __restrict__ out, int64_t ld_out) {
    const int w = VEC4 ? d >> 2 : d;                     // work items per row
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= n_rows * w) return;
    const int64_t i = e / w;
    const int c = (int)(e - i * w);
    const int32_t sl = slot[i];
    if (VEC4) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (sl >= 0) {
            float* g = gsum + sl * ld_gsum + 4 * c;
            v = ld_f4(g);
            v.x *= s; v.y *= s; v.z *= s; v.w *= s;
            st_f4(g, v);
        }
        st_f4(out + i * ld_out + 4 * c, v);
    } else {
        float v = 0.f;
        if (sl >= 0) {
            float* g = gsum + sl * ld_gsum + c;
            v = *g * s;
            *g = v;
        }
        out[i * ld_out + c] = v;
    }
}

int fill_mean(MeanArgs& a, const float* const* layers_host, int n_layers_plus1, int d, int64_t ld_out,
              const char* what) {
    NGCF_REQUIRE(layers_host, "%s: null layer array", what);
    NGCF_REQUIRE(n_layers_plus1 >= 1 && n_layers_plus1 <= NGCF_MAX_LAYERS + 1, "%s: %d layers", what, n_layers_plus1);
    NGCF_REQUIRE(d >= 1 && d <= NGCF_MAX_WIDTH, "%s: width %d not in [1, %d]", what, d, NGCF_MAX_WIDTH);
    NGCF_REQUIRE(ld_out >= d, "%s: ld_out %lld < width %d", what, (long long)ld_out, d);
    for (int k = 0; k < n_layers_plus1; ++k) {
        NGCF_REQUIRE(layers_host[k], "%s: null layer %d", what, k);
        a.layer[k] = layers_host[k];
    }
    a.n = n_layers_plus1;
    a.d = d;
    a.inv_n = 1.0f / (float)n_layers_plus1;
    a.ld_out = ld_out;
    return NGCF_OK;
}

int launch_mean(const MeanArgs& a, void* stream) {
    const int64_t total = a.base[a.n_sets];
    if (total == 0) return NGCF_OK;
    layer_mean_sets_kernel<<<(unsigned)ceil_div64(total * 32, 256), 256, 0, as_stream(stream)>>>(a);
    NGCF_LAUNCH_OK("layer_mean_sets_kernel");
    return NGCF_OK;
}

}  // namespace

extern "C" int ngcf_layer_mean(const float* const* layers_host, int n_layers_plus1, int d, const int64_t* rows,
                               int64_t row_offset, int64_t n_out, float* out, int64_t ld_out, void* stream) {
    MeanArgs a{};
    const int rc = fill_mean(a, layers_host, n_layers_plus1, d, ld_out, "layer_mean");
    if (rc != NGCF_OK) return rc;
    NGCF_REQUIRE(n_out >= 0, "layer_mean: n_out %lld", (long long)n_out);
    NGCF_REQUIRE(n_out == 0 || out, "layer_mean: null output");
    a.rows[0] = rows; a.row_offset[0] = row_offset; a.out[0] = out; a.n_sets = 1;
    for (int j = 1; j <= 4; ++j) a.base[j] = n_out;
    return launch_mean(a, stream);
}

extern "C" int ngcf_layer_mean_sets(const float* const* layers_host, int n_layers_plus1, int d,
                                    const int64_t* const* rows_host, const int64_t* offsets_host,
                                    const int64_t* sizes_host, float* const* outs_host, int n_sets, int64_t ld_out,
                                    void* stream) {
    MeanArgs a{};
    const int rc = fill_mean(a, layers_host, n_layers_plus1, d, ld_out, "layer_mean_sets");
    if (rc != NGCF_OK) return rc;
    NGCF_REQUIRE(rows_host && offsets_host && sizes_host && outs_host, "layer_mean_sets: null host array");
    NGCF_REQUIRE(n_sets >= 1 && n_sets <= 4, "layer_mean_sets: n_sets %d not in [1,4]", n_sets);
    int64_t total = 0;
    for (int j = 0; j < n_sets; ++j) {
        NGCF_REQUIRE(sizes_host[j] >= 0 && (sizes_host[j] == 0 || (rows_host[j] && outs_host[j])),
                     "layer_mean_sets: set %d", j);
        a.rows[j] = rows_host[j]; a.row_offset[j] = offsets_host[j]; a.out[j] = outs_host[j];
        a.base[j] = total;
        total += sizes_host[j];
    }
    for (int j = n_sets; j <= 4; ++j) a.base[j] = total;
    a.n_sets = n_sets;
    return launch_mean(a, stream);
}

extern "C" int ngcf_rowgrad_expand(const int32_t* slot, int64_t n_rows, float* gsum, int64_t ld_gsum, int d,
                                   float scale, float* out, int64_t ld_out, void* stream) {
    NGCF_REQUIRE(slot && gsum && out, "rowgrad_expand: null pointer");
    NGCF_REQUIRE(n_rows >= 0 && n_rows < ((int64_t)1 << 31), "rowgrad_expand: n_rows %lld", (long long)n_rows);
    NGCF_REQUIRE(d >= 1 && d <= NGCF_MAX_WIDTH, "rowgrad_expand: width %d not in [1, %d]", d, NGCF_MAX_WIDTH);
    NGCF_REQUIRE(ld_gsum >= d && ld_out >= d, "rowgrad_expand: row pitches %lld / %lld < width %d",
                 (long long)ld_gsum, (long long)ld_out, d);
    if (n_rows == 0) return NGCF_OK;
    const bool vec4 = d % 4 == 0 && ld_gsum % 4 == 0 && ld_out % 4 == 0 &&
                      (((uintptr_t)gsum | (uintptr_t)out) % 16 == 0);
    const int64_t work = n_rows * (vec4 ? d / 4 : d);
    const unsigned grid = (unsigned)ceil_div64(work, 256);
    if (vec4)
        rowgrad_expand_kernel<true><<<grid, 256, 0, as_stream(stream)>>>(slot, n_rows, gsum, ld_gsum, d, scale, out,
                                                                         ld_out);
    else
        rowgrad_expand_kernel<false><<<grid, 256, 0, as_stream(stream)>>>(slot, n_rows, gsum, ld_gsum, d, scale, out,
                                                                          ld_out);
    NGCF_LAUNCH_OK("rowgrad_expand_kernel");
    return NGCF_OK;
}
