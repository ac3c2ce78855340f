// XSimGCL's kernels of its own (the propagation is ngcf_spmm, the readouts ngcf_layer_mean(_sets)):
//   * the layer noise E += eps * sign(E) * normalize(U), U uniform on [0, 1) from the device RNG, one warp per row;
//   * the cosine InfoNCE over the distinct ids of a batch: first-occurrence flags and the row normalization in front of
//     the softmax loss's launches (softmax_core.cuh), the normalize backward behind them;
//   * the scatter of extra row gradients onto an existing slot map (or a dense matrix), for the view-2 rows.
#include <math.h>

#include "softmax_core.cuh"

namespace {

constexpr int PR_Q = NGCF_MAX_WIDTH / 32;               // columns per lane
constexpr int IN_MAX_B = 4096;                          // the softmax loss's limits
constexpr int IN_MAX_D = 1152;

// one warp per row r: u_c = (hash64(key, r, c, layer, 'NOIS').x >> 8) * 2^-24, then E[r, c] += sign(E[r, c]) * u_c *
// (eps / max(|u|, 1e-12)), sign(0) = 0
__global__ void __launch_bounds__(256) perturb_rows_kernel(float* __restrict__ E, int64_t N, int d, int64_t ld, float eps,
                                                           uint64_t seed, const uint64_t* __restrict__ seed_dev,
                                                           int layer) {
    const int64_t r = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= N) return;                                                   // whole warps
    const uint64_t key = ngcf_seed(seed, seed_dev);
    float u[PR_Q], ss = 0.f;
#pragma unroll
    for (int q = 0; q < PR_Q; ++q) {
        const int c = lane + 32 * q;
        u[q] = 0.f;
        if (c < d) {
            const uint2 h = ngcf_hash64(key, (uint32_t)r, (uint32_t)c, (uint32_t)layer, NGCF_STREAM_NOISE);
            u[q] = (float)(h.x >> 8) * 0x1p-24f;
            ss = fmaf(u[q], u[q], ss);
        }
    }
    ss = warp_sum(ss);
    const float s = eps / fmaxf(sqrtf(ss), 1e-12f);
    float* row = E + r * ld;
#pragma unroll
    for (int q = 0; q < PR_Q; ++q) {
        const int c = lane + 32 * q;
        if (c < d) {
            const float v = row[c];
            const float sg = v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f);
            row[c] = fmaf(sg, u[q] * s, v);
        }
    }
}

// one warp per row i of the batch: valid[i] = ids[i] occurs in no earlier row (fixed shape, no scratch: the same flags
// every time), and the normalized rows z = x / max(|x|, 1e-12) of both views with their norms
__global__ void __launch_bounds__(256) infonce_prep_kernel(const float* __restrict__ x1, const float* __restrict__ x2,
                                                           int64_t B, int D, const int64_t* __restrict__ ids,
                                                           uint8_t* __restrict__ valid, float* __restrict__ z1,
                                                           float* __restrict__ z2, float* __restrict__ nrm) {
    const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= B) return;
    const int64_t id = ids[i];
    bool dup = false;
    for (int64_t j0 = 0; j0 < i && !dup; j0 += 32) {
        const int64_t j = j0 + lane;
        dup = __any_sync(FULL_MASK, j < i && ids[j] == id);
    }
    if (lane == 0) valid[i] = dup ? 0 : 1;
#pragma unroll
    for (int v = 0; v < 2; ++v) {
        const float* x = (v ? x2 : x1) + i * D;
        float* z = (v ? z2 : z1) + i * D;
        float ss = 0.f;
        for (int c = lane; c < D; c += 32) ss = fmaf(x[c], x[c], ss);
        const float n = fmaxf(sqrtf(warp_sum(ss)), 1e-12f);
        for (int c = lane; c < D; c += 32) z[c] = x[c] / n;
        if (lane == 0) nrm[v * B + i] = n;
    }
}

// one warp per row of [g1; g2] (2B rows), in place: g <- (g' - z (z . g')) / n with g' = g / U (the gradient of
// z = x / n with respect to x; the softmax loss's G was left unscaled by 1 / U)
__global__ void __launch_bounds__(256) infonce_finish_kernel(float* __restrict__ g1, float* __restrict__ g2,
                                                             const float* __restrict__ z1, const float* __restrict__ z2,
                                                             const float* __restrict__ nrm,
                                                             const float* __restrict__ inv_count, int64_t B, int D) {
    const int64_t w = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= 2 * B) return;
    const bool second = w >= B;
    const int64_t i = second ? w - B : w;
    float* g = (second ? g2 : g1) + i * D;
    const float* z = (second ? z2 : z1) + i * D;
    const float s = *inv_count, n = nrm[w];
    float dot = 0.f;
    for (int c = lane; c < D; c += 32) dot = fmaf(z[c], g[c] * s, dot);
    dot = warp_sum(dot);
    for (int c = lane; c < D; c += 32) g[c] = (g[c] * s - z[c] * dot) / n;
}

struct AddSets {
    const int64_t* rows[2];
    int64_t offset[2];
    const float* g[2];
    int64_t base[3];     // first global row index of set j; base[n_sets] = total
};

// one warp per gradient row: dst[slot[r] or r] += g row (atomic: several rows may share a destination)
__global__ void __launch_bounds__(256) rowgrad_add_kernel(AddSets s, int d, const int32_t* __restrict__ slot,
                                                          float* __restrict__ dst, int64_t ld_dst) {
    const int64_t b = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (b >= s.base[2]) return;
    const bool second = b >= s.base[1];                                  // (selects: no local copy of the sets)
    const int64_t i = b - (second ? s.base[1] : 0);
    const int64_t r = (second ? s.rows[1] : s.rows[0])[i] + (second ? s.offset[1] : s.offset[0]);
    const int64_t t = slot ? (int64_t)slot[r] : r;
    const float* g = (second ? s.g[1] : s.g[0]) + i * d;
    float* o = dst + t * ld_dst;
    for (int c = lane; c < d; c += 32) atomicAdd(o + c, g[c]);
}

struct InfoLayout {
    size_t z1, z2, nrm, valid, inv, loss_ws, total;
};

inline size_t al1k(size_t x) { return (x + 1023) & ~(size_t)1023; }

InfoLayout info_layout(int64_t B, int D) {
    InfoLayout L;
    size_t o = 0;
    L.z1 = o;      o = al1k(o + (size_t)B * D * sizeof(float));
    L.z2 = o;      o = al1k(o + (size_t)B * D * sizeof(float));
    L.nrm = o;     o = al1k(o + (size_t)2 * B * sizeof(float));
    L.valid = o;   o = al1k(o + (size_t)B);
    L.inv = o;     o = al1k(o + sizeof(float));
    L.loss_ws = o; o += softmax_run_bytes(B, false, D);
    L.total = o + 1024;                                                   // slack to align the caller's base
    return L;
}

}  // namespace

extern "C" int ngcf_perturb_rows(float* E, int64_t n_rows, int d, int64_t ld, float eps, uint64_t seed,
                                 const uint64_t* seed_dev, int layer, void* stream) {
    NGCF_REQUIRE(E, "perturb_rows: null E");
    NGCF_REQUIRE(n_rows >= 0 && n_rows < ((int64_t)1 << 31), "perturb_rows: n_rows %lld", (long long)n_rows);
    NGCF_REQUIRE(d >= 1 && d <= NGCF_MAX_WIDTH, "perturb_rows: width %d not in [1, %d]", d, NGCF_MAX_WIDTH);
    NGCF_REQUIRE(ld >= d, "perturb_rows: ld %lld < width %d", (long long)ld, d);
    NGCF_REQUIRE(eps >= 0.f && isfinite(eps), "perturb_rows: eps %g is not >= 0", eps);
    NGCF_REQUIRE(layer >= 0 && layer <= NGCF_MAX_LAYERS, "perturb_rows: layer %d not in [0, %d]", layer, NGCF_MAX_LAYERS);
    if (n_rows == 0) return NGCF_OK;
    perturb_rows_kernel<<<(unsigned)ceil_div64(n_rows * 32, 256), 256, 0, as_stream(stream)>>>(E, n_rows, d, ld, eps, seed,
                                                                                                seed_dev, layer);
    NGCF_LAUNCH_OK("perturb_rows_kernel");
    return NGCF_OK;
}

extern "C" int ngcf_infonce_workspace(int64_t batch, int D, size_t* bytes_host) {
    NGCF_REQUIRE(bytes_host, "infonce_workspace: null pointer");
    NGCF_REQUIRE(batch >= 1 && batch <= IN_MAX_B, "infonce_workspace: batch %lld not in [1, %d]", (long long)batch,
                 IN_MAX_B);
    NGCF_REQUIRE(D >= 1 && D <= IN_MAX_D, "infonce_workspace: D %d not in [1, %d]", D, IN_MAX_D);
    *bytes_host = info_layout(batch, D).total;
    return NGCF_OK;
}

extern "C" int ngcf_infonce(const float* x1, const float* x2, int64_t batch, int D, const int64_t* ids,
                            float temperature, float* loss, float* g1, float* g2, void* workspace,
                            size_t workspace_bytes, void* stream) {
    NGCF_REQUIRE(x1 && x2 && ids && loss, "infonce: null x1, x2, ids or loss");
    NGCF_REQUIRE(batch >= 1 && batch <= IN_MAX_B, "infonce: batch %lld not in [1, %d]", (long long)batch, IN_MAX_B);
    NGCF_REQUIRE(D >= 1 && D <= IN_MAX_D, "infonce: D %d not in [1, %d]", D, IN_MAX_D);
    NGCF_REQUIRE(temperature > 0.f && isfinite(temperature), "infonce: temperature %g is not > 0", temperature);
    NGCF_REQUIRE((g1 && g2) || (!g1 && !g2), "infonce: give both gradient buffers or none");
    const InfoLayout L = info_layout(batch, D);
    if (!workspace || workspace_bytes < L.total) {
        ngcf_set_error("infonce: workspace of %zu bytes, %zu needed", workspace ? workspace_bytes : (size_t)0, L.total);
        return NGCF_ERR_WORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 1023) & ~(uintptr_t)1023);
    float* z1 = reinterpret_cast<float*>(ws + L.z1);
    float* z2 = reinterpret_cast<float*>(ws + L.z2);
    float* nrm = reinterpret_cast<float*>(ws + L.nrm);
    uint8_t* valid = ws + L.valid;
    float* inv = reinterpret_cast<float*>(ws + L.inv);
    infonce_prep_kernel<<<(unsigned)ceil_div64(batch * 32, 256), 256, 0, st>>>(x1, x2, batch, D, ids, valid, z1, z2, nrm);
    NGCF_LAUNCH_OK("infonce_prep_kernel");
    SoftmaxRun r{};
    r.u = z1; r.p = z2; r.batch = batch; r.D = D;
    r.temperature = temperature; r.batch_size = 1.f;
    r.valid = valid; r.inv_count = inv;
    r.loss = loss; r.gu = g1; r.gp = g2;
    const int rc = softmax_run(r, ws + L.loss_ws, st);
    if (rc != NGCF_OK || !g1) return rc;
    infonce_finish_kernel<<<(unsigned)ceil_div64(2 * batch * 32, 256), 256, 0, st>>>(g1, g2, z1, z2, nrm, inv, batch, D);
    NGCF_LAUNCH_OK("infonce_finish_kernel");
    return NGCF_OK;
}

extern "C" int ngcf_rowgrad_add(const int64_t* const* rows_host, const int64_t* offsets_host, const float* const* g_host,
                                const int64_t* batch_host, int n_sets, int d, const int32_t* slot, float* dst,
                                int64_t ld_dst, void* stream) {
    NGCF_REQUIRE(rows_host && offsets_host && g_host && batch_host && dst, "rowgrad_add: null pointer");
    NGCF_REQUIRE(n_sets >= 1 && n_sets <= 2, "rowgrad_add: n_sets %d not in [1, 2]", n_sets);
    NGCF_REQUIRE(d >= 1 && d <= NGCF_MAX_WIDTH, "rowgrad_add: width %d not in [1, %d]", d, NGCF_MAX_WIDTH);
    NGCF_REQUIRE(ld_dst >= d, "rowgrad_add: ld_dst %lld < width %d", (long long)ld_dst, d);
    AddSets s{};
    int64_t total = 0;
    for (int j = 0; j < 2; ++j) {
        s.base[j] = total;
        if (j >= n_sets) continue;
        NGCF_REQUIRE(batch_host[j] >= 0 && (batch_host[j] == 0 || (rows_host[j] && g_host[j])), "rowgrad_add: set %d", j);
        s.rows[j] = rows_host[j]; s.offset[j] = offsets_host[j]; s.g[j] = g_host[j];
        total += batch_host[j];
    }
    s.base[2] = total;
    if (total == 0) return NGCF_OK;
    rowgrad_add_kernel<<<(unsigned)ceil_div64(total * 32, 256), 256, 0, as_stream(stream)>>>(s, d, slot, dst, ld_dst);
    NGCF_LAUNCH_OK("rowgrad_add_kernel");
    return NGCF_OK;
}
