// Laplacian format conversion, edge-value (node-dropout) pass, and the in-place feature mix.
// Reference lines replaced: matrix.py:79-83 (format), NGCF.py:93-100 (sparse_dropout), NGCF.py:103-115.
#include <cub/device/device_radix_sort.cuh>
#include <stdarg.h>

#include "common.cuh"
#include "tmap.h"

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

void ngcf_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int ngcf_num_sms() {
    static int cached[64] = {};                        // per device
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    int& c = cached[dev & 63];
    if (c == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) c = n;
        else return 148;
    }
    return c;
}

// ---- TMA descriptors (tmap.h) ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int ngcf_encode_tmap_2d(CUtensorMap* out, const float* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_cols,
                        uint32_t box_rows, CUtensorMapSwizzle swizzle) {
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) return -1;
        encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    const cuuint64_t dims[2] = {cols, rows};
    const cuuint64_t strides[1] = {ld * sizeof(float)};
    const cuuint32_t box[2] = {box_cols, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return (int)encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

static unsigned long long g_launches = 0;
void ngcf_count_launch() { __atomic_add_fetch(&g_launches, 1ull, __ATOMIC_RELAXED); }
extern "C" uint64_t ngcf_launch_count(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }

extern "C" int ngcf_abi_version(void) { return NGCF_B200_ABI_VERSION; }
extern "C" const char* ngcf_last_error(void) { return g_err; }

// ------------------------------------------------------------------------------------------------
// COO (int64, uncoalesced) -> CSR (int32) with permutation
// ------------------------------------------------------------------------------------------------
__global__ void make_keys_kernel(const int64_t* __restrict__ row, const int64_t* __restrict__ col, int64_t nnz,
                                 int transpose, uint64_t* __restrict__ keys, uint32_t* __restrict__ iota) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= nnz) return;
    uint64_t major = (uint64_t)(transpose ? col[t] : row[t]);
    uint64_t minor = (uint64_t)(transpose ? row[t] : col[t]);
    keys[t] = (major << 32) | (minor & 0xffffffffull);
    iota[t] = (uint32_t)t;
}

// colidx from the sorted keys; rowptr[r] = first sorted position whose major index is >= r
__global__ void csr_from_sorted_kernel(const uint64_t* __restrict__ keys, int64_t nnz, int64_t n_major,
                                       int32_t* __restrict__ rowptr, int32_t* __restrict__ colidx) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t > nnz) return;
    if (t == nnz) {                                    // tail: rows after the last non-empty one
        int64_t last = nnz > 0 ? (int64_t)(keys[nnz - 1] >> 32) : -1;
        for (int64_t r = last + 1; r <= n_major; ++r) rowptr[r] = (int32_t)nnz;
        return;
    }
    uint64_t k = keys[t];
    colidx[t] = (int32_t)(k & 0xffffffffull);
    int64_t major = (int64_t)(k >> 32);
    int64_t prev = t > 0 ? (int64_t)(keys[t - 1] >> 32) : -1;
    for (int64_t r = prev + 1; r <= major; ++r) rowptr[r] = (int32_t)t;
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

static int bits_for(int64_t n) {
    int b = 1;
    while (b < 32 && ((int64_t)1 << b) < n) ++b;
    return b;
}

extern "C" int ngcf_coo_to_csr_workspace(int64_t nnz, int64_t n_rows, size_t* bytes_host) {
    NGCF_REQUIRE(bytes_host != nullptr, "coo_to_csr_workspace: bytes_host is null");
    NGCF_REQUIRE(nnz >= 0 && nnz < ((int64_t)1 << 31), "coo_to_csr_workspace: nnz %lld out of range", (long long)nnz);
    (void)n_rows;
    size_t cub_bytes = 0;
    NGCF_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                              (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)nnz, 0, 64,
                                              (cudaStream_t)0));
    size_t n = (size_t)(nnz > 0 ? nnz : 1);
    *bytes_host = align256(8 * n) * 2 + align256(4 * n) + align256(cub_bytes) + 256;
    return NGCF_OK;
}

extern "C" int ngcf_coo_to_csr(const int64_t* coo_row, const int64_t* coo_col, int64_t nnz, int64_t n_rows,
                               int64_t n_cols, int transpose, int32_t* rowptr, int32_t* colidx, int32_t* perm,
                               void* workspace, size_t workspace_bytes, void* stream) {
    NGCF_REQUIRE(nnz >= 0 && nnz < ((int64_t)1 << 31), "coo_to_csr: nnz %lld out of range", (long long)nnz);
    NGCF_REQUIRE(n_rows > 0 && n_cols > 0 && n_rows < ((int64_t)1 << 31) && n_cols < ((int64_t)1 << 31),
                 "coo_to_csr: bad shape %lld x %lld", (long long)n_rows, (long long)n_cols);
    NGCF_REQUIRE(rowptr && (nnz == 0 || (coo_row && coo_col && colidx && perm)), "coo_to_csr: null pointer");
    size_t need = 0;
    int rc = ngcf_coo_to_csr_workspace(nnz, n_rows, &need);
    if (rc != NGCF_OK) return rc;
    if (workspace == nullptr || workspace_bytes < need) {
        ngcf_set_error("coo_to_csr: workspace %zu bytes < required %zu", workspace_bytes, need);
        return NGCF_ERR_WORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    const int64_t n_major = transpose ? n_cols : n_rows;
    const int64_t n_minor = transpose ? n_rows : n_cols;
    size_t n = (size_t)(nnz > 0 ? nnz : 1);
    char* w = reinterpret_cast<char*>(workspace);
    uint64_t* keys_in = reinterpret_cast<uint64_t*>(w);   w += align256(8 * n);
    uint64_t* keys_out = reinterpret_cast<uint64_t*>(w);  w += align256(8 * n);
    uint32_t* iota = reinterpret_cast<uint32_t*>(w);      w += align256(4 * n);
    void* cub_tmp = w;
    size_t cub_bytes = workspace_bytes - (size_t)(w - reinterpret_cast<char*>(workspace));
    const int threads = 256;
    if (nnz > 0) {
        make_keys_kernel<<<(unsigned)ceil_div64(nnz, threads), threads, 0, st>>>(coo_row, coo_col, nnz, transpose,
                                                                                  keys_in, iota);
        NGCF_LAUNCH_OK("make_keys_kernel");
        (void)n_minor;
        int end_bit = 32 + bits_for(n_major);
        NGCF_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cub_bytes, keys_in, keys_out, iota,
                                                  reinterpret_cast<uint32_t*>(perm), (int)nnz, 0, end_bit, st));
    }
    csr_from_sorted_kernel<<<(unsigned)ceil_div64(nnz + 1, threads), threads, 0, st>>>(keys_out, nnz, n_major, rowptr,
                                                                                      colidx);
    NGCF_LAUNCH_OK("csr_from_sorted_kernel");
    return NGCF_OK;
}

// ------------------------------------------------------------------------------------------------
// edge values with node dropout folded in (NGCF.py:93-100, 124-126)
// ------------------------------------------------------------------------------------------------
__global__ void edge_entries_kernel(const int32_t* __restrict__ colidx, const float* __restrict__ coo_val,
                                    const int32_t* __restrict__ perm, const uint8_t* __restrict__ keep_mask,
                                    int2* __restrict__ out, int64_t nnz) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= nnz) return;
    int64_t e = perm ? (int64_t)perm[t] : t;
    float v = coo_val[e];
    if (keep_mask && !keep_mask[e]) v = 0.0f;
    out[t] = make_int2(colidx[t], __float_as_int(v));
}

extern "C" int ngcf_edge_entries(const int32_t* colidx, const float* coo_val, const int32_t* perm,
                                 const uint8_t* keep_mask, int32_t* ent_out, int64_t nnz, void* stream) {
    NGCF_REQUIRE(nnz >= 0 && (nnz == 0 || (colidx && coo_val && ent_out)), "edge_entries: null pointer");
    NGCF_REQUIRE((reinterpret_cast<uintptr_t>(ent_out) & 7) == 0, "edge_entries: ent_out must be 8-byte aligned");
    if (nnz == 0) return NGCF_OK;
    edge_entries_kernel<<<(unsigned)ceil_div64(nnz, 256), 256, 0, as_stream(stream)>>>(
        colidx, coo_val, perm, keep_mask, reinterpret_cast<int2*>(ent_out), nnz);
    NGCF_LAUNCH_OK("edge_entries_kernel");
    return NGCF_OK;
}

// ------------------------------------------------------------------------------------------------
// feature mix (NGCF.py:103-115): last occurrence of a user id in the batch wins
// ------------------------------------------------------------------------------------------------
struct FeatArgs {
    const float* tab[5];
    const int64_t* idx[5];
    int width[5];
};

__global__ void featmix_claim_kernel(const int64_t* __restrict__ u_id, int64_t batch, int64_t n_user,
                                     int32_t* __restrict__ winner) {
    int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (b >= batch) return;
    int64_t u = u_id[b];
    if (u >= 0 && u < n_user) atomicMax(&winner[u], (int32_t)b);
}

// one warp per batch element; the winning occurrence writes the row and releases the claim
__global__ void featmix_apply_kernel(float* __restrict__ user_w, int d, FeatArgs fa, const int64_t* __restrict__ u_id,
                                     int64_t batch, int64_t n_user, float ratio, int32_t* __restrict__ winner) {
    int64_t b = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (b >= batch) return;
    int64_t u = u_id[b];
    if (u < 0 || u >= n_user) return;
    if (winner[u] != (int32_t)b) return;
    float* row = user_w + u * (int64_t)d;
    for (int c = lane; c < d; c += 32) {
        int off = c, f = 0;
        while (f < 4 && off >= fa.width[f]) { off -= fa.width[f]; ++f; }
        float feat = fa.tab[f][fa.idx[f][b] * (int64_t)fa.width[f] + off];
        row[c] = row[c] * (1.0f - ratio) + feat * ratio;       // NGCF.py:114-115
    }
    __syncwarp();
    if (lane == 0) winner[u] = -1;
}

extern "C" int ngcf_feature_mix(float* user_w, int64_t n_user, int d, const float* const* tables_host,
                                const int* widths_host, const int64_t* const* idx_host, const int64_t* u_id,
                                int64_t batch, float ratio, int32_t* winner, void* stream) {
    NGCF_REQUIRE(user_w && tables_host && widths_host && idx_host && u_id && winner, "feature_mix: null pointer");
    NGCF_REQUIRE(batch >= 0 && batch < ((int64_t)1 << 31), "feature_mix: batch %lld", (long long)batch);
    FeatArgs fa;
    int sum = 0;
    for (int f = 0; f < 5; ++f) {
        NGCF_REQUIRE(tables_host[f] && idx_host[f] && widths_host[f] > 0, "feature_mix: bad feature table %d", f);
        fa.tab[f] = tables_host[f];
        fa.idx[f] = idx_host[f];
        fa.width[f] = widths_host[f];
        sum += widths_host[f];
    }
    NGCF_REQUIRE(sum == d, "feature_mix: feature widths sum to %d, embedding width is %d "
                           "(reference: size mismatch at NGCF.py:114)", sum, d);
    if (batch == 0) return NGCF_OK;
    cudaStream_t st = as_stream(stream);
    featmix_claim_kernel<<<(unsigned)ceil_div64(batch, 256), 256, 0, st>>>(u_id, batch, n_user, winner);
    NGCF_LAUNCH_OK("featmix_claim_kernel");
    featmix_apply_kernel<<<(unsigned)ceil_div64(batch * 32, 256), 256, 0, st>>>(user_w, d, fa, u_id, batch, n_user,
                                                                               ratio, winner);
    NGCF_LAUNCH_OK("featmix_apply_kernel");
    return NGCF_OK;
}

// ------------------------------------------------------------------------------------------------
// SpMM tiles on the device (plan.greedy_tiles for graphs whose tile count rules out a host loop): consecutive tiles of at
// most max_rows rows and max_ent entries.  next[r] = end of the tile that starts at row r, for every r in parallel; the
// tile list is the orbit of row 0 under next[], walked by one thread (one dependent load per tile).
// ------------------------------------------------------------------------------------------------
__global__ void tile_next_kernel(const int32_t* __restrict__ rowptr, int64_t n_rows, int max_rows, int max_ent,
                                 int32_t* __restrict__ next) {
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int64_t limit = (int64_t)rowptr[r] + max_ent;
    int64_t lo = r, hi = min(n_rows, r + max_rows);                    // last k in [r, hi] with rowptr[k] <= limit
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (rowptr[mid] <= limit) lo = mid; else hi = mid - 1;
    }
    next[r] = (int32_t)max(r + 1, lo);
}
__global__ void tile_chase_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ next, int64_t n_rows,
                                  int4* __restrict__ tiles, int64_t capacity, int32_t* __restrict__ count) {
    int64_t n = 0;
    for (int64_t r = 0; r < n_rows;) {
        const int32_t r1 = next[r];
        if (n < capacity) tiles[n] = make_int4((int)r, r1, rowptr[r], rowptr[r1]);
        ++n;
        r = r1;
    }
    *count = (int32_t)n;
}

extern "C" int ngcf_build_tiles(const int32_t* rowptr, int64_t n_rows, int max_rows, int max_ent, int32_t* next_scratch,
                                int32_t* tiles_out, int64_t capacity, int32_t* count_out, void* stream) {
    NGCF_REQUIRE(rowptr && next_scratch && tiles_out && count_out, "build_tiles: null pointer");
    NGCF_REQUIRE(n_rows >= 0 && n_rows < ((int64_t)1 << 31) && max_rows >= 1 && max_ent >= 1, "build_tiles: bad sizes");
    cudaStream_t st = as_stream(stream);
    if (n_rows > 0) {
        tile_next_kernel<<<(unsigned)ceil_div64(n_rows, 256), 256, 0, st>>>(rowptr, n_rows, max_rows, max_ent, next_scratch);
        NGCF_LAUNCH_OK("tile_next_kernel");
    }
    tile_chase_kernel<<<1, 1, 0, st>>>(rowptr, next_scratch, n_rows, reinterpret_cast<int4*>(tiles_out), capacity, count_out);
    NGCF_LAUNCH_OK("tile_chase_kernel");
    return NGCF_OK;
}
