// Shared device/host helpers for the NGCF B200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "ngcf_b200.h"

// ---- host-side error plumbing (thread-local message behind ngcf_last_error) ----------------------
void ngcf_set_error(const char* fmt, ...);

#define NGCF_REQUIRE(cond, ...)                      \
    do {                                             \
        if (!(cond)) {                               \
            ngcf_set_error(__VA_ARGS__);             \
            return NGCF_ERR_INVALID;                 \
        }                                            \
    } while (0)

#define NGCF_CUDA(call)                                                                   \
    do {                                                                                  \
        cudaError_t e__ = (call);                                                         \
        if (e__ != cudaSuccess) {                                                         \
            ngcf_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return NGCF_ERR_CUDA;                                                         \
        }                                                                                 \
    } while (0)

void ngcf_count_launch();   // bumps the counter behind ngcf_launch_count()

#define NGCF_LAUNCH_OK(name)                                                              \
    do {                                                                                  \
        ngcf_count_launch();                                                              \
        cudaError_t e__ = cudaGetLastError();                                             \
        if (e__ != cudaSuccess) {                                                         \
            ngcf_set_error("launch of %s failed: %s", name, cudaGetErrorString(e__));     \
            return NGCF_ERR_CUDA;                                                         \
        }                                                                                 \
    } while (0)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

int ngcf_num_sms();   // cached cudaDevAttrMultiProcessorCount of the current device

// ---- programmatic dependent launch ---------------------------------------------------------------------------------
// A training step is ~30 dependent launches of 5-50 us: the launch latency and the ramp-up / drain of every kernel are a
// sizeable share of it.  The large kernels are launched with programmatic stream serialization: each signals
// launch_dependents at its top, so the NEXT kernel's CTAs become resident while this one drains and run their
// prologue (barriers, TMEM allocation, tile descriptors, weight tiles); they stop at pdl_wait() — which returns once
// the preceding kernel has completed and its writes are visible — before touching anything a predecessor produced and
// before writing anything at all.

template <typename... KArgs, typename... Args>
static inline cudaError_t ngcf_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                          Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- device helpers ------------------------------------------------------------------------------
#define FULL_MASK 0xffffffffu

__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
    return v;
}

// first position in [lo, hi) of the ascending list a whose value is >= v (hi if there is none)
__device__ __forceinline__ int64_t lower_bound_i32(const int32_t* __restrict__ a, int64_t lo, int64_t hi, int v) {
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ float4 ld_f4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st_f4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

// streaming 128-bit load of data this kernel only reads once: no L1 line is allocated.  In the tensor-core kernels
// ~216 KB of the SM's 256 KB are shared memory, the L1 that remains is a few tens of KB, and every outstanding
// allocating load pins a line of it: 8 loader warps x 8 loads x 4 lines could not even be in flight together.
// Asks the memory system to bring [p, p + bytes) into L2 (no registers, no completion to wait for): one thread of a
// persistent CTA issues it for the tile it will need a few tiles from now, so that the tile's loads meet L2 latency
// instead of DRAM latency.  p 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void l2_prefetch_bulk(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ float4 ld_stream_f4(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}

// streaming (read-once) loads: keep CSR arrays out of L1 so gathered embedding rows stay resident
__device__ __forceinline__ int ld_stream_i32(const int* p) {
    int v;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float ld_stream_f32(const float* p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

// Counter-based dropout RNG: stateless, so forward and backward regenerate the same decisions from
// (seed, stream, layer, coordinates) without storing masks.  Three rounds of the murmur3 32-bit finalizer over the
// counter words plus one more round give 64 bits = four 16-bit uniforms per call (probabilities are resolved to
// 2^-16).  (The first version used Philox4x32-10: its 40 dependent 32x32->64 high multiplies run at a quarter of the
// integer rate on sm_100, and the per-step decision pass alone cost 40 us at Gowalla shape.)
__device__ __forceinline__ uint32_t ngcf_mix(uint32_t h) {
    h ^= h >> 16; h *= 0x85ebca6bu; h ^= h >> 13; h *= 0xc2b2ae35u; h ^= h >> 16;
    return h;
}
__device__ __forceinline__ uint2 ngcf_hash64(uint64_t seed, uint32_t a, uint32_t b, uint32_t c, uint32_t stream) {
    uint32_t h = ngcf_mix(a ^ (uint32_t)seed ^ stream);
    h = ngcf_mix(h ^ (b + 0x9E3779B9u) ^ (uint32_t)(seed >> 32));
    h = ngcf_mix(h + c * 0x632BE5ABu + 0x7F4A7C15u);
    return make_uint2(h, ngcf_mix(h ^ 0x68E31DA4u));
}
#define NGCF_STREAM_NODE 0x4e4f4445u   // 'NODE'
#define NGCF_STREAM_MESS 0x4d455353u   // 'MESS'
#define NGCF_STREAM_NOISE 0x4e4f4953u  // 'NOIS': XSimGCL's layer noise (ngcf_perturb_rows)
__device__ __forceinline__ uint32_t ngcf_threshold16(float p) { return (uint32_t)(p * 65536.0f); }   // keep iff u16 >= it

// Per-step randomness: `seed` is a host value baked into the launch, `seed_dev` an optional device counter
// added to it, so a captured CUDA graph draws fresh decisions on every replay.
__device__ __forceinline__ uint64_t ngcf_seed(uint64_t seed, const uint64_t* seed_dev) {
    return seed + (seed_dev ? *seed_dev : 0ull);
}

// Node dropout (NGCF.py:93-100,124-126) in device-RNG mode.  An entry (row, col) of L has a STATIC 32-bit key (it
// depends on the coordinates only, so the plan can store it per entry: the per-step pass then needs neither the
// entry's row nor a hash of two coordinates); the step's draws are two mixes of key ^ seed: four 16-bit uniforms per
// group of four layers.  Bit k of the result = the entry survives layer k, i.e. its draws for layers 0..k are all
// >= p (cumulative over layers, values unscaled).  Keyed on the coordinates IN L, so the forward CSR and the CSR of
// L^T agree without a permutation.
__device__ __forceinline__ uint32_t ngcf_node_key(uint32_t row, uint32_t col) {
    return ngcf_mix(ngcf_mix(row + 0x9E3779B9u) ^ (col * 0x85EBCA77u + 0xC2B2AE3Du));
}
__device__ __forceinline__ uint32_t node_keep_bits_key(uint32_t thr, uint64_t seed, int n_layers, uint32_t key) {
    uint32_t bits = 0;
    bool keep = true;
    for (int g = 0; g * 4 < n_layers && keep; ++g) {
        const uint32_t h = ngcf_mix(key ^ (uint32_t)seed ^ ((uint32_t)g * 0x632BE5ABu) ^ NGCF_STREAM_NODE);
        const uint32_t y = ngcf_mix(h ^ (uint32_t)(seed >> 32));
        const uint32_t u[4] = {h & 0xffffu, h >> 16, y & 0xffffu, y >> 16};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            keep = keep && (u[j] >= thr);
            if (keep && g * 4 + j < n_layers) bits |= 1u << (g * 4 + j);
        }
    }
    return bits;
}
__device__ __forceinline__ uint32_t node_keep_bits(float p, uint64_t seed, int n_layers, uint32_t row, uint32_t col) {
    return node_keep_bits_key(ngcf_threshold16(p), seed, n_layers, ngcf_node_key(row, col));
}
__device__ __forceinline__ bool node_keep(float p, uint64_t seed, int layer, uint32_t row, uint32_t col) {
    return (node_keep_bits(p, seed, layer + 1, row, col) >> layer) & 1u;
}

// 64 bits for the message-dropout decisions of one quad: three mixes (the layer is folded into the first word) instead
// of ngcf_hash64's four - the dense epilogues spend most of their per-tile time on this chain (profiles/
// r02_dense_fwd_timeline.txt)
__device__ __forceinline__ uint2 ngcf_mess_hash(uint64_t seed, int layer, uint64_t quad) {
    uint32_t h = ngcf_mix((uint32_t)quad ^ (uint32_t)seed ^ NGCF_STREAM_MESS ^ ((uint32_t)layer * 0x632BE5ABu));
    h = ngcf_mix(h ^ ((uint32_t)(quad >> 32) + 0x9E3779B9u) ^ (uint32_t)(seed >> 32));
    return make_uint2(h, ngcf_mix(h ^ 0x68E31DA4u));
}
// inverted-dropout multipliers of message dropout (NGCF.py:142) in device-RNG mode: one call covers the four
// consecutive elements 4*quad .. 4*quad+3 of the flattened [N, d_out] layer output
__device__ __forceinline__ float4 mess_multiplier4(float p, uint64_t seed, int layer, uint64_t quad) {
    const uint2 r = ngcf_mess_hash(seed, layer, quad);
    const uint32_t thr = ngcf_threshold16(p);
    const float s = 1.0f / (1.0f - p);
    return make_float4((r.x & 0xffffu) >= thr ? s : 0.f, (r.x >> 16) >= thr ? s : 0.f, (r.y & 0xffffu) >= thr ? s : 0.f,
                       (r.y >> 16) >= thr ? s : 0.f);
}
// the same decisions with the threshold and 1/(1-p) hoisted out of the caller's loop
__device__ __forceinline__ float4 mess_multiplier4_pre(uint32_t thr, float s, uint64_t seed, int layer, uint64_t quad) {
    const uint2 r = ngcf_mess_hash(seed, layer, quad);
    return make_float4((r.x & 0xffffu) >= thr ? s : 0.f, (r.x >> 16) >= thr ? s : 0.f, (r.y & 0xffffu) >= thr ? s : 0.f,
                       (r.y >> 16) >= thr ? s : 0.f);
}
__device__ __forceinline__ float mess_multiplier(float p, uint64_t seed, int layer, uint64_t elem) {
    const float4 m = mess_multiplier4(p, seed, layer, elem >> 2);
    const int j = (int)(elem & 3);
    return j == 0 ? m.x : j == 1 ? m.y : j == 2 ? m.z : m.w;
}

// message-dropout decisions precomputed per step (ngcf_mess_dropout_bits): bit (col & 31) of word
// [row, col >> 5] of a [n_rows, ceil(d_out/32)] array = keep; same RNG stream as mess_multiplier4
__device__ __forceinline__ float mess_multiplier_bits(const uint32_t* bits, float p, int64_t row, int d_out, int col) {
    const uint32_t w = bits[row * ((d_out + 31) >> 5) + (col >> 5)];
    return (w >> (col & 31)) & 1u ? 1.0f / (1.0f - p) : 0.0f;
}
