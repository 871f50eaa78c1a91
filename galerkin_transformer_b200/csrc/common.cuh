// Shared device/host helpers for libgalerkin_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/galerkin_b200.h"

namespace gb200 {

// ---- error plumbing: C entry points return 0 / non-zero and keep a thread-local message ----
void set_error(const char* fmt, ...);
int check_launch(const char* what, int nkernels = 1);  // cudaGetLastError -> error string; counts launches
void use_device(int device);                 // thread-local cached cudaSetDevice
const unsigned long long* rng_offset_ptr();  // device counter added to every dropout seed (graph-safe RNG)

#define GB_REQUIRE(cond, ...)                                  \
    do {                                                       \
        if (!(cond)) {                                         \
            gb200::set_error(__VA_ARGS__);                     \
            return GB200_ERR_INVALID;                          \
        }                                                      \
    } while (0)

// ---- programmatic dependent launch (PDL) ---------------------------------------------------
// Every kernel of this library starts with pdl_enter(): `launch_dependents` lets the NEXT kernel in the stream be
// scheduled as soon as all CTAs of this one are resident (its CTAs fill SMs as ours retire, run their prologue and
// park), `wait` then blocks until the PREVIOUS kernel has completed and flushed.  No global memory is touched before
// the wait, so ordering is exactly that of a plain stream.  The library's own kernels are launched WITHOUT the
// programmatic attribute: inside the CUDA-graph replay of the C3 step, programmatic edges measured 4-8 % SLOWER than
// plain kernel edges in every trigger placement tried (entry, after the MMAs, none).  The entry trigger still matters:
// the fused encoder chain (encoder_common.cuh) is launched with the attribute, and its first kernel starts early only
// once the library kernel before it has triggered.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_enter() { pdl_trigger(); pdl_wait(); }

// errors surface in check_launch()
template <typename... KArgs, typename... Args>
static inline void launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                 Args&&... args) {
    kernel<<<grid, block, smem, st>>>(static_cast<KArgs>(args)...);
}

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// ---- activations --------------------------------------------------------------------------
enum { ACT_NONE = GB200_ACT_NONE, ACT_RELU = GB200_ACT_RELU, ACT_SILU = GB200_ACT_SILU };

__device__ __forceinline__ float act_apply(int act, float v) {
    if (act == ACT_RELU) return v > 0.f ? v : 0.f;
    if (act == ACT_SILU) return v / (1.f + __expf(-v));
    return v;
}
// derivative w.r.t. the pre-activation z
__device__ __forceinline__ float act_grad(int act, float z) {
    if (act == ACT_RELU) return z > 0.f ? 1.f : 0.f;
    if (act == ACT_SILU) {
        float s = 1.f / (1.f + __expf(-z));
        return s * (1.f + z * (1.f - s));
    }
    return 1.f;
}

// ---- counter-based RNG for fused dropout: Philox4x32-7 keyed by (seed, element index / 8) ------
// One Philox block yields eight 16-bit uniforms, one per element: element idx uses halfword (idx & 7) of block
// (idx >> 3).  The same (seed, index) reproduces the same keep decision in forward and backward, so no mask tensor ever
// touches HBM.  Seven rounds are the Crush-resistant minimum of Salmon et al. (SC'11); the drop probability is quantised
// to thr / 65536 and the keep scale is its exact inverse complement 65536 / (65536 - thr), so the mask stays unbiased
// (p = 0.5 -> scale exactly 2, as libs/layers.py:730-731 needs).
__device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) { return __umulhi(a, b); }

__device__ __forceinline__ uint4 philox4x32(uint64_t seed, uint64_t idx) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    uint32_t c0 = (uint32_t)idx, c1 = (uint32_t)(idx >> 32), c2 = 0x9E3779B9u, c3 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 7; ++r) {
        const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
        uint32_t h0 = mulhi32(M0, c0), l0 = M0 * c0;
        uint32_t h1 = mulhi32(M1, c2), l1 = M1 * c2;
        uint32_t n0 = h1 ^ c1 ^ k0, n1 = l1, n2 = h0 ^ c3 ^ k1, n3 = l0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ uint32_t dropout_threshold(float p) { return (uint32_t)(p * 65536.f + 0.5f); }
__device__ __forceinline__ float dropout_keep_scale(uint32_t thr) { return 65536.f / (65536.f - (float)thr); }

// keep-scale for element `idx`: 0 if dropped, 1/(1-p) if kept.  p in [0,1).
__device__ __forceinline__ float dropout_scale(float p, uint64_t seed, uint64_t idx) {
    if (p <= 0.f) return 1.f;
    const uint4 r = philox4x32(seed, idx >> 3);
    const uint32_t e = (uint32_t)idx & 7u;
    const uint32_t w = (e >> 1) == 0 ? r.x : (e >> 1) == 1 ? r.y : (e >> 1) == 2 ? r.z : r.w;
    const uint32_t u = (e & 1u) ? (w >> 16) : (w & 0xffffu);
    const uint32_t thr = dropout_threshold(p);
    return u < thr ? 0.f : dropout_keep_scale(thr);
}

// eight consecutive elements idx..idx+7 (idx % 8 == 0) from ONE Philox block -- same stream as dropout_scale
__device__ __forceinline__ void dropout_scale8(float p, uint64_t seed, uint64_t idx, float (&s)[8]) {
    const uint4 r = philox4x32(seed, idx >> 3);
    const uint32_t thr = dropout_threshold(p);
    const float keep = dropout_keep_scale(thr);
    s[0] = (r.x & 0xffffu) < thr ? 0.f : keep; s[1] = (r.x >> 16) < thr ? 0.f : keep;
    s[2] = (r.y & 0xffffu) < thr ? 0.f : keep; s[3] = (r.y >> 16) < thr ? 0.f : keep;
    s[4] = (r.z & 0xffffu) < thr ? 0.f : keep; s[5] = (r.z >> 16) < thr ? 0.f : keep;
    s[6] = (r.w & 0xffffu) < thr ? 0.f : keep; s[7] = (r.w >> 16) < thr ? 0.f : keep;
}

// out[c] (+)= scale * sum_{p < nparts} part[p * stride + c]   for c < width: a (32 x 32)-thread CTA per 32
// columns, rows strided over threadIdx.y, fixed-order shared-memory finish (deterministic).
__device__ __forceinline__ void reduce_partials_2d(const float* __restrict__ part, int nparts, long long stride,
                                                   int width, float scale, int accumulate,
                                                   float* __restrict__ out) {
    __shared__ float red[32][33];
    const int c = blockIdx.x * 32 + threadIdx.x;
    float s = 0.f;
    if (c < width)
        for (int p = threadIdx.y; p < nparts; p += 32) s += part[(long long)p * stride + c];
    red[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && c < width) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) t += red[i][threadIdx.x];
        t *= scale;
        out[c] = accumulate ? out[c] + t : t;
    }
}

// four consecutive elements idx..idx+3 (idx % 4 == 0): half a Philox block -- same stream as dropout_scale
__device__ __forceinline__ float4 dropout_scale4(float p, uint64_t seed, uint64_t idx) {
    const uint4 r = philox4x32(seed, idx >> 3);
    const uint32_t thr = dropout_threshold(p);
    const float keep = dropout_keep_scale(thr);
    const uint32_t w0 = (idx & 4) ? r.z : r.x, w1 = (idx & 4) ? r.w : r.y;
    return make_float4((w0 & 0xffffu) < thr ? 0.f : keep, (w0 >> 16) < thr ? 0.f : keep,
                       (w1 & 0xffffu) < thr ? 0.f : keep, (w1 >> 16) < thr ? 0.f : keep);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace gb200
