// tcgen05 (5th-gen tensor core) TF32 GEMM for sm_100a with the library's fused epilogue.
//
//   C = R + rscale * drop( act( alpha * op(A) . op(B) + bias ) )           fp32 in, fp32 out
//
//   * operands are fp32 in HBM and are consumed as TF32 by `tcgen05.mma.kind::tf32`
//     (10-bit mantissa; ~4e-4 relative error per contraction, SURVEY section 7 item 6);
//   * tiles are staged global -> shared by TMA (`cp.async.bulk.tensor.2d`, SWIZZLE_128B,
//     out-of-range rows/columns zero-filled so ragged M/N/K need no special casing);
//   * accumulators live in TMEM (128 lanes x BN fp32 columns), read back with `tcgen05.ld`;
//   * both operand majors are supported through the UMMA descriptors, so the three GEMMs of a
//     Linear layer (y = x W^T, dx = g W, dW = g^T x) all run here without any transpose copy:
//         A K-major : stored [M, K]      A MN-major : stored [K, M]
//         B K-major : stored [N, K]      B MN-major : stored [K, N]
//   * warp roles (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer (one lane),
//     warps 2-5 = TF32 round-to-nearest converters during the main loop, then the epilogue (each owns
//     one 32-lane TMEM quarter); 3-stage mbarrier ring (full -> converted -> empty); two CTAs fit per
//     SM so one tile's epilogue overlaps another tile's main loop;
//   * split-K (weight gradients reduce over all tokens) writes fp32 partials that
//     `splitk_reduce_kernel` sums in fixed order (deterministic).
//
// All waits are bounded: a descriptor/protocol bug traps instead of hanging the device.
#include <cuda.h>

#include "common.cuh"
#include "gemm_epilogue.cuh"
#include "tc_prims.cuh"

namespace gb200 {

constexpr int TC_BM = 128, TC_BK = 32, TC_THREADS = 192;
// pipeline depth: 3 stages let two CTAs share an SM (one tile's epilogue overlaps another's main loop); a 6-stage,
// one-CTA-per-SM ring for the long-K weight-gradient GEMMs was measured and is slower (tools/bench_gemm.py)
// (6 for MN/MN measured slower).  Narrow tiles (BN <= 64, 24 KB stages) afford a 4th stage at the same occupancy;
// the 192-wide tile (N = 384 in one wave of 232 CTAs instead of 348 in two) has room for two.
// split (3xTF32) stages are twice as large: two of them keep the CTA under half an SM's shared memory for BN <= 64, so two
// CTAs co-reside and one's prologue / epilogue overlaps the other's main loop (the tall-skinny decoder GEMMs are 8 waves of
// single-tile CTAs: with one CTA per SM those phases were serialised, 62 us for a 16 us problem)
// SPLIT ("3xTF32"): every operand tile also keeps its TF32 residual lo = rna(x - hi) in a second buffer and each k-step
// issues hi.hi + hi.lo + lo.hi -- fp32-grade products (2^-22) for the forward / input-gradient GEMMs of 'x3' mode that no
// fused kernel covers; stages are twice as large, so the ring is one stage shorter
template <int BN, bool SPLIT = false> __host__ __device__ constexpr int tc_stages() {
    return SPLIT ? 2 : (BN == 192 ? 2 : (BN <= 64 ? 4 : 3));
}
template <int BN> __host__ __device__ constexpr int tc_tmem_cols() { return BN == 192 ? 256 : BN; }     // power of two >= 32
template <int BN, bool SPLIT = false> __host__ __device__ constexpr int tc_smem_bytes() {
    constexpr int ring = tc_stages<BN, SPLIT>() * (SPLIT ? 2 : 1) * (TC_BM * TC_BK * 4 + BN * TC_BK * 4);
    constexpr int staging = TC_BM * (BN + 4) * 4;                                   // epilogue reuses the ring
    return (ring > staging ? ring : staging) + 1024 + 256;
}
struct TcArgs {
    GemmEpilogue ep;      // shared with the SIMT kernel: bias/act/dropout/residual/Z/C
    int M, N, K;
    int ksplit, kchunk;   // kchunk is a multiple of TC_BK
    float* ws;
    int vec4;             // C/R/Z/ws rows are 16-byte aligned and N % 4 == 0: float4 epilogue
    unsigned long long* trace;   // diagnostics: 8 globaltimer stamps per CTA (gb200_gemm_tc_set_trace), else null
};

__device__ __forceinline__ void tc_stamp(const TcArgs& g, int slot) {
    if (g.trace) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        const long long cta = ((long long)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
        g.trace[cta * 8 + slot] = t;
    }
}

// activation with fast intrinsics (the TF32 path is not bit-exact fp32 anyway)
template <int ACT>
__device__ __forceinline__ float act_fast(float v) {
    if (ACT == ACT_RELU) return fmaxf(v, 0.f);
    if (ACT == ACT_SILU) return __fdividef(v, 1.f + __expf(-v));
    return v;
}

// Coalesced float4 epilogue for one warp's 32 accumulator rows staged in shared memory.
// Compile-time activation / dropout; residual, Z and accumulate are warp-uniform runtime switches.
// GATE != 0 (host guarantees no residual / accumulate then): the rv registers carry the gate operand G instead and
// v *= act'(G) before the dropout scale -- the elementwise backward between two Linear layers, fused.
template <int ACT, bool DROP, int GATE = 0>
__device__ __forceinline__ void tc_epilogue_vec4(const TcArgs& g, const float* __restrict__ stage, int DS, int lane,
                                                 int rbase, int n0, int ncols, unsigned long long seed) {
    const GemmEpilogue& ep = g.ep;
    constexpr int RB = 8;                        // rows in flight per thread
    const bool hasR = ep.R != nullptr, hasZ = ep.Z != nullptr, accum = ep.accumulate != 0;
    const float alpha = ep.alpha, rscale = ep.rscale, p = ep.drop_p;
    const int nrows = min(32, g.M - rbase);
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int c = lane * 4; c < ncols; c += 128) {
        const int n = n0 + c;
        float4 bv = zero4;
        if (ep.bias) bv = *reinterpret_cast<const float4*>(ep.bias + n);
        const float* rp = GATE ? ep.G + (long long)rbase * ep.ldg + n : (hasR ? ep.R + (long long)rbase * ep.ldr + n : nullptr);
        const int ldr = GATE ? ep.ldg : ep.ldr;
        float* cp = ep.C + (long long)rbase * ep.ldc + n;
        float* zp = hasZ ? ep.Z + (long long)rbase * ep.ldz + n : nullptr;
#pragma unroll 1
        for (int r0 = 0; r0 < nrows; r0 += RB) {
            float4 acc[RB], rv[RB];
#pragma unroll
            for (int i = 0; i < RB; ++i) {
                acc[i] = *reinterpret_cast<const float4*>(&stage[(r0 + i) * DS + c]);
                rv[i] = zero4;
                if (r0 + i < nrows) {
                    if (GATE || hasR) rv[i] = *reinterpret_cast<const float4*>(rp + (long long)(r0 + i) * ldr);
                    if (!GATE && accum) {
                        const float4 cvv = *reinterpret_cast<const float4*>(cp + (long long)(r0 + i) * ep.ldc);
                        rv[i].x += cvv.x; rv[i].y += cvv.y; rv[i].z += cvv.z; rv[i].w += cvv.w;
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < RB; ++i) {
                if (r0 + i >= nrows) break;                                  // uniform across the warp
                float4 z = make_float4(fmaf(alpha, acc[i].x, bv.x), fmaf(alpha, acc[i].y, bv.y),
                                       fmaf(alpha, acc[i].z, bv.z), fmaf(alpha, acc[i].w, bv.w));
                if (hasZ) *reinterpret_cast<float4*>(zp + (long long)(r0 + i) * ep.ldz) = z;
                float4 v = make_float4(act_fast<ACT>(z.x), act_fast<ACT>(z.y), act_fast<ACT>(z.z), act_fast<ACT>(z.w));
                if (GATE == ACT_RELU) {
                    v.x = rv[i].x > 0.f ? v.x : 0.f; v.y = rv[i].y > 0.f ? v.y : 0.f;
                    v.z = rv[i].z > 0.f ? v.z : 0.f; v.w = rv[i].w > 0.f ? v.w : 0.f;
                } else if (GATE == ACT_SILU) {
                    v.x *= act_grad(ACT_SILU, rv[i].x); v.y *= act_grad(ACT_SILU, rv[i].y);
                    v.z *= act_grad(ACT_SILU, rv[i].z); v.w *= act_grad(ACT_SILU, rv[i].w);
                }
                if (DROP) {
                    const float4 ds = dropout_scale4(p, seed, (unsigned long long)(rbase + r0 + i) * g.N + n);
                    v.x *= ds.x; v.y *= ds.y; v.z *= ds.z; v.w *= ds.w;
                }
                if (GATE) rv[i] = zero4;
                *reinterpret_cast<float4*>(cp + (long long)(r0 + i) * ep.ldc) =
                    make_float4(fmaf(rscale, v.x, rv[i].x), fmaf(rscale, v.y, rv[i].y), fmaf(rscale, v.z, rv[i].z),
                                fmaf(rscale, v.w, rv[i].w));
            }
        }
    }
}

template <int BN, bool A_MN, bool B_MN, bool SPLIT = false>
__device__ __forceinline__ void gemm_tc_body(const CUtensorMap& mapA, const CUtensorMap& mapB, const TcArgs& g, int bx, int by,
                                             int bz) {
    constexpr int A_BYTES = TC_BM * TC_BK * 4;          // 16 KB
    constexpr int B_BYTES = BN * TC_BK * 4;
    constexpr int TILE_PAIR = A_BYTES + B_BYTES;        // what TMA lands per k-block
    constexpr int STAGE_BYTES = (SPLIT ? 2 : 1) * TILE_PAIR;   // SPLIT: [A hi | B hi | A lo | B lo]
    constexpr int TC_STAGES = tc_stages<BN, SPLIT>();
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // 1024-byte alignment is required by SWIZZLE_128B atoms
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + tc_smem_bytes<BN, SPLIT>() - 1024 - 256);   // past ring AND staging
    uint64_t* empty_bar = full_bar + TC_STAGES;
    uint64_t* conv_bar = empty_bar + TC_STAGES;
    uint64_t* tmem_full = conv_bar + TC_STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const int m0 = by * TC_BM, n0 = bx * BN;
    const int split = bz;
    const int kbeg = split * g.kchunk;
    const int kend = min(g.K, kbeg + g.kchunk);
    const int nkb = (kend - kbeg + TC_BK - 1) / TC_BK;
    pdl_trigger();
    if (threadIdx.x == 64) tc_stamp(g, 0);                                   // CTA entry

    if (threadIdx.x == 0) {
        for (int s = 0; s < TC_STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
            mbar_init(&conv_bar[s], 4);          // one arrival per converter warp
        }
        mbar_init(tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&mapA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&mapB) : "memory");
    }
    if (warp == 2) {   // TMEM allocation: BN fp32 columns x 128 lanes (power of two >= 32)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "n"(tc_tmem_cols<BN>())
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // Everything above (barrier init, TMEM allocation, tensor-map prefetch) touched no global memory and has
    // overlapped the tail of the previous kernel; from here on its results are needed.
    pdl_wait();
    if (threadIdx.x == 64) tc_stamp(g, 1);                                   // barriers + TMEM ready

    if (warp == 0) {
        if (lane == 0) {   // ---------------- TMA producer ----------------
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % TC_STAGES;
                const uint32_t ph = (kb / TC_STAGES) & 1;
                mbar_wait(&empty_bar[s], ph ^ 1);
                uint8_t* sa = smem + s * STAGE_BYTES;
                uint8_t* sb = sa + A_BYTES;
                mbar_expect_tx(&full_bar[s], TILE_PAIR);
                const int k0 = kbeg + kb * TC_BK;
                if (!A_MN) {
                    tma_load_2d(sa, &mapA, &full_bar[s], k0, m0);                    // box {32 k, 128 m}
                } else {
#pragma unroll
                    for (int j = 0; j < TC_BM / 32; ++j)                                // box {32 m, 32 k}
                        tma_load_2d(sa + j * 4096, &mapA, &full_bar[s], m0 + 32 * j, k0);
                }
                if (!B_MN) {
                    tma_load_2d(sb, &mapB, &full_bar[s], k0, n0);                    // box {32 k, BN n}
                } else {
#pragma unroll
                    for (int j = 0; j < BN / 32; ++j)
                        tma_load_2d(sb + j * 4096, &mapB, &full_bar[s], n0 + 32 * j, k0);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {   // ---------------- MMA issuer ----------------
            // instruction descriptor (cute UMMA::InstrDescriptor): D=F32, A=B=TF32, majors, N>>3, M>>4
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((A_MN ? 1u : 0u) << 15) |
                                   ((B_MN ? 1u : 0u) << 16) | ((uint32_t)(BN >> 3) << 17) |
                                   ((uint32_t)(TC_BM >> 4) << 24);
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % TC_STAGES;
                const uint32_t ph = (kb / TC_STAGES) & 1;
                mbar_wait(&conv_bar[s], ph);     // tile landed (TMA) and rounded to TF32
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + s * STAGE_BYTES);
                const uint32_t sb = sa + A_BYTES;
#pragma unroll
                for (int k = 0; k < TC_BK / 8; ++k) {
                    // K-major (SW128): 8 tf32 = 32 bytes further along the 128-byte swizzled row; 8-row groups
                    //   are 1024 B apart (SBO).
                    // MN-major (SW128 base-32B): rows are k, 128 B each; 4-row swizzle atoms 512 B apart (SBO);
                    //   8 k-rows per MMA = 1024 B; 32-wide MN blocks are 4096 B apart (LBO).
                    const uint64_t ad = A_MN ? umma_desc<1>(sa + k * 1024, 4096, 512) : umma_desc<2>(sa + k * 32, 16, 1024);
                    const uint64_t bd = B_MN ? umma_desc<1>(sb + k * 1024, 4096, 512) : umma_desc<2>(sb + k * 32, 16, 1024);
                    tc_mma_tf32(tmem_base, ad, bd, idesc, (kb | k) != 0);
                    if (SPLIT) {
                        const uint32_t la = sa + TILE_PAIR, lb = sb + TILE_PAIR;
                        const uint64_t adl = A_MN ? umma_desc<1>(la + k * 1024, 4096, 512) : umma_desc<2>(la + k * 32, 16, 1024);
                        const uint64_t bdl = B_MN ? umma_desc<1>(lb + k * 1024, 4096, 512) : umma_desc<2>(lb + k * 32, 16, 1024);
                        tc_mma_tf32(tmem_base, ad, bdl, idesc, 1u);
                        tc_mma_tf32(tmem_base, adl, bd, idesc, 1u);
                    }
                }
                tc_commit(&empty_bar[s]);        // frees the stage once these MMAs have read it
            }
            tc_commit(tmem_full);                // accumulator complete
        }
    } else {               // ---------------- epilogue warps 2..5 ----------------
        // TMEM -> registers (thread = accumulator row) -> shared memory (the pipeline stages are idle once
        // tmem_full has fired) -> coalesced global epilogue (lane = output column).  Each warp only touches
        // its own 32 rows, so no cross-warp synchronisation is needed.
        // Main-loop duty: round every landed fp32 tile to TF32 with round-to-nearest (cvt.rna), in place.
        // tcgen05.mma kind::tf32 would otherwise just drop the 13 low mantissa bits (truncation: a
        // systematic -1e-3 relative bias per product); rounding makes the error zero-mean like cuBLAS TF32.
        {
            const int ct = threadIdx.x - 64;     // 0..127
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % TC_STAGES;
                const uint32_t ph = (kb / TC_STAGES) & 1;
                mbar_wait(&full_bar[s], ph);
                if (ct == 0 && kb == 0) tc_stamp(g, 2);                      // first tile landed
                if (ct == 0 && kb == nkb - 1) tc_stamp(g, 3);                // last tile landed
                float4* tile = reinterpret_cast<float4*>(smem + s * STAGE_BYTES);
#pragma unroll 4
                for (int i = ct; i < TILE_PAIR / 16; i += 128) {
                    float4 v = tile[i];
                    uint32_t x, y, z, w;
                    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(x) : "f"(v.x));
                    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(y) : "f"(v.y));
                    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(z) : "f"(v.z));
                    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(w) : "f"(v.w));
                    tile[i] = make_float4(__uint_as_float(x), __uint_as_float(y), __uint_as_float(z),
                                          __uint_as_float(w));
                    if (SPLIT) {       // residual, itself rounded to TF32 (same swizzled position in the lo buffer)
                        uint32_t a, b, c, d;
                        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(a) : "f"(v.x - __uint_as_float(x)));
                        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(b) : "f"(v.y - __uint_as_float(y)));
                        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(c) : "f"(v.z - __uint_as_float(z)));
                        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(d) : "f"(v.w - __uint_as_float(w)));
                        tile[i + TILE_PAIR / 16] = make_float4(__uint_as_float(a), __uint_as_float(b), __uint_as_float(c),
                                                               __uint_as_float(d));
                    }
                }
                // generic-proxy writes -> visible to the tensor core's async-proxy reads
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0)
                    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&conv_bar[s])) : "memory");
            }
            if (ct == 0) tc_stamp(g, 4);                                     // last tile rounded
        }
        const int q = warp % 4;                  // TMEM lane quarter this warp may access
        constexpr int DS = BN + 4;               // row pitch = 1 (mod 8) float4s: conflict-free float4 stores (thread = row)
                                                 // and float4 loads (lane = 4 columns)
        float* stage = reinterpret_cast<float*>(smem) + q * 32 * DS;
        if (nkb > 0) {
            mbar_wait(tmem_full, 0);
            tc_fence_after();
        }
        if (threadIdx.x == 64) tc_stamp(g, 5);                               // accumulator complete
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
            uint32_t v[32];
            if (nkb > 0) {
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                    : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                      "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
                      "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),
                      "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),
                      "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                    : "r"(taddr)
                    : "memory");
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = 0u;
            }
#pragma unroll
            for (int j = 0; j < 32; j += 4)
                *reinterpret_cast<float4*>(&stage[lane * DS + c0 + j]) =
                    make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                                __uint_as_float(v[j + 3]));
        }
        tc_fence_before();
        __syncwarp();
        if (threadIdx.x == 64) tc_stamp(g, 6);                               // TMEM drained to shared memory
        const int ncols = min(BN, g.N - n0);
        const GemmEpilogue& ep = g.ep;
        const unsigned long long seed = ep.seed + ((ep.drop_p > 0.f && ep.seed_off) ? *ep.seed_off : 0ull);
        constexpr int RB = 8;                    // rows in flight per thread: 8 independent global loads
        const int rbase = m0 + q * 32;
        if (g.ksplit > 1 && g.vec4) {
            // split-K: raw fp32 partials, coalesced float4 rows
            const int nrows = min(32, g.M - rbase);
            for (int c = lane * 4; c < ncols; c += 128)
                for (int r = 0; r < nrows; ++r)
                    *reinterpret_cast<float4*>(g.ws + ((long long)split * g.M + rbase + r) * g.N + n0 + c) =
                        *reinterpret_cast<const float4*>(&stage[r * DS + c]);
        } else if (g.vec4) {
            const bool drop = ep.drop_p > 0.f;
            if (ep.G) {     // gated backward GEMM (host guarantees act none, no residual / accumulate)
                if (ep.gate == ACT_RELU) {
                    if (drop) tc_epilogue_vec4<ACT_NONE, true, ACT_RELU>(g, stage, DS, lane, rbase, n0, ncols, seed);
                    else tc_epilogue_vec4<ACT_NONE, false, ACT_RELU>(g, stage, DS, lane, rbase, n0, ncols, seed);
                } else {
                    if (drop) tc_epilogue_vec4<ACT_NONE, true, ACT_SILU>(g, stage, DS, lane, rbase, n0, ncols, seed);
                    else tc_epilogue_vec4<ACT_NONE, false, ACT_SILU>(g, stage, DS, lane, rbase, n0, ncols, seed);
                }
            } else if (ep.act == ACT_NONE) {
                if (drop) tc_epilogue_vec4<ACT_NONE, true>(g, stage, DS, lane, rbase, n0, ncols, seed);
                else tc_epilogue_vec4<ACT_NONE, false>(g, stage, DS, lane, rbase, n0, ncols, seed);
            } else if (ep.act == ACT_RELU) {
                if (drop) tc_epilogue_vec4<ACT_RELU, true>(g, stage, DS, lane, rbase, n0, ncols, seed);
                else tc_epilogue_vec4<ACT_RELU, false>(g, stage, DS, lane, rbase, n0, ncols, seed);
            } else {
                if (drop) tc_epilogue_vec4<ACT_SILU, true>(g, stage, DS, lane, rbase, n0, ncols, seed);
                else tc_epilogue_vec4<ACT_SILU, false>(g, stage, DS, lane, rbase, n0, ncols, seed);
            }
        } else {
            for (int c = lane; c < ncols; c += 32) {
                const int n = n0 + c;
                const float bv = (g.ksplit == 1 && ep.bias) ? ep.bias[n] : 0.f;
#pragma unroll 1
                for (int r0 = 0; r0 < 32; r0 += RB) {
                    float acc[RB], rv[RB], cv[RB];
#pragma unroll
                    for (int i = 0; i < RB; ++i) {
                        const int row = rbase + r0 + i;
                        acc[i] = stage[(r0 + i) * DS + c];
                        const bool ok = row < g.M && g.ksplit == 1;
                        rv[i] = (ok && ep.R) ? ep.R[(long long)row * ep.ldr + n] : 0.f;
                        cv[i] = (ok && ep.accumulate) ? ep.C[(long long)row * ep.ldc + n] : 0.f;
                    }
#pragma unroll
                    for (int i = 0; i < RB; ++i) {
                        const int row = rbase + r0 + i;
                        if (row >= g.M) continue;
                        if (g.ksplit > 1) {
                            g.ws[((long long)split * g.M + row) * g.N + n] = acc[i];
                            continue;
                        }
                        float v = ep.alpha * acc[i] + bv;
                        if (ep.Z) ep.Z[(long long)row * ep.ldz + n] = v;
                        v = act_apply(ep.act, v);
                        if (ep.G) {
                            const float gv = ep.G[(long long)row * ep.ldg + n];
                            v = ep.gate == ACT_RELU ? (gv > 0.f ? v : 0.f) : v * act_grad(ep.gate, gv);
                        }
                        if (ep.drop_p > 0.f)
                            v *= dropout_scale(ep.drop_p, seed, (unsigned long long)row * g.N + n);
                        v = ep.R ? rv[i] + ep.rscale * v : ep.rscale * v;
                        ep.C[(long long)row * ep.ldc + n] = v + cv[i];
                    }
                }
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 64) tc_stamp(g, 7);                                   // all epilogue stores issued
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(tc_tmem_cols<BN>())
                     : "memory");
    }
}

template <int BN, bool A_MN, bool B_MN, bool SPLIT = false>
__global__ void __launch_bounds__(TC_THREADS) gemm_tc_kernel(const __grid_constant__ CUtensorMap mapA,
                                                             const __grid_constant__ CUtensorMap mapB, TcArgs g) {
    gemm_tc_body<BN, A_MN, B_MN, SPLIT>(mapA, mapB, g, blockIdx.x, blockIdx.y, blockIdx.z);
}

// Grouped launch: up to TC_GROUP_MAX independent split-K problems (the weight gradients of one encoder layer) in ONE grid,
// so their CTAs fill the GPU together instead of queueing behind one another on side streams.
constexpr int TC_GROUP_MAX = 6;
struct TcGroup {
    CUtensorMap mapA[TC_GROUP_MAX], mapB[TC_GROUP_MAX];
    TcArgs g[TC_GROUP_MAX];
    int first[TC_GROUP_MAX + 1];      // CTA index range of each problem
    int tn[TC_GROUP_MAX], tm[TC_GROUP_MAX];
    int n;
};
template <int BN>
__global__ void __launch_bounds__(TC_THREADS) gemm_tc_group_kernel(const __grid_constant__ TcGroup G) {
    int p = 0;
    while (p + 1 < G.n && (int)blockIdx.x >= G.first[p + 1]) ++p;
    const int local = blockIdx.x - G.first[p];
    const int bx = local % G.tn[p], by = (local / G.tn[p]) % G.tm[p], bz = local / (G.tn[p] * G.tm[p]);
    gemm_tc_body<BN, true, true, false>(G.mapA[p], G.mapB[p], G.g[p], bx, by, bz);
}
__global__ void tc_splitk_reduce_group_kernel(const __grid_constant__ TcGroup G) {
    const TcArgs& g = G.g[blockIdx.y];
    if (g.ksplit <= 1) return;          // that problem's CTAs wrote the final values themselves
    const long long total = (long long)g.M * g.N;
    if (g.vec4) {       // float4 columns, eight split partials in flight per thread; the sum stays in split order (deterministic)
        const float4* w4 = reinterpret_cast<const float4*>(g.ws);
        const long long total4 = total / 4;
        const int n4 = g.N / 4;
        for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total4; e += (long long)gridDim.x * blockDim.x) {
            float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int k0 = 0; k0 < g.ksplit; k0 += 8) {
                float4 v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    v[j] = k0 + j < g.ksplit ? w4[(long long)(k0 + j) * total4 + e] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int j = 0; j < 8; ++j) { s.x += v[j].x; s.y += v[j].y; s.z += v[j].z; s.w += v[j].w; }
            }
            const int m = (int)(e / n4), n = (int)(e % n4) * 4;
            *reinterpret_cast<float4*>(g.ep.C + (long long)m * g.ep.ldc + n) = s;
        }
        return;
    }
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int n = (int)(e % g.N);
        const int m = (int)(e / g.N);
        float s = 0.f;
        for (int k = 0; k < g.ksplit; ++k) s += g.ws[(long long)k * total + e];
        g.ep.C[(long long)m * g.ep.ldc + n] = s;
    }
}

// ---------------------------------------------------------------------------------------------------------
// Persistent variant for split (3xTF32) GEMMs with a K-major A and ksplit == 1: one CTA per SM walks a static list of
// output tiles.  The shared-memory ring runs continuously across tile boundaries and the accumulator is double-buffered
// in TMEM, so the epilogue of tile i (TMEM -> smem -> global) overlaps the TMA / convert / MMA work of tile i+1, and the
// fixed per-CTA costs (barrier init, TMEM allocation, tensor-map fetch) are paid once per SM instead of once per tile.
//   warp 0: TMA producer | warp 1: MMA issuer | warps 2-5: TF32 round-to-nearest converters |
//   warps 6-13: epilogue (two warps per 32-lane TMEM quarter, each taking half of the tile's columns)
// ---------------------------------------------------------------------------------------------------------
constexpr int TCP_EPI_WARPS = 8, TCP_THREADS = (6 + TCP_EPI_WARPS) * 32;
// ring depth: as many stages as fit beside the epilogue staging tile; every stage carries a hi and a lo copy
template <int BN> __host__ __device__ constexpr int tcp_stages() { return BN <= 32 ? 4 : (BN <= 64 ? 3 : 2); }
template <int BN> __host__ __device__ constexpr int tcp_smem_bytes() {
    return tcp_stages<BN>() * 2 * (TC_BM * TC_BK * 4 + BN * TC_BK * 4) + TC_BM * (BN + 4) * 4 + 1024 + 256;
}

template <int BN, bool B_MN>
__global__ void __launch_bounds__(TCP_THREADS, 1) gemm_tc_persistent_kernel(const __grid_constant__ CUtensorMap mapA,
                                                                            const __grid_constant__ CUtensorMap mapB,
                                                                            TcArgs g) {
    constexpr int A_BYTES = TC_BM * TC_BK * 4;
    constexpr int B_BYTES = BN * TC_BK * 4;
    constexpr int TILE_PAIR = A_BYTES + B_BYTES;               // what TMA lands per k-block
    constexpr int STAGE_BYTES = 2 * TILE_PAIR;                 // [A hi | B hi | A lo | B lo]
    constexpr int TCP_STAGES = tcp_stages<BN>();
    constexpr int DS = BN + 4;
    constexpr int TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;      // two accumulator buffers (power of two >= 32)
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    float* staging = reinterpret_cast<float*>(smem + TCP_STAGES * STAGE_BYTES);            // [128][DS]
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(staging + TC_BM * DS);
    uint64_t* empty_bar = full_bar + TCP_STAGES;
    uint64_t* conv_bar = empty_bar + TCP_STAGES;
    uint64_t* tmem_full = conv_bar + TCP_STAGES;       // [2]
    uint64_t* tmem_empty = tmem_full + 2;              // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const int ntn = (g.N + BN - 1) / BN, ntm = (g.M + TC_BM - 1) / TC_BM;
    const int ntiles = ntn * ntm;
    const int nkb = (g.K + TC_BK - 1) / TC_BK;
    pdl_trigger();

    if (threadIdx.x == 0) {
        for (int s = 0; s < TCP_STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
            mbar_init(&conv_bar[s], 4);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tmem_full[b], 1);
            mbar_init(&tmem_empty[b], TCP_EPI_WARPS);   // one arrival per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&mapA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&mapB) : "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "n"(TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();

    if (warp == 0) {
        if (lane == 0) {   // ---------------- TMA producer ----------------
            uint32_t it = 0;
            for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
                const int m0 = (t / ntn) * TC_BM, n0 = (t % ntn) * BN;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % TCP_STAGES;
                    const uint32_t ph = (it / TCP_STAGES) & 1;
                    mbar_wait(&empty_bar[s], ph ^ 1);
                    uint8_t* sa = smem + s * STAGE_BYTES;
                    uint8_t* sb = sa + A_BYTES;
                    mbar_expect_tx(&full_bar[s], TILE_PAIR);
                    const int k0 = kb * TC_BK;
                    tma_load_2d(sa, &mapA, &full_bar[s], k0, m0);
                    if (!B_MN) {
                        tma_load_2d(sb, &mapB, &full_bar[s], k0, n0);
                    } else {
#pragma unroll
                        for (int j = 0; j < BN / 32; ++j) tma_load_2d(sb + j * 4096, &mapB, &full_bar[s], n0 + 32 * j, k0);
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {   // ---------------- MMA issuer ----------------
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((B_MN ? 1u : 0u) << 16) |
                                   ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
            uint32_t it = 0, j = 0;
            for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++j) {
                const uint32_t buf = j & 1;
                mbar_wait(&tmem_empty[buf], ((j >> 1) & 1) ^ 1);     // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t tacc = tmem_base + buf * BN;
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % TCP_STAGES;
                    const uint32_t ph = (it / TCP_STAGES) & 1;
                    mbar_wait(&conv_bar[s], ph);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + s * STAGE_BYTES);
                    const uint32_t sb = sa + A_BYTES;
#pragma unroll
                    for (int k = 0; k < TC_BK / 8; ++k) {
                        const uint64_t ad = umma_desc<2>(sa + k * 32, 16, 1024);
                        const uint64_t bd = B_MN ? umma_desc<1>(sb + k * 1024, 4096, 512) : umma_desc<2>(sb + k * 32, 16, 1024);
                        tc_mma_tf32(tacc, ad, bd, idesc, (kb | k) != 0);
                        const uint32_t la = sa + TILE_PAIR, lb = sb + TILE_PAIR;       // residual (lo) copies
                        const uint64_t adl = umma_desc<2>(la + k * 32, 16, 1024);
                        const uint64_t bdl = B_MN ? umma_desc<1>(lb + k * 1024, 4096, 512) : umma_desc<2>(lb + k * 32, 16, 1024);
                        tc_mma_tf32(tacc, ad, bdl, idesc, 1u);
                        tc_mma_tf32(tacc, adl, bd, idesc, 1u);
                    }
                    tc_commit(&empty_bar[s]);
                }
                tc_commit(&tmem_full[buf]);
            }
        }
    } else if (warp < 6) {   // ---------------- converters (warps 2-5) ----------------
        const int ct = threadIdx.x - 64;
        uint32_t it = 0;
        for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int s = it % TCP_STAGES;
                const uint32_t ph = (it / TCP_STAGES) & 1;
                mbar_wait(&full_bar[s], ph);
                float4* tile = reinterpret_cast<float4*>(smem + s * STAGE_BYTES);
#pragma unroll 4
                for (int i = ct; i < TILE_PAIR / 16; i += 128) {
                    float4 v = tile[i];
                    uint32_t x, y, z, w;
                    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(x) : "f"(v.x));
                    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(y) : "f"(v.y));
                    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(z) : "f"(v.z));
                    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(w) : "f"(v.w));
                    tile[i] = make_float4(__uint_as_float(x), __uint_as_float(y), __uint_as_float(z),
                                          __uint_as_float(w));
                    // residual, itself rounded to TF32 (same swizzled position in the lo copy)
                    uint32_t a, b, c, d;
                    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(a) : "f"(v.x - __uint_as_float(x)));
                    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(b) : "f"(v.y - __uint_as_float(y)));
                    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(c) : "f"(v.z - __uint_as_float(z)));
                    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(d) : "f"(v.w - __uint_as_float(w)));
                    tile[i + TILE_PAIR / 16] = make_float4(__uint_as_float(a), __uint_as_float(b), __uint_as_float(c),
                                                           __uint_as_float(d));
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0)
                    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&conv_bar[s])) : "memory");
            }
        }
    } else {                 // ---------------- epilogue (warps 6-9) ----------------
        const int q = warp % 4;                                  // TMEM lane quarter
        constexpr int HALF = BN >= 64 ? BN / 2 : BN;             // columns per epilogue warp
        const int cbase = (BN >= 64 && warp >= 10) ? HALF : 0;
        const bool idle = BN < 64 && warp >= 10;                 // 32-wide tiles: one warp per quarter is enough
        float* stage = staging + q * 32 * DS + cbase;
        const GemmEpilogue& ep = g.ep;
        const unsigned long long seed = ep.seed + ((ep.drop_p > 0.f && ep.seed_off) ? *ep.seed_off : 0ull);
        uint32_t j = 0;
        for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++j) {
            const int m0 = (t / ntn) * TC_BM, n0 = (t % ntn) * BN;
            const uint32_t buf = j & 1;
            mbar_wait(&tmem_full[buf], (j >> 1) & 1);
            tc_fence_after();
#pragma unroll 1
            for (int c0 = 0; c0 < (idle ? 0 : HALF); c0 += 32) {
                uint32_t v[32];
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + cbase + c0);
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                    : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                      "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
                      "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),
                      "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),
                      "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                    : "r"(taddr)
                    : "memory");
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int jj = 0; jj < 32; jj += 4)
                    *reinterpret_cast<float4*>(&stage[lane * DS + c0 + jj]) =
                        make_float4(__uint_as_float(v[jj]), __uint_as_float(v[jj + 1]), __uint_as_float(v[jj + 2]),
                                    __uint_as_float(v[jj + 3]));
            }
            // accumulator is now in shared memory: hand the TMEM buffer back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0)
                asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&tmem_empty[buf])) : "memory");
            const int nc0 = n0 + cbase;                                     // this warp's first output column
            const int ncols = idle ? 0 : max(0, min(HALF, g.N - nc0));
            const int rbase = m0 + q * 32;
            if (rbase < g.M && ncols > 0) {
                if (g.vec4) {
                    const bool drop = ep.drop_p > 0.f;
                    if (ep.G) {            // gated backward GEMM (host guarantees act none, no residual / accumulate)
                        if (ep.gate == ACT_RELU) {
                            if (drop) tc_epilogue_vec4<ACT_NONE, true, ACT_RELU>(g, stage, DS, lane, rbase, nc0, ncols, seed);
                            else tc_epilogue_vec4<ACT_NONE, false, ACT_RELU>(g, stage, DS, lane, rbase, nc0, ncols, seed);
                        } else {
                            if (drop) tc_epilogue_vec4<ACT_NONE, true, ACT_SILU>(g, stage, DS, lane, rbase, nc0, ncols, seed);
                            else tc_epilogue_vec4<ACT_NONE, false, ACT_SILU>(g, stage, DS, lane, rbase, nc0, ncols, seed);
                        }
                    } else if (ep.act == ACT_NONE) {
                        if (drop) tc_epilogue_vec4<ACT_NONE, true>(g, stage, DS, lane, rbase, nc0, ncols, seed);
                        else tc_epilogue_vec4<ACT_NONE, false>(g, stage, DS, lane, rbase, nc0, ncols, seed);
                    } else if (ep.act == ACT_RELU) {
                        if (drop) tc_epilogue_vec4<ACT_RELU, true>(g, stage, DS, lane, rbase, nc0, ncols, seed);
                        else tc_epilogue_vec4<ACT_RELU, false>(g, stage, DS, lane, rbase, nc0, ncols, seed);
                    } else {
                        if (drop) tc_epilogue_vec4<ACT_SILU, true>(g, stage, DS, lane, rbase, nc0, ncols, seed);
                        else tc_epilogue_vec4<ACT_SILU, false>(g, stage, DS, lane, rbase, nc0, ncols, seed);
                    }
                } else {
                    const int nrows = min(32, g.M - rbase);
                    for (int r = 0; r < nrows; ++r)
                        for (int c = lane; c < ncols; c += 32)
                            ep.store(0, rbase + r, nc0 + c, g.M, g.N, stage[r * DS + c]);
                }
            }
            __syncwarp();          // staging rows are rewritten by this warp for its next tile
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}

__global__ void tc_splitk_reduce_kernel(TcArgs g) {
    pdl_enter();
    const long long total = (long long)g.M * g.N;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        const int n = (int)(e % g.N);
        const int m = (int)(e / g.N);
        float s = 0.f;
        for (int k = 0; k < g.ksplit; ++k) s += g.ws[(long long)k * total + e];
        g.ep.store(0, m, n, g.M, g.N, s);
    }
}

// 2-D fp32 tensor map: `inner` contiguous elements per row, `outer` rows, row pitch ld floats.
static bool make_map(CUtensorMap* m, const float* base, long long inner, long long outer, long long ld, int box_inner,
                     int box_outer, CUtensorMapSwizzle swizzle) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

template <int BN, bool A_MN, bool B_MN, bool SPLIT = false>
static int launch_tc(const CUtensorMap& ma, const CUtensorMap& mb, const TcArgs& g, cudaStream_t st) {
    constexpr int smem = tc_smem_bytes<BN, SPLIT>();
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(gemm_tc_kernel<BN, A_MN, B_MN, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        configured = true;
    }
    dim3 grid(cdiv(g.N, BN), cdiv(g.M, TC_BM), g.ksplit);
    launch_kernel(gemm_tc_kernel<BN, A_MN, B_MN, SPLIT>, grid, TC_THREADS, smem, st, ma, mb, g);
    return 0;
}

template <int BN, bool B_MN>
static int launch_tc_persistent(const CUtensorMap& ma, const CUtensorMap& mb, const TcArgs& g, cudaStream_t st) {
    constexpr int smem = tcp_smem_bytes<BN>();
    static_assert(smem <= 232448, "persistent GEMM: shared memory");
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(gemm_tc_persistent_kernel<BN, B_MN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        configured = true;
    }
    static int num_sms = 0;
    if (!num_sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
        if (num_sms <= 0) num_sms = 148;
    }
    const int tiles = cdiv(g.N, BN) * cdiv(g.M, TC_BM);
    const int grid = tiles < num_sms ? tiles : num_sms;
    launch_kernel(gemm_tc_persistent_kernel<BN, B_MN>, grid, TCP_THREADS, smem, st, ma, mb, g);
    return 0;
}

}  // namespace gb200

using namespace gb200;

extern "C" int gb200_gemm_tc_supported(const float* A, int lda, const float* B, int ldb, int M, int N, int K) {
    if (M < 1 || N < 8 || K < 8) return 0;
    if (((uintptr_t)A % 16) || ((uintptr_t)B % 16) || (lda % 4) || (ldb % 4)) return 0;
    return encode_fn() != nullptr;
}

// widest N tile that still gives every SM a CTA (two co-reside per SM); narrow outputs get narrow tiles
static int pick_bn(int M, int N) {
    const long long mt = cdiv(M, TC_BM);
    if (N >= 192 && N % 192 == 0 && mt * cdiv(N, 128) > 2 * 148 && mt * (N / 192) <= 2 * 148)
        return 192;      // one resident wave instead of two (the Q|K|V projection at C3: 232 CTAs, not 348)
    if (N >= 128 && mt * cdiv(N, 128) >= 148) return 128;
    if (N >= 64 && mt * cdiv(N, 64) >= 148) return 64;
    if (N >= 128) return mt * cdiv(N, 32) >= 148 ? 32 : 128;   // tiny problems: fewer, fatter CTAs
    return N >= 64 ? 64 : 32;
}

extern "C" int gb200_gemm_tc_suggest_ksplit(int M, int N, int K) {
    const int bn = pick_bn(M, N);
    long long tiles = (long long)cdiv(M, TC_BM) * cdiv(N, bn);
    if (tiles >= 120 || K < 1024) return 1;
    int want = (int)((2 * 148 + tiles - 1) / tiles);
    int maxs = K / 256;                  // at least 256 of K per split
    int s = want < maxs ? want : maxs;
    return s < 1 ? 1 : (s > 64 ? 64 : s);
}

namespace gb200 {
static unsigned long long* g_tc_trace = nullptr;
extern "C" int gb200_gemm_tc_set_trace(unsigned long long* device_buffer) {
    g_tc_trace = device_buffer;
    return 0;
}

// gb200_gemm_tc and gb200_gemm_tc_gated: gate == nullptr is the plain GEMM
static int gemm_tc(int device, const float* A, int lda, int transA, const float* B, int ldb, int transB, float* C, int ldc,
                   int M, int N, int K, float alpha, const float* bias, int act, float* Zout, int ldz, float drop_p,
                   unsigned long long seed, const float* R, int ldr, float rscale, int accumulate, const float* gate, int ldg,
                   int gate_act, int ksplit, float* workspace, size_t workspace_bytes, int split, void* stream) {
    use_device(device);
    GB_REQUIRE(A && B && C, "gb200_gemm_tc: null operand");
    GB_REQUIRE(gb200_gemm_tc_supported(A, lda, B, ldb, M, N, K),
               "gb200_gemm_tc: unsupported shape/alignment (M=%d N=%d K=%d lda=%d ldb=%d); use gb200_gemm", M, N, K,
               lda, ldb);
    GB_REQUIRE(act == ACT_NONE || act == ACT_RELU || act == ACT_SILU, "gb200_gemm_tc: unknown activation %d", act);
    GB_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "gb200_gemm_tc: dropout p=%f outside [0,1)", drop_p);
    if (ksplit < 1) ksplit = 1;
    const bool a_mn = transA != 0;      // A stored [K, M]
    const bool b_mn = transB == 0;      // B stored [K, N]
    int bn = pick_bn(M, N);
    TcArgs g;
    g.ep.C = C; g.ep.ldc = ldc; g.ep.sC = 0; g.ep.alpha = alpha; g.ep.bias = bias; g.ep.act = act; g.ep.Z = Zout;
    g.ep.ldz = ldz; g.ep.drop_p = drop_p; g.ep.seed = seed; g.ep.seed_off = rng_offset_ptr(); g.trace = g_tc_trace; g.ep.R = R; g.ep.ldr = ldr; g.ep.rscale = rscale;
    g.ep.accumulate = accumulate;
    g.ep.G = gate; g.ep.ldg = ldg; g.ep.gate = gate_act;
    GB_REQUIRE(!gate || ((gate_act == ACT_RELU || gate_act == ACT_SILU) && act == ACT_NONE),
               "gb200_gemm_tc: bad gate (act %d)", gate_act);
    g.M = M; g.N = N; g.K = K; g.ksplit = ksplit;
    g.kchunk = cdiv(cdiv(K, TC_BK), ksplit) * TC_BK;
    g.ksplit = cdiv(K, g.kchunk);
    g.ws = workspace;
    auto al16 = [](const void* p) { return ((uintptr_t)p % 16) == 0; };
    g.vec4 = (N % 4 == 0) && al16(C) && (ldc % 4 == 0) && (!R || (al16(R) && ldr % 4 == 0)) &&
             (!Zout || (al16(Zout) && ldz % 4 == 0)) && (!bias || al16(bias)) && (!workspace || al16(workspace)) &&
             (!gate || (al16(gate) && ldg % 4 == 0 && !R && !accumulate));
    if (g.ksplit > 1)
        GB_REQUIRE(workspace && workspace_bytes >= (size_t)g.ksplit * M * N * sizeof(float),
                   "gb200_gemm_tc: split-K workspace too small");
    // split (3xTF32) tall-skinny problems -- the decoder's per-pixel linears, 1243 row tiles of a K <= 130 GEMM -- are bound by
    // per-tile latency (prologue, first TMA, epilogue) in the one-tile-per-CTA kernel: the persistent kernel keeps the ring
    // streaming across tiles and drains tile i while tile i+1 is loading.  For single-pass TF32 it measured equal or slower
    // in the full step, so only split problems take it.
    const bool persistent = split && !a_mn && g.ksplit == 1 && g.vec4 && (long long)cdiv(M, TC_BM) * cdiv(N, 128) >= 2 * 148;
    if (bn == 192 && split) bn = 128;
    if (split && !persistent && bn > 64 && (long long)cdiv(M, TC_BM) * cdiv(N, 64) >= 2 * 148) bn = 64;
    if (persistent) bn = N >= 128 ? 128 : (N >= 64 ? 64 : 32);
    CUtensorMap ma, mb;
    const CUtensorMapSwizzle SWK = CU_TENSOR_MAP_SWIZZLE_128B, SWMN = CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;
    bool ok = a_mn ? make_map(&ma, A, M, K, lda, 32, 32, SWMN) : make_map(&ma, A, K, M, lda, 32, TC_BM, SWK);
    ok = ok && (b_mn ? make_map(&mb, B, N, K, ldb, 32, 32, SWMN) : make_map(&mb, B, K, N, ldb, 32, bn, SWK));
    GB_REQUIRE(ok, "gb200_gemm_tc: cuTensorMapEncodeTiled failed (M=%d N=%d K=%d lda=%d ldb=%d)", M, N, K, lda, ldb);
    cudaStream_t st = as_stream(stream);
#define TC_LAYOUT(BNV, SPLITV)                                                             \
    do {                                                                                   \
        if (!a_mn && !b_mn) launch_tc<BNV, false, false, SPLITV>(ma, mb, g, st);          \
        else if (!a_mn && b_mn) launch_tc<BNV, false, true, SPLITV>(ma, mb, g, st);       \
        else if (a_mn && !b_mn) launch_tc<BNV, true, false, SPLITV>(ma, mb, g, st);       \
        else launch_tc<BNV, true, true, SPLITV>(ma, mb, g, st);                           \
    } while (0)
#define TC_PERSISTENT(BNV)                                                                 \
    do {                                                                                   \
        if (!b_mn) launch_tc_persistent<BNV, false>(ma, mb, g, st);                        \
        else launch_tc_persistent<BNV, true>(ma, mb, g, st);                               \
    } while (0)
    if (persistent) {
        if (bn == 128) TC_PERSISTENT(128);
        else if (bn == 64) TC_PERSISTENT(64);
        else TC_PERSISTENT(32);
    } else if (split) {
        if (bn == 128) TC_LAYOUT(128, true);
        else if (bn == 64) TC_LAYOUT(64, true);
        else TC_LAYOUT(32, true);
    } else if (bn == 192) TC_LAYOUT(192, false);
    else if (bn == 128) TC_LAYOUT(128, false);
    else if (bn == 64) TC_LAYOUT(64, false);
    else TC_LAYOUT(32, false);
#undef TC_PERSISTENT
#undef TC_LAYOUT
    if (g.ksplit > 1) {
        long long total = (long long)M * N;
        int blocks = (int)((total + 255) / 256);
        if (blocks > 148 * 8) blocks = 148 * 8;
        launch_kernel(tc_splitk_reduce_kernel, blocks, 256, 0, st, g);
    }
    return check_launch("gb200_gemm_tc", g.ksplit > 1 ? 2 : 1);
}
}  // namespace gb200

extern "C" int gb200_gemm_tc(int device, const float* A, int lda, int transA, const float* B, int ldb, int transB,
                             float* C, int ldc, int M, int N, int K, float alpha, const float* bias, int act,
                             float* Zout, int ldz, float drop_p, unsigned long long seed, const float* R, int ldr,
                             float rscale, int accumulate, int ksplit, float* workspace, size_t workspace_bytes,
                             int split, void* stream) {
    return gemm_tc(device, A, lda, transA, B, ldb, transB, C, ldc, M, N, K, alpha, bias, act, Zout, ldz, drop_p, seed, R,
                   ldr, rscale, accumulate, nullptr, 0, ACT_NONE, ksplit, workspace, workspace_bytes, split, stream);
}

extern "C" int gb200_gemm_tc_gated(int device, const float* A, int lda, int transA, const float* B, int ldb, int transB,
                                   float* C, int ldc, int M, int N, int K, float alpha, float drop_p,
                                   unsigned long long seed, float rscale, const float* gate, int ldg, int gate_act,
                                   int ksplit, float* workspace, size_t workspace_bytes, int split, void* stream) {
    return gemm_tc(device, A, lda, transA, B, ldb, transB, C, ldc, M, N, K, alpha, nullptr, ACT_NONE, nullptr, 0, drop_p,
                   seed, nullptr, 0, rscale, 0, gate, ldg, gate_act, ksplit, workspace, workspace_bytes, split, stream);
}

extern "C" size_t gb200_gemm_tc_wgrad_group_workspace_bytes(int n, const gb200_wgrad_problem* probs) {
    size_t total = 0;
    for (int i = 0; i < n; ++i) total += (size_t)64 * probs[i].M * probs[i].N * sizeof(float);   // upper bound: ksplit <= 64
    return total;
}

/* dW_i (M_i, N_i) = G_i^T X_i for i < n <= 4: the weight gradients of one layer (contractions over all T tokens) as ONE
 * tcgen05 TF32 split-K launch plus ONE fixed-order reduction (deterministic). */
extern "C" int gb200_gemm_tc_wgrad_group(int device, int n, const gb200_wgrad_problem* probs, float* workspace,
                                         size_t workspace_bytes, void* stream) {
    use_device(device);
    GB_REQUIRE(n >= 1 && n <= TC_GROUP_MAX && probs && workspace, "gb200_gemm_tc_wgrad_group: 1..%d problems", TC_GROUP_MAX);
    TcGroup G;
    memset(&G, 0, sizeof(G));
    G.n = n;
    int tiles = 0;
    for (int i = 0; i < n; ++i) {
        const gb200_wgrad_problem& q = probs[i];
        GB_REQUIRE(q.G && q.X && q.dW && q.T >= 1, "gb200_gemm_tc_wgrad_group: null operand in problem %d", i);
        GB_REQUIRE(gb200_gemm_tc_supported(q.G, q.ldg, q.X, q.ldx, q.M, q.N, (int)q.T) && q.N % 4 == 0 && q.ldw % 4 == 0 &&
                       ((uintptr_t)q.dW % 16) == 0,
                   "gb200_gemm_tc_wgrad_group: problem %d is not TMA / float4 aligned", i);
        tiles += cdiv(q.M, TC_BM) * cdiv(q.N, 128);
    }
    // Grid size: two CTAs per SM over the whole GPU.  A smaller grid that would fit on the 28 SMs the fused encoder kernels
    // leave free was measured (56 / 112 CTAs: 4.66 / 4.68 ms per C3 step against 4.61) -- filling the GPU wins.
    int S = 2 * 148 / tiles;
    if (S < 1) S = 1;
    if (S > 64) S = 64;
    size_t woff = 0;
    int cta = 0;
    const CUtensorMapSwizzle SWMN = CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;
    for (int i = 0; i < n; ++i) {
        const gb200_wgrad_problem& q = probs[i];
        TcArgs& g = G.g[i];
        const int K = (int)q.T;
        g.ep.C = q.dW; g.ep.ldc = q.ldw; g.ep.alpha = 1.f; g.ep.rscale = 1.f; g.ep.act = ACT_NONE;
        g.M = q.M; g.N = q.N; g.K = K;
        g.kchunk = cdiv(cdiv(K, TC_BK), S) * TC_BK;
        g.ksplit = cdiv(K, g.kchunk);
        g.ws = workspace + woff;
        g.vec4 = 1;
        woff += (size_t)g.ksplit * q.M * q.N;
        GB_REQUIRE(make_map(&G.mapA[i], q.G, q.M, K, q.ldg, 32, 32, SWMN) && make_map(&G.mapB[i], q.X, q.N, K, q.ldx, 32, 32, SWMN),
                   "gb200_gemm_tc_wgrad_group: cuTensorMapEncodeTiled failed (problem %d)", i);
        G.tn[i] = cdiv(q.N, 128);
        G.tm[i] = cdiv(q.M, TC_BM);
        G.first[i] = cta;
        cta += G.tn[i] * G.tm[i] * g.ksplit;
    }
    G.first[n] = cta;
    GB_REQUIRE(workspace_bytes >= woff * sizeof(float), "gb200_gemm_tc_wgrad_group: workspace too small");
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(gemm_tc_group_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem_bytes<128>());
        configured = true;
    }
    cudaStream_t st = as_stream(stream);
    gemm_tc_group_kernel<128><<<cta, TC_THREADS, tc_smem_bytes<128>(), st>>>(G);
    tc_splitk_reduce_group_kernel<<<dim3(64, n), 256, 0, st>>>(G);
    return check_launch("gb200_gemm_tc_wgrad_group", 2);
}
