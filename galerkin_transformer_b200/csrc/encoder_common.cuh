// Building blocks of the fused encoder-layer kernels (encoder_fwd.cu / encoder_bwd.cu), sm_100a.
//
// Arithmetic: every GEMM of these kernels is an error-compensated bf16 split on the 5th-generation tensor cores
//     a = a_hi + a_lo (two bf16),   a.b ~= a_hi.b_hi + a_hi.b_lo + a_lo.b_hi      (fp32 accumulate in TMEM)
// i.e. three `tcgen05.mma.kind::f16` products per logical product.  hi + lo carries 16-17 significand bits, the dropped
// lo.lo term is 2^-18 relative: ~30x tighter than single-pass TF32 at 1.5x its tensor time (the "bf16x3" mode,
// DESIGN.md section 3).
//
// Operand tiles are K-major SWIZZLE_128B images: a "chunk" holds 64 consecutive K elements of every row,
//     element (r, k) at byte   r * 128 + (((k >> 3) ^ (r & 7)) << 4) + (k & 7) * 2        (rows of 128 B, 16-byte units)
// which is exactly what TMA's CU_TENSOR_MAP_SWIZZLE_128B produces and what the UMMA shared-memory descriptor
// (layout 2, SBO = 1024) reads.  Weight tiles are written in this image ONCE per step by enc_pack_kernel and
// streamed with 1-D bulk TMA copies; activation tiles arrive as fp32 through tensor-map TMA and are split in place.
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"
#include "tc_prims.cuh"

namespace gb200 {
namespace enc {

constexpr int TM = 128;                 // tokens per CTA tile (= UMMA M)
constexpr int TILE_BYTES = 16384;       // 128 rows x 64 bf16
constexpr int NWORK = 8;                // worker warps (fp32 -> bf16 split, epilogues)
constexpr int THREADS = (2 + NWORK) * 32;
constexpr int STAGE_PITCH = 36;         // floats per row of a warp's 32 x 32 staging block (conflict-free float4)
constexpr int STAGE_BYTES = 32 * STAGE_PITCH * 4;

// ---- PTX wrappers not in tc_prims.cuh ---------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// 1-D bulk copy global -> shared (bytes % 16 == 0, 16-byte aligned), completion on an mbarrier
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// instruction descriptor: D = f32, A = B = bf16, both K-major, M = 128, N = n
__device__ __forceinline__ uint32_t idesc_bf16(int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
}
__device__ __forceinline__ uint64_t kdesc(uint32_t smem_addr) { return umma_desc<2>(smem_addr, 16, 1024); }
// MN-major operand (contraction over the ROWS of a chunk image: rows = K index, 128-byte rows = 64 MN elements):
// 8-row groups 1024 B apart (SBO), 64-wide MN blocks `lbo` bytes apart; one k-step = 16 rows = 2048 B.  The byte image
// is the same as a K-major chunk, so one tile can feed both kinds of contraction.
__device__ __forceinline__ uint64_t mndesc(uint32_t smem_addr, uint32_t lbo) { return umma_desc<2>(smem_addr, lbo, 1024); }
__device__ __forceinline__ uint32_t idesc_bf16_mn(int n) { return idesc_bf16(n) | (1u << 15) | (1u << 16); }
// three products of one k-step, both operands MN-major
__device__ __forceinline__ void mma3_mn(uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t lbo_a, uint32_t b_hi, uint32_t b_lo,
                                        uint32_t lbo_b, uint32_t idesc, bool first) {
    tc_mma_bf16(d, mndesc(a_hi, lbo_a), mndesc(b_hi, lbo_b), idesc, first ? 0u : 1u);
    tc_mma_bf16(d, mndesc(a_hi, lbo_a), mndesc(b_lo, lbo_b), idesc, 1u);
    tc_mma_bf16(d, mndesc(a_lo, lbo_a), mndesc(b_hi, lbo_b), idesc, 1u);
}

// the three products of one 16-wide k-step (a_* / b_* are shared-memory byte addresses of the k-step)
__device__ __forceinline__ void mma3(uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo,
                                     uint32_t idesc, bool first) {
    tc_mma_bf16(d, kdesc(a_hi), kdesc(b_hi), idesc, first ? 0u : 1u);
    tc_mma_bf16(d, kdesc(a_hi), kdesc(b_lo), idesc, 1u);
    tc_mma_bf16(d, kdesc(a_lo), kdesc(b_hi), idesc, 1u);
}
// one streamed weight tile (the hi or the lo image of a [128 x 64] block) against the A chunk (a_hi, a_lo):
// hi image -> a_hi.b_hi + a_lo.b_hi, lo image -> a_hi.b_lo
__device__ __forceinline__ void mma_weight_tile(uint32_t d, uint32_t a_hi, uint32_t a_lo, uint32_t b, bool b_is_hi,
                                                uint32_t idesc, bool first) {
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        if (b_is_hi) {
            tc_mma_bf16(d, kdesc(a_hi + ks * 32), kdesc(b + ks * 32), idesc, (first && ks == 0) ? 0u : 1u);
            tc_mma_bf16(d, kdesc(a_lo + ks * 32), kdesc(b + ks * 32), idesc, 1u);
        } else {
            tc_mma_bf16(d, kdesc(a_hi + ks * 32), kdesc(b + ks * 32), idesc, 1u);
        }
    }
}

// ---- TMEM -> registers ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
}
__device__ __forceinline__ void tmem_ld2(uint32_t taddr, float& a, float& b) {
    uint32_t r0, r1;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    a = __uint_as_float(r0);
    b = __uint_as_float(r1);
}

// ---- bf16 split helpers -------------------------------------------------------------------------------------------
__device__ __forceinline__ void split2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);           // .x = x0 (low half), .y = x1
    const float2 hf = __bfloat1622float2(h);
    const __nv_bfloat162 l = __floats2bfloat162_rn(x0 - hf.x, x1 - hf.y);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ void split1(float x, unsigned short& hi, unsigned short& lo) {
    const __nv_bfloat16 h = __float2bfloat16_rn(x);
    const __nv_bfloat16 l = __float2bfloat16_rn(x - __bfloat162float(h));
    hi = *reinterpret_cast<const unsigned short*>(&h);
    lo = *reinterpret_cast<const unsigned short*>(&l);
}
// byte offset of 16-byte unit u (0..7) of row r inside a chunk image
__device__ __forceinline__ uint32_t unit_off(int r, int u) { return (uint32_t)(r * 128 + ((u ^ (r & 7)) << 4)); }

// eight consecutive K elements of row r -> unit u of the hi and lo chunk images
__device__ __forceinline__ void store_unit(uint8_t* chunk_hi, uint8_t* chunk_lo, int r, int u, const float* x8) {
    uint4 h, l;
    split2(x8[0], x8[1], h.x, l.x);
    split2(x8[2], x8[3], h.y, l.y);
    split2(x8[4], x8[5], h.z, l.z);
    split2(x8[6], x8[7], h.w, l.w);
    const uint32_t off = unit_off(r, u);
    *reinterpret_cast<uint4*>(chunk_hi + off) = h;
    *reinterpret_cast<uint4*>(chunk_lo + off) = l;
}

// A 128 x 128 fp32 tile landed by TMA as four [128 x 32] SWIZZLE_128B blocks of 16 KB (block j = columns 32j..32j+31)
// is split IN PLACE: blocks (2kc, 2kc+1) become the (hi, lo) bf16 chunk images of K chunk kc.  One thread owns one
// (row, kc): it reads its 64 floats, then overwrites the same two 128-byte rows -- no cross-thread hazard.
__device__ __forceinline__ void split_tile_inplace(uint8_t* tile, int r, int kc) {
    uint8_t* ba = tile + (2 * kc) * TILE_BYTES;
    uint8_t* bb = ba + TILE_BYTES;
    float4 v[16];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        v[c] = *reinterpret_cast<const float4*>(ba + unit_off(r, c));
        v[8 + c] = *reinterpret_cast<const float4*>(bb + unit_off(r, c));
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        uint4 h, l;
        split2(v[2 * u].x, v[2 * u].y, h.x, l.x);
        split2(v[2 * u].z, v[2 * u].w, h.y, l.y);
        split2(v[2 * u + 1].x, v[2 * u + 1].y, h.z, l.z);
        split2(v[2 * u + 1].z, v[2 * u + 1].w, h.w, l.w);
        *reinterpret_cast<uint4*>(ba + unit_off(r, u)) = h;
        *reinterpret_cast<uint4*>(bb + unit_off(r, u)) = l;
    }
}

// ---- coalesced 32 x 32 fp32 block traffic through a per-warp staging block ------------------------------------------
// thread `lane` owns row `lane` (32 values in registers); global rows are written / read as 128-byte segments
__device__ __forceinline__ void warp_store_block(float* stage, const float (&v)[32], int lane, float* g, long long ld,
                                                 int nrows) {
#pragma unroll
    for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<float4*>(&stage[lane * STAGE_PITCH + j]) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    __syncwarp();
    const int rr = lane >> 3, c4 = (lane & 7) * 4;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int r = it * 4 + rr;
        if (r < nrows)
            *reinterpret_cast<float4*>(g + (long long)r * ld + c4) =
                *reinterpret_cast<const float4*>(&stage[r * STAGE_PITCH + c4]);
    }
    __syncwarp();
}
// [32 x 34] block (one head of the head-merged attention output, 136-byte row segments): lanes take consecutive float2
// of the staged block, so one store instruction covers ~2 rows instead of 32 scattered words
__device__ __forceinline__ void warp_store_rows34(float* stage, const float (&v)[32], float e0, float e1, int lane,
                                                  float* g, long long ld, int nrows, int width) {
#pragma unroll
    for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<float4*>(&stage[lane * STAGE_PITCH + j]) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    *reinterpret_cast<float2*>(&stage[lane * STAGE_PITCH + 32]) = make_float2(e0, e1);
    __syncwarp();
    if ((width & 1) == 0) {
        const int w2 = width >> 1;
        for (int f = lane; f < 32 * w2; f += 32) {
            const int r = f / w2, c = (f - r * w2) * 2;
            if (r < nrows)
                *reinterpret_cast<float2*>(g + (long long)r * ld + c) = *reinterpret_cast<const float2*>(&stage[r * STAGE_PITCH + c]);
        }
    } else {
        for (int f = lane; f < 32 * width; f += 32) {
            const int r = f / width, c = f - r * width;
            if (r < nrows) g[(long long)r * ld + c] = stage[r * STAGE_PITCH + c];
        }
    }
    __syncwarp();
}
__device__ __forceinline__ void warp_load_block(float* stage, float (&v)[32], int lane, const float* g, long long ld,
                                                int nrows) {
    const int rr = lane >> 3, c4 = (lane & 7) * 4;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int r = it * 4 + rr;
        float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < nrows) t = *reinterpret_cast<const float4*>(g + (long long)r * ld + c4);
        *reinterpret_cast<float4*>(&stage[r * STAGE_PITCH + c4]) = t;
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
        const float4 t = *reinterpret_cast<const float4*>(&stage[lane * STAGE_PITCH + j]);
        v[j] = t.x; v[j + 1] = t.y; v[j + 2] = t.z; v[j + 3] = t.w;
    }
    __syncwarp();
}

// fused dropout over 32 consecutive elements of one row (first flat element index idx0, idx0 % 8 == 0): same Philox
// stream as the unfused GEMM epilogues, so a fused forward and an unfused backward agree on the mask
__device__ __forceinline__ void dropout32(float (&v)[32], float p, unsigned long long seed, unsigned long long idx0) {
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
        float ds[8];
        dropout_scale8(p, seed, idx0 + j, ds);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[j + i] *= ds[i];
    }
}

__device__ __forceinline__ void worker_bar() { asm volatile("bar.sync 1, %0;" ::"n"(NWORK * 32) : "memory"); }

// ---- diagnostics: per-CTA clock stamps (gb200_encoder_set_trace); 32 slots per CTA, slot 31 = globaltimer at entry ----
static __device__ unsigned long long* g_enc_trace = nullptr;    // one copy per translation unit
__device__ __forceinline__ void trace(int slot) {
    if (g_enc_trace) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%clock64;" : "=l"(t));
        g_enc_trace[(size_t)blockIdx.x * 32 + slot] = t;
    }
}
__device__ __forceinline__ void trace_entry() {
    if (g_enc_trace) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        g_enc_trace[(size_t)blockIdx.x * 32 + 31] = t;
    }
}
// 1024-aligned dynamic shared memory base that keeps the shared address space visible to the compiler (LDS / STS)
__device__ __forceinline__ uint8_t* smem_base(uint8_t* raw) { return raw + ((1024u - (smem_u32(raw) & 1023u)) & 1023u); }

// ---- one-time CTA setup shared by every kernel: barriers, TMEM allocation --------------------------------------
__device__ __forceinline__ uint32_t tmem_alloc_512(uint32_t* slot, int warp) {
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    return *slot;
}
__device__ __forceinline__ void tmem_free_512(uint32_t base, int warp) {
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(base) : "memory");
    }
}

// ---- programmatic dependent launch for the fused kernel chain ------------------------------------------------------------------
// Every fused kernel calls grid_dep_sync() once its barriers and TMEM are set up: `launch_dependents` lets the NEXT kernel of
// the stream start its CTAs as SMs free up (its own setup then overlaps this kernel's tail instead of following it) and
// `wait` blocks until the PREVIOUS kernel has completed and flushed.  Measured 4.99 -> 4.78 ms per C3 step.
__device__ __forceinline__ void grid_dep_sync() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}
template <typename... KArgs, typename... Args>
static inline void launch_enc(void (*kernel)(KArgs...), int grid, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- layer geometry (BASELINE config 3) and the packed-parameter layout shared by forward and backward ----------
constexpr int DM = 128, NH = 4, DK = 32, DFF = 256, HP = 48;     // HP: padded head width of the fc operand (>= DK + 2)
constexpr int VEC_BQKV = 0, VEC_GK = 384, VEC_BK = 512, VEC_GV = 640, VEC_BV = 768, VEC_BFC = 896, VEC_B1 = 1024,
              VEC_B2 = 1280, VEC_FLOATS = 1408;
// forward tile stream (tiles of TILE_BYTES): W_qkv 12 | W_fc' 6 | W1 8 | W2 8
constexpr int TS_QKV = 0, TS_FC = 12, TS_W1 = 18, TS_W2 = 26;
// backward stream: W2^T 8 | W1^T 8 | W_fc'^T 8 | W_qkv^T 12
constexpr int TS_W2T = 34, TS_W1T = 42, TS_FCT = 50, TS_QKVT = 58;

struct Bars {
    uint64_t xfull, xconv, full[6], empty[6], dfull[4], hand[4], done;
    uint32_t tmem_slot;
};

// ---- tile-partial reduction through shared memory -------------------------------------------------------------------
// The per-sample attention-shaped matrices (4 x d x d) are summed over the sample's tiles in TILE ORDER (deterministic).
// One producer lane streams the 15 x 18.5 KB of partials through a 3-slot ring with 1-D bulk copies
// (Bars::full/empty[3..5]) and the workers add slot after slot from shared memory -- no registers tied up in flight.
// The step is L2-bandwidth bound: all 120 CTAs pull their sample's partials at once (33 MB per kernel, ~9 us either way).
// Summing once per sample instead (the tile CTA that finishes last, ticket counter) was built and measured: its serial
// tail on the previous kernel costs more than the 15-fold traffic it saves (3.89 vs 3.82 ms per C3 step); so was a
// cluster-of-15 DSMEM reduction (only 7 such clusters fit the GPU at one CTA per SM, tools/probes/cluster_probe.cu).
constexpr int PART_SLOTS = 3;
constexpr int PART_SLOT_BYTES = 18560;                       // >= 4 * 34 * 34 * 4, multiple of 128

__device__ __forceinline__ void partials_init(Bars* bar) {   // by the thread that initialises the other barriers
    for (int s = 0; s < PART_SLOTS; ++s) { mbar_init(&bar->full[3 + s], 1); mbar_init(&bar->empty[3 + s], NWORK); }
}
__device__ __forceinline__ void partials_produce(Bars* bar, uint8_t* pbuf, const float* pb, int tiles, int ne) {
    const uint32_t bytes = (uint32_t)ne * 4u;
    for (int k = 0; k < tiles; ++k) {
        const int s = k % PART_SLOTS;
        mbar_wait(&bar->empty[3 + s], ((k / PART_SLOTS) & 1) ^ 1);
        mbar_expect_tx(&bar->full[3 + s], bytes);
        bulk_load(pbuf + s * PART_SLOT_BYTES, pb + (long long)k * ne, bytes, &bar->full[3 + s]);
    }
    // the ring memory is reused afterwards: wait until the workers have read the last fill of every slot
    for (int s = 0; s < PART_SLOTS && s < tiles; ++s) {
        const int uses = (tiles - s + PART_SLOTS - 1) / PART_SLOTS;
        mbar_wait(&bar->empty[3 + s], (uses - 1) & 1);
    }
}
template <int EPT>
__device__ __forceinline__ void partials_consume(Bars* bar, const uint8_t* pbuf, int tiles, int ne, int wt, int lane,
                                                 float (&acc)[EPT]) {
#pragma unroll
    for (int i = 0; i < EPT; ++i) acc[i] = 0.f;
    for (int k = 0; k < tiles; ++k) {
        const int s = k % PART_SLOTS;
        mbar_wait(&bar->full[3 + s], (k / PART_SLOTS) & 1);
        const float* pslot = reinterpret_cast<const float*>(pbuf + s * PART_SLOT_BYTES);
#pragma unroll
        for (int i = 0; i < EPT; ++i) {
            const int e = wt + i * NWORK * 32;
            if (e < ne) acc[i] += pslot[e];
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar->empty[3 + s]);
    }
}

static inline bool make_tile_map(CUtensorMap* m, const float* base, int ld, int n, int B) {
    cuuint64_t dims[3] = {(cuuint64_t)ld, (cuuint64_t)n, (cuuint64_t)B};
    cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)ld * 4 * (cuuint64_t)n};
    cuuint32_t box[3] = {32, (cuuint32_t)TM, 1};
    return make_map_nd(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <typename K>
static inline void set_smem(K kernel, int bytes) {
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}


}  // namespace enc
}  // namespace gb200
