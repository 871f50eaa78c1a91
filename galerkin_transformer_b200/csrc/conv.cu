// 3x3 convolution blocks of the interpolation scalers (SURVEY 8f row 1; reference: Conv2dResBlock libs/layers.py:88-150,
// used by Interp2dEncoder :431-512 and Interp2dUpsample :624-670):   y = act( dropout( conv3x3(x) ) ),  no bias, stride 1,
// padding 1, channel-last (B, H, W, C) fp32.
//
//   conv3x3_tc_kernel   implicit GEMM on tcgen05, bf16x3 (encoder_common.cuh): CTA = an 8 x 16 patch of output pixels
//                       (UMMA M = 128) x all output channels; the nine taps are nine SHIFTED 4-D TMA tile loads of the
//                       (hi, lo) bf16 images of the input -- out-of-image coordinates are zero-filled by TMA, which IS the
//                       padding -- against the matching [C_out x 64] weight tiles streamed with bulk copies.
//                       The same kernel computes the input gradient (weights transposed + flipped by the pack kernel).
//   conv_split_kernel   fp32 channel-last -> (hi, lo) bf16 images padded to 64-channel chunks; in backward mode it first
//                       applies the activation / dropout derivative  g = dy * act'(.) * mask  and also keeps g in fp32.
//   conv1_* kernels     the single-input-channel first convolution (1 -> 128) as a streaming stencil (fwd / dgrad / wgrad).
// The weight gradient of the multi-channel blocks (a contraction over all pixels) stays a library call (cuDNN TF32).
#include <cuda.h>

#include "encoder_common.cuh"

namespace gb200 {
namespace enc {

__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[32]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
#pragma unroll
    for (int j = 16; j < 32; ++j) v[j] = 0.f;
}

constexpr int CV_RING = 3, CV_STAGE = 4 * TILE_BYTES;          // stage: A hi | A lo | W hi | W lo
constexpr int CV_SMEM = CV_RING * CV_STAGE + 512 + 1024;
constexpr int PATCH_W = 16, PATCH_H = 8;

struct ConvArgs {
    const uint8_t* wtiles;      // per (tap, 64-channel chunk): [W hi tile][W lo tile], tile = [128 rows (C_out, zero past it)][64 k]
    float* out;                 // (B, H, W, ldo) channel-last, channels [co0, co0 + Cout)
    float* zout;                // pre-activation (after dropout) for SiLU backward, same layout as out, or null
    const float* resid;         // added to the accumulator (gradient accumulation of the input-gradient pass) or null
    int ldo, co0, ldr, r0;
    int Cout, N;                // N = Cout rounded up to 48 / 128
    int nchunk;                 // input channel chunks of 64
    int act;                    // ACT_NONE / ACT_RELU / ACT_SILU applied after dropout
    float p;
    unsigned long long seed;
    const unsigned long long* seed_off;
    int B, H, W, tiles_x, tiles_y;
};

struct ConvBars {
    uint64_t full[CV_RING], empty[CV_RING], dfull;
    uint32_t tmem_slot;
};

__global__ void __launch_bounds__(THREADS, 1) conv3x3_tc_kernel(const __grid_constant__ CUtensorMap mapHi,
                                                                const __grid_constant__ CUtensorMap mapLo, ConvArgs a) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_base(smem_raw);
    uint8_t* ring = smem;
    ConvBars* bar = reinterpret_cast<ConvBars*>(ring + CV_RING * CV_STAGE);
    float* staging = reinterpret_cast<float*>(ring);           // epilogue only

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tx_ = blockIdx.x % a.tiles_x, ty_ = (blockIdx.x / a.tiles_x) % a.tiles_y, b = blockIdx.x / (a.tiles_x * a.tiles_y);
    const int x0 = tx_ * PATCH_W, y0 = ty_ * PATCH_H;
    const int nit = 9 * a.nchunk;

    if (threadIdx.x == 0) {
        for (int s = 0; s < CV_RING; ++s) { mbar_init(&bar->full[s], 1); mbar_init(&bar->empty[s], 1); }
        mbar_init(&bar->dfull, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&mapHi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&mapLo) : "memory");
    }
    const uint32_t tmem = tmem_alloc_512(&bar->tmem_slot, warp);

    if (warp == 0) {
        if (lane == 0) {
            for (int it = 0; it < nit; ++it) {
                const int s = it % CV_RING;
                const int tap = it / a.nchunk, ck = it - tap * a.nchunk;
                const int dy = tap / 3 - 1, dx = tap % 3 - 1;
                mbar_wait(&bar->empty[s], ((it / CV_RING) & 1) ^ 1);
                uint8_t* st = ring + s * CV_STAGE;
                mbar_expect_tx(&bar->full[s], CV_STAGE);
                tma_load_4d(st, &mapHi, &bar->full[s], ck * 64, x0 + dx, y0 + dy, b);
                tma_load_4d(st + TILE_BYTES, &mapLo, &bar->full[s], ck * 64, x0 + dx, y0 + dy, b);
                bulk_load(st + 2 * TILE_BYTES, a.wtiles + (size_t)(2 * it) * TILE_BYTES, 2 * TILE_BYTES, &bar->full[s]);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t rb = smem_u32(ring);
            const uint32_t idn = idesc_bf16(a.N);
            for (int it = 0; it < nit; ++it) {
                const int s = it % CV_RING;
                mbar_wait(&bar->full[s], (it / CV_RING) & 1);
                tc_fence_after();
                const uint32_t ah = rb + s * CV_STAGE, al = ah + TILE_BYTES, bh = ah + 2 * TILE_BYTES, bl = ah + 3 * TILE_BYTES;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
                    mma3(tmem, ah + ks * 32, al + ks * 32, bh + ks * 32, bl + ks * 32, idn, it == 0 && ks == 0);
                tc_commit(&bar->empty[s]);
            }
            tc_commit(&bar->dfull);
        }
    } else {
        const int w = warp - 2, q = warp & 3, hf = w >> 2;
        float* stage = staging + w * 32 * STAGE_PITCH;
        const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);
        const unsigned long long so = (a.p > 0.f && a.seed_off) ? *a.seed_off : 0ull;
        // this thread's accumulator row = patch pixel m; the rows it STORES after the staging transpose are r_st
        const int m = q * 32 + lane;
        const int gy = y0 + (m >> 4), gx = x0 + (m & 15);
        const long long px = ((long long)b * a.H + gy) * a.W + gx;
        mbar_wait(&bar->dfull, 0);
        tc_fence_after();
        const int nchunks = a.N == 128 ? 2 : 1;
        for (int cc = 0; cc < nchunks; ++cc) {
            int c0, wcols;
            if (a.N == 128) { c0 = hf * 64 + cc * 32; wcols = 32; }
            else { c0 = hf * 32; wcols = hf == 0 ? 32 : 16; }
            float v[32];
            if (wcols == 32) tmem_ld32(tlane + c0, v);
            else tmem_ld16(tlane + c0, v);
            const int ncols = max(0, min(wcols, a.Cout - c0));  // valid output channels in this chunk
            if (a.resid) {                                      // gradient accumulation: scattered but L2-resident
                const bool ok = gy < a.H && gx < a.W;
#pragma unroll 8
                for (int j = 0; j < 32; ++j)
                    if (ok && j < ncols) v[j] += a.resid[px * a.ldr + a.r0 + c0 + j];
            }
            if (a.p > 0.f) dropout32(v, a.p, a.seed + so, (unsigned long long)px * 128 + c0);
            // staged, row-wise stores: lane pairs a row with 16 float2 columns
            auto store_rows = [&](float* dst_base) {
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4*>(&stage[lane * STAGE_PITCH + j]) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                __syncwarp();
#pragma unroll
                for (int it = 0; it < 16; ++it) {
                    const int r = it * 2 + (lane >> 4), c = (lane & 15) * 2;
                    const int mm = q * 32 + r;
                    const int yy = y0 + (mm >> 4), xx = x0 + (mm & 15);
                    if (yy < a.H && xx < a.W && c < ncols) {
                        float* dp = dst_base + (((long long)b * a.H + yy) * a.W + xx) * a.ldo + a.co0 + c0 + c;
                        const float2 t = *reinterpret_cast<const float2*>(&stage[r * STAGE_PITCH + c]);
                        if (c + 1 < ncols) *reinterpret_cast<float2*>(dp) = t;
                        else dp[0] = t.x;
                    }
                }
                __syncwarp();
            };
            if (a.zout) store_rows(a.zout);
            if (a.act == ACT_RELU) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
            } else if (a.act == ACT_SILU) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = __fdividef(v[j], 1.f + __expf(-v[j]));
            }
            store_rows(a.out);
        }
        tc_fence_before();
    }
    tmem_free_512(tmem, warp);
}

// ---------------------------------------------------------------------------------------------------------------
// fp32 -> (hi, lo) bf16 images, channel-padded; optional activation / dropout backward first
// ---------------------------------------------------------------------------------------------------------------
struct SplitArgs {
    const float* x;             // (npix, ldx) channels [c0, c0 + C)
    int ldx, c0, C, CP;
    long long npix;
    __nv_bfloat16* hi;          // (npix, CP)
    __nv_bfloat16* lo;
    // backward mode (yz != null): x is dy; g = dy * act'(yz) * mask
    const float* yz;            // forward output y (ReLU) or pre-activation u = mask * conv (SiLU), (npix, ldyz) at yz_c0
    int ldyz, yz_c0, act;
    float p;
    unsigned long long seed;
    const unsigned long long* seed_off;
    float* gout;                // (npix, C) fp32 or null
};

__global__ void __launch_bounds__(256) conv_split_kernel(SplitArgs a) {
    const int upr = a.CP >> 3;                                  // 16-byte units per pixel
    const long long total = a.npix * upr;
    const unsigned long long so = (a.p > 0.f && a.seed_off) ? *a.seed_off : 0ull;
    const float keep = a.p > 0.f ? dropout_keep_scale(dropout_threshold(a.p)) : 1.f;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long px = e / upr;
        const int u = (int)(e - px * upr);
        float v[8];
        float ds[8];
        if (a.yz && a.act == ACT_SILU && a.p > 0.f) dropout_scale8(a.p, a.seed + so, (unsigned long long)px * 128 + 8 * u, ds);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int c = 8 * u + i;
            float t = c < a.C ? a.x[px * a.ldx + a.c0 + c] : 0.f;
            if (a.yz && c < a.C) {
                const float s = a.yz[px * a.ldyz + a.yz_c0 + c];
                if (a.act == ACT_RELU) t = s > 0.f ? t * keep : 0.f;             // y > 0  <=>  kept and conv > 0
                else if (a.act == ACT_SILU) t *= act_grad(ACT_SILU, s) * (a.p > 0.f ? ds[i] : 1.f);
                else if (a.p > 0.f) t *= dropout_scale(a.p, a.seed + so, (unsigned long long)px * 128 + c);
                if (a.gout) a.gout[px * a.C + c] = t;
            }
            v[i] = t;
        }
        uint4 h, l;
        split2(v[0], v[1], h.x, l.x);
        split2(v[2], v[3], h.y, l.y);
        split2(v[4], v[5], h.z, l.z);
        split2(v[6], v[7], h.w, l.w);
        *reinterpret_cast<uint4*>(a.hi + px * a.CP + 8 * u) = h;
        *reinterpret_cast<uint4*>(a.lo + px * a.CP + 8 * u) = l;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// weight packing for the implicit GEMM: tile (tap, chunk) = [128 rows][64 k] (hi, lo), zero padded
//   forward : T[r = co][k = ci] = W[co][ci][tap]
//   dgrad   : T[r = ci][k = co] = W[co][ci][8 - tap]
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) conv_pack_kernel(const float* __restrict__ w, int Cout, int Cin, int nchunk, int dgrad,
                                                        uint8_t* __restrict__ tiles) {
    const int tap = blockIdx.x / nchunk, ck = blockIdx.x % nchunk;
    uint8_t* hi = tiles + (size_t)blockIdx.x * 2 * TILE_BYTES;
    uint8_t* lo = hi + TILE_BYTES;
    for (int e = threadIdx.x; e < 128 * 8; e += blockDim.x) {
        const int r = e >> 3, u = e & 7;
        float x8[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int k = ck * 64 + u * 8 + i;
            float val = 0.f;
            if (!dgrad) {
                if (r < Cout && k < Cin) val = w[((long long)r * Cin + k) * 9 + tap];
            } else {
                if (r < Cin && k < Cout) val = w[((long long)k * Cin + r) * 9 + (8 - tap)];
            }
            x8[i] = val;
        }
        store_unit(hi, lo, r, u, x8);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// 1 -> C first convolution: streaming stencils
// ---------------------------------------------------------------------------------------------------------------
struct Conv1Args {
    const float* x;             // (B, H, W)
    const float* w;             // (C, 1, 3, 3)
    float* y;                   // (B, H, W, C)
    int B, H, W, C, act;
    float p;
    unsigned long long seed;
    const unsigned long long* seed_off;
};

__global__ void __launch_bounds__(256) conv1_fwd_kernel(Conv1Args a) {
    extern __shared__ float wsm[];                              // [9][C]
    for (int i = threadIdx.x; i < 9 * a.C; i += blockDim.x) wsm[(i % 9) * a.C + i / 9] = a.w[i];
    __syncthreads();
    const unsigned long long so = (a.p > 0.f && a.seed_off) ? *a.seed_off : 0ull;
    const int c4n = a.C >> 2;
    const long long total = (long long)a.B * a.H * a.W * c4n;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long px = e / c4n;
        const int c = (int)(e - px * c4n) * 4;
        const int xx = (int)(px % a.W), yy = (int)((px / a.W) % a.H);
        const float* img = a.x + (px - xx - (long long)yy * a.W);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const int y2 = yy + t / 3 - 1, x2 = xx + t % 3 - 1;
            if (y2 >= 0 && y2 < a.H && x2 >= 0 && x2 < a.W) {
                const float xv = img[(long long)y2 * a.W + x2];
                const float4 wv = *reinterpret_cast<const float4*>(&wsm[t * a.C + c]);
                acc.x = fmaf(xv, wv.x, acc.x); acc.y = fmaf(xv, wv.y, acc.y);
                acc.z = fmaf(xv, wv.z, acc.z); acc.w = fmaf(xv, wv.w, acc.w);
            }
        }
        if (a.p > 0.f) {
            const float4 ds = dropout_scale4(a.p, a.seed + so, (unsigned long long)px * a.C + c);
            acc.x *= ds.x; acc.y *= ds.y; acc.z *= ds.z; acc.w *= ds.w;
        }
        acc.x = act_apply(a.act, acc.x); acc.y = act_apply(a.act, acc.y);
        acc.z = act_apply(a.act, acc.z); acc.w = act_apply(a.act, acc.w);
        *reinterpret_cast<float4*>(a.y + px * a.C + c) = acc;
    }
}

// Row-structured variant (C <= 128): CTA = one image row, the three input rows it needs sit zero-padded in shared memory,
// a thread keeps the nine taps of its four channels in registers and walks the row eight pixels apart.  The grid-stride
// kernel above spent its time on 64-bit index arithmetic and per-tap bounds tests (83 us for an 81 MB output).
__global__ void __launch_bounds__(256) conv1_fwd_row_kernel(Conv1Args a) {
    extern __shared__ float xs[];                               // [3][W + 2]
    const int W = a.W, WP = W + 2;
    const int cq = threadIdx.x & 31, ph = threadIdx.x >> 5, c = cq * 4;
    const bool cok = c < a.C;
    float4 wr[9];
#pragma unroll
    for (int t = 0; t < 9; ++t)
        wr[t] = cok ? make_float4(a.w[(c + 0) * 9 + t], a.w[(c + 1) * 9 + t], a.w[(c + 2) * 9 + t], a.w[(c + 3) * 9 + t])
                    : make_float4(0.f, 0.f, 0.f, 0.f);
    const unsigned long long so = (a.p > 0.f && a.seed_off) ? *a.seed_off : 0ull;
    for (int row = blockIdx.x; row < a.B * a.H; row += gridDim.x) {
        const int b = row / a.H, yy = row % a.H;
        __syncthreads();
        for (int i = threadIdx.x; i < 3 * WP; i += blockDim.x) {
            const int r = i / WP, xx = i % WP - 1, y2 = yy + r - 1;
            xs[i] = (y2 >= 0 && y2 < a.H && xx >= 0 && xx < W) ? a.x[((long long)b * a.H + y2) * W + xx] : 0.f;
        }
        __syncthreads();
        if (!cok) continue;
        for (int xx = ph; xx < W; xx += 8) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                const float xv = xs[(t / 3) * WP + xx + t % 3];
                acc.x = fmaf(xv, wr[t].x, acc.x); acc.y = fmaf(xv, wr[t].y, acc.y);
                acc.z = fmaf(xv, wr[t].z, acc.z); acc.w = fmaf(xv, wr[t].w, acc.w);
            }
            const long long px = (long long)row * W + xx;
            if (a.p > 0.f) {
                const float4 ds = dropout_scale4(a.p, a.seed + so, (unsigned long long)px * a.C + c);
                acc.x *= ds.x; acc.y *= ds.y; acc.z *= ds.z; acc.w *= ds.w;
            }
            acc.x = act_apply(a.act, acc.x); acc.y = act_apply(a.act, acc.y);
            acc.z = act_apply(a.act, acc.z); acc.w = act_apply(a.act, acc.w);
            *reinterpret_cast<float4*>(a.y + px * a.C + c) = acc;
        }
    }
}

// g = dy * act'(y) * mask (ReLU only: y > 0 <=> kept and positive), then
//   dx[px]        = sum_{tap, c} g[px - tap][c] w[c][tap]                     (one warp per pixel)
//   dw[c][tap]    = sum_px g[px][c] x[px + tap]                                (thread = channel, CTA = pixel range)
struct Conv1BwdArgs {
    const float* dy;            // (B, H, W, C)
    const float* y;             // forward output (ReLU gate)
    const float* x;             // (B, H, W)
    const float* w;
    float* dx;                  // (B, H, W) or null
    float* dwpart;              // (gridDim.x, 9, C)
    int B, H, W, C;
    float keep;
};

__global__ void __launch_bounds__(256) conv1_dgrad_kernel(Conv1BwdArgs a) {
    extern __shared__ float wsm[];                              // [9][C]
    for (int i = threadIdx.x; i < 9 * a.C; i += blockDim.x) wsm[(i % 9) * a.C + i / 9] = a.w[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long npix = (long long)a.B * a.H * a.W;
    for (long long px = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5); px < npix;
         px += (long long)gridDim.x * (blockDim.x >> 5)) {
        const int xx = (int)(px % a.W), yy = (int)((px / a.W) % a.H);
        float s = 0.f;
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            // output pixel q = px - (tap offset) used x[px] with weight tap t
            const int y2 = yy - (t / 3 - 1), x2 = xx - (t % 3 - 1);
            if (y2 >= 0 && y2 < a.H && x2 >= 0 && x2 < a.W) {
                const long long qx = px + (long long)(y2 - yy) * a.W + (x2 - xx);
                for (int c = lane; c < a.C; c += 32) {
                    const float yv = a.y[qx * a.C + c];
                    if (yv > 0.f) s = fmaf(a.dy[qx * a.C + c] * a.keep, wsm[t * a.C + c], s);
                }
            }
        }
        s = warp_sum(s);
        if (lane == 0) a.dx[px] = s;
    }
}

__global__ void __launch_bounds__(256) conv1_wgrad_kernel(Conv1BwdArgs a) {
    // CTA = a range of pixels; thread = (channel quad, pixel phase): 32 channel quads x 8 phases -> float4 loads of g,
    // eight independent pixels in flight per quad; the phases are summed through shared memory in fixed order
    __shared__ float red[8][9][128 + 4];
    const int cq = threadIdx.x & 31, ph = threadIdx.x >> 5;
    const int c = cq * 4;
    const long long npix = (long long)a.B * a.H * a.W;
    const long long per = (npix + gridDim.x - 1) / gridDim.x;
    const long long beg = blockIdx.x * per, end = min(npix, beg + per);
    float acc[9][4];
#pragma unroll
    for (int t = 0; t < 9; ++t) acc[t][0] = acc[t][1] = acc[t][2] = acc[t][3] = 0.f;
    if (c < a.C) {
        for (long long px = beg + ph; px < end; px += 8) {
            const float4 yv = *reinterpret_cast<const float4*>(a.y + px * a.C + c);
            float4 g = *reinterpret_cast<const float4*>(a.dy + px * a.C + c);
            g.x = yv.x > 0.f ? g.x * a.keep : 0.f; g.y = yv.y > 0.f ? g.y * a.keep : 0.f;
            g.z = yv.z > 0.f ? g.z * a.keep : 0.f; g.w = yv.w > 0.f ? g.w * a.keep : 0.f;
            const int xx = (int)(px % a.W), yy = (int)((px / a.W) % a.H);
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                const int y2 = yy + t / 3 - 1, x2 = xx + t % 3 - 1;
                const float xv = (y2 >= 0 && y2 < a.H && x2 >= 0 && x2 < a.W) ? a.x[px + (long long)(y2 - yy) * a.W + (x2 - xx)] : 0.f;
                acc[t][0] = fmaf(g.x, xv, acc[t][0]); acc[t][1] = fmaf(g.y, xv, acc[t][1]);
                acc[t][2] = fmaf(g.z, xv, acc[t][2]); acc[t][3] = fmaf(g.w, xv, acc[t][3]);
            }
        }
    }
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
        for (int i = 0; i < 4; ++i) red[ph][t][c + i] = acc[t][i];
    __syncthreads();
    for (int i = threadIdx.x; i < 9 * a.C; i += blockDim.x) {
        const int t = i / a.C, cc = i % a.C;
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) s += red[k][t][cc];
        a.dwpart[((long long)blockIdx.x * 9 + t) * a.C + cc] = s;
    }
}

// Row-structured weight gradient: CTA = `rows_per_cta` consecutive image rows, input rows staged in shared memory, two
// pixels (four float4 loads) in flight per thread, no 64-bit index arithmetic in the loop.
__global__ void __launch_bounds__(256) conv1_wgrad_row_kernel(Conv1BwdArgs a, int rows_per_cta) {
    __shared__ float red[8][9][128 + 4];
    extern __shared__ float xs[];                               // [3][W + 2]
    const int W = a.W, WP = W + 2;
    const int cq = threadIdx.x & 31, ph = threadIdx.x >> 5, c = cq * 4;
    const bool cok = c < a.C;
    float acc[9][4];
#pragma unroll
    for (int t = 0; t < 9; ++t) acc[t][0] = acc[t][1] = acc[t][2] = acc[t][3] = 0.f;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r = 0; r < rows_per_cta; ++r) {
        const int row = blockIdx.x * rows_per_cta + r;
        if (row >= a.B * a.H) break;
        const int b = row / a.H, yy = row % a.H;
        __syncthreads();
        for (int i = threadIdx.x; i < 3 * WP; i += blockDim.x) {
            const int rr = i / WP, xx = i % WP - 1, y2 = yy + rr - 1;
            xs[i] = (y2 >= 0 && y2 < a.H && xx >= 0 && xx < W) ? a.x[((long long)b * a.H + y2) * W + xx] : 0.f;
        }
        __syncthreads();
        if (!cok) continue;
        const float* yrow = a.y + (long long)row * W * a.C + c;
        const float* grow = a.dy + (long long)row * W * a.C + c;
        for (int xx = ph; xx < W; xx += 16) {
            const bool two = xx + 8 < W;
            const float4 y0 = *reinterpret_cast<const float4*>(yrow + (long long)xx * a.C);
            float4 g0 = *reinterpret_cast<const float4*>(grow + (long long)xx * a.C);
            const float4 y1 = two ? *reinterpret_cast<const float4*>(yrow + (long long)(xx + 8) * a.C) : zero4;
            float4 g1 = two ? *reinterpret_cast<const float4*>(grow + (long long)(xx + 8) * a.C) : zero4;
            g0.x = y0.x > 0.f ? g0.x * a.keep : 0.f; g0.y = y0.y > 0.f ? g0.y * a.keep : 0.f;
            g0.z = y0.z > 0.f ? g0.z * a.keep : 0.f; g0.w = y0.w > 0.f ? g0.w * a.keep : 0.f;
            g1.x = y1.x > 0.f ? g1.x * a.keep : 0.f; g1.y = y1.y > 0.f ? g1.y * a.keep : 0.f;
            g1.z = y1.z > 0.f ? g1.z * a.keep : 0.f; g1.w = y1.w > 0.f ? g1.w * a.keep : 0.f;
            const int x1 = two ? xx + 8 : xx;                     // g1 is zero when there is no second pixel
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                const float xv0 = xs[(t / 3) * WP + xx + t % 3], xv1 = xs[(t / 3) * WP + x1 + t % 3];
                acc[t][0] = fmaf(g1.x, xv1, fmaf(g0.x, xv0, acc[t][0])); acc[t][1] = fmaf(g1.y, xv1, fmaf(g0.y, xv0, acc[t][1]));
                acc[t][2] = fmaf(g1.z, xv1, fmaf(g0.z, xv0, acc[t][2])); acc[t][3] = fmaf(g1.w, xv1, fmaf(g0.w, xv0, acc[t][3]));
            }
        }
    }
    __syncthreads();
    if (cok) {
#pragma unroll
        for (int t = 0; t < 9; ++t)
#pragma unroll
            for (int i = 0; i < 4; ++i) red[ph][t][c + i] = acc[t][i];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 9 * a.C; i += blockDim.x) {
        const int t = i / a.C, cc = i % a.C;
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) s += red[k][t][cc];
        a.dwpart[((long long)blockIdx.x * 9 + t) * a.C + cc] = s;
    }
}

__global__ void conv1_wgrad_final_kernel(const float* __restrict__ part, int nparts, int C, float* __restrict__ dw) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;        // i = t * C + c
    if (i >= 9 * C) return;
    float s = 0.f;
    for (int k = 0; k < nparts; ++k) s += part[(long long)k * 9 * C + i];
    dw[(i % C) * 9 + i / C] = s;                                // (C, 1, 3, 3)
}

static bool make_image_map(CUtensorMap* m, const void* base, int CP, int W, int H, int B) {
    cuuint64_t dims[4] = {(cuuint64_t)CP, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
    cuuint64_t strides[3] = {(cuuint64_t)CP * 2, (cuuint64_t)CP * 2 * W, (cuuint64_t)CP * 2 * W * H};
    cuuint32_t box[4] = {64, (cuuint32_t)PATCH_W, (cuuint32_t)PATCH_H, 1};
    return make_map_nd(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

}  // namespace enc
}  // namespace gb200

using namespace gb200;
using namespace gb200::enc;

static int chunks_of(int c) { return (c + 63) / 64; }

extern "C" int gb200_conv3x3_supported(int Cin, int Cout) {
    return Cin >= 1 && Cin <= 128 && Cout >= 1 && Cout <= 128 && encode_fn() != nullptr;
}
extern "C" size_t gb200_conv3x3_pack_bytes(int Cin, int Cout, int dgrad) {
    return (size_t)9 * chunks_of(dgrad ? Cout : Cin) * 2 * TILE_BYTES;
}
/* weight (Cout, Cin, 3, 3) fp32 contiguous -> operand tile stream of the forward (dgrad = 0) or input-gradient pass */
extern "C" int gb200_conv3x3_pack(int device, const float* w, int Cin, int Cout, int dgrad, void* tiles, void* stream) {
    use_device(device);
    GB_REQUIRE(w && tiles && gb200_conv3x3_supported(Cin, Cout), "gb200_conv3x3_pack: bad arguments");
    const int nchunk = chunks_of(dgrad ? Cout : Cin);
    conv_pack_kernel<<<9 * nchunk, 256, 0, as_stream(stream)>>>(w, Cout, Cin, nchunk, dgrad, reinterpret_cast<uint8_t*>(tiles));
    return check_launch("gb200_conv3x3_pack");
}

/* x (npix, ldx)[c0 : c0 + C] -> (hi, lo) bf16 images (npix, CP = 64 * ceil(C / 64)).  Backward mode (yz != null):
 * x is dy, g = dy * act'(yz) * dropmask is what gets split, and gout (npix, C) receives g in fp32. */
extern "C" int gb200_conv_split(int device, const float* x, int ldx, int c0, int C, long long npix, void* hi, void* lo,
                                const float* yz, int ldyz, int yz_c0, int act, float p, unsigned long long seed, float* gout,
                                void* stream) {
    use_device(device);
    GB_REQUIRE(x && hi && lo && C >= 1 && npix >= 1, "gb200_conv_split: bad arguments");
    SplitArgs a;
    a.x = x; a.ldx = ldx; a.c0 = c0; a.C = C; a.CP = 64 * chunks_of(C); a.npix = npix;
    a.hi = reinterpret_cast<__nv_bfloat16*>(hi); a.lo = reinterpret_cast<__nv_bfloat16*>(lo);
    a.yz = yz; a.ldyz = ldyz; a.yz_c0 = yz_c0; a.act = act; a.p = p; a.seed = seed; a.seed_off = rng_offset_ptr(); a.gout = gout;
    const long long total = npix * (a.CP / 8);
    int blocks = (int)((total + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    conv_split_kernel<<<blocks, 256, 0, as_stream(stream)>>>(a);
    return check_launch("gb200_conv_split");
}

/* out[.., co0 : co0 + Cout] = act( dropout( conv3x3(in) + resid ) ) from the (hi, lo) images of the input
 * (B, H, W, 64 * nchunk) and a packed weight stream (gb200_conv3x3_pack). */
extern "C" int gb200_conv3x3(int device, const void* in_hi, const void* in_lo, int Cin, const void* wtiles, int Cout, int B, int H,
                             int W, float* out, int ldo, int co0, float* zout, const float* resid, int ldr, int r0, int act,
                             float p, unsigned long long seed, void* stream) {
    use_device(device);
    GB_REQUIRE(in_hi && in_lo && wtiles && out, "gb200_conv3x3: null buffer");
    GB_REQUIRE(gb200_conv3x3_supported(Cin, Cout), "gb200_conv3x3: unsupported channel counts %d -> %d", Cin, Cout);
    GB_REQUIRE(act == ACT_NONE || act == ACT_RELU || act == ACT_SILU, "gb200_conv3x3: unknown activation");
    GB_REQUIRE(p >= 0.f && p < 1.f, "gb200_conv3x3: dropout p outside [0,1)");
    GB_REQUIRE(((co0 | ldo) & 1) == 0 && ((uintptr_t)out % 8) == 0 && (!zout || ((uintptr_t)zout % 8) == 0),
               "gb200_conv3x3: output must be 8-byte aligned with even channel offsets");
    static bool configured = false;
    if (!configured) {
        set_smem(conv3x3_tc_kernel, CV_SMEM);
        configured = true;
    }
    const int nchunk = chunks_of(Cin);
    CUtensorMap mh, ml;
    GB_REQUIRE(make_image_map(&mh, in_hi, 64 * nchunk, W, H, B) && make_image_map(&ml, in_lo, 64 * nchunk, W, H, B),
               "gb200_conv3x3: tensor map failed");
    ConvArgs a;
    a.wtiles = reinterpret_cast<const uint8_t*>(wtiles); a.out = out; a.zout = zout; a.resid = resid; a.ldo = ldo; a.co0 = co0;
    a.ldr = ldr; a.r0 = r0; a.Cout = Cout; a.N = Cout <= 48 ? 48 : 128; a.nchunk = nchunk; a.act = act; a.p = p; a.seed = seed;
    a.seed_off = rng_offset_ptr(); a.B = B; a.H = H; a.W = W; a.tiles_x = (W + PATCH_W - 1) / PATCH_W;
    a.tiles_y = (H + PATCH_H - 1) / PATCH_H;
    conv3x3_tc_kernel<<<B * a.tiles_x * a.tiles_y, THREADS, CV_SMEM, as_stream(stream)>>>(mh, ml, a);
    return check_launch("gb200_conv3x3");
}

extern "C" int gb200_conv1_fwd(int device, const float* x, const float* w, float* y, int B, int H, int W, int C, int act, float p,
                               unsigned long long seed, void* stream) {
    use_device(device);
    GB_REQUIRE(x && w && y && C % 4 == 0 && C <= 256, "gb200_conv1_fwd: bad arguments (C %% 4, C <= 256)");
    Conv1Args a;
    a.x = x; a.w = w; a.y = y; a.B = B; a.H = H; a.W = W; a.C = C; a.act = act; a.p = p; a.seed = seed; a.seed_off = rng_offset_ptr();
    const long long total = (long long)B * H * W * (C / 4);
    int blocks = (int)((total + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (C <= 128 && W <= 2048) {
        int rb = B * H;
        if (rb > 148 * 16) rb = 148 * 16;
        conv1_fwd_row_kernel<<<rb, 256, 3 * (W + 2) * sizeof(float), as_stream(stream)>>>(a);
        return check_launch("gb200_conv1_fwd");
    }
    conv1_fwd_kernel<<<blocks, 256, 9 * C * sizeof(float), as_stream(stream)>>>(a);
    return check_launch("gb200_conv1_fwd");
}

extern "C" size_t gb200_conv1_bwd_workspace_bytes(int C) { return (size_t)148 * 4 * 9 * C * sizeof(float); }

/* ReLU block only (the shipped down-scaler): dx (B,H,W) (optional) and dw (C,1,3,3) from dy, the forward output y and x */
extern "C" int gb200_conv1_bwd(int device, const float* dy, const float* y, const float* x, const float* w, float* dx, float* dw,
                               int B, int H, int W, int C, float p, float* workspace, size_t workspace_bytes, void* stream) {
    use_device(device);
    GB_REQUIRE(dy && y && x && w && dw && workspace && C <= 128 && C % 4 == 0, "gb200_conv1_bwd: bad arguments");
    GB_REQUIRE(workspace_bytes >= gb200_conv1_bwd_workspace_bytes(C), "gb200_conv1_bwd: workspace too small");
    Conv1BwdArgs a;
    a.dy = dy; a.y = y; a.x = x; a.w = w; a.dx = dx; a.dwpart = workspace; a.B = B; a.H = H; a.W = W; a.C = C;
    a.keep = p > 0.f ? 65536.f / (65536.f - (float)(unsigned)(p * 65536.f + 0.5f)) : 1.f;
    cudaStream_t st = as_stream(stream);
    int launched = 2;
    if (dx) {
        conv1_dgrad_kernel<<<148 * 8, 256, 9 * C * sizeof(float), st>>>(a);
        ++launched;
    }
    int nparts = 148 * 4;
    if (W <= 512) {
        const int nrows = B * H;
        const int rpc = (nrows + nparts - 1) / nparts;          // the workspace holds 148 * 4 partials
        nparts = (nrows + rpc - 1) / rpc;
        conv1_wgrad_row_kernel<<<nparts, 256, 3 * (W + 2) * sizeof(float), st>>>(a, rpc);
    } else {
        conv1_wgrad_kernel<<<nparts, 256, 0, st>>>(a);
    }
    conv1_wgrad_final_kernel<<<(9 * C + 127) / 128, 128, 0, st>>>(workspace, nparts, C, dw);
    return check_launch("gb200_conv1_bwd", launched);
}
