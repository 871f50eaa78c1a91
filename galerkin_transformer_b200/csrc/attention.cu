// Softmax-free attention core (Galerkin Q(K^T V)/n and linear-form Fourier (Q K^T) V/(sqrt(d) n)).
//
// Layout: tokens stay token-major.  The projection GEMM writes one (T, 3*d_model) buffer
// [Q | K | V]; head h of each operand is the d_k-wide column slice h*d_k.. of its block.  No
// head-major transposes, no torch.cat of the position columns, no torch.stack of per-head
// LayerNorm outputs ever exist in HBM: the kernels read an "augmented head operand"
//       X~[t, h, :] = [ pos[t, 0..p) , gamma[h] * xhat[t, h, :] + beta[h] ]          (d = p + d_k)
// straight from the token-major buffers (xhat = the per-head normalised rows written in
// place by headnorm_fwd, or the raw rows when the operand has no norm).
//
// Reference semantics replaced here (scaomath/galerkin-transformer):
//   libs/layers.py:846-851, 859-864   per-head LayerNorm loop + torch.stack
//   libs/layers.py:869-874            pos.repeat + torch.cat([pos, x]) for q, k, v
//   libs/layers.py:723, 728, 733      K^T V, /n, Q.(.)           (linear_attention)
//   libs/layers.py:730-731            F.dropout(p_attn), p=0.5, always on (mask input)
//   libs/layers.py:892-894            transpose(1,2).contiguous().view  (head merge)
#include "common.cuh"
#include "head_operand.cuh"
#include "attention_mma.cuh"
namespace gb200 {

// -------------------------------------------------------------------------------------------
// per-head LayerNorm, forward: x -> xhat (in place), rstd (T, H) saved for backward.
// One CTA stages ROWS token rows (all heads) through shared memory with coalesced loads,
// then one thread normalises one (token, head) group (biased variance, two-pass).
// -------------------------------------------------------------------------------------------
constexpr int HN_ROWS = 32;

__global__ void headnorm_fwd_kernel(float* __restrict__ x, int ld, int col0, long long T, int H, int dk,
                                    float eps, float* __restrict__ rstd_out) {
    pdl_enter();
    extern __shared__ float sm[];
    const int W = H * dk, WS = W + 1;
    const long long t0 = (long long)blockIdx.x * HN_ROWS;
    const int nrows = (int)min((long long)HN_ROWS, T - t0);
    for (int e = threadIdx.x; e < nrows * W; e += blockDim.x) {
        int r = e / W, c = e % W;
        sm[r * WS + c] = x[(t0 + r) * ld + col0 + c];
    }
    __syncthreads();
    for (int gidx = threadIdx.x; gidx < nrows * H; gidx += blockDim.x) {
        int r = gidx / H, h = gidx % H;
        float* row = sm + r * WS + h * dk;
        float mean = 0.f;
        for (int c = 0; c < dk; ++c) mean += row[c];
        mean /= dk;
        float var = 0.f;
        for (int c = 0; c < dk; ++c) { float d = row[c] - mean; var += d * d; }
        var /= dk;
        float rs = rsqrtf(var + eps);
        for (int c = 0; c < dk; ++c) row[c] = (row[c] - mean) * rs;
        rstd_out[(t0 + r) * H + h] = rs;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < nrows * W; e += blockDim.x) {
        int r = e / W, c = e % W;
        x[(t0 + r) * ld + col0 + c] = sm[r * WS + c];
    }
}

// per-head LayerNorm, backward.  dy (grad w.r.t. gamma*xhat+beta) is overwritten by the grad
// w.r.t. the raw projection output; per-CTA partial sums of dgamma/dbeta go to `part`.
__global__ void headnorm_bwd_kernel(float* __restrict__ dy, int lddy, int dcol0,
                                    const float* __restrict__ xhat, int ldx, int xcol0,
                                    const float* __restrict__ rstd, const float* __restrict__ gamma,
                                    long long T, int H, int dk, float* __restrict__ part) {
    pdl_enter();
    extern __shared__ float sm[];
    const int W = H * dk, WS = W + 1;
    float* sdy = sm;
    float* sxh = sm + HN_ROWS * WS;
    const long long t0 = (long long)blockIdx.x * HN_ROWS;
    const int nrows = (int)min((long long)HN_ROWS, T - t0);
    for (int e = threadIdx.x; e < nrows * W; e += blockDim.x) {
        int r = e / W, c = e % W;
        sdy[r * WS + c] = dy[(t0 + r) * lddy + dcol0 + c];
        sxh[r * WS + c] = xhat[(t0 + r) * ldx + xcol0 + c];
    }
    __syncthreads();
    // dgamma / dbeta partials: one thread per column, fixed row order
    for (int c = threadIdx.x; c < W; c += blockDim.x) {
        float sg = 0.f, sb = 0.f;
        for (int r = 0; r < nrows; ++r) {
            float d = sdy[r * WS + c];
            sg += d * sxh[r * WS + c];
            sb += d;
        }
        part[((long long)blockIdx.x * 2 + 0) * W + c] = sg;
        part[((long long)blockIdx.x * 2 + 1) * W + c] = sb;
    }
    __syncthreads();
    for (int gidx = threadIdx.x; gidx < nrows * H; gidx += blockDim.x) {
        int r = gidx / H, h = gidx % H;
        float* d = sdy + r * WS + h * dk;
        const float* xh = sxh + r * WS + h * dk;
        const float* gm = gamma + h * dk;
        float c1 = 0.f, c2 = 0.f;
        for (int c = 0; c < dk; ++c) {
            float gd = gm[c] * d[c];
            c1 += gd;
            c2 += gd * xh[c];
        }
        c1 /= dk; c2 /= dk;
        float rs = rstd[(t0 + r) * H + h];
        for (int c = 0; c < dk; ++c) d[c] = rs * (gm[c] * d[c] - c1 - xh[c] * c2);
    }
    __syncthreads();
    for (int e = threadIdx.x; e < nrows * W; e += blockDim.x) {
        int r = e / W, c = e % W;
        dy[(t0 + r) * lddy + dcol0 + c] = sdy[r * WS + c];
    }
}

// -------------------------------------------------------------------------------------------
// Coalesced variants (d_k/4 a power of two <= 32 and 256 % (H*d_k/4) == 0): one float4 per lane, the
// d_k/4 lanes of a head group combine their statistics with warp shuffles; no shared-memory staging.
// blockIdx.y selects the operand block (K and V, or Q and K, normalised by ONE launch).
// -------------------------------------------------------------------------------------------
struct HeadNormBlocks {
    int col0[2];
    float* rstd[2];
    const float* gamma[2];
    float* part[2];
    int dcol0[2];
};

template <int LG>   // lanes per head group = d_k / 4
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int o = LG / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int LG>
__global__ void __launch_bounds__(256) headnorm_fwd_vec_kernel(float* __restrict__ x, int ld, HeadNormBlocks blk,
                                                               long long T, int H, int dk, float eps) {
    pdl_enter();
    const int col0 = blk.col0[blockIdx.y];
    float* rstd_out = blk.rstd[blockIdx.y];
    const int rowq = H * LG;                              // float4s per row
    const int q = threadIdx.x % rowq, rsub = threadIdx.x / rowq, rpb = 256 / rowq;
    const float inv = 1.f / dk;
    // uniform trip count: every lane of a warp takes part in every shuffle (rows past T are predicated)
    const long long stride = (long long)gridDim.x * rpb;
    const long long iters = (T + stride - 1) / stride;
    for (long long it = 0; it < iters; ++it) {
        const long long r = (long long)blockIdx.x * rpb + rsub + it * stride;
        const bool ok = r < T;
        float4* p = reinterpret_cast<float4*>(x + (ok ? r : 0) * ld + col0) + q;
        float4 v = ok ? *p : make_float4(0.f, 0.f, 0.f, 0.f);
        const float mean = group_sum<LG>(v.x + v.y + v.z + v.w) * inv;
        v.x -= mean; v.y -= mean; v.z -= mean; v.w -= mean;
        const float var = group_sum<LG>(v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w) * inv;
        const float rs = rsqrtf(var + eps);
        if (ok) {
            *p = make_float4(v.x * rs, v.y * rs, v.z * rs, v.w * rs);
            if (q % LG == 0) rstd_out[r * H + q / LG] = rs;
        }
    }
}

template <int LG>
__global__ void __launch_bounds__(256) headnorm_bwd_vec_kernel(float* __restrict__ dy, int lddy,
                                                               const float* __restrict__ xhat, int ldx,
                                                               HeadNormBlocks blk, long long T, int H, int dk) {
    pdl_enter();
    __shared__ float4 sg[256], sb[256];
    const int bi = blockIdx.y;
    const int rowq = H * LG;
    const int q = threadIdx.x % rowq, rsub = threadIdx.x / rowq, rpb = 256 / rowq;
    const float inv = 1.f / dk;
    const float4 gm = reinterpret_cast<const float4*>(blk.gamma[bi])[q];
    const float* rstd = blk.rstd[bi];
    float4 ag = make_float4(0.f, 0.f, 0.f, 0.f), ab = ag;
    const long long stride = (long long)gridDim.x * rpb;
    const long long iters = (T + stride - 1) / stride;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (long long it = 0; it < iters; ++it) {
        const long long r = (long long)blockIdx.x * rpb + rsub + it * stride;
        const bool ok = r < T;
        float4* dp = reinterpret_cast<float4*>(dy + (ok ? r : 0) * lddy + blk.dcol0[bi]) + q;
        const float4 d = ok ? *dp : zero4;
        const float4 xh = ok ? *(reinterpret_cast<const float4*>(xhat + r * ldx + blk.col0[bi]) + q) : zero4;
        ag.x += d.x * xh.x; ag.y += d.y * xh.y; ag.z += d.z * xh.z; ag.w += d.w * xh.w;
        ab.x += d.x; ab.y += d.y; ab.z += d.z; ab.w += d.w;
        const float4 gd = make_float4(gm.x * d.x, gm.y * d.y, gm.z * d.z, gm.w * d.w);
        const float c1 = group_sum<LG>(gd.x + gd.y + gd.z + gd.w) * inv;
        const float c2 = group_sum<LG>(gd.x * xh.x + gd.y * xh.y + gd.z * xh.z + gd.w * xh.w) * inv;
        const float rs = ok ? rstd[r * H + q / LG] : 0.f;
        if (ok) *dp = make_float4(rs * (gd.x - c1 - xh.x * c2), rs * (gd.y - c1 - xh.y * c2), rs * (gd.z - c1 - xh.z * c2),
                          rs * (gd.w - c1 - xh.w * c2));
    }
    // fixed-order sum over the rpb row-threads that share a column quad, then the CTA partial
    sg[threadIdx.x] = ag; sb[threadIdx.x] = ab;
    __syncthreads();
    if (threadIdx.x < rowq) {
        float4 tg = sg[threadIdx.x], tb = sb[threadIdx.x];
        for (int k = 1; k < rpb; ++k) {
            const float4 a = sg[threadIdx.x + k * rowq], b2 = sb[threadIdx.x + k * rowq];
            tg.x += a.x; tg.y += a.y; tg.z += a.z; tg.w += a.w;
            tb.x += b2.x; tb.y += b2.y; tb.z += b2.z; tb.w += b2.w;
        }
        float* part = blk.part[bi];
        const int W = H * dk;
        reinterpret_cast<float4*>(part + ((long long)blockIdx.x * 2 + 0) * W)[threadIdx.x] = tg;
        reinterpret_cast<float4*>(part + ((long long)blockIdx.x * 2 + 1) * W)[threadIdx.x] = tb;
    }
}

static int headnorm_vec_lanes(int H, int dk, int ld, int col0, const void* base) {
    if (dk % 4) return 0;
    const int lg = dk / 4;
    if (lg < 1 || lg > 32 || (lg & (lg - 1))) return 0;
    const int rowq = H * lg;
    if (rowq > 256 || 256 % rowq) return 0;
    if ((ld % 4) || (col0 % 4) || ((uintptr_t)base % 16)) return 0;
    return lg;
}
constexpr int HN_VEC_BLOCKS = 296;

// out[j][c] (+)= sum_blocks part[blk][j][c]   (j = 0: dgamma, 1: dbeta), fixed order
__global__ void headnorm_bwd_reduce_kernel(const float* __restrict__ part, int nblocks, int W,
                                           float* __restrict__ dgamma, float* __restrict__ dbeta,
                                           int accumulate) {
    pdl_enter();
    // blockIdx.y = 0: dgamma, 1: dbeta
    reduce_partials_2d(part + (long long)blockIdx.y * W, nblocks, 2LL * W, W, 1.f, accumulate,
                       blockIdx.y == 0 ? dgamma : dbeta);
}

// -------------------------------------------------------------------------------------------
// xty:  P[b,h,s][i][j] = sum_{t in split s} L~[b,t,h,i] * R~[b,t,h,j]          (d x d per head)
// CTA = one (b,h) x one token split; TC tokens staged per step; 16x16 threads, (DP/16)^2
// accumulators each.  Partials are summed in fixed order by xty_reduce (deterministic).
// -------------------------------------------------------------------------------------------
template <int DP>
__global__ void __launch_bounds__(256) xty_kernel(HeadOperand L, HeadOperand R, const float* __restrict__ pos,
                                                  int p, int dk, int H, int n, int nsplit, int chunk,
                                                  float* __restrict__ part) {
    pdl_enter();
    constexpr int TC = 32, MT = DP / 16;
    __shared__ float Ls[TC][DP + 1];
    __shared__ float Rs[TC][DP + 1];
    const int d = p + dk;
    const int bh = blockIdx.y, b = bh / H, h = bh % H, split = blockIdx.x;
    const int tbeg = split * chunk, tend = min(n, tbeg + chunk);
    const int ty = threadIdx.x / 16, tx = threadIdx.x % 16;
    float acc[MT][MT];
#pragma unroll
    for (int a = 0; a < MT; ++a)
#pragma unroll
        for (int c = 0; c < MT; ++c) acc[a][c] = 0.f;

    for (int t0 = tbeg; t0 < tend; t0 += TC) {
        const int nt = min(TC, tend - t0);
        for (int e = threadIdx.x; e < TC * DP; e += 256) {
            int r = e / DP, i = e % DP;
            float lv = 0.f, rv = 0.f;
            if (r < nt && i < d) {
                long long t = (long long)b * n + t0 + r;
                lv = load_aug(L, pos, p, dk, h, t, i);
                rv = load_aug(R, pos, p, dk, h, t, i);
            }
            Ls[r][i] = lv;
            Rs[r][i] = rv;
        }
        __syncthreads();
#pragma unroll 4
        for (int r = 0; r < TC; ++r) {
            float lv[MT], rv[MT];
#pragma unroll
            for (int a = 0; a < MT; ++a) lv[a] = Ls[r][ty + 16 * a];
#pragma unroll
            for (int c = 0; c < MT; ++c) rv[c] = Rs[r][tx + 16 * c];
#pragma unroll
            for (int a = 0; a < MT; ++a)
#pragma unroll
                for (int c = 0; c < MT; ++c) acc[a][c] = fmaf(lv[a], rv[c], acc[a][c]);
        }
        __syncthreads();
    }
    float* out = part + ((long long)bh * nsplit + split) * d * d;
#pragma unroll
    for (int a = 0; a < MT; ++a)
#pragma unroll
        for (int c = 0; c < MT; ++c) {
            int i = ty + 16 * a, j = tx + 16 * c;
            if (i < d && j < d) out[i * d + j] = acc[a][c];
        }
}

// A[bh][i][j] = scale * sum_s P[bh][s][i][j] * (mask ? 2*mask : 1); optionally also the
// un-masked value (needed by nothing downstream; kept null) -- fixed summation order.
__global__ void xty_reduce_kernel(const float* __restrict__ part, int nsplit, int dd, long long total,
                                  float scale, const unsigned char* __restrict__ mask, float mask_p,
                                  unsigned long long mask_seed, const unsigned long long* seed_off,
                                  float* __restrict__ out) {
    pdl_enter();
    if (mask_p > 0.f && seed_off) mask_seed += *seed_off;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        long long bh = e / dd;
        int ij = (int)(e % dd);
        const float* p = part + bh * nsplit * dd + ij;
        float s = 0.f;
        for (int k = 0; k < nsplit; ++k) s += p[(long long)k * dd];
        s *= scale;
        if (mask) s *= 2.f * (float)mask[e];
        else if (mask_p > 0.f) s *= dropout_scale(mask_p, mask_seed, (unsigned long long)e);   // 0 or 1/(1-p)
        out[e] = s;
    }
}

// -------------------------------------------------------------------------------------------
// xm:  O[b,t,h,j] = sum_i L~[b,t,h,i] * M[b,h][i][j]      (or M^T), token tile x d x d.
// Output either in augmented layout (T, H*d) -- the head-merged tensor the fc Linear reads --
// or scattered into a token-major (T, ld) buffer dropping the p position columns (gradients
// w.r.t. q, k, v: position coordinates carry no gradient).
// -------------------------------------------------------------------------------------------
template <int DP>
__global__ void __launch_bounds__(256) xm_kernel(HeadOperand L, const float* __restrict__ pos,
                                                 const float* __restrict__ Mat, int transM, int p, int dk,
                                                 int H, int n, float* __restrict__ out, int ldo, int ocol0,
                                                 int out_augmented, float oscale) {
    pdl_enter();
    constexpr int TT = 64, MT = DP / 16;
    extern __shared__ float sm[];
    float* Ms = sm;                    // [DP][DP+1]   Ms[i][j]
    float* Ls = sm + DP * (DP + 1);    // [TT][DP+1]
    const int d = p + dk;
    const int bh = blockIdx.y, b = bh / H, h = bh % H;
    const int t0 = blockIdx.x * TT;
    const int nt = min(TT, n - t0);
    const float* M = Mat + (long long)bh * d * d;
    for (int e = threadIdx.x; e < DP * DP; e += 256) {
        int i = e / DP, j = e % DP;
        float v = 0.f;
        if (i < d && j < d) v = transM ? M[j * d + i] : M[i * d + j];
        Ms[i * (DP + 1) + j] = v;
    }
    for (int e = threadIdx.x; e < TT * DP; e += 256) {
        int r = e / DP, i = e % DP;
        float v = 0.f;
        if (r < nt && i < d) v = load_aug(L, pos, p, dk, h, (long long)b * n + t0 + r, i);
        Ls[r * (DP + 1) + i] = v;
    }
    __syncthreads();
    const int ty = threadIdx.x / 16, tx = threadIdx.x % 16;
    float acc[4][MT];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < MT; ++c) acc[a][c] = 0.f;
    for (int i = 0; i < d; ++i) {
        float lv[4], mv[MT];
#pragma unroll
        for (int a = 0; a < 4; ++a) lv[a] = Ls[(ty + 16 * a) * (DP + 1) + i];
#pragma unroll
        for (int c = 0; c < MT; ++c) mv[c] = Ms[i * (DP + 1) + tx + 16 * c];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int c = 0; c < MT; ++c) acc[a][c] = fmaf(lv[a], mv[c], acc[a][c]);
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        int r = ty + 16 * a;
        if (r >= nt) continue;
        long long t = (long long)b * n + t0 + r;
#pragma unroll
        for (int c = 0; c < MT; ++c) {
            int j = tx + 16 * c;
            if (j >= d) continue;
            float v = acc[a][c] * oscale;
            if (out_augmented) out[t * ldo + ocol0 + h * d + j] = v;
            else if (j >= p) out[t * ldo + ocol0 + h * dk + (j - p)] = v;
        }
    }
}

static int pick_dp(int d) { return d <= 32 ? 32 : d <= 64 ? 64 : d <= 128 ? 128 : 0; }

}  // namespace gb200

using namespace gb200;

static HeadOperand make_op(const gb200_head_operand* o) { return make_head_operand(o); }

extern "C" int gb200_headnorm_fwd(int device, float* x, int ld, int col0, int col0b, long long T, int H, int dk,
                                  float eps, float* rstd, float* rstd_b, void* stream) {
    use_device(device);
    GB_REQUIRE(x && rstd && T >= 0 && H >= 1 && dk >= 1, "gb200_headnorm_fwd: bad arguments");
    GB_REQUIRE(col0b < 0 || rstd_b, "gb200_headnorm_fwd: second block needs its own rstd buffer");
    if (T == 0) return GB200_OK;
    cudaStream_t st = as_stream(stream);
    const int nblk = col0b >= 0 ? 2 : 1;
    int lg = headnorm_vec_lanes(H, dk, ld, col0, x);
    if (lg && nblk == 2 && !headnorm_vec_lanes(H, dk, ld, col0b, x)) lg = 0;
    if (lg) {
        HeadNormBlocks blk = {};
        blk.col0[0] = col0; blk.col0[1] = col0b; blk.rstd[0] = rstd; blk.rstd[1] = rstd_b;
        const int rpb = 256 / (H * lg);
        int blocks = cdiv(T, rpb);
        if (blocks > HN_VEC_BLOCKS) blocks = HN_VEC_BLOCKS;
        dim3 grid(blocks, nblk);
#define HN_FWD(LG) launch_kernel(headnorm_fwd_vec_kernel<LG>, grid, 256, 0, st, x, ld, blk, T, H, dk, eps)
        switch (lg) { case 1: HN_FWD(1); break; case 2: HN_FWD(2); break; case 4: HN_FWD(4); break;
                      case 8: HN_FWD(8); break; case 16: HN_FWD(16); break; default: HN_FWD(32); }
#undef HN_FWD
        return check_launch("gb200_headnorm_fwd");
    }
    size_t smem = (size_t)HN_ROWS * (H * dk + 1) * sizeof(float);
    GB_REQUIRE(smem <= 200 * 1024, "gb200_headnorm_fwd: H*d_k=%d too wide", H * dk);
    if (smem > 48 * 1024)
        cudaFuncSetAttribute(headnorm_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    launch_kernel(headnorm_fwd_kernel, cdiv(T, HN_ROWS), 256, smem, st, x, ld, col0, T, H, dk, eps, rstd);
    if (nblk == 2) launch_kernel(headnorm_fwd_kernel, cdiv(T, HN_ROWS), 256, smem, st, x, ld, col0b, T, H, dk, eps, rstd_b);
    return check_launch("gb200_headnorm_fwd", nblk);
}

extern "C" size_t gb200_headnorm_bwd_workspace_bytes(long long T, int H, int dk) {
    long long nb = cdiv(T, HN_ROWS);
    if (nb < HN_VEC_BLOCKS) nb = HN_VEC_BLOCKS;
    return (size_t)2 * nb * 2 * H * dk * sizeof(float);          // room for two operand blocks
}

extern "C" int gb200_headnorm_bwd(int device, float* dy, int lddy, int dcol0, int dcol0b, const float* xhat, int ldx,
                                  int xcol0, int xcol0b, const float* rstd, const float* rstd_b, const float* gamma,
                                  const float* gamma_b, long long T, int H, int dk, float* dgamma, float* dbeta,
                                  float* dgamma_b, float* dbeta_b, int accumulate, float* workspace,
                                  size_t workspace_bytes, void* stream) {
    use_device(device);
    GB_REQUIRE(dy && xhat && rstd && gamma && dgamma && dbeta, "gb200_headnorm_bwd: null argument");
    const int nblk = dcol0b >= 0 ? 2 : 1;
    GB_REQUIRE(nblk == 1 || (rstd_b && gamma_b && dgamma_b && dbeta_b && xcol0b >= 0),
               "gb200_headnorm_bwd: second block is incomplete");
    if (T == 0) return GB200_OK;
    GB_REQUIRE(workspace && workspace_bytes >= gb200_headnorm_bwd_workspace_bytes(T, H, dk),
               "gb200_headnorm_bwd: workspace too small");
    cudaStream_t st = as_stream(stream);
    const int W = H * dk;
    int lg = headnorm_vec_lanes(H, dk, lddy, dcol0, dy);
    if (lg && (!headnorm_vec_lanes(H, dk, ldx, xcol0, xhat) || ((uintptr_t)gamma % 16))) lg = 0;
    if (lg && nblk == 2 && (!headnorm_vec_lanes(H, dk, lddy, dcol0b, dy) || !headnorm_vec_lanes(H, dk, ldx, xcol0b, xhat) ||
                            ((uintptr_t)gamma_b % 16)))
        lg = 0;
    float* part_a = workspace;
    if (lg) {
        const int rpb = 256 / (H * lg);
        int blocks = cdiv(T, rpb);
        if (blocks > HN_VEC_BLOCKS) blocks = HN_VEC_BLOCKS;
        float* part_b = workspace + (size_t)blocks * 2 * W;
        HeadNormBlocks blk = {};
        blk.col0[0] = xcol0; blk.col0[1] = xcol0b; blk.dcol0[0] = dcol0; blk.dcol0[1] = dcol0b;
        blk.rstd[0] = const_cast<float*>(rstd); blk.rstd[1] = const_cast<float*>(rstd_b);
        blk.gamma[0] = gamma; blk.gamma[1] = gamma_b; blk.part[0] = part_a; blk.part[1] = part_b;
        dim3 grid(blocks, nblk);
#define HN_BWD(LG) launch_kernel(headnorm_bwd_vec_kernel<LG>, grid, 256, 0, st, dy, lddy, xhat, ldx, blk, T, H, dk)
        switch (lg) { case 1: HN_BWD(1); break; case 2: HN_BWD(2); break; case 4: HN_BWD(4); break;
                      case 8: HN_BWD(8); break; case 16: HN_BWD(16); break; default: HN_BWD(32); }
#undef HN_BWD
        launch_kernel(headnorm_bwd_reduce_kernel, dim3(cdiv(W, 32), 2), dim3(32, 32), 0, st, part_a, blocks, W, dgamma, dbeta,
                                                                                accumulate);
        if (nblk == 2)
            launch_kernel(headnorm_bwd_reduce_kernel, dim3(cdiv(W, 32), 2), dim3(32, 32), 0, st, part_b, blocks, W, dgamma_b,
                                                                                    dbeta_b, accumulate);
        return check_launch("gb200_headnorm_bwd", 1 + nblk);
    }
    size_t smem = (size_t)2 * HN_ROWS * (W + 1) * sizeof(float);
    GB_REQUIRE(smem <= 200 * 1024, "gb200_headnorm_bwd: H*d_k=%d too wide", W);
    if (smem > 48 * 1024)
        cudaFuncSetAttribute(headnorm_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int nblocks = cdiv(T, HN_ROWS);
    float* part_b = workspace + (size_t)nblocks * 2 * W;
    launch_kernel(headnorm_bwd_kernel, nblocks, 256, smem, st, dy, lddy, dcol0, xhat, ldx, xcol0, rstd, gamma, T, H, dk, part_a);
    launch_kernel(headnorm_bwd_reduce_kernel, dim3(cdiv(W, 32), 2), dim3(32, 32), 0, st, part_a, nblocks, W, dgamma, dbeta,
                                                                            accumulate);
    if (nblk == 2) {
        launch_kernel(headnorm_bwd_kernel, nblocks, 256, smem, st, dy, lddy, dcol0b, xhat, ldx, xcol0b, rstd_b, gamma_b, T, H, dk,
                                                        part_b);
        launch_kernel(headnorm_bwd_reduce_kernel, dim3(cdiv(W, 32), 2), dim3(32, 32), 0, st, part_b, nblocks, W, dgamma_b,
                                                                                dbeta_b, accumulate);
    }
    return check_launch("gb200_headnorm_bwd", 2 * nblk);
}

extern "C" int gb200_attn_suggest_nsplit(int B, int H, int n) {
    // The kernel is latency-bound (stage tokens -> sync -> contract): give every 64-token stage its own CTA so all
    // loads of the launch are in flight at once, instead of a few CTAs looping over stages.
    int s = (n + 63) / 64;
    if (s > 64) s = 64;
    return s < 1 ? 1 : s;
}

extern "C" size_t gb200_attn_xty_workspace_bytes(int B, int H, int d, int nsplit) {
    return (size_t)B * H * nsplit * d * d * sizeof(float);
}

extern "C" int gb200_attn_xty(int device, const gb200_head_operand* L, const gb200_head_operand* R,
                              const float* pos, int B, int H, int n, int dk, int p, float scale,
                              const unsigned char* keep_mask, float mask_p, unsigned long long mask_seed,
                              float* out, int nsplit, float* workspace, size_t workspace_bytes, int tensor_cores,
                              void* stream) {
    use_device(device);
    GB_REQUIRE(L && R && out && L->ptr && R->ptr, "gb200_attn_xty: null operand");
    GB_REQUIRE(B >= 1 && H >= 1 && n >= 1 && dk >= 1 && p >= 0, "gb200_attn_xty: bad shape");
    GB_REQUIRE(p == 0 || pos || (L->augmented && R->augmented), "gb200_attn_xty: pos is null but pos_dim=%d", p);
    const int d = dk + p, dp = pick_dp(d);
    GB_REQUIRE(dp != 0, "gb200_attn_xty: head width d_k+pos_dim=%d > 128 unsupported", d);
    if (nsplit < 1) nsplit = 1;
    GB_REQUIRE(workspace && workspace_bytes >= gb200_attn_xty_workspace_bytes(B, H, d, nsplit),
               "gb200_attn_xty: workspace too small");
    GB_REQUIRE(B * H <= 65535, "gb200_attn_xty: B*H too large");
    const int chunk = cdiv(n, nsplit);
    dim3 grid(nsplit, B * H);
    cudaStream_t st = as_stream(stream);
    HeadOperand l = make_op(L), r = make_op(R);
    if (tensor_cores && d <= 64) {       // warp-level TF32 MMA, tiles right-sized to d
        if (d <= 24) launch_kernel(xty_mma_kernel<2, 3>, grid, 256, 0, st, l, r, pos, p, dk, H, n, nsplit, chunk, workspace);
        else if (d <= 40) launch_kernel(xty_mma_kernel<3, 5>, grid, 256, 0, st, l, r, pos, p, dk, H, n, nsplit, chunk, workspace);
        else if (d <= 56) launch_kernel(xty_mma_kernel<4, 7>, grid, 256, 0, st, l, r, pos, p, dk, H, n, nsplit, chunk, workspace);
        else launch_kernel(xty_mma_kernel<4, 8>, grid, 256, 0, st, l, r, pos, p, dk, H, n, nsplit, chunk, workspace);
    } else
    if (dp == 32) launch_kernel(xty_kernel<32>, grid, 256, 0, st, l, r, pos, p, dk, H, n, nsplit, chunk, workspace);
    else if (dp == 64) launch_kernel(xty_kernel<64>, grid, 256, 0, st, l, r, pos, p, dk, H, n, nsplit, chunk, workspace);
    else launch_kernel(xty_kernel<128>, grid, 256, 0, st, l, r, pos, p, dk, H, n, nsplit, chunk, workspace);
    long long total = (long long)B * H * d * d;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    GB_REQUIRE(mask_p >= 0.f && mask_p < 1.f, "gb200_attn_xty: mask_p=%f outside [0,1)", mask_p);
    launch_kernel(xty_reduce_kernel, blocks, 256, 0, st, workspace, nsplit, d * d, total, scale, keep_mask, mask_p, mask_seed,
                                              rng_offset_ptr(), out);
    return check_launch("gb200_attn_xty", 2);
}

// scale tensor of the in-kernel attention dropout: out[e] = 0 or 1/(1-p), same stream as gb200_attn_xty
__global__ void philox_scale_kernel(float* __restrict__ out, long long total, float p, unsigned long long seed,
                                    const unsigned long long* seed_off) {
    pdl_enter();
    if (seed_off) seed += *seed_off;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x)
        out[e] = dropout_scale(p, seed, (unsigned long long)e);
}

extern "C" int gb200_philox_scale(int device, float* out, long long total, float p, unsigned long long seed,
                                  void* stream) {
    use_device(device);
    GB_REQUIRE(out && total >= 0 && p >= 0.f && p < 1.f, "gb200_philox_scale: bad arguments");
    if (total == 0) return GB200_OK;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    launch_kernel(philox_scale_kernel, blocks, 256, 0, as_stream(stream), out, total, p, seed, rng_offset_ptr());
    return check_launch("gb200_philox_scale");
}

extern "C" int gb200_attn_xm(int device, const gb200_head_operand* L, const float* pos, const float* M,
                             int transM, int B, int H, int n, int dk, int p, float* out, int ldo, int ocol0,
                             int out_augmented, float out_scale, int tensor_cores, void* stream) {
    use_device(device);
    GB_REQUIRE(L && L->ptr && M && out, "gb200_attn_xm: null operand");
    GB_REQUIRE(p == 0 || pos || L->augmented, "gb200_attn_xm: pos is null but pos_dim=%d", p);
    const int d = dk + p, dp = pick_dp(d);
    GB_REQUIRE(dp != 0, "gb200_attn_xm: head width d_k+pos_dim=%d > 128 unsupported", d);
    GB_REQUIRE(B * H <= 65535, "gb200_attn_xm: B*H too large");
    dim3 grid(cdiv(n, 64), B * H);
    size_t smem = (size_t)(dp + 64) * (dp + 1) * sizeof(float);
    cudaStream_t st = as_stream(stream);
    HeadOperand l = make_op(L);
    if (tensor_cores && d <= 64) {
#define LAUNCH_XMM(KT, NT, TT)                                                                               \
    launch_kernel(xm_mma_kernel<KT, NT, TT>, dim3(cdiv(n, TT), B * H), TT * 2, 0, st, l, pos, M, transM, p, dk, H, n, out, ldo, \
                                                                           ocol0, out_augmented, out_scale)
        if (d <= 24) LAUNCH_XMM(3, 3, 128);
        else if (d <= 40) LAUNCH_XMM(5, 5, 128);
        else if (d <= 56) LAUNCH_XMM(7, 7, 64);
        else LAUNCH_XMM(8, 8, 64);
#undef LAUNCH_XMM
        return check_launch("gb200_attn_xm");
    }
#define LAUNCH_XM(DPV)                                                                                  \
    do {                                                                                                \
        if (smem > 48 * 1024)                                                                           \
            cudaFuncSetAttribute(xm_kernel<DPV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        launch_kernel(xm_kernel<DPV>, grid, 256, smem, st, l, pos, M, transM, p, dk, H, n, out, ldo, ocol0,          \
                                               out_augmented, out_scale);                               \
    } while (0)
    if (dp == 32) LAUNCH_XM(32);
    else if (dp == 64) LAUNCH_XM(64);
    else LAUNCH_XM(128);
#undef LAUNCH_XM
    return check_launch("gb200_attn_xm");
}
