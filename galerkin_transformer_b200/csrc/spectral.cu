// Spectral convolution (FNO layer) as a mode-truncated DFT pipeline.
//
// The reference (libs/layers.py:1077-1106 SpectralConv1d, :1153-1197 SpectralConv2d) runs a
// full-size rfft -> keeps `modes` (2 x modes^2 in 2-D) coefficients -> complex channel mix ->
// zero-pads -> full-size irfft, with permute / stack / zeros / slice-assign / torch.complex
// copies in between (~375 MB of traffic per 2-D layer at Darcy 141^2 against 43 MB of
// algorithmic bytes).  Only m << n modes survive, so the transform pair is evaluated
// directly on the kept modes, channel-last, with precomputed twiddles:
//
//   ydft        T1[R,ky,c]   = s * c_ky? * sum_Y x[R,Y,c] e^{-i 2pi ky Y/n}      (rows R = (b,X) or b)
//   xdft        X^[b,r,ky,c] = s * sum_X T1[b,X,ky,c] e^{-i 2pi kx(r) X/n}       kx(r) = r | n-2m+r
//   mode_mix    O^[b,q,o]    = sum_i X^[b,q,i] * W[i,o,q]                         (complex, per mode q)
//   xidft       Z[b,X,ky,o]  = s * sum_r O^[b,r,ky,o] e^{+i 2pi kx(r) X/n}
//   yidft_epi   y[R,Y,o]     = act( s * sum_ky c_ky Re(Z[R,ky,o] e^{+i 2pi ky Y/n})
//                                   + sum_i x2[R,Y,i] Wm[i,o] + bias[o] )
//
// c_ky = 1 for ky = 0 (and Nyquist), 2 otherwise: the Hermitian fold that irfft applies; the
// imaginary part of the ky = 0 column is dropped exactly as pocketfft / cuFFT C2R do.  The
// backward pass is the same five kernels with the adjoint scalings (see functional.py), which
// reproduces autograd-through-rfft2/irfft2 to round-off (checked in tests against the oracle).
#include "common.cuh"
#include "spectral_mma.cuh"

namespace gb200 {

__device__ __forceinline__ float herm_weight(int ky, int n) {
    return (ky == 0 || (2 * ky == n)) ? 1.f : 2.f;
}

// ---------------------------------------------------------------- ydft ----------------------
constexpr int KYG = 16;   // ky handled per thread pass
constexpr int YCH = 64;   // Y values whose twiddles are staged per step

__global__ void __launch_bounds__(128) ydft_kernel(const float* __restrict__ x, long long RC, int C, int n, int m,
                                                   const float2* __restrict__ twY, float scale, int hermitian,
                                                   int nsplit, int ychunk, float2* __restrict__ out,
                                                   float2* __restrict__ part) {
    pdl_enter();
    __shared__ float2 tws[KYG][YCH];
    const int kg0 = blockIdx.z * KYG;
    const int nk = min(KYG, m - kg0);
    const int split = blockIdx.y;
    const int ybeg = split * ychunk, yend = min(n, ybeg + ychunk);
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = g < RC;
    const long long R = active ? g / C : 0;
    const int c = active ? (int)(g % C) : 0;
    float are[KYG], aim[KYG];
#pragma unroll
    for (int k = 0; k < KYG; ++k) { are[k] = 0.f; aim[k] = 0.f; }
    for (int y0 = ybeg; y0 < yend; y0 += YCH) {
        const int ny = min(YCH, yend - y0);
        __syncthreads();
        for (int e = threadIdx.x; e < KYG * YCH; e += blockDim.x) {
            int k = e / YCH, yy = e % YCH;
            tws[k][yy] = (k < nk && yy < ny) ? twY[(long long)(kg0 + k) * n + y0 + yy] : make_float2(0.f, 0.f);
        }
        __syncthreads();
        if (active) {
            // sixteen independent loads in flight per thread (the grid is only ~8 warps per SM: latency, not bandwidth, binds)
            const float* xp = x + (R * n + y0) * C + c;
            for (int yb = 0; yb < ny; yb += 16) {
                float v[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = (yb + j < ny) ? xp[(long long)(yb + j) * C] : 0.f;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
#pragma unroll
                    for (int k = 0; k < KYG; ++k) {
                        const float2 t = tws[k][yb + j];
                        are[k] = fmaf(v[j], t.x, are[k]);
                        aim[k] = fmaf(-v[j], t.y, aim[k]);
                    }
                }
            }
        }
    }
    if (!active) return;
#pragma unroll
    for (int k = 0; k < KYG; ++k) {
        if (k >= nk) break;
        const int ky = kg0 + k;
        if (nsplit == 1) {
            const float s = scale * (hermitian ? herm_weight(ky, n) : 1.f);
            out[(R * m + ky) * C + c] = make_float2(are[k] * s, aim[k] * s);
        } else {
            part[(((long long)split * (RC / C) + R) * m + ky) * C + c] = make_float2(are[k], aim[k]);
        }
    }
}

__global__ void ydft_reduce_kernel(const float2* __restrict__ part, int nsplit, long long total, int C, int m,
                                   int n, float scale, int hermitian, float2* __restrict__ out) {
    pdl_enter();
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        const int ky = (int)((e / C) % m);
        float sr = 0.f, si = 0.f;
        for (int s = 0; s < nsplit; ++s) {
            float2 v = part[(long long)s * total + e];
            sr += v.x; si += v.y;
        }
        const float sc = scale * (hermitian ? herm_weight(ky, n) : 1.f);
        out[e] = make_float2(sr * sc, si * sc);
    }
}

// ---------------------------------------------------------------- xdft / xidft --------------
// thread per (b, r, ky, c); loops over X
__global__ void xdft_kernel(const float2* __restrict__ T1, int B, int n, int m, int C,
                            const float2* __restrict__ twX, float scale, float2* __restrict__ out) {
    pdl_enter();
    const long long total = (long long)B * 2 * m * m * C;
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const int c = (int)(e % C);
    const int ky = (int)((e / C) % m);
    const int r = (int)((e / ((long long)C * m)) % (2 * m));
    const int b = (int)(e / ((long long)C * m * 2 * m));
    const float2* tp = T1 + (((long long)b * n) * m + ky) * C + c;
    const float2* tw = twX + (long long)r * n;
    const long long xstride = (long long)m * C;
    float are = 0.f, aim = 0.f;
#pragma unroll 4
    for (int X = 0; X < n; ++X) {
        const float2 t = tp[X * xstride];
        const float2 w = __ldg(tw + X);
        are = fmaf(t.x, w.x, fmaf(t.y, w.y, are));
        aim = fmaf(t.y, w.x, fmaf(-t.x, w.y, aim));
    }
    out[e] = make_float2(are * scale, aim * scale);
}

// thread per (b, X, ky, c); loops over r
__global__ void xidft_kernel(const float2* __restrict__ Oft, int B, int n, int m, int C,
                             const float2* __restrict__ twX, float scale, float2* __restrict__ Z) {
    pdl_enter();
    const long long total = (long long)B * n * m * C;
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const int c = (int)(e % C);
    const int ky = (int)((e / C) % m);
    const int X = (int)((e / ((long long)C * m)) % n);
    const int b = (int)(e / ((long long)C * m * n));
    const float2* op = Oft + (((long long)b * 2 * m) * m + ky) * C + c;
    const long long rstride = (long long)m * C;
    float zre = 0.f, zim = 0.f;
    for (int r0 = 0; r0 < 2 * m; r0 += 8) {
        float2 o[8], w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const bool ok = r0 + j < 2 * m;
            o[j] = ok ? op[(r0 + j) * rstride] : make_float2(0.f, 0.f);
            w[j] = ok ? __ldg(twX + (long long)(r0 + j) * n + X) : make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            zre = fmaf(o[j].x, w[j].x, fmaf(-o[j].y, w[j].y, zre));
            zim = fmaf(o[j].x, w[j].y, fmaf(o[j].y, w[j].x, zim));
        }
    }
    Z[e] = make_float2(zre * scale, zim * scale);
}

// ---------------------------------------------------------------- mode mix ------------------
// X^: (B, halves*M2, Ci) complex; W_half: (Ci, Co, M2) complex; O^: (B, halves*M2, Co) complex.
// One thread per mode: the weight read W[i,o,:] is a contiguous run of M2 complex numbers, so
// the 2*Ci*Co*M2 weight floats stream through exactly once, fully coalesced.
constexpr int MIXB = 2;    // batch entries per thread: small, so the grid has enough CTAs to stream W

__global__ void mix_fwd_kernel(const float2* __restrict__ Xf, const float2* __restrict__ W0,
                               const float2* __restrict__ W1, int B, int halves, int M2, int Ci, int Co,
                               float2* __restrict__ Of) {
    pdl_enter();
    const int mode = blockIdx.x * blockDim.x + threadIdx.x;
    const int o = blockIdx.y, half = blockIdx.z % halves, b0 = (blockIdx.z / halves) * MIXB;
    if (mode >= M2) return;
    const int nb = min(MIXB, B - b0);
    const float2* W = half == 0 ? W0 : W1;
    float are[MIXB], aim[MIXB];
#pragma unroll
    for (int b = 0; b < MIXB; ++b) { are[b] = 0.f; aim[b] = 0.f; }
    for (int i = 0; i < Ci; ++i) {
        const float2 w = W[((long long)i * Co + o) * M2 + mode];
#pragma unroll
        for (int b = 0; b < MIXB; ++b) {
            if (b < nb) {
                const float2 x = Xf[(((long long)(b0 + b) * halves + half) * M2 + mode) * Ci + i];
                are[b] = fmaf(x.x, w.x, fmaf(-x.y, w.y, are[b]));
                aim[b] = fmaf(x.x, w.y, fmaf(x.y, w.x, aim[b]));
            }
        }
    }
    for (int b = 0; b < nb; ++b)
        Of[(((long long)(b0 + b) * halves + half) * M2 + mode) * Co + o] = make_float2(are[b], aim[b]);
}

// dX^[b,q,i] = sum_o dO^[b,q,o] * conj(W[i,o,q])
__global__ void mix_bwd_x_kernel(const float2* __restrict__ dO, const float2* __restrict__ W0,
                                 const float2* __restrict__ W1, int B, int halves, int M2, int Ci, int Co,
                                 float2* __restrict__ dX) {
    pdl_enter();
    const int mode = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = blockIdx.y, half = blockIdx.z % halves, b0 = (blockIdx.z / halves) * MIXB;
    if (mode >= M2) return;
    const int nb = min(MIXB, B - b0);
    const float2* W = half == 0 ? W0 : W1;
    float are[MIXB], aim[MIXB];
#pragma unroll
    for (int b = 0; b < MIXB; ++b) { are[b] = 0.f; aim[b] = 0.f; }
    for (int o = 0; o < Co; ++o) {
        const float2 w = W[((long long)i * Co + o) * M2 + mode];
#pragma unroll
        for (int b = 0; b < MIXB; ++b) {
            if (b < nb) {
                const float2 g = dO[(((long long)(b0 + b) * halves + half) * M2 + mode) * Co + o];
                are[b] = fmaf(g.x, w.x, fmaf(g.y, w.y, are[b]));
                aim[b] = fmaf(g.y, w.x, fmaf(-g.x, w.y, aim[b]));
            }
        }
    }
    for (int b = 0; b < nb; ++b)
        dX[(((long long)(b0 + b) * halves + half) * M2 + mode) * Ci + i] = make_float2(are[b], aim[b]);
}

// dW[i,o,q] = sum_b conj(X^[b,q,i]) * dO^[b,q,o]      (written as (re, im) pairs, coalesced)
__global__ void mix_bwd_w_kernel(const float2* __restrict__ Xf, const float2* __restrict__ dO, int B,
                                 int halves, int M2, int Ci, int Co, float2* __restrict__ dW0,
                                 float2* __restrict__ dW1, int accumulate) {
    pdl_enter();
    const int mode = blockIdx.x * blockDim.x + threadIdx.x;
    const int o = blockIdx.y, half = blockIdx.z;
    if (mode >= M2) return;
    float2* dW = half == 0 ? dW0 : dW1;
    // batch entries in groups of 8: their dO values are loaded once, and for every input channel the 8 X^ loads are issued
    // together (the grid is small -- a few hundred warps -- so loads in flight per thread are what hides the latency)
    for (int i = 0; i < Ci; ++i) {
        float are = 0.f, aim = 0.f;
        for (int b0 = 0; b0 < B; b0 += 8) {
            float2 x[8], g[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const bool ok = b0 + j < B;
                const long long q = ((long long)(ok ? b0 + j : b0) * halves + half) * M2 + mode;
                x[j] = ok ? Xf[q * Ci + i] : make_float2(0.f, 0.f);
                g[j] = ok ? dO[q * Co + o] : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                are = fmaf(x[j].x, g[j].x, fmaf(x[j].y, g[j].y, are));
                aim = fmaf(x[j].x, g[j].y, fmaf(-x[j].y, g[j].x, aim));
            }
        }
        float2* dst = dW + ((long long)i * Co + o) * M2 + mode;
        if (accumulate) { float2 old = *dst; are += old.x; aim += old.y; }
        *dst = make_float2(are, aim);
    }
}

// ---------------------------------------------------------------- yidft + epilogue ----------
// CTA = one row R x a run of Y tiles.  Z[R] (m x Co complex) and the pointwise weight (Ci x Co)
// stay in shared memory; every thread produces 4 consecutive Y for one output channel so each
// weight / coefficient read from shared memory feeds 4 (resp. 8) FMAs.
constexpr int YT = 32;
constexpr int XP = YT + 4;   // pitch of the transposed x tile: float4-aligned, 4-way instead of 32-way store conflicts

__global__ void __launch_bounds__(256) yidft_epi_kernel(
    const float2* __restrict__ Z, int n, int m, int Co, const float2* __restrict__ twY, float scale,
    int hermitian, const float* __restrict__ x2, int Ci, const float* __restrict__ Wm,
    const float* __restrict__ bias, int act, float* __restrict__ y, float* __restrict__ zout,
    int tiles_per_cta) {
    pdl_enter();
    extern __shared__ __align__(16) float sm[];
    float* twc = sm;                                            // [m][YT]  cos * c_ky * scale
    float* tws = twc + m * YT;                                  // [m][YT]  sin * c_ky * scale
    float* xsT = tws + m * YT;                                  // [Ci][XP] (float4 reads: 16B aligned)
    float2* Zs = reinterpret_cast<float2*>(xsT + Ci * XP);      // [m][Co]
    float* Ws = xsT + Ci * XP + 2 * m * Co;                     // [Ci][Co]
    const long long R = blockIdx.x;
    for (int e = threadIdx.x; e < m * Co; e += blockDim.x) Zs[e] = Z[R * m * Co + e];
    for (int e = threadIdx.x; e < Ci * Co; e += blockDim.x) Ws[e] = Wm[e];
    const int tile0 = blockIdx.y * tiles_per_cta;
    for (int tile = tile0; tile < tile0 + tiles_per_cta; ++tile) {
        const int y0 = tile * YT;
        if (y0 >= n) break;
        const int ny = min(YT, n - y0);
        __syncthreads();
        for (int e = threadIdx.x; e < m * YT; e += blockDim.x) {
            int ky = e / YT, yy = e % YT;
            float2 t = make_float2(0.f, 0.f);
            if (yy < ny) t = twY[(long long)ky * n + y0 + yy];
            const float s = scale * (hermitian ? herm_weight(ky, n) : 1.f);
            twc[e] = t.x * s;
            tws[e] = t.y * s;
        }
        for (int e = threadIdx.x; e < YT * Ci; e += blockDim.x) {
            int yy = e / Ci, i = e % Ci;
            xsT[i * XP + yy] = (yy < ny) ? x2[((R * n) + y0 + yy) * Ci + i] : 0.f;
        }
        __syncthreads();
        for (int w = threadIdx.x; w < (YT / 4) * Co; w += blockDim.x) {
            const int o = w % Co, q = w / Co;
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
            for (int ky = 0; ky < m; ++ky) {
                const float2 z = Zs[ky * Co + o];
                const float4 cc = *reinterpret_cast<const float4*>(twc + ky * YT + q * 4);
                const float4 ss = *reinterpret_cast<const float4*>(tws + ky * YT + q * 4);
                a0 = fmaf(z.x, cc.x, fmaf(-z.y, ss.x, a0));
                a1 = fmaf(z.x, cc.y, fmaf(-z.y, ss.y, a1));
                a2 = fmaf(z.x, cc.z, fmaf(-z.y, ss.z, a2));
                a3 = fmaf(z.x, cc.w, fmaf(-z.y, ss.w, a3));
            }
            for (int i = 0; i < Ci; ++i) {
                const float wv = Ws[i * Co + o];
                const float4 xv = *reinterpret_cast<const float4*>(xsT + i * XP + q * 4);
                a0 = fmaf(xv.x, wv, a0);
                a1 = fmaf(xv.y, wv, a1);
                a2 = fmaf(xv.z, wv, a2);
                a3 = fmaf(xv.w, wv, a3);
            }
            const float bb = bias ? bias[o] : 0.f;
            const float av[4] = {a0 + bb, a1 + bb, a2 + bb, a3 + bb};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int yy = q * 4 + k;
                if (yy < ny) {
                    const long long idx = ((R * n) + y0 + yy) * Co + o;
                    if (zout) zout[idx] = av[k];
                    y[idx] = act_apply(act, av[k]);
                }
            }
        }
    }
}


// ---------------------------------------------------------------------------------------------------------------------
// Row kernels for 2-D grids (many short rows: R = B*n rows of n <= ~1000 points).  Same arithmetic as the kernels above
// (fp32 FMAs, sequential sums), restructured so that shared-memory traffic and load latency stop binding:
//   ydft_row    CTA = one row: the whole row and the twiddle table are staged once (all global loads in flight together),
//               a thread owns 3 modes of one channel and consumes 4 points per step with float4 twiddle reads
//   xdft_rows   CTA = (b, ky, 6 modes kx): 4 thread groups split X, 4 loads in flight each, shared-memory reduction
//   xidft_rows  CTA = (b, ky, 36 X): the (2m x C) coefficient column is staged once and reused for every X
//   yidft_row   register tile of 4 points x 4 channels per thread: each float4 read from shared memory feeds 16 FMAs
//               (the kernel above: 4) -- it was bound by shared-memory bandwidth at 18% of the FMA rate
// ---------------------------------------------------------------------------------------------------------------------
constexpr int YR_KPT = 3;

__global__ void __launch_bounds__(128) ydft_row_kernel(const float* __restrict__ x, int n, int NP, int C, int m,
                                                       const float2* __restrict__ twY, float scale, int hermitian,
                                                       float2* __restrict__ out) {
    pdl_enter();
    extern __shared__ __align__(16) float sm[];
    float* xs = sm;                  // [NP][C], rows >= n are zero
    float* twc = xs + NP * C;        // [m][NP]
    float* tws = twc + m * NP;       // [m][NP]
    const long long R = blockIdx.x;
    const float4* x4 = reinterpret_cast<const float4*>(x + R * n * C);
    const int n4 = n * C / 4, np4 = NP * C / 4;
#pragma unroll 4
    for (int e = threadIdx.x; e < np4; e += 128)
        reinterpret_cast<float4*>(xs)[e] = e < n4 ? x4[e] : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int e = threadIdx.x; e < m * NP; e += 128) {
        const int ky = e / NP, y = e % NP;
        const float2 t = y < n ? twY[(long long)ky * n + y] : make_float2(0.f, 0.f);
        twc[e] = t.x;
        tws[e] = t.y;
    }
    __syncthreads();
    const int nkg = (m + YR_KPT - 1) / YR_KPT;
    for (int item = threadIdx.x; item < C * nkg; item += 128) {
        const int c = item % C, k0 = (item / C) * YR_KPT;
        float are[YR_KPT], aim[YR_KPT];
        const float *pc[YR_KPT], *ps[YR_KPT];
#pragma unroll
        for (int j = 0; j < YR_KPT; ++j) {
            are[j] = 0.f; aim[j] = 0.f;
            const int kk = min(k0 + j, m - 1);
            pc[j] = twc + kk * NP;
            ps[j] = tws + kk * NP;
        }
        const float* xp = xs + c;
#pragma unroll 2
        for (int y = 0; y < NP; y += 4) {
            const float v0 = xp[y * C], v1 = xp[(y + 1) * C], v2 = xp[(y + 2) * C], v3 = xp[(y + 3) * C];
#pragma unroll
            for (int j = 0; j < YR_KPT; ++j) {
                const float4 cc = *reinterpret_cast<const float4*>(pc[j] + y);
                const float4 ss = *reinterpret_cast<const float4*>(ps[j] + y);
                are[j] = fmaf(v0, cc.x, are[j]); aim[j] = fmaf(-v0, ss.x, aim[j]);
                are[j] = fmaf(v1, cc.y, are[j]); aim[j] = fmaf(-v1, ss.y, aim[j]);
                are[j] = fmaf(v2, cc.z, are[j]); aim[j] = fmaf(-v2, ss.z, aim[j]);
                are[j] = fmaf(v3, cc.w, are[j]); aim[j] = fmaf(-v3, ss.w, aim[j]);
            }
        }
#pragma unroll
        for (int j = 0; j < YR_KPT; ++j) {
            const int ky = k0 + j;
            if (ky < m) {
                const float sc = scale * (hermitian ? herm_weight(ky, n) : 1.f);
                out[(R * m + ky) * C + c] = make_float2(are[j] * sc, aim[j] * sc);
            }
        }
    }
}

// Channel-blocked forward transform: a thread owns 4 channels x YQ_KPT modes of one row and every YQ-th point of it, so each
// twiddle word read from shared memory (a broadcast: 1 word per cycle, however wide the load) feeds 4 FMAs and each x
// value (one float4 straight from global memory) feeds 2*YQ_KPT.  ncu showed the first version latency-bound (long-scoreboard
// stalls at 23% occupancy): the x loads are double-buffered one batch ahead, and the twiddle table is filled with six
// independent loads per thread in flight.  The point split is 4-way (8-way, twice the warps, measured 35 against 21 us).
// The YQ point groups are reduced through shared memory in fixed order.
constexpr int YQ = 4;
constexpr int YQ_KPT = 6;
constexpr int YQ_UN = 6;

__global__ void __launch_bounds__(128) ydft_rowq_kernel(const float* __restrict__ x, long long R, int n, int P, int C, int m,
                                                        int CG, int KG, const float2* __restrict__ twY, float scale,
                                                        int hermitian, float2* __restrict__ out) {
    pdl_enter();
    extern __shared__ __align__(16) float sm[];
    constexpr int SLOTS = 128 / YQ;           // (row, cg, kg) slots per CTA
    constexpr int ACC = 2 * YQ_KPT * 4;
    float* twc = sm;                          // [KG*YQ_KPT][P]   rows >= m are zero
    float* tws = twc + KG * YQ_KPT * P;
    float* red = tws + KG * YQ_KPT * P;       // [YQ-1][SLOTS][ACC]
    const int TPR = CG * KG;                  // threads per (row, point group): a power of two <= SLOTS
    const int rows = SLOTS / TPR;
    for (int k0 = 0; k0 < KG * YQ_KPT; k0 += YQ_KPT) {
        for (int y = threadIdx.x; y < P; y += 128) {
            float2 t[YQ_KPT];
#pragma unroll
            for (int j = 0; j < YQ_KPT; ++j)
                t[j] = (k0 + j < m && y < n) ? twY[(long long)(k0 + j) * n + y] : make_float2(0.f, 0.f);
#pragma unroll
            for (int j = 0; j < YQ_KPT; ++j) {
                twc[(k0 + j) * P + y] = t[j].x;
                tws[(k0 + j) * P + y] = t[j].y;
            }
        }
    }
    __syncthreads();
    const int slot = threadIdx.x / YQ;
    const int yq = threadIdx.x % YQ;
    const int rl = slot / TPR, cg = (slot % TPR) % CG, kg = (slot % TPR) / CG;
    const long long row = (long long)blockIdx.x * rows + rl;
    const bool live = row < R;
    float are[YQ_KPT][4], aim[YQ_KPT][4];
#pragma unroll
    for (int k = 0; k < YQ_KPT; ++k)
#pragma unroll
        for (int j = 0; j < 4; ++j) { are[k][j] = 0.f; aim[k][j] = 0.f; }
    const float* xp = x + (live ? row : 0) * n * C + 4 * cg;
    const float* pc = twc + kg * YQ_KPT * P;
    const float* ps = tws + kg * YQ_KPT * P;
    constexpr int STEP = YQ * YQ_UN;
    auto load = [&](float4 (&v)[YQ_UN], int y0) {
#pragma unroll
        for (int u = 0; u < YQ_UN; ++u) {
            const int y = y0 + YQ * u;
            v[u] = (live && y < n) ? *reinterpret_cast<const float4*>(xp + (long long)y * C) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto consume = [&](const float4 (&v)[YQ_UN], int y0) {
#pragma unroll
        for (int u = 0; u < YQ_UN; ++u) {
            const int y = min(y0 + YQ * u, P - 1);          // v[u] is zero past the end of the row
#pragma unroll
            for (int k = 0; k < YQ_KPT; ++k) {
                const float c = pc[k * P + y], sn = ps[k * P + y];
                are[k][0] = fmaf(v[u].x, c, are[k][0]); aim[k][0] = fmaf(-v[u].x, sn, aim[k][0]);
                are[k][1] = fmaf(v[u].y, c, are[k][1]); aim[k][1] = fmaf(-v[u].y, sn, aim[k][1]);
                are[k][2] = fmaf(v[u].z, c, are[k][2]); aim[k][2] = fmaf(-v[u].z, sn, aim[k][2]);
                are[k][3] = fmaf(v[u].w, c, are[k][3]); aim[k][3] = fmaf(-v[u].w, sn, aim[k][3]);
            }
        }
    };
    float4 va[YQ_UN], vb[YQ_UN];
    load(va, yq);
    for (int y0 = yq; y0 < n; y0 += 2 * STEP) {
        load(vb, y0 + STEP);                 // next batch in flight while this one is consumed (zero past the end)
        consume(va, y0);
        if (y0 + STEP < n) {
            load(va, y0 + 2 * STEP);
            consume(vb, y0 + STEP);
        }
    }
    if (yq > 0) {
        float* r = red + ((yq - 1) * SLOTS + slot) * ACC;
#pragma unroll
        for (int k = 0; k < YQ_KPT; ++k)
#pragma unroll
            for (int j = 0; j < 4; ++j) { r[k * 8 + j] = are[k][j]; r[k * 8 + 4 + j] = aim[k][j]; }
    }
    __syncthreads();
    if (yq == 0 && live) {
#pragma unroll 1
        for (int q = 0; q < YQ - 1; ++q) {
            const float* r = red + (q * SLOTS + slot) * ACC;
#pragma unroll
            for (int k = 0; k < YQ_KPT; ++k)
#pragma unroll
                for (int j = 0; j < 4; ++j) { are[k][j] += r[k * 8 + j]; aim[k][j] += r[k * 8 + 4 + j]; }
        }
#pragma unroll
        for (int k = 0; k < YQ_KPT; ++k) {
            const int ky = kg * YQ_KPT + k;
            if (ky < m) {
                const float sc = scale * (hermitian ? herm_weight(ky, n) : 1.f);
                float4* o = reinterpret_cast<float4*>(out + (row * m + ky) * C + 4 * cg);
                o[0] = make_float4(are[k][0] * sc, aim[k][0] * sc, are[k][1] * sc, aim[k][1] * sc);
                o[1] = make_float4(are[k][2] * sc, aim[k][2] * sc, are[k][3] * sc, aim[k][3] * sc);
            }
        }
    }
}

constexpr int XD_RG = 6;    // modes kx per CTA

constexpr int XD_XQ = 8;    // thread groups splitting X (one warp each)

__global__ void __launch_bounds__(32 * XD_XQ) xdft_rows_kernel(const float2* __restrict__ T1, int n, int m, int C,
                                                               const float2* __restrict__ twX, float scale,
                                                               float2* __restrict__ out) {
    pdl_enter();
    __shared__ float2 red[XD_XQ - 1][XD_RG][32];
    extern __shared__ __align__(16) float2 tw2[];          // [XD_RG][n]
    const int r0 = blockIdx.x * XD_RG, ky = blockIdx.y, b = blockIdx.z;
    const int nr = min(XD_RG, 2 * m - r0);
    for (int X = threadIdx.x; X < n; X += blockDim.x) {
        float2 t[XD_RG];
#pragma unroll
        for (int j = 0; j < XD_RG; ++j) t[j] = j < nr ? twX[(long long)(r0 + j) * n + X] : make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < XD_RG; ++j) tw2[j * n + X] = t[j];
    }
    __syncthreads();
    const int cl = threadIdx.x % 32, xq = threadIdx.x / 32;
    const long long xstride = (long long)m * C;
    constexpr int STEP = 4 * XD_XQ;
    for (int c0 = 0; c0 < C; c0 += 32) {
        const int c = c0 + cl;
        const bool cok = c < C;
        float are[XD_RG], aim[XD_RG];
#pragma unroll
        for (int j = 0; j < XD_RG; ++j) { are[j] = 0.f; aim[j] = 0.f; }
        const float2* tp = T1 + (((long long)b * n) * m + ky) * C + (cok ? c : 0);
        auto load = [&](float2 (&t)[4], int X0) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int X = X0 + XD_XQ * u;
                t[u] = (cok && X < n) ? tp[X * xstride] : make_float2(0.f, 0.f);
            }
        };
        auto consume = [&](const float2 (&t)[4], int X0) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int X = min(X0 + XD_XQ * u, n - 1);          // t[u] is zero past the end
#pragma unroll
                for (int j = 0; j < XD_RG; ++j) {
                    const float2 w = tw2[j * n + X];
                    are[j] = fmaf(t[u].x, w.x, fmaf(t[u].y, w.y, are[j]));
                    aim[j] = fmaf(t[u].y, w.x, fmaf(-t[u].x, w.y, aim[j]));
                }
            }
        };
        float2 ta[4], tb[4];
        load(ta, xq);
        for (int X0 = xq; X0 < n; X0 += 2 * STEP) {
            load(tb, X0 + STEP);
            consume(ta, X0);
            if (X0 + STEP < n) {
                load(ta, X0 + 2 * STEP);
                consume(tb, X0 + STEP);
            }
        }
        if (xq > 0) {
#pragma unroll
            for (int j = 0; j < XD_RG; ++j) red[xq - 1][j][cl] = make_float2(are[j], aim[j]);
        }
        __syncthreads();
        if (xq == 0 && cok) {
#pragma unroll
            for (int j = 0; j < XD_RG; ++j) {
                if (j < nr) {
                    float sr = are[j], si = aim[j];
#pragma unroll
                    for (int q = 0; q < XD_XQ - 1; ++q) { sr += red[q][j][cl].x; si += red[q][j][cl].y; }
                    out[(((long long)b * 2 * m + r0 + j) * m + ky) * C + c] = make_float2(sr * scale, si * scale);
                }
            }
        }
        __syncthreads();
    }
}

constexpr int XI_XC = 36;   // X per CTA: 4 thread groups x 3 passes x 3 X per pass

__global__ void __launch_bounds__(128) xidft_rows_kernel(const float2* __restrict__ Oft, int n, int m, int C,
                                                         const float2* __restrict__ twX, float scale,
                                                         float2* __restrict__ Z) {
    pdl_enter();
    extern __shared__ __align__(16) float2 sm2[];
    float2* Os = sm2;                       // [2m][32]   one 32-channel block of O^[b, :, ky, :]
    float2* tw = Os + 2 * m * 32;           // [2m][XI_XC]
    const int x0 = blockIdx.x * XI_XC, ky = blockIdx.y, b = blockIdx.z;
    const int m2 = 2 * m;
    for (int e = threadIdx.x; e < m2 * XI_XC; e += 128) {
        const int r = e / XI_XC, X = x0 + e % XI_XC;
        tw[e] = X < n ? twX[(long long)r * n + X] : make_float2(0.f, 0.f);
    }
    const int cl = threadIdx.x % 32, xq = threadIdx.x / 32;
    for (int c0 = 0; c0 < C; c0 += 32) {
        __syncthreads();
        for (int e = threadIdx.x; e < m2 * 32; e += 128) {
            const int r = e / 32, cc = c0 + e % 32;
            Os[e] = cc < C ? Oft[(((long long)b * m2 + r) * m + ky) * C + cc] : make_float2(0.f, 0.f);
        }
        __syncthreads();
        const int c = c0 + cl;
        for (int i0 = xq; i0 < XI_XC; i0 += 12) {
            float zr[3] = {0.f, 0.f, 0.f}, zi[3] = {0.f, 0.f, 0.f};
#pragma unroll 4
            for (int r = 0; r < m2; ++r) {
                const float2 o = Os[r * 32 + cl];
#pragma unroll
                for (int u = 0; u < 3; ++u) {
                    const float2 w = tw[r * XI_XC + i0 + 4 * u];
                    zr[u] = fmaf(o.x, w.x, fmaf(-o.y, w.y, zr[u]));
                    zi[u] = fmaf(o.x, w.y, fmaf(o.y, w.x, zi[u]));
                }
            }
#pragma unroll
            for (int u = 0; u < 3; ++u) {
                const int X = x0 + i0 + 4 * u;
                if (X < n && c < C) Z[(((long long)b * n + X) * m + ky) * C + c] = make_float2(zr[u] * scale, zi[u] * scale);
            }
        }
    }
}

template <int YG>
__global__ void __launch_bounds__(512) yidft_row_kernel(
    const float2* __restrict__ Z, int n, int m, int Co, const float2* __restrict__ twY, float scale, int hermitian,
    const float* __restrict__ x2, int Ci, const float* __restrict__ Wm, const float* __restrict__ bias, int act,
    float* __restrict__ y, float* __restrict__ zout, int tiles_per_cta) {
    pdl_enter();
    constexpr int YT = 4 * YG;
    extern __shared__ __align__(16) float sm[];
    const int XP = Ci + 4;                 // row pitch of the x tile: rows yg..yg+3 of a warp fall in distinct banks
    float* zre = sm;                       // [m][Co]   c_ky * scale * Re Z
    float* zim = zre + m * Co;             // [m][Co]  -c_ky * scale * Im Z
    float* Ws = zim + m * Co;              // [Ci][Co]
    float* twc = Ws + Ci * Co;             // [m][YT]   column p = 4*yg + j  <->  point yg + YG*j
    float* tws = twc + m * YT;             // [m][YT]
    float* xs = tws + m * YT;              // [YT][XP]
    const int OG = Co / 4;
    const int og = threadIdx.x % OG, yg = threadIdx.x / OG;
    const long long R = blockIdx.x;
    for (int e = threadIdx.x; e < m * Co; e += blockDim.x) {
        const int ky = e / Co;
        const float s = scale * (hermitian ? herm_weight(ky, n) : 1.f);
        const float2 z = Z[R * m * Co + e];
        zre[e] = z.x * s;
        zim[e] = -z.y * s;
    }
    for (int e = threadIdx.x; e < Ci * Co / 4; e += blockDim.x)
        reinterpret_cast<float4*>(Ws)[e] = reinterpret_cast<const float4*>(Wm)[e];
    const float4 bb = bias ? *reinterpret_cast<const float4*>(bias + 4 * og) : make_float4(0.f, 0.f, 0.f, 0.f);
    const int c4 = Ci / 4;
    const int tile0 = blockIdx.y * tiles_per_cta;
    for (int tile = tile0; tile < tile0 + tiles_per_cta; ++tile) {
        const int y0 = tile * YT;
        if (y0 >= n) break;
        __syncthreads();
        for (int e = threadIdx.x; e < m * YT; e += blockDim.x) {
            const int ky = e / YT, p = e % YT;
            const int Y = y0 + (p >> 2) + YG * (p & 3);
            const float2 t = Y < n ? twY[(long long)ky * n + Y] : make_float2(0.f, 0.f);
            twc[e] = t.x;
            tws[e] = t.y;
        }
        for (int e = threadIdx.x; e < YT * c4; e += blockDim.x) {
            const int r = e / c4, q = e % c4;
            const int Y = y0 + r;
            *reinterpret_cast<float4*>(xs + r * XP + 4 * q) =
                Y < n ? *reinterpret_cast<const float4*>(x2 + ((R * n) + Y) * Ci + 4 * q) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        __syncthreads();
        float acc[4][4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int o = 0; o < 4; ++o) acc[j][o] = 0.f;
        for (int ky = 0; ky < m; ++ky) {
            const float4 zr = *reinterpret_cast<const float4*>(zre + ky * Co + 4 * og);
            const float4 zi = *reinterpret_cast<const float4*>(zim + ky * Co + 4 * og);
            const float4 cc = *reinterpret_cast<const float4*>(twc + ky * YT + 4 * yg);
            const float4 ss = *reinterpret_cast<const float4*>(tws + ky * YT + 4 * yg);
            const float cj[4] = {cc.x, cc.y, cc.z, cc.w}, sj[4] = {ss.x, ss.y, ss.z, ss.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                acc[j][0] = fmaf(zr.x, cj[j], fmaf(zi.x, sj[j], acc[j][0]));
                acc[j][1] = fmaf(zr.y, cj[j], fmaf(zi.y, sj[j], acc[j][1]));
                acc[j][2] = fmaf(zr.z, cj[j], fmaf(zi.z, sj[j], acc[j][2]));
                acc[j][3] = fmaf(zr.w, cj[j], fmaf(zi.w, sj[j], acc[j][3]));
            }
        }
        for (int i4 = 0; i4 < c4; ++i4) {
            float xv[4][4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 v = *reinterpret_cast<const float4*>(xs + (yg + YG * j) * XP + 4 * i4);
                xv[j][0] = v.x; xv[j][1] = v.y; xv[j][2] = v.z; xv[j][3] = v.w;
            }
#pragma unroll
            for (int ii = 0; ii < 4; ++ii) {
                const float4 w = *reinterpret_cast<const float4*>(Ws + (4 * i4 + ii) * Co + 4 * og);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    acc[j][0] = fmaf(xv[j][ii], w.x, acc[j][0]);
                    acc[j][1] = fmaf(xv[j][ii], w.y, acc[j][1]);
                    acc[j][2] = fmaf(xv[j][ii], w.z, acc[j][2]);
                    acc[j][3] = fmaf(xv[j][ii], w.w, acc[j][3]);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int Y = y0 + yg + YG * j;
            if (Y < n) {
                const float4 v = make_float4(acc[j][0] + bb.x, acc[j][1] + bb.y, acc[j][2] + bb.z, acc[j][3] + bb.w);
                const long long idx = ((R * n) + Y) * Co + 4 * og;
                if (zout) *reinterpret_cast<float4*>(zout + idx) = v;
                *reinterpret_cast<float4*>(y + idx) =
                    make_float4(act_apply(act, v.x), act_apply(act, v.y), act_apply(act, v.z), act_apply(act, v.w));
            }
        }
    }
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace gb200

using namespace gb200;

extern "C" int gb200_spectral_suggest_ysplit(long long R, int C, int n) {
    long long ctas = (R * C + 127) / 128;
    if (ctas >= 148 || n < 4 * YCH) return 1;
    int want = (int)((2 * 148 + ctas - 1) / ctas);
    int maxs = n / (2 * YCH);
    int s = want < maxs ? want : maxs;
    return s < 1 ? 1 : s;
}

extern "C" size_t gb200_spectral_ydft_workspace_bytes(long long R, int C, int m, int nsplit) {
    return nsplit > 1 ? (size_t)nsplit * R * m * C * 2 * sizeof(float) : 0;
}

extern "C" int gb200_spectral_ydft(int device, const float* x, long long R, int n, int C, int m,
                                   const float* twY, float scale, int hermitian, float* out, int nsplit,
                                   float* workspace, size_t workspace_bytes, int tensor_cores, void* stream) {
    use_device(device);
    GB_REQUIRE(x && twY && out && R >= 1 && n >= 1 && C >= 1 && m >= 1, "gb200_spectral_ydft: bad arguments");
    GB_REQUIRE(m <= n / 2 + 1, "gb200_spectral_ydft: modes=%d exceeds n/2+1 for n=%d", m, n);
    if (nsplit < 1) nsplit = 1;
    if (nsplit > 1)
        GB_REQUIRE(workspace && workspace_bytes >= gb200_spectral_ydft_workspace_bytes(R, C, m, nsplit),
                   "gb200_spectral_ydft: workspace too small");
    cudaStream_t st = as_stream(stream);
    if (tensor_cores && 2 * m <= 32 && C % 8 == 0 && C <= 64 && R >= 128 && n <= 1024) {
        // per-row twiddle GEMM on warp-level TF32 MMA (2-D grids: many rows, short transform length)
        const int KP = (n + 7) / 8 * 8;
        const int AP = KP + ((4 - KP % 32 + 32) % 32);
        const size_t smem = (size_t)32 * AP * sizeof(float);
        dim3 grid(cdiv(R, SM_WARPS));
#define YD(NT)                                                                                                 \
    do {                                                                                                       \
        if (smem > 48 * 1024)                                                                                  \
            cudaFuncSetAttribute(ydft_mma_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        launch_kernel(ydft_mma_kernel<NT>, grid, SM_WARPS * 32, smem, st, x, R, n, C, m, reinterpret_cast<const float2*>(twY), \
                                                              scale, hermitian, reinterpret_cast<float2*>(out)); \
    } while (0)
        switch (C / 8) { case 1: YD(1); break; case 2: YD(2); break; case 3: YD(3); break; case 4: YD(4); break;
                         case 5: YD(5); break; case 6: YD(6); break; case 7: YD(7); break; default: YD(8); }
#undef YD
        return check_launch("gb200_spectral_ydft");
    }
    if (nsplit == 1 && C % 4 == 0 && R >= 148 && R <= 0x7fffffffLL && aligned16(x) && aligned16(out)) {
        const int CG = C / 4, KG = cdiv(m, YQ_KPT), TPR = CG * KG;
        const int P = n | 1;                              // odd pitch: the KG mode groups of a warp fall in distinct banks
        const size_t smem = (size_t)(2 * KG * YQ_KPT * P + (YQ - 1) * (128 / YQ) * 2 * YQ_KPT * 4) * sizeof(float);
        if (TPR <= 32 && (TPR & (TPR - 1)) == 0 && smem <= 96 * 1024) {
            const int rows = (128 / YQ) / TPR;
            if (smem > 48 * 1024)
                cudaFuncSetAttribute(ydft_rowq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            launch_kernel(ydft_rowq_kernel, dim3((unsigned)cdiv(R, rows)), 128, smem, st, x, R, n, P, C, m, CG, KG,
                          reinterpret_cast<const float2*>(twY), scale, hermitian, reinterpret_cast<float2*>(out));
            return check_launch("gb200_spectral_ydft");
        }
    }
    {
        const int NP = (n + 3) / 4 * 4;
        const size_t smem = (size_t)(NP * C + 2 * m * NP) * sizeof(float);
        if (nsplit == 1 && C % 4 == 0 && R >= 148 && R <= 0x7fffffffLL && smem <= 96 * 1024 && aligned16(x)) {
            if (smem > 48 * 1024)
                cudaFuncSetAttribute(ydft_row_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            launch_kernel(ydft_row_kernel, dim3((unsigned)R), 128, smem, st, x, n, NP, C, m,
                       reinterpret_cast<const float2*>(twY), scale, hermitian, reinterpret_cast<float2*>(out));
            return check_launch("gb200_spectral_ydft");
        }
    }
    const long long RC = R * C;
    int ychunk = cdiv(cdiv(n, nsplit), YCH) * YCH;
    nsplit = cdiv(n, ychunk);
    dim3 grid(cdiv(RC, 128), nsplit, cdiv(m, KYG));
    GB_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "gb200_spectral_ydft: grid too large");
    launch_kernel(ydft_kernel, grid, 128, 0, st, x, RC, C, n, m, reinterpret_cast<const float2*>(twY), scale, hermitian,
                                      nsplit, ychunk, reinterpret_cast<float2*>(out),
                                      reinterpret_cast<float2*>(workspace));
    if (nsplit > 1) {
        long long total = R * m * C;
        int blocks = (int)((total + 255) / 256);
        if (blocks > 148 * 8) blocks = 148 * 8;
        launch_kernel(ydft_reduce_kernel, blocks, 256, 0, st, reinterpret_cast<const float2*>(workspace), nsplit, total, C,
                                                   m, n, scale, hermitian, reinterpret_cast<float2*>(out));
    }
    return check_launch("gb200_spectral_ydft", nsplit > 1 ? 2 : 1);
}

extern "C" int gb200_spectral_xdft(int device, const float* T1, int B, int n, int m, int C, const float* twX,
                                   float scale, int inverse, float* out, void* stream) {
    use_device(device);
    GB_REQUIRE(T1 && twX && out && B >= 1 && n >= 1 && m >= 1 && C >= 1, "gb200_spectral_xdft: bad arguments");
    GB_REQUIRE(2 * m <= n, "gb200_spectral_xdft: 2*modes=%d exceeds n=%d (mode blocks would overlap)", 2 * m, n);
    cudaStream_t st = as_stream(stream);
    if (B <= 65535 && m <= 65535) {
        if (!inverse) {
            const size_t smem = (size_t)XD_RG * n * sizeof(float2);
            if (smem <= 36 * 1024) {          // + 10.5 KB of static reduction buffer: stays under the 48 KB default limit
                launch_kernel(xdft_rows_kernel, dim3(cdiv(2 * m, XD_RG), m, B), 32 * XD_XQ, smem, st,
                           reinterpret_cast<const float2*>(T1), n, m, C, reinterpret_cast<const float2*>(twX), scale,
                           reinterpret_cast<float2*>(out));
                return check_launch("gb200_spectral_xdft");
            }
        } else {
            const size_t smem = (size_t)2 * m * (32 + XI_XC) * sizeof(float2);
            if (smem <= 48 * 1024) {
                launch_kernel(xidft_rows_kernel, dim3(cdiv(n, XI_XC), m, B), 128, smem, st,
                           reinterpret_cast<const float2*>(T1), n, m, C, reinterpret_cast<const float2*>(twX), scale,
                           reinterpret_cast<float2*>(out));
                return check_launch("gb200_spectral_xdft");
            }
        }
    }
    if (!inverse) {
        long long total = (long long)B * 2 * m * m * C;
        launch_kernel(xdft_kernel, cdiv(total, 128), 128, 0, st, reinterpret_cast<const float2*>(T1), B, n, m, C,
                                                      reinterpret_cast<const float2*>(twX), scale,
                                                      reinterpret_cast<float2*>(out));
    } else {
        long long total = (long long)B * n * m * C;
        launch_kernel(xidft_kernel, cdiv(total, 256), 256, 0, st, reinterpret_cast<const float2*>(T1), B, n, m, C,
                                                       reinterpret_cast<const float2*>(twX), scale,
                                                       reinterpret_cast<float2*>(out));
    }
    return check_launch("gb200_spectral_xdft");
}

static int mix_threads(int M2) { int t = ((M2 + 31) / 32) * 32; return t > 256 ? 256 : t; }

extern "C" int gb200_spectral_mix_fwd(int device, const float* Xf, const float* W0, const float* W1, int B,
                                      int halves, int M2, int Ci, int Co, float* Of, void* stream) {
    use_device(device);
    GB_REQUIRE(Xf && W0 && Of && (halves == 1 || (halves == 2 && W1)), "gb200_spectral_mix_fwd: bad arguments");
    int th = mix_threads(M2);
    dim3 grid(cdiv(M2, th), Co, halves * cdiv(B, MIXB));
    GB_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "gb200_spectral_mix_fwd: grid too large");
    launch_kernel(mix_fwd_kernel, grid, th, 0, as_stream(stream), reinterpret_cast<const float2*>(Xf),
                                                       reinterpret_cast<const float2*>(W0),
                                                       reinterpret_cast<const float2*>(W1), B, halves, M2, Ci, Co,
                                                       reinterpret_cast<float2*>(Of));
    return check_launch("gb200_spectral_mix_fwd");
}

extern "C" int gb200_spectral_mix_bwd(int device, const float* Xf, const float* dO, const float* W0,
                                      const float* W1, int B, int halves, int M2, int Ci, int Co, float* dX,
                                      float* dW0, float* dW1, int accumulate_dw, void* stream) {
    use_device(device);
    GB_REQUIRE(Xf && dO && W0 && (halves == 1 || (halves == 2 && W1)), "gb200_spectral_mix_bwd: bad arguments");
    int th = mix_threads(M2);
    cudaStream_t st = as_stream(stream);
    if (dX) {
        dim3 grid(cdiv(M2, th), Ci, halves * cdiv(B, MIXB));
        launch_kernel(mix_bwd_x_kernel, grid, th, 0, st, reinterpret_cast<const float2*>(dO),
                                              reinterpret_cast<const float2*>(W0),
                                              reinterpret_cast<const float2*>(W1), B, halves, M2, Ci, Co,
                                              reinterpret_cast<float2*>(dX));
    }
    if (dW0) {
        GB_REQUIRE(halves == 1 || dW1, "gb200_spectral_mix_bwd: dW1 is null");
        dim3 grid(cdiv(M2, th), Co, halves);
        launch_kernel(mix_bwd_w_kernel, grid, th, 0, st, reinterpret_cast<const float2*>(Xf),
                                              reinterpret_cast<const float2*>(dO), B, halves, M2, Ci, Co,
                                              reinterpret_cast<float2*>(dW0), reinterpret_cast<float2*>(dW1),
                                              accumulate_dw);
    }
    return check_launch("gb200_spectral_mix_bwd", (dX ? 1 : 0) + (dW0 ? 1 : 0));
}

extern "C" int gb200_spectral_yidft_epilogue(int device, const float* Z, long long R, int n, int m, int Co,
                                             const float* twY, float scale, int hermitian, const float* x2,
                                             int Ci, const float* Wm, const float* bias, int act, float* y,
                                             float* zout, int tensor_cores, void* stream) {
    use_device(device);
    GB_REQUIRE(Z && twY && x2 && Wm && y, "gb200_spectral_yidft_epilogue: null argument");
    GB_REQUIRE(R >= 1 && R <= 0x7fffffffLL && n >= 1 && m >= 1 && Co >= 1 && Ci >= 1,
               "gb200_spectral_yidft_epilogue: bad shape");
    if (tensor_cores && 2 * m <= 32 && Co <= 64 && Ci <= 64 && n <= 16384) {
        const int KS = (2 * m + 7) / 8 * 8, MP = (n + 15) / 16 * 16;
        const int SP = KS + ((4 - KS % 32 + 32) % 32);
        const size_t smem2 = (size_t)MP * SP * sizeof(float);
        if (smem2 <= 200 * 1024) {
            const int mtiles = MP / 16;
            int tiles_per_warp = mtiles;               // one warp per row unless rows alone cannot fill the GPU
            while (tiles_per_warp > 4 && R * cdiv(mtiles, tiles_per_warp) < 8 * 148 * SM_WARPS)
                tiles_per_warp = (tiles_per_warp + 1) / 2;
            const int chunks = cdiv(mtiles, tiles_per_warp);
            const long long warps = R * chunks;
            dim3 grid((unsigned)cdiv(warps, SM_WARPS));
            const int nt = (Co + 7) / 8;
            cudaStream_t st2 = as_stream(stream);
#define YI(NT)                                                                                                   \
    do {                                                                                                         \
        if (smem2 > 48 * 1024)                                                                                   \
            cudaFuncSetAttribute(yidft_mma_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2); \
        launch_kernel(yidft_mma_kernel<NT>, grid, SM_WARPS * 32, smem2, st2, \
            reinterpret_cast<const float2*>(Z), R, n, m, Co, reinterpret_cast<const float2*>(twY), scale, hermitian, \
            x2, Ci, Wm, bias, act, y, zout, tiles_per_warp, chunks);                                             \
    } while (0)
            switch (nt) { case 1: YI(1); break; case 2: YI(2); break; case 3: YI(3); break; case 4: YI(4); break;
                          case 5: YI(5); break; case 6: YI(6); break; case 7: YI(7); break; default: YI(8); }
#undef YI
            return check_launch("gb200_spectral_yidft_epilogue");
        }
    }
    if (Co % 8 == 0 && Co <= 128 && Ci % 4 == 0 && R >= 148 && aligned16(x2) && aligned16(Wm) &&
        aligned16(y) && (!zout || aligned16(zout)) && (!bias || aligned16(bias))) {
        const int OG = Co / 4;
        const int pad12 = cdiv(n, 48) * 48, pad16 = cdiv(n, 64) * 64;
        const int YG = (pad12 <= pad16 && (12 * OG) % 32 == 0 && 12 * OG <= 512) ? 12 : 16;
        const int YTr = 4 * YG, threads = YG * OG;
        const size_t smr = (size_t)(2 * m * Co + Ci * Co + 2 * m * YTr + YTr * (Ci + 4)) * sizeof(float);
        if (threads <= 512 && threads % 32 == 0 && smr <= 64 * 1024) {
            const int ntl = cdiv(n, YTr);
            int tpc = ntl;
            while (tpc > 1 && R * cdiv(ntl, tpc) < 4 * 148) tpc = (tpc + 1) / 2;
            dim3 gridr((unsigned)R, cdiv(ntl, tpc));
            cudaStream_t str = as_stream(stream);
            if (YG == 12) {
                if (smr > 48 * 1024)
                    cudaFuncSetAttribute(yidft_row_kernel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smr);
                launch_kernel(yidft_row_kernel<12>, gridr, threads, smr, str, reinterpret_cast<const float2*>(Z), n, m, Co,
                           reinterpret_cast<const float2*>(twY), scale, hermitian, x2, Ci, Wm, bias, act, y, zout, tpc);
            } else {
                if (smr > 48 * 1024)
                    cudaFuncSetAttribute(yidft_row_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smr);
                launch_kernel(yidft_row_kernel<16>, gridr, threads, smr, str, reinterpret_cast<const float2*>(Z), n, m, Co,
                           reinterpret_cast<const float2*>(twY), scale, hermitian, x2, Ci, Wm, bias, act, y, zout, tpc);
            }
            return check_launch("gb200_spectral_yidft_epilogue");
        }
    }
    size_t smem = (size_t)(2 * m * Co + Ci * Co + 2 * m * YT + Ci * XP) * sizeof(float);
    GB_REQUIRE(smem <= 200 * 1024, "gb200_spectral_yidft_epilogue: tile needs %zu B of shared memory", smem);
    if (smem > 48 * 1024)
        cudaFuncSetAttribute(yidft_epi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int ntiles = cdiv(n, YT);
    // enough CTAs to fill the machine a few times over; rows first, then Y tiles
    int tiles_per_cta = ntiles;
    while (tiles_per_cta > 1 && R * cdiv(ntiles, tiles_per_cta) < 4 * 148) tiles_per_cta = (tiles_per_cta + 1) / 2;
    dim3 grid((unsigned)R, cdiv(ntiles, tiles_per_cta));
    launch_kernel(yidft_epi_kernel, grid, 256, smem, as_stream(stream), reinterpret_cast<const float2*>(Z), n, m, Co,
                                                            reinterpret_cast<const float2*>(twY), scale, hermitian,
                                                            x2, Ci, Wm, bias, act, y, zout, tiles_per_cta);
    return check_launch("gb200_spectral_yidft_epilogue");
}
