// Exact-fp32 SIMT GEMM with a fused epilogue (bias, activation, Philox dropout, signed
// residual, pre-activation side output) and deterministic split-K.
//
// This is the precise path of the library (fp32 FMA, no TF32 rounding): it serves the
// contractions whose shapes do not fit a tcgen05 tile (K = 2 grid columns, N = 1 output
// head, weight-gradient reductions over tokens) and is the on-device cross-check for the
// tensor-core GEMM in gemm_tc.cu.
//
//   C[b] = R[b] + rscale * drop( act( alpha * op(A[b]) . op(B[b]) + bias ) )      (+= if accumulate)
//
// Replaces, on the reference side, every nn.Linear / torch.matmul on the hot path:
// libs/layers.py:837-839 (Q,K,V projections), :896-897 (fc), :980-986 (FeedForward),
// :1083/:1172 (SpectralConv residual Linear) and libs/model.py:615-617, 629 (regressor).
#include "common.cuh"
#include "gemm_epilogue.cuh"

namespace gb200 {

constexpr int BM = 64, BN = 64, BK = 16, PAD = 4, NT = 256;

struct GemmArgs {
    const float* A; const float* B;
    int M, N, K, lda, ldb;
    long long sA, sB;
    int nbatch, ksplit, kchunk;
    GemmEpilogue ep;
    float* ws;
    int vecA, vecB;
};

// 4 consecutive elements along the contiguous storage dimension, zero-filled out of range.
__device__ __forceinline__ float4 load4(const float* base, long long row, int ld, int col, int nrows,
                                        int ncols, bool vec) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row >= nrows) return v;
    const float* p = base + row * ld + col;
    if (vec && col + 3 < ncols) return *reinterpret_cast<const float4*>(p);
    if (col + 0 < ncols) v.x = p[0];
    if (col + 1 < ncols) v.y = p[1];
    if (col + 2 < ncols) v.z = p[2];
    if (col + 3 < ncols) v.w = p[3];
    return v;
}

template <bool TA, bool TB>
__global__ void __launch_bounds__(NT) gemm_simt_kernel(GemmArgs g) {
    pdl_enter();
    __shared__ __align__(16) float As[2][BK][BM + PAD];
    __shared__ __align__(16) float Bs[2][BK][BN + PAD];
    const int tid = threadIdx.x;
    const int batch = blockIdx.z / g.ksplit, split = blockIdx.z % g.ksplit;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const float* A = g.A + (long long)batch * g.sA;
    const float* B = g.B + (long long)batch * g.sB;
    const int kbeg = split * g.kchunk;
    const int kend = min(g.K, kbeg + g.kchunk);
    const int nkt = (kend - kbeg + BK - 1) / BK;

    float4 ra, rb;
    auto gload = [&](int kt) {
        const int k0 = kbeg + kt * BK;
        if (!TA) ra = load4(A, m0 + tid / 4, g.lda, k0 + (tid % 4) * 4, g.M, kend, g.vecA);
        else     ra = load4(A, k0 + tid / 16, g.lda, m0 + (tid % 16) * 4, kend, g.M, g.vecA);
        if (!TB) rb = load4(B, k0 + tid / 16, g.ldb, n0 + (tid % 16) * 4, kend, g.N, g.vecB);
        else     rb = load4(B, n0 + tid / 4, g.ldb, k0 + (tid % 4) * 4, g.N, kend, g.vecB);
    };
    auto sstore = [&](int buf) {
        if (!TA) {
            int r = tid / 4, kq = (tid % 4) * 4;
            As[buf][kq + 0][r] = ra.x; As[buf][kq + 1][r] = ra.y;
            As[buf][kq + 2][r] = ra.z; As[buf][kq + 3][r] = ra.w;
        } else {
            *reinterpret_cast<float4*>(&As[buf][tid / 16][(tid % 16) * 4]) = ra;
        }
        if (!TB) {
            *reinterpret_cast<float4*>(&Bs[buf][tid / 16][(tid % 16) * 4]) = rb;
        } else {
            int r = tid / 4, kq = (tid % 4) * 4;
            Bs[buf][kq + 0][r] = rb.x; Bs[buf][kq + 1][r] = rb.y;
            Bs[buf][kq + 2][r] = rb.z; Bs[buf][kq + 3][r] = rb.w;
        }
    };

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    const int ty = tid / 16, tx = tid % 16;
    if (nkt > 0) {
        gload(0);
        sstore(0);
    }
    __syncthreads();
    for (int kt = 0; kt < nkt; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nkt) gload(kt + 1);
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float4 a = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
            float4 b = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        if (kt + 1 < nkt) sstore(buf ^ 1);
        __syncthreads();
    }

#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= g.M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= g.N) continue;
            if (g.ksplit > 1)
                g.ws[(((long long)batch * g.ksplit + split) * g.M + m) * g.N + n] = acc[i][j];
            else
                g.ep.store(batch, m, n, g.M, g.N, acc[i][j]);
        }
    }
}

// fixed-order sum of the split-K partials followed by the epilogue (run-to-run deterministic)
__global__ void splitk_reduce_kernel(GemmArgs g) {
    pdl_enter();
    const long long total = (long long)g.nbatch * g.M * g.N;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        const int n = (int)(e % g.N);
        const int m = (int)((e / g.N) % g.M);
        const int batch = (int)(e / ((long long)g.M * g.N));
        float s = 0.f;
        const float* p = g.ws + ((long long)batch * g.ksplit * g.M + m) * g.N + n;
        for (int k = 0; k < g.ksplit; ++k) s += p[(long long)k * g.M * g.N];
        g.ep.store(batch, m, n, g.M, g.N, s);
    }
}

// ---------------------------------------------------------------------------------------------------------
// Degenerate shapes (single batch).  A 64 x 64 tile wastes 63/64 of its work on an N = 1 output head and cannot
// spread a 159 048-long reduction with a 128-element result over the machine; these three kernels are pure
// streaming passes over the one large operand (the C3 regressor: libs/model.py:615-617 `fc(cat[x, grid])` grid
// columns, :629 `out` Linear(dim_feedforward, 1), and their gradients).
//   op(A)(m,k) = A[m*sam + k*sak],  op(B)(k,n) = B[k*sbk + n*sbn]
// ---------------------------------------------------------------------------------------------------------
struct SkinnyArgs {
    const float* A; const float* B;
    int M, N, K;
    long long sam, sak, sbk, sbn;
    int ksplit, kchunk;
    GemmEpilogue ep;
    float* ws;
};

// (1) tiny inner dimension (K <= 8): one output element per thread, op(A) row held in registers
__global__ void __launch_bounds__(256) gemm_thin_k_kernel(SkinnyArgs g) {
    pdl_enter();
    const unsigned total = (unsigned)g.M * (unsigned)g.N;          // host guarantees M*N < 2^31
    for (unsigned e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int m = (int)(e / (unsigned)g.N), n = (int)(e % (unsigned)g.N);
        float acc = 0.f;
        for (int k = 0; k < g.K; ++k) acc = fmaf(g.A[m * g.sam + k * g.sak], g.B[k * g.sbk + n * g.sbn], acc);
        g.ep.store(0, m, n, g.M, g.N, acc);
    }
}

// float4 variant: four consecutive output columns per thread (N % 4 == 0, every [M,N] operand 16-byte aligned)
template <int KMAX>
__global__ void __launch_bounds__(256) gemm_thin_k_vec4_kernel(SkinnyArgs g) {
    pdl_enter();
    const unsigned nq = (unsigned)g.N / 4u, total = (unsigned)g.M * nq;
    for (unsigned e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int m = (int)(e / nq), n = (int)(e % nq) * 4;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < KMAX; ++k)
            if (k < g.K) {
                const float a = g.A[m * g.sam + k * g.sak];
                const float* b = g.B + k * g.sbk + n * g.sbn;
                acc.x = fmaf(a, b[0], acc.x); acc.y = fmaf(a, b[g.sbn], acc.y);
                acc.z = fmaf(a, b[2 * g.sbn], acc.z); acc.w = fmaf(a, b[3 * g.sbn], acc.w);
            }
        g.ep.store4(m, n, g.N, acc);
    }
}

// (2) tiny output width (N <= 8), row-major A: one warp per output row, lanes stride the contraction
template <int NMAX>
__global__ void __launch_bounds__(256) gemm_thin_n_kernel(SkinnyArgs g) {
    pdl_enter();
    const int lane = threadIdx.x % 32;
    const int wglobal = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32, nwarps = gridDim.x * (blockDim.x / 32);
    for (int m = wglobal; m < g.M; m += nwarps) {
        float acc[NMAX];
#pragma unroll
        for (int n = 0; n < NMAX; ++n) acc[n] = 0.f;
        const float* a = g.A + m * g.sam;
        for (int k = lane; k < g.K; k += 32) {
            const float av = a[k];
#pragma unroll
            for (int n = 0; n < NMAX; ++n)
                if (n < g.N) acc[n] = fmaf(av, g.B[k * g.sbk + n * g.sbn], acc[n]);
        }
#pragma unroll
        for (int n = 0; n < NMAX; ++n) {
            const float s = warp_sum(acc[n]);
            if (lane == n && n < g.N) g.ep.store(0, m, n, g.M, g.N, s);
        }
    }
}

// N = 1..2 with K % 4 == 0, 16-byte aligned rows and k-contiguous B (transB): float4 along the contraction, four
// rows of A in flight per warp
template <int NMAX>
__global__ void __launch_bounds__(256) gemm_thin_n_vec4_kernel(SkinnyArgs g) {
    pdl_enter();
    constexpr int RU = 4;
    const int lane = threadIdx.x % 32;
    const int wglobal = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32, nwarps = gridDim.x * (blockDim.x / 32);
    const int kq = g.K / 4;
    for (int m0 = wglobal * RU; m0 < g.M; m0 += nwarps * RU) {
        float acc[RU][NMAX];
#pragma unroll
        for (int r = 0; r < RU; ++r)
#pragma unroll
            for (int n = 0; n < NMAX; ++n) acc[r][n] = 0.f;
        for (int q = lane; q < kq; q += 32) {
            float4 av[RU];
#pragma unroll
            for (int r = 0; r < RU; ++r)
                av[r] = m0 + r < g.M ? *reinterpret_cast<const float4*>(g.A + (long long)(m0 + r) * g.sam + 4 * q)
                                     : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int n = 0; n < NMAX; ++n)
                if (n < g.N) {
                    const float4 bv = *reinterpret_cast<const float4*>(g.B + n * g.sbn + 4 * q);
#pragma unroll
                    for (int r = 0; r < RU; ++r)
                        acc[r][n] = fmaf(av[r].x, bv.x, fmaf(av[r].y, bv.y, fmaf(av[r].z, bv.z, fmaf(av[r].w, bv.w, acc[r][n]))));
                }
        }
#pragma unroll
        for (int r = 0; r < RU; ++r)
#pragma unroll
            for (int n = 0; n < NMAX; ++n) {
                const float s = warp_sum(acc[r][n]);
                if (lane == r * NMAX + n && n < g.N && m0 + r < g.M) g.ep.store(0, m0 + r, n, g.M, g.N, s);
            }
    }
}

// (3) tiny output (M*N <= 1024), very long contraction, both operands stored k-major (the weight-gradient layout
// dY^T X): CTA `split` owns k in [split*kchunk, ...), threads own output elements, several k-rows in flight per CTA;
// partial sums go to ws[split][M*N] and are finished in fixed order by tall_final_kernel.
__global__ void __launch_bounds__(256) gemm_tall_partial_kernel(SkinnyArgs g) {
    pdl_enter();
    __shared__ float red[256];
    const int E = g.M * g.N;
    const int le = E < 256 ? E : 256;                 // threads along the output
    const int KP = 256 / le;                          // k-rows processed concurrently
    const int kk = threadIdx.x / le, e0 = threadIdx.x % le;
    const bool active = kk < KP;
    const int kbeg = blockIdx.x * g.kchunk, kend = min(g.K, kbeg + g.kchunk);
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    const float* ap[4]; const float* bp[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int e = e0 + j * le;
        const int m = e < E ? e / g.N : 0, n = e < E ? e % g.N : 0;
        ap[j] = g.A + m * g.sam;
        bp[j] = g.B + n * g.sbn;
    }
    const int nj = (E + le - 1) / le;                 // <= 4
    if (active) {
        int k = kbeg + kk;
        for (; k + 3 * KP < kend; k += 4 * KP) {      // four independent k-rows per thread in flight
            float av[4][4], bv[4][4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (j < nj) {
                        av[u][j] = ap[j][(long long)(k + u * KP) * g.sak];
                        bv[u][j] = bp[j][(long long)(k + u * KP) * g.sbk];
                    }
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (j < nj) acc[j] = fmaf(av[u][j], bv[u][j], acc[j]);
        }
        for (; k < kend; k += KP)
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (j < nj) acc[j] = fmaf(ap[j][(long long)k * g.sak], bp[j][(long long)k * g.sbk], acc[j]);
    }
    // fold the KP concurrent k-rows (fixed order), one output slot j at a time
    for (int j = 0; j < nj; ++j) {
        red[threadIdx.x] = active ? acc[j] : 0.f;
        __syncthreads();
        if (kk == 0) {
            float s = 0.f;
            for (int q = 0; q < KP; ++q) s += red[q * le + e0];
            const int e = e0 + j * le;
            if (e < E) g.ws[(long long)blockIdx.x * E + e] = s;
        }
        __syncthreads();
    }
}
// float4 along n (N % 4 == 0, B rows 16-byte aligned, M*N/4 <= 256): one B row = N/4 lanes, 256/(M*N/4) k-rows per pass
__global__ void __launch_bounds__(256) gemm_tall_partial_vec4_kernel(SkinnyArgs g) {
    pdl_enter();
    __shared__ float4 red[256];
    const int E4 = g.M * g.N / 4;
    const int KP = 256 / E4;
    const int kk = threadIdx.x / E4, e4 = threadIdx.x % E4;
    const bool active = kk < KP;
    const int m = (e4 * 4) / g.N, n = (e4 * 4) % g.N;
    const int kbeg = blockIdx.x * g.kchunk, kend = min(g.K, kbeg + g.kchunk);
    const float* ap = g.A + m * g.sam;
    const float* bp = g.B + n;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (active) {
        int k = kbeg + kk;
        for (; k + 7 * KP < kend; k += 8 * KP) {      // eight independent k-rows per thread in flight
            float av[8]; float4 bv[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                av[u] = ap[(long long)(k + u * KP) * g.sak];
                bv[u] = *reinterpret_cast<const float4*>(bp + (long long)(k + u * KP) * g.sbk);
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                acc.x = fmaf(av[u], bv[u].x, acc.x); acc.y = fmaf(av[u], bv[u].y, acc.y);
                acc.z = fmaf(av[u], bv[u].z, acc.z); acc.w = fmaf(av[u], bv[u].w, acc.w);
            }
        }
        for (; k < kend; k += KP) {
            const float a = ap[(long long)k * g.sak];
            const float4 b = *reinterpret_cast<const float4*>(bp + (long long)k * g.sbk);
            acc.x = fmaf(a, b.x, acc.x); acc.y = fmaf(a, b.y, acc.y); acc.z = fmaf(a, b.z, acc.z); acc.w = fmaf(a, b.w, acc.w);
        }
    }
    red[threadIdx.x] = active ? acc : make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();
    if (kk == 0) {
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int q = 0; q < KP; ++q) {
            const float4 t = red[q * E4 + e4];
            s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w;
        }
        *reinterpret_cast<float4*>(g.ws + (long long)blockIdx.x * (E4 * 4) + e4 * 4) = s;
    }
}
__global__ void gemm_tall_final_kernel(SkinnyArgs g) {
    pdl_enter();
    __shared__ float red[32][33];
    const int E = g.M * g.N;
    const int e = blockIdx.x * 32 + threadIdx.x;
    float s = 0.f;
    if (e < E)
        for (int p = threadIdx.y; p < g.ksplit; p += 32) s += g.ws[(long long)p * E + e];
    red[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && e < E) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) t += red[i][threadIdx.x];
        g.ep.store(0, e / g.N, e % g.N, g.M, g.N, t);
    }
}

// column sums of a row-major [M,N] matrix (bias gradients), two deterministic stages
__global__ void colsum_partial_kernel(const float* __restrict__ X, int M, int N, int ld,
                                      int rows_per_block, float* __restrict__ part) {
    pdl_enter();
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    const int r0 = blockIdx.y * rows_per_block;
    const int r1 = min(M, r0 + rows_per_block);
    __shared__ float red[32][33];
    float s = 0.f;
    if (n < N)
        for (int r = r0 + threadIdx.y; r < r1; r += blockDim.y) s += X[(long long)r * ld + n];
    red[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && n < N) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i) t += red[i][threadIdx.x];
        part[(long long)blockIdx.y * N + n] = t;
    }
}
__global__ void colsum_final_kernel(const float* __restrict__ part, int nparts, int N, float scale,
                                    int accumulate, float* __restrict__ out) {
    pdl_enter();
    reduce_partials_2d(part, nparts, N, N, scale, accumulate, out);
}

// g = dy * rscale * dropmask * act'(z)   (backward of the GEMM epilogue, elementwise)
__global__ void epilogue_bwd_kernel(const float* __restrict__ dy, int lddy, const float* __restrict__ z,
                                    int ldz, const float* __restrict__ y, int ldy, float* __restrict__ gout,
                                    int ldg, long long M, int N, int act, float rscale, float drop_p,
                                    unsigned long long seed, const unsigned long long* seed_off) {
    pdl_enter();
    const long long total = M * N;
    if (drop_p > 0.f && seed_off) seed += *seed_off;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        const long long m = e / N;
        const int n = (int)(e % N);
        float v = dy[m * lddy + n] * rscale;
        if (drop_p > 0.f) v *= dropout_scale(drop_p, seed, (unsigned long long)e);
        if (act == ACT_RELU) {
            // relu'(z) from the stored output: y > 0 <=> z > 0 and kept (dropped => v already 0)
            float ref = z ? z[m * ldz + n] : y[m * ldy + n];
            v = ref > 0.f ? v : 0.f;
        } else if (act == ACT_SILU) {
            v *= act_grad(ACT_SILU, z[m * ldz + n]);
        }
        gout[m * ldg + n] = v;
    }
}

// float4 variant: contiguous rows (ld == N), N % 4 == 0, 16-byte aligned pointers; 32-bit indexing
template <int ACT>
__global__ void epilogue_bwd_vec4_kernel(const float4* __restrict__ dy, const float4* __restrict__ ref,
                                         float4* __restrict__ gout, unsigned int total4, float rscale, float drop_p,
                                         unsigned long long seed, const unsigned long long* seed_off) {
    pdl_enter();
    if (drop_p > 0.f && seed_off) seed += *seed_off;
    for (unsigned int e = blockIdx.x * blockDim.x + threadIdx.x; e < total4; e += gridDim.x * blockDim.x) {
        float4 v = dy[e];
        v.x *= rscale; v.y *= rscale; v.z *= rscale; v.w *= rscale;
        if (drop_p > 0.f) {
            const float4 ds = dropout_scale4(drop_p, seed, (unsigned long long)e * 4);
            v.x *= ds.x; v.y *= ds.y; v.z *= ds.z; v.w *= ds.w;
        }
        if (ACT == ACT_RELU) {
            const float4 r = ref[e];
            v.x = r.x > 0.f ? v.x : 0.f; v.y = r.y > 0.f ? v.y : 0.f;
            v.z = r.z > 0.f ? v.z : 0.f; v.w = r.w > 0.f ? v.w : 0.f;
        } else if (ACT == ACT_SILU) {
            const float4 r = ref[e];
            v.x *= act_grad(ACT_SILU, r.x); v.y *= act_grad(ACT_SILU, r.y);
            v.z *= act_grad(ACT_SILU, r.z); v.w *= act_grad(ACT_SILU, r.w);
        }
        gout[e] = v;
    }
}

// epilogue backward fused with the bias gradient: thread = fixed column quad, rows strided, so the column sums of
// g accumulate in registers while g is written; per-CTA partials are finished by colsum_final_kernel.
constexpr int EB_BLOCKS = 296;
template <int ACT>
__global__ void __launch_bounds__(256) epilogue_bwd_bias_kernel(const float4* __restrict__ dy,
                                                                const float4* __restrict__ ref,
                                                                float4* __restrict__ gout, int M, int N, float rscale,
                                                                float drop_p, unsigned long long seed,
                                                                const unsigned long long* seed_off,
                                                                float* __restrict__ part) {
    pdl_enter();
    __shared__ float4 red[256];
    if (drop_p > 0.f && seed_off) seed += *seed_off;
    const int rowq = N / 4, q = threadIdx.x % rowq, rsub = threadIdx.x / rowq, rpb = 256 / rowq;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    constexpr int RU = 4;                       // rows in flight per thread: all loads issued before the Philox math
    const int stride = gridDim.x * rpb;
    for (int r0 = blockIdx.x * rpb + rsub; r0 < M; r0 += RU * stride) {
        float4 v[RU], rr[RU];
#pragma unroll
        for (int u = 0; u < RU; ++u) {
            const int r = r0 + u * stride;
            if (r < M) {
                v[u] = dy[(long long)r * rowq + q];
                if (ACT != ACT_NONE) rr[u] = ref[(long long)r * rowq + q];
            }
        }
#pragma unroll
        for (int u = 0; u < RU; ++u) {
            const int r = r0 + u * stride;
            if (r >= M) break;
            const long long e = (long long)r * rowq + q;
            float4 w = v[u];
            w.x *= rscale; w.y *= rscale; w.z *= rscale; w.w *= rscale;
            if (drop_p > 0.f) {
                const float4 ds = dropout_scale4(drop_p, seed, (unsigned long long)e * 4);
                w.x *= ds.x; w.y *= ds.y; w.z *= ds.z; w.w *= ds.w;
            }
            if (ACT == ACT_RELU) {
                w.x = rr[u].x > 0.f ? w.x : 0.f; w.y = rr[u].y > 0.f ? w.y : 0.f;
                w.z = rr[u].z > 0.f ? w.z : 0.f; w.w = rr[u].w > 0.f ? w.w : 0.f;
            } else if (ACT == ACT_SILU) {
                w.x *= act_grad(ACT_SILU, rr[u].x); w.y *= act_grad(ACT_SILU, rr[u].y);
                w.z *= act_grad(ACT_SILU, rr[u].z); w.w *= act_grad(ACT_SILU, rr[u].w);
            }
            gout[e] = w;
            acc.x += w.x; acc.y += w.y; acc.z += w.z; acc.w += w.w;
        }
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x < rowq) {
        float4 t = red[threadIdx.x];
        for (int k = 1; k < rpb; ++k) {
            const float4 o = red[threadIdx.x + k * rowq];
            t.x += o.x; t.y += o.y; t.z += o.z; t.w += o.w;
        }
        reinterpret_cast<float4*>(part + (long long)blockIdx.x * N)[threadIdx.x] = t;
    }
}

}  // namespace gb200

using namespace gb200;

extern "C" size_t gb200_gemm_workspace_bytes(int M, int N, int K, int nbatch, int ksplit) {
    (void)K;
    return ksplit > 1 ? (size_t)nbatch * ksplit * M * N * sizeof(float) : 0;
}

extern "C" int gb200_gemm_suggest_ksplit(int M, int N, int K, int nbatch) {
    if (nbatch == 1 && (long long)M * N <= 1024 && K >= 8192) {      // streaming reduction: ~8 CTAs per SM
        const int s = K / 128;
        return s > 148 * 8 ? 148 * 8 : s;
    }
    long long tiles = (long long)cdiv(M, BM) * cdiv(N, BN) * nbatch;
    if (tiles >= 148 || K < 512) return 1;
    int want = (int)((2 * 148 + tiles - 1) / tiles);
    int maxs = K / 256;
    if (maxs < 1) maxs = 1;
    int s = want < maxs ? want : maxs;
    return s < 1 ? 1 : (s > 128 ? 128 : s);
}

// gb200_gemm and gb200_gemm_gated: gate == nullptr is the plain GEMM
static int gemm_simt(int device, const float* A, int lda, int transA, const float* B, int ldb, int transB, float* C,
                     int ldc, int M, int N, int K, int nbatch, long long strideA, long long strideB, long long strideC,
                     float alpha, const float* bias, int act, float* Zout, int ldz, float drop_p, unsigned long long seed,
                     const float* R, int ldr, float rscale, int accumulate, const float* gate, int ldg, int gate_act,
                     int ksplit, float* workspace, size_t workspace_bytes, void* stream) {
    use_device(device);
    GB_REQUIRE(M >= 0 && N >= 0 && K >= 0 && nbatch >= 1, "gb200_gemm: bad shape M=%d N=%d K=%d nb=%d", M, N, K, nbatch);
    if (M == 0 || N == 0) return GB200_OK;
    GB_REQUIRE(A && B && C, "gb200_gemm: null operand");
    GB_REQUIRE(act == ACT_NONE || act == ACT_RELU || act == ACT_SILU, "gb200_gemm: unknown activation %d", act);
    GB_REQUIRE(drop_p >= 0.f && drop_p < 1.f, "gb200_gemm: dropout p=%f outside [0,1)", drop_p);
    if (ksplit < 1) ksplit = 1;
    if (K == 0) ksplit = 1;
    GemmArgs g;
    g.A = A; g.B = B; g.M = M; g.N = N; g.K = K; g.lda = lda; g.ldb = ldb;
    g.sA = strideA; g.sB = strideB; g.nbatch = nbatch; g.ksplit = ksplit;
    g.ep.C = C; g.ep.ldc = ldc; g.ep.sC = strideC;
    int ktiles = cdiv(K > 0 ? K : 1, BK);
    g.kchunk = cdiv(ktiles, ksplit) * BK;
    g.ep.alpha = alpha; g.ep.bias = bias; g.ep.act = act; g.ep.Z = Zout; g.ep.ldz = ldz; g.ep.drop_p = drop_p;
    g.ep.seed = seed; g.ep.seed_off = rng_offset_ptr(); g.ep.R = R; g.ep.ldr = ldr; g.ep.rscale = rscale; g.ep.accumulate = accumulate;
    g.ep.G = gate; g.ep.ldg = ldg; g.ep.gate = gate_act;
    GB_REQUIRE(!gate || gate_act == ACT_RELU || gate_act == ACT_SILU, "gb200_gemm: unknown gate %d", gate_act);
    g.ws = workspace;
    g.vecA = ((uintptr_t)A % 16 == 0) && (lda % 4 == 0) && (strideA % 4 == 0);
    g.vecB = ((uintptr_t)B % 16 == 0) && (ldb % 4 == 0) && (strideB % 4 == 0);
    if (ksplit > 1)
        GB_REQUIRE(workspace && workspace_bytes >= gb200_gemm_workspace_bytes(M, N, K, nbatch, ksplit),
                   "gb200_gemm: split-K workspace too small (%zu bytes)", workspace_bytes);
    cudaStream_t st = as_stream(stream);
    if (nbatch == 1) {      // degenerate shapes: streaming kernels instead of 64 x 64 tiles
        SkinnyArgs s;
        s.A = A; s.B = B; s.M = M; s.N = N; s.K = K; s.ep = g.ep; s.ws = workspace;
        s.sam = transA ? 1 : lda; s.sak = transA ? lda : 1;
        s.sbk = transB ? 1 : ldb; s.sbn = transB ? ldb : 1;
        s.ksplit = ksplit;
        s.kchunk = cdiv(K > 0 ? K : 1, ksplit);
        const long long total = (long long)M * N;
        auto al16 = [](const void* p) { return ((uintptr_t)p % 16) == 0; };
        const GemmEpilogue& e = g.ep;
        const bool out4 = N % 4 == 0 && al16(C) && ldc % 4 == 0 && (!e.bias || al16(e.bias)) &&
                          (!e.Z || (al16(e.Z) && ldz % 4 == 0)) && (!e.R || (al16(e.R) && ldr % 4 == 0)) &&
                          (!e.G || (al16(e.G) && e.ldg % 4 == 0));
        if (K <= 8 && total < (1ll << 31) && out4) {
            const long long quads = total / 4;
            const int blocks = (int)(quads / 256 + 1 < 148 * 16 ? quads / 256 + 1 : 148 * 16);
            if (K <= 2) launch_kernel(gemm_thin_k_vec4_kernel<2>, blocks, 256, 0, st, s);
            else launch_kernel(gemm_thin_k_vec4_kernel<8>, blocks, 256, 0, st, s);
            return check_launch("gb200_gemm(thin K, float4)", 1);
        }
        if (K <= 8 && total < (1ll << 31)) {
            launch_kernel(gemm_thin_k_kernel, (int)(total / 256 + 1 < 148 * 16 ? total / 256 + 1 : 148 * 16), 256, 0, st, s);
            return check_launch("gb200_gemm(thin K)", 1);
        }
        if (N <= 2 && !transA && transB && M >= 1024 && K % 4 == 0 && al16(A) && al16(B) && lda % 4 == 0 && ldb % 4 == 0) {
            const int blocks = cdiv(M, 32) < 148 * 16 ? cdiv(M, 32) : 148 * 16;
            if (N == 1) launch_kernel(gemm_thin_n_vec4_kernel<1>, blocks, 256, 0, st, s);
            else launch_kernel(gemm_thin_n_vec4_kernel<2>, blocks, 256, 0, st, s);
            return check_launch("gb200_gemm(thin N, float4)", 1);
        }
        if (N <= 8 && !transA && M >= 1024) {
            const int blocks = cdiv(M, 8) < 148 * 16 ? cdiv(M, 8) : 148 * 16;
            if (N <= 2) launch_kernel(gemm_thin_n_kernel<2>, blocks, 256, 0, st, s);
            else launch_kernel(gemm_thin_n_kernel<8>, blocks, 256, 0, st, s);
            return check_launch("gb200_gemm(thin N)", 1);
        }
        if (transA && !transB && total <= 1024 && ksplit > 1) {
            s.ksplit = cdiv(K, s.kchunk);
            if (N % 4 == 0 && total / 4 <= 256 && al16(B) && ldb % 4 == 0 && al16(workspace))
                launch_kernel(gemm_tall_partial_vec4_kernel, s.ksplit, 256, 0, st, s);
            else
                launch_kernel(gemm_tall_partial_kernel, s.ksplit, 256, 0, st, s);
            launch_kernel(gemm_tall_final_kernel, cdiv(total, 32), dim3(32, 32), 0, st, s);
            return check_launch("gb200_gemm(tall)", 2);
        }
    }
    dim3 grid(cdiv(N, BN), cdiv(M, BM), nbatch * ksplit);
    GB_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "gb200_gemm: grid too large");
    if (!transA && !transB) launch_kernel(gemm_simt_kernel<false, false>, grid, NT, 0, st, g);
    else if (!transA && transB) launch_kernel(gemm_simt_kernel<false, true>, grid, NT, 0, st, g);
    else if (transA && !transB) launch_kernel(gemm_simt_kernel<true, false>, grid, NT, 0, st, g);
    else launch_kernel(gemm_simt_kernel<true, true>, grid, NT, 0, st, g);
    if (ksplit > 1) {
        long long total = (long long)nbatch * M * N;
        int blocks = (int)((total + 255) / 256);
        if (blocks > 148 * 8) blocks = 148 * 8;
        launch_kernel(splitk_reduce_kernel, blocks, 256, 0, st, g);
    }
    return check_launch("gb200_gemm", ksplit > 1 ? 2 : 1);
}

extern "C" int gb200_gemm(int device, const float* A, int lda, int transA, const float* B, int ldb,
                          int transB, float* C, int ldc, int M, int N, int K, int nbatch,
                          long long strideA, long long strideB, long long strideC, float alpha,
                          const float* bias, int act, float* Zout, int ldz, float drop_p,
                          unsigned long long seed, const float* R, int ldr, float rscale,
                          int accumulate, int ksplit, float* workspace, size_t workspace_bytes,
                          void* stream) {
    return gemm_simt(device, A, lda, transA, B, ldb, transB, C, ldc, M, N, K, nbatch, strideA, strideB, strideC, alpha,
                     bias, act, Zout, ldz, drop_p, seed, R, ldr, rscale, accumulate, nullptr, 0, ACT_NONE, ksplit,
                     workspace, workspace_bytes, stream);
}

extern "C" int gb200_gemm_gated(int device, const float* A, int lda, int transA, const float* B, int ldb,
                                int transB, float* C, int ldc, int M, int N, int K, float alpha, float drop_p,
                                unsigned long long seed, float rscale, const float* gate, int ldg, int gate_act,
                                int ksplit, float* workspace, size_t workspace_bytes, void* stream) {
    return gemm_simt(device, A, lda, transA, B, ldb, transB, C, ldc, M, N, K, 1, 0, 0, 0, alpha, nullptr, ACT_NONE, nullptr,
                     0, drop_p, seed, nullptr, 0, rscale, 0, gate, ldg, gate_act, ksplit, workspace, workspace_bytes,
                     stream);
}

extern "C" size_t gb200_colsum_workspace_bytes(long long M, int N) {
    int rows_per_block = 128;
    return (size_t)cdiv(M, rows_per_block) * N * sizeof(float);
}

extern "C" int gb200_colsum(int device, const float* X, int ld, long long M, int N, float scale,
                            int accumulate, float* out, float* workspace, size_t workspace_bytes,
                            void* stream) {
    use_device(device);
    GB_REQUIRE(X && out && M >= 1 && N >= 1, "gb200_colsum: bad arguments");
    const int rows_per_block = 128;
    int nparts = cdiv(M, rows_per_block);
    GB_REQUIRE(workspace && workspace_bytes >= (size_t)nparts * N * sizeof(float),
               "gb200_colsum: workspace too small");
    GB_REQUIRE(nparts <= 65535, "gb200_colsum: too many rows");
    cudaStream_t st = as_stream(stream);
    launch_kernel(colsum_partial_kernel, dim3(cdiv(N, 32), nparts), dim3(32, 32), 0, st, X, (int)M, N, ld, rows_per_block,
                                                                               workspace);
    launch_kernel(colsum_final_kernel, cdiv(N, 32), dim3(32, 32), 0, st, workspace, nparts, N, scale, accumulate, out);
    return check_launch("gb200_colsum", 2);
}

extern "C" int gb200_epilogue_bwd(int device, const float* dy, int lddy, const float* z, int ldz,
                                  const float* y, int ldy, float* g, int ldg, long long M, int N, int act,
                                  float rscale, float drop_p, unsigned long long seed, void* stream) {
    use_device(device);
    GB_REQUIRE(dy && g && M >= 0 && N >= 1, "gb200_epilogue_bwd: bad arguments");
    GB_REQUIRE(act != ACT_SILU || z, "gb200_epilogue_bwd: SiLU backward needs the pre-activation");
    GB_REQUIRE(act != ACT_RELU || z || y, "gb200_epilogue_bwd: ReLU backward needs z or y");
    if (M == 0) return GB200_OK;
    long long total = M * N;
    const float* ref = z ? z : y;
    const int ldref = z ? ldz : ldy;
    auto al16 = [](const void* p) { return ((uintptr_t)p % 16) == 0; };
    if (N % 4 == 0 && lddy == N && ldg == N && (act == ACT_NONE || ldref == N) && al16(dy) && al16(g) &&
        (act == ACT_NONE || al16(ref)) && total / 4 < 0x7fffffffLL) {
        const unsigned int total4 = (unsigned int)(total / 4);
        int blocks = (int)((total4 + 255) / 256);
        if (blocks > 148 * 8) blocks = 148 * 8;
        const float4* d4 = reinterpret_cast<const float4*>(dy);
        const float4* r4 = reinterpret_cast<const float4*>(ref);
        float4* g4 = reinterpret_cast<float4*>(g);
        cudaStream_t st = as_stream(stream);
        if (act == ACT_RELU)
            launch_kernel(epilogue_bwd_vec4_kernel<ACT_RELU>, blocks, 256, 0, st, d4, r4, g4, total4, rscale, drop_p, seed, rng_offset_ptr());
        else if (act == ACT_SILU)
            launch_kernel(epilogue_bwd_vec4_kernel<ACT_SILU>, blocks, 256, 0, st, d4, r4, g4, total4, rscale, drop_p, seed, rng_offset_ptr());
        else
            launch_kernel(epilogue_bwd_vec4_kernel<ACT_NONE>, blocks, 256, 0, st, d4, r4, g4, total4, rscale, drop_p, seed, rng_offset_ptr());
        return check_launch("gb200_epilogue_bwd");
    }
    int blocks = (int)((total + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    launch_kernel(epilogue_bwd_kernel, blocks, 256, 0, as_stream(stream), dy, lddy, z, ldz, y, ldy, g, ldg, M, N, act,
                                                               rscale, drop_p, seed, rng_offset_ptr());
    return check_launch("gb200_epilogue_bwd");
}

extern "C" size_t gb200_epilogue_bwd_bias_workspace_bytes(long long M, int N) {
    size_t a = (size_t)EB_BLOCKS * N * sizeof(float), b = gb200_colsum_workspace_bytes(M, N);
    return a > b ? a : b;
}

// g = dy * rscale * dropmask * act'(.)  AND  dbias[n] = sum_m g[m, n]   in one pass over g
extern "C" int gb200_epilogue_bwd_bias(int device, const float* dy, int lddy, const float* z, int ldz, const float* y,
                                       int ldy, float* g, int ldg, long long M, int N, int act, float rscale,
                                       float drop_p, unsigned long long seed, float* dbias, float* workspace,
                                       size_t workspace_bytes, void* stream) {
    use_device(device);
    GB_REQUIRE(dy && g && dbias && M >= 1 && N >= 1, "gb200_epilogue_bwd_bias: bad arguments");
    GB_REQUIRE(workspace && workspace_bytes >= gb200_epilogue_bwd_bias_workspace_bytes(M, N),
               "gb200_epilogue_bwd_bias: workspace too small");
    const float* ref = z ? z : y;
    const int ldref = z ? ldz : ldy;
    GB_REQUIRE(act == ACT_NONE || ref, "gb200_epilogue_bwd_bias: activation backward needs z or y");
    GB_REQUIRE(act != ACT_SILU || z, "gb200_epilogue_bwd_bias: SiLU backward needs the pre-activation");
    auto al16 = [](const void* p) { return ((uintptr_t)p % 16) == 0; };
    const int rowq = N / 4;
    const bool vec = N % 4 == 0 && rowq <= 256 && 256 % rowq == 0 && lddy == N && ldg == N &&
                     (act == ACT_NONE || ldref == N) && al16(dy) && al16(g) && (act == ACT_NONE || al16(ref)) &&
                     al16(workspace) && M < 0x7fffffffLL / (rowq > 0 ? rowq : 1);
    cudaStream_t st = as_stream(stream);
    if (!vec) {
        int rc = gb200_epilogue_bwd(device, dy, lddy, z, ldz, y, ldy, g, ldg, M, N, act, rscale, drop_p, seed, stream);
        if (rc) return rc;
        return gb200_colsum(device, g, ldg, M, N, 1.f, 0, dbias, workspace, workspace_bytes, stream);
    }
    const int rpb = 256 / rowq;
    int blocks = cdiv(M, rpb);
    if (blocks > EB_BLOCKS) blocks = EB_BLOCKS;
    const float4* d4 = reinterpret_cast<const float4*>(dy);
    const float4* r4 = reinterpret_cast<const float4*>(ref);
    float4* g4 = reinterpret_cast<float4*>(g);
    if (act == ACT_RELU)
        launch_kernel(epilogue_bwd_bias_kernel<ACT_RELU>, blocks, 256, 0, st, d4, r4, g4, (int)M, N, rscale, drop_p, seed,
                                                                   rng_offset_ptr(), workspace);
    else if (act == ACT_SILU)
        launch_kernel(epilogue_bwd_bias_kernel<ACT_SILU>, blocks, 256, 0, st, d4, r4, g4, (int)M, N, rscale, drop_p, seed,
                                                                   rng_offset_ptr(), workspace);
    else
        launch_kernel(epilogue_bwd_bias_kernel<ACT_NONE>, blocks, 256, 0, st, d4, r4, g4, (int)M, N, rscale, drop_p, seed,
                                                                   rng_offset_ptr(), workspace);
    launch_kernel(colsum_final_kernel, cdiv(N, 32), dim3(32, 32), 0, st, workspace, blocks, N, 1.f, 0, dbias);
    return check_launch("gb200_epilogue_bwd_bias", 2);
}
