// Quadratic-form Fourier-type attention  O = drop(Q~ K~^T / (sqrt(d) n)) V~  without materialising the
// (B,H,n,n) matrix (the reference does, and keeps it alive: libs/layers.py:687-703, :887).
//
// Needed only when an n x n dropout mask sits between the two products -- the reference's unconditional
// F.dropout(p_attn) (libs/layers.py:700-701) or an explicit keep-mask; without it the products reassociate
// and SimpleAttention uses the O(n d^2) linear-form kernels (attention.cu).  Flash-style tiling: one CTA owns a
// 64-row tile and streams 64-row tiles of the other side through shared memory; the score tile is masked,
// scaled and immediately consumed.  The dropout mask is either an explicit uint8 (B,H,n,n) tensor or a Philox
// draw keyed by (seed, flat (b,h,i,j) index), regenerated identically by the two backward passes:
//     S   = c * drop (.) (Q~ K~^T)                      c = 1/(sqrt(d) n),  drop in {0, 1/(1-p)}
//     O   = S V~           dV~ = S^T dO
//     dSp = c * drop (.) (dO V~^T)        dQ~ = dSp K~        dK~ = dSp^T Q~
// Exact fp32 FMAs (this is the precise path; a tcgen05 version of this tensor-bound kernel is the next step).
#include "common.cuh"
#include "head_operand.cuh"

namespace gb200 {

constexpr int QT = 64;     // tile rows (queries and keys)

struct QuadArgs {
    HeadOperand q, k, v, dO;
    const float* pos;
    int B, H, n, dk, p;
    float c;                              // 1 / (sqrt(d) n)
    const unsigned char* mask;            // (B,H,n,n) keep-mask or null
    float mask_p; unsigned long long seed; const unsigned long long* seed_off;
    float* out; int ldo; int ocol0;       // forward: augmented (T, H*d); backward: token-major, pos columns dropped
    float* out2; int ocol2;               // dK/dV pass: second output block
    float* attn;                          // optional (B,H,n,n) post-dropout matrix
};

template <int DP>
__device__ __forceinline__ void load_tile(float* __restrict__ S, const HeadOperand& op, const QuadArgs& a, int h,
                                          long long tok0, int nt) {
    const int d = a.p + a.dk;
    for (int e = threadIdx.x; e < QT * DP; e += blockDim.x) {
        const int r = e / DP, i = e % DP;
        S[r * (DP + 1) + i] = (r < nt && i < d) ? load_aug(op, a.pos, a.p, a.dk, h, tok0 + r, i) : 0.f;
    }
}

__device__ __forceinline__ float drop_factor(const QuadArgs& a, unsigned long long seed, long long bh, int i, int j) {
    const unsigned long long e = ((unsigned long long)bh * a.n + i) * a.n + j;
    if (a.mask) return 2.f * (float)a.mask[e];
    if (a.mask_p > 0.f) return dropout_scale(a.mask_p, seed, e);
    return 1.f;
}

// scores: P[i][j] = c * drop(i0+i, j0+j) * sum_k X[i][k] * Y[j][k]   (64 x 64, thread = 4 x 4 micro-tile)
template <int DP>
__device__ __forceinline__ void score_tile(float* __restrict__ P, const float* __restrict__ X, const float* __restrict__ Y,
                                           const QuadArgs& a, unsigned long long seed, long long bh, int i0, int ni,
                                           int j0, int nj) {
    const int ty = threadIdx.x / 16, tx = threadIdx.x % 16;
    float s[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int w = 0; w < 4; ++w) s[u][w] = 0.f;
    for (int k = 0; k < DP; ++k) {
        float xv[4], yv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) xv[u] = X[(ty * 4 + u) * (DP + 1) + k];
#pragma unroll
        for (int w = 0; w < 4; ++w) yv[w] = Y[(tx * 4 + w) * (DP + 1) + k];
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int w = 0; w < 4; ++w) s[u][w] = fmaf(xv[u], yv[w], s[u][w]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const int i = ty * 4 + u, j = tx * 4 + w;
            float v = 0.f;
            if (i < ni && j < nj) v = s[u][w] * a.c * drop_factor(a, seed, bh, i0 + i, j0 + j);
            P[i * (QT + 1) + j] = v;
        }
}

// acc[u][c] += sum_j P[row(u)][j] * Y[j][col(c)]      rows ty*4+u, cols tx + 16 c
template <int DP, bool TRANS_P>
__device__ __forceinline__ void accum_tile(float (&acc)[4][DP / 16], const float* __restrict__ P,
                                           const float* __restrict__ Y) {
    const int ty = threadIdx.x / 16, tx = threadIdx.x % 16;
    for (int j = 0; j < QT; ++j) {
        float pv[4], yv[DP / 16];
#pragma unroll
        for (int u = 0; u < 4; ++u) pv[u] = TRANS_P ? P[j * (QT + 1) + ty * 4 + u] : P[(ty * 4 + u) * (QT + 1) + j];
#pragma unroll
        for (int c = 0; c < DP / 16; ++c) yv[c] = Y[j * (DP + 1) + tx + 16 * c];
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int c = 0; c < DP / 16; ++c) acc[u][c] = fmaf(pv[u], yv[c], acc[u][c]);
    }
}

template <int DP>
__device__ __forceinline__ void store_rows(const float (&acc)[4][DP / 16], const QuadArgs& a, float* out, int ocol0,
                                           bool augmented, int h, long long tok0, int nt) {
    const int ty = threadIdx.x / 16, tx = threadIdx.x % 16;
    const int d = a.p + a.dk;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int r = ty * 4 + u;
        if (r >= nt) continue;
#pragma unroll
        for (int c = 0; c < DP / 16; ++c) {
            const int j = tx + 16 * c;
            if (j >= d) continue;
            if (augmented) out[(tok0 + r) * a.ldo + ocol0 + h * d + j] = acc[u][c];
            else if (j >= a.p) out[(tok0 + r) * a.ldo + ocol0 + h * a.dk + (j - a.p)] = acc[u][c];
        }
    }
}

// mode 0: forward (rows = queries, streams K,V): O = S V       [+ optional attn matrix]
// mode 1: dQ pass  (rows = queries, streams K,V): dQ = dSp K,  dSp from (dO, V)
template <int DP, int MODE>
__global__ void __launch_bounds__(256) quad_rows_kernel(QuadArgs a) {
    pdl_enter();
    extern __shared__ float sm[];
    float* Xs = sm;                          // Q tile (mode 0) / dO tile (mode 1)
    float* Ks = Xs + QT * (DP + 1);
    float* Vs = Ks + QT * (DP + 1);
    float* Ps = Vs + QT * (DP + 1);          // [QT][QT+1]
    const long long bh = blockIdx.y;
    const int b = (int)(bh / a.H), h = (int)(bh % a.H);
    const int i0 = blockIdx.x * QT, ni = min(QT, a.n - i0);
    const unsigned long long seed = a.seed + ((a.mask_p > 0.f && a.seed_off) ? *a.seed_off : 0ull);
    const long long base = (long long)b * a.n;
    load_tile<DP>(Xs, MODE == 0 ? a.q : a.dO, a, h, base + i0, ni);
    float acc[4][DP / 16];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int c = 0; c < DP / 16; ++c) acc[u][c] = 0.f;
    for (int j0 = 0; j0 < a.n; j0 += QT) {
        const int nj = min(QT, a.n - j0);
        __syncthreads();
        load_tile<DP>(Ks, a.k, a, h, base + j0, nj);
        load_tile<DP>(Vs, a.v, a, h, base + j0, nj);
        __syncthreads();
        score_tile<DP>(Ps, Xs, MODE == 0 ? Ks : Vs, a, seed, bh, i0, ni, j0, nj);
        __syncthreads();
        if (MODE == 0 && a.attn) {
            for (int e = threadIdx.x; e < QT * QT; e += blockDim.x) {
                const int i = e / QT, j = e % QT;
                if (i < ni && j < nj) a.attn[((long long)bh * a.n + i0 + i) * a.n + j0 + j] = Ps[i * (QT + 1) + j];
            }
        }
        accum_tile<DP, false>(acc, Ps, MODE == 0 ? Vs : Ks);
    }
    store_rows<DP>(acc, a, a.out, a.ocol0, MODE == 0, h, base + i0, ni);
}

// dK/dV pass (rows = keys, streams Q, dO):  dV = S^T dO,  dK = dSp^T Q
template <int DP>
__global__ void __launch_bounds__(256) quad_cols_kernel(QuadArgs a) {
    pdl_enter();
    extern __shared__ float sm[];
    float* Ks = sm;
    float* Vs = Ks + QT * (DP + 1);
    float* Qs = Vs + QT * (DP + 1);
    float* Ds = Qs + QT * (DP + 1);
    float* Ss = Ds + QT * (DP + 1);          // [i][j] scores
    float* Ps = Ss + QT * (QT + 1);          // [i][j] dSp
    const long long bh = blockIdx.y;
    const int b = (int)(bh / a.H), h = (int)(bh % a.H);
    const int j0 = blockIdx.x * QT, nj = min(QT, a.n - j0);
    const unsigned long long seed = a.seed + ((a.mask_p > 0.f && a.seed_off) ? *a.seed_off : 0ull);
    const long long base = (long long)b * a.n;
    load_tile<DP>(Ks, a.k, a, h, base + j0, nj);
    load_tile<DP>(Vs, a.v, a, h, base + j0, nj);
    float dk_acc[4][DP / 16], dv_acc[4][DP / 16];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int c = 0; c < DP / 16; ++c) { dk_acc[u][c] = 0.f; dv_acc[u][c] = 0.f; }
    for (int i0 = 0; i0 < a.n; i0 += QT) {
        const int ni = min(QT, a.n - i0);
        __syncthreads();
        load_tile<DP>(Qs, a.q, a, h, base + i0, ni);
        load_tile<DP>(Ds, a.dO, a, h, base + i0, ni);
        __syncthreads();
        score_tile<DP>(Ss, Qs, Ks, a, seed, bh, i0, ni, j0, nj);      // S[i][j]
        score_tile<DP>(Ps, Ds, Vs, a, seed, bh, i0, ni, j0, nj);      // dSp[i][j]
        __syncthreads();
        accum_tile<DP, true>(dv_acc, Ss, Ds);                         // dV[j] += sum_i S[i][j] dO[i]
        accum_tile<DP, true>(dk_acc, Ps, Qs);                         // dK[j] += sum_i dSp[i][j] Q[i]
    }
    store_rows<DP>(dk_acc, a, a.out, a.ocol0, false, h, base + j0, nj);
    store_rows<DP>(dv_acc, a, a.out2, a.ocol2, false, h, base + j0, nj);
}

}  // namespace gb200

using namespace gb200;

static HeadOperand mk(const gb200_head_operand* o) { return make_head_operand(o); }

static int quad_common(QuadArgs& a, const gb200_head_operand* q, const gb200_head_operand* k,
                       const gb200_head_operand* v, const gb200_head_operand* dO, const float* pos, int B, int H, int n,
                       int dk, int p, float scale, const unsigned char* mask, float mask_p, unsigned long long seed) {
    GB_REQUIRE(q && k && v && q->ptr && k->ptr && v->ptr, "gb200_fourier_quad: null operand");
    GB_REQUIRE(B >= 1 && H >= 1 && n >= 1 && dk >= 1 && p >= 0, "gb200_fourier_quad: bad shape");
    GB_REQUIRE(p == 0 || pos, "gb200_fourier_quad: pos is null but pos_dim=%d", p);
    GB_REQUIRE(dk + p <= 64, "gb200_fourier_quad: head width d_k+pos_dim=%d > 64 unsupported", dk + p);
    GB_REQUIRE((long long)B * H <= 65535, "gb200_fourier_quad: B*H too large");
    GB_REQUIRE(mask_p >= 0.f && mask_p < 1.f, "gb200_fourier_quad: mask_p=%f outside [0,1)", mask_p);
    a.q = mk(q); a.k = mk(k); a.v = mk(v); a.dO = mk(dO); a.pos = pos; a.B = B; a.H = H; a.n = n; a.dk = dk; a.p = p;
    a.c = scale; a.mask = mask; a.mask_p = mask ? 0.f : mask_p; a.seed = seed; a.seed_off = rng_offset_ptr();
    a.out = nullptr; a.ldo = 0; a.ocol0 = 0; a.out2 = nullptr; a.ocol2 = 0; a.attn = nullptr;
    return GB200_OK;
}

template <typename K>
static void launch_quad(K kernel, const QuadArgs& a, size_t smem, cudaStream_t st) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    dim3 grid(cdiv(a.n, QT), a.B * a.H);
    launch_kernel(kernel, grid, 256, smem, st, a);
}

extern "C" int gb200_fourier_quad_fwd(int device, const gb200_head_operand* q, const gb200_head_operand* k,
                                      const gb200_head_operand* v, const float* pos, int B, int H, int n, int dk, int p,
                                      float scale, const unsigned char* keep_mask, float mask_p,
                                      unsigned long long mask_seed, float* out, float* attn_or_null, void* stream) {
    use_device(device);
    QuadArgs a;
    int rc = quad_common(a, q, k, v, nullptr, pos, B, H, n, dk, p, scale, keep_mask, mask_p, mask_seed);
    if (rc) return rc;
    GB_REQUIRE(out, "gb200_fourier_quad_fwd: null output");
    a.out = out; a.ldo = H * (dk + p); a.ocol0 = 0; a.attn = attn_or_null;
    const int d = dk + p;
    cudaStream_t st = as_stream(stream);
    if (d <= 32) launch_quad(quad_rows_kernel<32, 0>, a, (size_t)(3 * QT * 33 + QT * (QT + 1)) * 4, st);
    else launch_quad(quad_rows_kernel<64, 0>, a, (size_t)(3 * QT * 65 + QT * (QT + 1)) * 4, st);
    return check_launch("gb200_fourier_quad_fwd");
}

extern "C" int gb200_fourier_quad_bwd(int device, const gb200_head_operand* q, const gb200_head_operand* k,
                                      const gb200_head_operand* v, const gb200_head_operand* dO, const float* pos, int B,
                                      int H, int n, int dk, int p, float scale, const unsigned char* keep_mask,
                                      float mask_p, unsigned long long mask_seed, float* dqkv, int ld, int qcol0,
                                      int kcol0, int vcol0, void* stream) {
    use_device(device);
    QuadArgs a;
    int rc = quad_common(a, q, k, v, dO, pos, B, H, n, dk, p, scale, keep_mask, mask_p, mask_seed);
    if (rc) return rc;
    GB_REQUIRE(dO && dO->ptr && dqkv, "gb200_fourier_quad_bwd: null gradient buffer");
    const int d = dk + p;
    cudaStream_t st = as_stream(stream);
    a.ldo = ld;
    a.out = dqkv; a.ocol0 = qcol0;
    if (d <= 32) launch_quad(quad_rows_kernel<32, 1>, a, (size_t)(3 * QT * 33 + QT * (QT + 1)) * 4, st);
    else launch_quad(quad_rows_kernel<64, 1>, a, (size_t)(3 * QT * 65 + QT * (QT + 1)) * 4, st);
    a.out = dqkv; a.ocol0 = kcol0; a.out2 = dqkv; a.ocol2 = vcol0;
    if (d <= 32) launch_quad(quad_cols_kernel<32>, a, (size_t)(4 * QT * 33 + 2 * QT * (QT + 1)) * 4, st);
    else launch_quad(quad_cols_kernel<64>, a, (size_t)(4 * QT * 65 + 2 * QT * (QT + 1)) * 4, st);
    return check_launch("gb200_fourier_quad_bwd", 2);
}
