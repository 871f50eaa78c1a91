// Tail of the training step (SURVEY.md 8(f) row 3): the weighted L2 / H1 loss with its gradient, and the
// clip-by-global-norm + Adam update, as four streaming launches over flat fp32 buffers with no host synchronisation.
//
// Reference: libs/ft.py:983-1105 (WeightedL2Loss2d: relative L2 loss per sample, sqrt, batch mean; optional
// central-difference H1 regulariser gamma*h*|K (grad u - D_h N(u))|^2 / |K grad u|^2) and libs/utils_ft.py:656-681
// (train_batch_darcy: loss + reg -> backward -> clip_grad_norm_(0.99) -> Adam.step -> OneCycleLR.step).  The reference
// spends ~40 elementwise launches on the loss and its autograd, one foreach pass per Adam sub-expression and a host
// sync in clip_grad_norm_; here:
//
//   loss_partial_kernel   per (sample, chunk): sum (p-t)^2, sum t^2, sum K tp^2, sum (K (tp - D_h p))^2        1 read of each
//   loss_grad_kernel      per-sample scalars from the partials (fixed order), then d(loss)/dp and d(reg)/dp as a GATHER of
//                         the four central-difference neighbours (deterministic), plus the scalar outputs
//   sumsq_partial_kernel  sum g^2 partials over the flat gradient bucket
//   adam_kernel           every CTA re-reduces the <= 1024 partials in the same order -> clip coefficient -> m, v, p update
//
// All reductions are fixed-order (bitwise reproducible run to run).  Hyper-parameters that change every step (lr, beta1 of
// the one-cycle schedule, the two bias corrections) are read from a 4-float device array so the launches can sit inside a
// captured CUDA graph.
#include "common.cuh"

namespace gb200 {

constexpr int LOSS_THREADS = 256;

struct LossArgs {
    const float *p, *t, *tp, *K;   // preds (B,n,n), targets (B,n,n), targets_prime (B,n,n,2) | null, K (B,n,n) | null
    int B, n, s;                   // s = dilation / 2
    float h, beta, gamma, eps;
    int regularizer, return_norm, chunks;
    float* ws;                     // [B][chunks][4]
    float* out;                    // loss, regularizer, metric (L1), loss + regularizer
    float *dl, *dr;                // d loss / d preds, d regularizer / d preds  (B,n,n) each, or null
};

__device__ __forceinline__ float block_sum(float v, float* red) {
    // fixed-order: lanes by xor-shuffle, then warps sequentially
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float s = 0.f;
    for (int w = 0; w < LOSS_THREADS / 32; ++w) s += red[w];
    return s;
}

// K^2 (D_h p - tp) at an interior pixel, both components; zero outside the interior
__device__ __forceinline__ float2 h1_residual(const LossArgs& a, const float* pb, const float* tpb, const float* Kb, int i,
                                              int j) {
    const int n = a.n, s = a.s;
    if (i < s || i >= n - s || j < s || j >= n - s) return make_float2(0.f, 0.f);
    const float inv = 1.f / (2.f * s * a.h);
    const float dx = (pb[(i + s) * n + j] - pb[(i - s) * n + j]) * inv;
    const float dy = (pb[i * n + j + s] - pb[i * n + j - s]) * inv;
    const float2 tp = *reinterpret_cast<const float2*>(tpb + 2 * (i * n + j));
    const float k = Kb ? Kb[i * n + j] : 1.f;
    return make_float2(k * k * (dx - tp.x), k * k * (dy - tp.y));
}

__global__ void __launch_bounds__(LOSS_THREADS) loss_partial_kernel(LossArgs a) {
    pdl_enter();
    __shared__ float red[LOSS_THREADS / 32];
    const int b = blockIdx.y, chunk = blockIdx.x, n = a.n, N = n * n, s = a.s;
    const int per = (N + a.chunks - 1) / a.chunks;
    const int e0 = chunk * per, e1 = min(N, e0 + per);
    const float* pb = a.p + (long long)b * N;
    const float* tb = a.t + (long long)b * N;
    const float* tpb = a.tp ? a.tp + (long long)b * N * 2 : nullptr;
    const float* Kb = a.K ? a.K + (long long)b * N : nullptr;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    const float inv = 1.f / (2.f * s * a.h);
    for (int e = e0 + threadIdx.x; e < e1; e += LOSS_THREADS) {
        const float p = pb[e], t = tb[e];
        s0 = fmaf(p - t, p - t, s0);
        s1 = fmaf(t, t, s1);
        if (tpb) {
            const float2 tp = *reinterpret_cast<const float2*>(tpb + 2 * e);
            const float k = Kb ? Kb[e] : 1.f;
            s2 += k * (tp.x * tp.x + tp.y * tp.y);
            if (a.regularizer) {
                const int i = e / n, j = e % n;
                if (i >= s && i < n - s && j >= s && j < n - s) {
                    const float dx = (pb[e + s * n] - pb[e - s * n]) * inv;
                    const float dy = (pb[e + s] - pb[e - s]) * inv;
                    const float rx = k * (tp.x - dx), ry = k * (tp.y - dy);
                    s3 += rx * rx + ry * ry;
                }
            }
        }
    }
    s0 = block_sum(s0, red);
    s1 = block_sum(s1, red);
    s2 = block_sum(s2, red);
    s3 = block_sum(s3, red);
    if (threadIdx.x == 0)
        *reinterpret_cast<float4*>(a.ws + ((long long)b * a.chunks + chunk) * 4) = make_float4(s0, s1, s2, s3);
}

struct SampleScalars { float loss, reg, metric, cl, cr; };   // per-sample loss / regulariser terms and the gradient coefficients

__device__ __forceinline__ SampleScalars sample_scalars(const LossArgs& a, int b) {
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    for (int c = 0; c < a.chunks; ++c) {
        const float4 v = *reinterpret_cast<const float4*>(a.ws + ((long long)b * a.chunks + c) * 4);
        s0 += v.x; s1 += v.y; s2 += v.z; s3 += v.w;
    }
    const float N = (float)a.n * (float)a.n;
    const float ni = (float)(a.n - 2 * a.s);
    const float Nint2 = ni * ni * 2.f;
    const float tnorm = s1 / N + a.eps;
    const float tpnorm = a.tp ? 2.f * (s2 / (2.f * N)) + a.eps : 1.f;   // d * mean_{(1,2,3)}(K tp^2) + eps, d = 2
    SampleScalars r;
    const float lb = a.beta * (s0 / N) / tnorm;
    const bool reg_on = a.regularizer && a.tp;
    const float rb = reg_on ? a.gamma * a.h * (s3 / Nint2) / tpnorm : 0.f;
    r.loss = a.return_norm ? sqrtf(lb) : lb;
    r.reg = a.return_norm ? sqrtf(rb) : rb;
    r.metric = sqrtf(lb);           // 'L1' metric_reduction: sqrt per sample, then the batch mean (libs/ft.py:1075-1076)
    // d(mean_b f(lb)) / dp = (1/B) f'(lb) * beta * 2 (p - t) / (N tnorm)
    const float fl = a.return_norm ? 0.5f / sqrtf(lb) : 1.f;
    const float fr = a.return_norm ? 0.5f / sqrtf(rb) : 1.f;
    r.cl = fl * a.beta * 2.f / (N * tnorm) / (float)a.B;
    // regulariser: gamma h / (Nint2 tpnorm) * 2 * K^2 (D_h p - tp) . d(D_h p)/dp, with d(D_h p)/dp = +-1 / (2 s h)
    r.cr = reg_on ? fr * a.gamma * a.h * 2.f / (Nint2 * tpnorm) / (2.f * a.s * a.h) / (float)a.B : 0.f;
    return r;
}

__global__ void __launch_bounds__(LOSS_THREADS) loss_grad_kernel(LossArgs a) {
    pdl_enter();
    __shared__ SampleScalars sc;
    const int b = blockIdx.y, chunk = blockIdx.x, n = a.n, N = n * n, s = a.s;
    if (threadIdx.x == 0) sc = sample_scalars(a, b);
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 32) {
        float L = 0.f, R = 0.f, Mt = 0.f;
        for (int bb = 0; bb < a.B; ++bb) {
            const SampleScalars q = sample_scalars(a, bb);
            L += q.loss;
            R += q.reg;
            Mt += q.metric;
        }
        L /= (float)a.B;
        R /= (float)a.B;
        a.out[0] = L;
        a.out[1] = R;
        a.out[2] = Mt / (float)a.B;
        a.out[3] = L + R;
    }
    __syncthreads();
    if (!a.dl) return;
    const int per = (N + a.chunks - 1) / a.chunks;
    const int e0 = chunk * per, e1 = min(N, e0 + per);
    const float* pb = a.p + (long long)b * N;
    const float* tb = a.t + (long long)b * N;
    const float* tpb = a.tp ? a.tp + (long long)b * N * 2 : nullptr;
    const float* Kb = a.K ? a.K + (long long)b * N : nullptr;
    const bool reg_on = a.regularizer && a.tp;
    for (int e = e0 + threadIdx.x; e < e1; e += LOSS_THREADS) {
        a.dl[(long long)b * N + e] = sc.cl * (pb[e] - tb[e]);
        if (a.dr) {
            float g = 0.f;
            if (reg_on) {
                const int i = e / n, j = e % n;
                // p[i][j] enters D_x at (i-s, j) with +, at (i+s, j) with -, D_y at (i, j-s) with +, at (i, j+s) with -
                g = h1_residual(a, pb, tpb, Kb, i - s, j).x - h1_residual(a, pb, tpb, Kb, i + s, j).x +
                    h1_residual(a, pb, tpb, Kb, i, j - s).y - h1_residual(a, pb, tpb, Kb, i, j + s).y;
            }
            a.dr[(long long)b * N + e] = sc.cr * g;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
constexpr int ADAM_THREADS = 256, ADAM_MAX_PARTS = 1024;

__global__ void __launch_bounds__(ADAM_THREADS) sumsq_partial_kernel(const float* __restrict__ g, long long n,
                                                                     float* __restrict__ parts) {
    pdl_enter();
    __shared__ float red[ADAM_THREADS / 32];
    const long long per = ((n + gridDim.x - 1) / gridDim.x + 3) / 4 * 4;
    const long long e0 = blockIdx.x * per, e1 = min(n, e0 + per);
    float s = 0.f;
    if (e1 > e0) {
        if (((uintptr_t)g & 15) == 0) {          // chunk starts are multiples of 4 elements
            const long long nvec = (e1 - e0) / 4;
            const float4* g4 = reinterpret_cast<const float4*>(g + e0);
            for (long long q = threadIdx.x; q < nvec; q += ADAM_THREADS) {
                const float4 v = g4[q];
                s = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, s))));
            }
            if (threadIdx.x == 0)
                for (long long e = e0 + 4 * nvec; e < e1; ++e) s = fmaf(g[e], g[e], s);
        } else {
            for (long long e = e0 + threadIdx.x; e < e1; e += ADAM_THREADS) s = fmaf(g[e], g[e], s);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (threadIdx.x % 32 == 0) red[threadIdx.x / 32] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < ADAM_THREADS / 32; ++w) t += red[w];
        parts[blockIdx.x] = t;
    }
}

struct AdamArgs {
    float *p, *m, *v;
    const float* g;
    long long n;
    const float* hyper;     // device: lr, beta1, bias_correction1, bias_correction2
    float beta2, eps, weight_decay, max_norm;
    const float* parts;
    int nparts;
    float* norm_out;        // total gradient norm before clipping, or null
};

__global__ void __launch_bounds__(ADAM_THREADS) adam_kernel(AdamArgs a) {
    pdl_enter();
    __shared__ float red[ADAM_THREADS];
    float s = 0.f;
    for (int i = threadIdx.x; i < a.nparts; i += ADAM_THREADS) s += a.parts[i];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = ADAM_THREADS / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    const float total = sqrtf(red[0]);
    if (blockIdx.x == 0 && threadIdx.x == 0 && a.norm_out) *a.norm_out = total;
    // torch.nn.utils.clip_grad_norm_: clip_coef = max_norm / (total_norm + 1e-6), clamped to 1
    const float clip = a.max_norm > 0.f ? fminf(1.f, a.max_norm / (total + 1e-6f)) : 1.f;
    const float lr = a.hyper[0], beta1 = a.hyper[1], bc1 = a.hyper[2], bc2 = a.hyper[3];
    const float step_size = lr / bc1, rs2 = 1.f / sqrtf(bc2);
    const long long stride = (long long)gridDim.x * ADAM_THREADS;
    for (long long e = (long long)blockIdx.x * ADAM_THREADS + threadIdx.x; e < a.n; e += stride) {
        float g = a.g[e] * clip;
        const float p = a.p[e];
        if (a.weight_decay != 0.f) g = fmaf(a.weight_decay, p, g);
        // torch/optim/adam.py (_single_tensor_adam): exp_avg.lerp_(grad, 1 - beta1); exp_avg_sq.mul_(beta2).addcmul_(g, g, 1 - beta2);
        // denom = exp_avg_sq.sqrt() / sqrt(bias_correction2) + eps; param.addcdiv_(exp_avg, denom, value=-step_size)
        const float m = fmaf(g - a.m[e], 1.f - beta1, a.m[e]);
        const float v = fmaf(a.v[e], a.beta2, (1.f - a.beta2) * g * g);
        a.m[e] = m;
        a.v[e] = v;
        const float denom = sqrtf(v) * rs2 + a.eps;
        a.p[e] = p - step_size * (m / denom);
    }
}

}  // namespace gb200

using namespace gb200;

static int loss_chunks(int B, int n) {
    const long long N = (long long)n * n;
    int c = (int)((4 * 148 + B - 1) / B);                       // a few CTAs per SM over the batch
    const int maxc = (int)((N + 2047) / 2048);                  // at least 2048 pixels per chunk
    if (c > maxc) c = maxc;
    if (c > 64) c = 64;
    return c < 1 ? 1 : c;
}

extern "C" size_t gb200_weighted_l2_loss2d_workspace_bytes(int B, int n) {
    return (size_t)B * loss_chunks(B, n) * 4 * sizeof(float);
}

extern "C" int gb200_weighted_l2_loss2d(int device, const float* preds, const float* targets, const float* targets_prime,
                                        const float* K, int B, int n, float h, float beta, float gamma, float eps,
                                        int dilation, int regularizer, int return_norm, float* out4, float* dloss,
                                        float* dreg, float* workspace, size_t workspace_bytes, void* stream) {
    use_device(device);
    GB_REQUIRE(preds && targets && out4 && workspace, "gb200_weighted_l2_loss2d: null argument");
    GB_REQUIRE(B >= 1 && B <= 65535 && n >= 1 && (long long)n * n < (1LL << 30), "gb200_weighted_l2_loss2d: bad shape");
    GB_REQUIRE(dilation >= 2 && dilation % 2 == 0 && n > dilation, "gb200_weighted_l2_loss2d: dilation %d (even, < n)",
               dilation);
    GB_REQUIRE(workspace_bytes >= gb200_weighted_l2_loss2d_workspace_bytes(B, n),
               "gb200_weighted_l2_loss2d: workspace too small");
    GB_REQUIRE(!targets_prime || ((uintptr_t)targets_prime % 8) == 0, "gb200_weighted_l2_loss2d: targets_prime alignment");
    GB_REQUIRE(((uintptr_t)workspace % 16) == 0, "gb200_weighted_l2_loss2d: workspace alignment");
    LossArgs a;
    a.p = preds; a.t = targets; a.tp = targets_prime; a.K = K; a.B = B; a.n = n; a.s = dilation / 2;
    a.h = h; a.beta = beta; a.gamma = gamma; a.eps = eps; a.regularizer = regularizer; a.return_norm = return_norm;
    a.chunks = loss_chunks(B, n); a.ws = workspace; a.out = out4; a.dl = dloss; a.dr = dreg;
    cudaStream_t st = as_stream(stream);
    dim3 grid(a.chunks, B);
    launch_kernel(loss_partial_kernel, grid, LOSS_THREADS, 0, st, a);
    launch_kernel(loss_grad_kernel, grid, LOSS_THREADS, 0, st, a);
    return check_launch("gb200_weighted_l2_loss2d", 2);
}

static int adam_parts(long long n) {
    long long p = (n + 16383) / 16384;
    if (p > ADAM_MAX_PARTS) p = ADAM_MAX_PARTS;
    return p < 1 ? 1 : (int)p;
}

extern "C" size_t gb200_adam_clip_step_workspace_bytes(long long n) { return (size_t)adam_parts(n) * sizeof(float); }

extern "C" int gb200_adam_clip_step(int device, float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                                    long long n, const float* hyper, float beta2, float eps, float weight_decay,
                                    float max_norm, float* grad_norm_out, float* workspace, size_t workspace_bytes,
                                    void* stream) {
    use_device(device);
    GB_REQUIRE(param && grad && exp_avg && exp_avg_sq && hyper && workspace, "gb200_adam_clip_step: null argument");
    GB_REQUIRE(n >= 1, "gb200_adam_clip_step: empty parameter bucket");
    GB_REQUIRE(workspace_bytes >= gb200_adam_clip_step_workspace_bytes(n), "gb200_adam_clip_step: workspace too small");
    cudaStream_t st = as_stream(stream);
    const int parts = adam_parts(n);
    launch_kernel(sumsq_partial_kernel, parts, ADAM_THREADS, 0, st, grad, n, workspace);
    AdamArgs a;
    a.p = param; a.m = exp_avg; a.v = exp_avg_sq; a.g = grad; a.n = n; a.hyper = hyper; a.beta2 = beta2; a.eps = eps;
    a.weight_decay = weight_decay; a.max_norm = max_norm; a.parts = workspace; a.nparts = parts; a.norm_out = grad_norm_out;
    long long blocks = (n + ADAM_THREADS * 4 - 1) / (ADAM_THREADS * 4);
    if (blocks > 148 * 8) blocks = 148 * 8;
    launch_kernel(adam_kernel, (int)blocks, ADAM_THREADS, 0, st, a);
    return check_launch("gb200_adam_clip_step", 2);
}
