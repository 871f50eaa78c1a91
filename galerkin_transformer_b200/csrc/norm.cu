// Row LayerNorm over d_model (the post-LN encoder variant, libs/model.py:128-129, 134-135,
// used by the Navier-Stokes configuration, examples/ex4_navier_stokes_2+1d.py:40-41).
// One warp per row, two-pass statistics, deterministic two-stage dgamma/dbeta reduction.
#include "common.cuh"

namespace gb200 {

constexpr int LN_WARPS = 8;
constexpr int LN_MAXW = 1024;

__global__ void __launch_bounds__(LN_WARPS * 32) layernorm_fwd_kernel(
    const float* __restrict__ x, long long rows, int width, const float* __restrict__ gamma,
    const float* __restrict__ beta, float eps, float* __restrict__ y, float* __restrict__ mean_out,
    float* __restrict__ rstd_out) {
    pdl_enter();
    const int lane = threadIdx.x % 32, warp = threadIdx.x / 32;
    for (long long r = (long long)blockIdx.x * LN_WARPS + warp; r < rows; r += (long long)gridDim.x * LN_WARPS) {
        const float* xr = x + r * width;
        float s = 0.f;
        for (int c = lane; c < width; c += 32) s += xr[c];
        const float mean = warp_sum(s) / width;
        float v = 0.f;
        for (int c = lane; c < width; c += 32) { float d = xr[c] - mean; v += d * d; }
        const float rstd = rsqrtf(warp_sum(v) / width + eps);
        float* yr = y + r * width;
        for (int c = lane; c < width; c += 32) yr[c] = (xr[c] - mean) * rstd * gamma[c] + beta[c];
        if (lane == 0) { mean_out[r] = mean; rstd_out[r] = rstd; }
    }
}

__global__ void __launch_bounds__(LN_WARPS * 32) layernorm_bwd_kernel(
    const float* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ mean,
    const float* __restrict__ rstd, const float* __restrict__ gamma, long long rows, int width,
    float* __restrict__ dx, float* __restrict__ part) {
    pdl_enter();
    extern __shared__ float sm[];   // [LN_WARPS][2][width]
    const int lane = threadIdx.x % 32, warp = threadIdx.x / 32;
    float* sg = sm + (size_t)warp * 2 * width;
    float* sb = sg + width;
    for (int c = lane; c < width; c += 32) { sg[c] = 0.f; sb[c] = 0.f; }
    for (long long r = (long long)blockIdx.x * LN_WARPS + warp; r < rows; r += (long long)gridDim.x * LN_WARPS) {
        const float* xr = x + r * width;
        const float* dr = dy + r * width;
        const float mu = mean[r], rs = rstd[r];
        float c1 = 0.f, c2 = 0.f;
        for (int c = lane; c < width; c += 32) {
            float xh = (xr[c] - mu) * rs, gd = gamma[c] * dr[c];
            c1 += gd; c2 += gd * xh;
            sg[c] += dr[c] * xh;
            sb[c] += dr[c];
        }
        c1 = warp_sum(c1) / width; c2 = warp_sum(c2) / width;
        float* dxr = dx + r * width;
        for (int c = lane; c < width; c += 32) {
            float xh = (xr[c] - mu) * rs;
            dxr[c] = rs * (gamma[c] * dr[c] - c1 - xh * c2);
        }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < width; c += blockDim.x) {
        float tg = 0.f, tb = 0.f;
        for (int w = 0; w < LN_WARPS; ++w) {
            tg += sm[(size_t)w * 2 * width + c];
            tb += sm[(size_t)w * 2 * width + width + c];
        }
        part[((long long)blockIdx.x * 2 + 0) * width + c] = tg;
        part[((long long)blockIdx.x * 2 + 1) * width + c] = tb;
    }
}

__global__ void layernorm_bwd_reduce_kernel(const float* __restrict__ part, int nblocks, int width,
                                            float* __restrict__ dgamma, float* __restrict__ dbeta,
                                            int accumulate) {
    pdl_enter();
    reduce_partials_2d(part + (long long)blockIdx.y * width, nblocks, 2LL * width, width, 1.f, accumulate,
                       blockIdx.y == 0 ? dgamma : dbeta);
}

static int ln_blocks(long long rows) {
    long long b = (rows + LN_WARPS - 1) / LN_WARPS;
    return (int)(b < 148 * 4 ? b : 148 * 4);
}

}  // namespace gb200

using namespace gb200;

extern "C" int gb200_layernorm_fwd(int device, const float* x, long long rows, int width, const float* gamma,
                                   const float* beta, float eps, float* y, float* mean, float* rstd,
                                   void* stream) {
    use_device(device);
    GB_REQUIRE(x && gamma && beta && y && mean && rstd && width >= 1, "gb200_layernorm_fwd: bad arguments");
    if (rows == 0) return GB200_OK;
    launch_kernel(layernorm_fwd_kernel, ln_blocks(rows), LN_WARPS * 32, 0, as_stream(stream), x, rows, width, gamma, beta,
                                                                                  eps, y, mean, rstd);
    return check_launch("gb200_layernorm_fwd");
}

extern "C" size_t gb200_layernorm_bwd_workspace_bytes(long long rows, int width) {
    return (size_t)ln_blocks(rows) * 2 * width * sizeof(float);
}

extern "C" int gb200_layernorm_bwd(int device, const float* dy, const float* x, const float* mean,
                                   const float* rstd, const float* gamma, long long rows, int width, float* dx,
                                   float* dgamma, float* dbeta, int accumulate, float* workspace,
                                   size_t workspace_bytes, void* stream) {
    use_device(device);
    GB_REQUIRE(dy && x && mean && rstd && gamma && dx && dgamma && dbeta, "gb200_layernorm_bwd: null argument");
    GB_REQUIRE(width >= 1 && width <= LN_MAXW, "gb200_layernorm_bwd: width %d unsupported (max %d)", width, LN_MAXW);
    if (rows == 0) return GB200_OK;
    GB_REQUIRE(workspace && workspace_bytes >= gb200_layernorm_bwd_workspace_bytes(rows, width),
               "gb200_layernorm_bwd: workspace too small");
    const int nblocks = ln_blocks(rows);
    size_t smem = (size_t)LN_WARPS * 2 * width * sizeof(float);
    if (smem > 48 * 1024)
        cudaFuncSetAttribute(layernorm_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaStream_t st = as_stream(stream);
    launch_kernel(layernorm_bwd_kernel, nblocks, LN_WARPS * 32, smem, st, dy, x, mean, rstd, gamma, rows, width, dx, workspace);
    launch_kernel(layernorm_bwd_reduce_kernel, dim3(cdiv(width, 32), 2), dim3(32, 32), 0, st, workspace, nblocks, width, dgamma,
                                                                                dbeta, accumulate);
    return check_launch("gb200_layernorm_bwd", 2);
}
