// Library-level plumbing: error strings, device selection, launch accounting.
#include <atomic>
#include <cstdarg>

#include "common.cuh"

namespace gb200 {

static thread_local char g_err[512] = "";
static thread_local int g_device = -1;
static std::atomic<unsigned long long> g_launches{0};
static const unsigned long long* g_rng_offset = nullptr;

const unsigned long long* rng_offset_ptr() { return g_rng_offset; }

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

void use_device(int device) {
    // the caller (PyTorch) may have switched this thread's current device since the last call: ask, do not cache
    if (device < 0) return;
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess || cur != device) cudaSetDevice(device);
    g_device = device;
}

int check_launch(const char* what, int nkernels) {
    g_launches.fetch_add((unsigned long long)nkernels, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: CUDA error %d (%s)", what, (int)e, cudaGetErrorString(e));
        return GB200_ERR_CUDA;
    }
    return GB200_OK;
}

}  // namespace gb200

extern "C" int gb200_version(void) { return 102; }
extern "C" int gb200_set_rng_offset_ptr(const unsigned long long* device_counter) {
    gb200::g_rng_offset = device_counter;
    return GB200_OK;
}
extern "C" const char* gb200_last_error(void) { return gb200::g_err; }
extern "C" unsigned long long gb200_launch_count(void) { return gb200::g_launches.load(); }

// ---- parameter packing: many small tensors -> one contiguous buffer, ONE launch -------------------------------
// (replaces the torch.cat / torch.stack calls that assemble W_qkv, b_qkv and the per-head LayerNorm affine tables
//  from the reference's separate nn.Linear / nn.LayerNorm parameters on every forward)
namespace gb200 {
constexpr int PACK_MAX = 64;
struct PackArgs { const float* src[PACK_MAX]; long long off[PACK_MAX + 1]; };
__global__ void pack_kernel(PackArgs a, float* __restrict__ dst) {
    pdl_enter();
    const int seg = blockIdx.x;
    const float* s = a.src[seg];
    float* d = dst + a.off[seg];
    const long long n = a.off[seg + 1] - a.off[seg];
    for (long long i = blockIdx.y * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.y * blockDim.x)
        d[i] = s[i];
}
}  // namespace gb200

extern "C" int gb200_pack(int device, float* dst, const float* const* srcs, const long long* sizes, int n, void* stream) {
    using namespace gb200;
    use_device(device);
    GB_REQUIRE(dst && srcs && sizes && n >= 1 && n <= PACK_MAX, "gb200_pack: 1..%d segments", PACK_MAX);
    PackArgs a;
    long long off = 0, biggest = 0;
    for (int i = 0; i < n; ++i) {
        GB_REQUIRE(srcs[i] && sizes[i] >= 0, "gb200_pack: bad segment %d", i);
        a.src[i] = srcs[i]; a.off[i] = off; off += sizes[i];
        if (sizes[i] > biggest) biggest = sizes[i];
    }
    a.off[n] = off;
    int by = (int)((biggest + 256 * 8 - 1) / (256 * 8));
    if (by < 1) by = 1;
    if (by > 32) by = 32;
    launch_kernel(pack_kernel, dim3(n, by), 256, 0, as_stream(stream), a, dst);
    return check_launch("gb200_pack");
}
