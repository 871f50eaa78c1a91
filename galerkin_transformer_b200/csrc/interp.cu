// Bilinear resize of channel-last grids, align_corners = True (the interpolation steps of the reference's
// Interp2dEncoder / Interp2dUpsample scalers: libs/layers.py:431-512, 624-670 call F.interpolate(mode='bilinear',
// align_corners=True) on (B, C, H, W); here the grid stays (B, H, W, C) in memory).
//
//   src_y = oy * (Hin - 1) / (Hout - 1),  y0 = floor(src_y), y1 = min(y0 + 1, Hin - 1), ly = src_y - y0
//   out[b, oy, ox, :] = (1-ly) (1-lx) in[y0,x0] + (1-ly) lx in[y0,x1] + ly (1-lx) in[y1,x0] + ly lx in[y1,x1]
//
// Both directions are pure streaming passes: one thread per (pixel, 4 channels), float4 memory operations.  The
// backward is a GATHER over the few output pixels whose stencil touches an input pixel (no atomics: deterministic).
#include "common.cuh"

namespace gb200 {

struct InterpArgs {
    const float* in; float* out;
    int B, Hin, Win, Hout, Wout, C;
    float sy, sx;            // (in - 1) / (out - 1), or 0 when out == 1
};

__device__ __forceinline__ void src_index(float scale, int dst, int nin, int& i0, int& i1, float& l) {
    const float s = scale * dst;
    i0 = min((int)s, nin - 1);
    i1 = i0 + (i0 < nin - 1 ? 1 : 0);
    l = s - (float)i0;
}

template <bool VEC>
__global__ void __launch_bounds__(256) interp_fwd_kernel(InterpArgs a) {
    pdl_enter();
    // one output row (b, oy) per CTA pass; threads stride over (ox, channel quad): 32-bit index arithmetic only
    const int cq = VEC ? a.C / 4 : a.C;
    const int rowlen = a.Wout * cq;
    for (int row = blockIdx.x; row < a.B * a.Hout; row += gridDim.x) {
      const int b = row / a.Hout, oy = row % a.Hout;
      int y0, y1; float ly;
      src_index(a.sy, oy, a.Hin, y0, y1, ly);
      for (int t = threadIdx.x; t < rowlen; t += blockDim.x) {
        const int ox = t / cq, c = t % cq;
        const long long e = (long long)row * rowlen + t;
        int x0, x1; float lx;
        src_index(a.sx, ox, a.Win, x0, x1, lx);
        const float hy = 1.f - ly, hx = 1.f - lx;
        const long long base = (long long)b * a.Hin * a.Win;
        if (VEC) {
            const float4* in4 = reinterpret_cast<const float4*>(a.in);
            const float4 v00 = in4[(base + (long long)y0 * a.Win + x0) * cq + c];
            const float4 v01 = in4[(base + (long long)y0 * a.Win + x1) * cq + c];
            const float4 v10 = in4[(base + (long long)y1 * a.Win + x0) * cq + c];
            const float4 v11 = in4[(base + (long long)y1 * a.Win + x1) * cq + c];
            float4 o;
            o.x = hy * (hx * v00.x + lx * v01.x) + ly * (hx * v10.x + lx * v11.x);
            o.y = hy * (hx * v00.y + lx * v01.y) + ly * (hx * v10.y + lx * v11.y);
            o.z = hy * (hx * v00.z + lx * v01.z) + ly * (hx * v10.z + lx * v11.z);
            o.w = hy * (hx * v00.w + lx * v01.w) + ly * (hx * v10.w + lx * v11.w);
            reinterpret_cast<float4*>(a.out)[e] = o;
        } else {
            const float v00 = a.in[(base + (long long)y0 * a.Win + x0) * cq + c];
            const float v01 = a.in[(base + (long long)y0 * a.Win + x1) * cq + c];
            const float v10 = a.in[(base + (long long)y1 * a.Win + x0) * cq + c];
            const float v11 = a.in[(base + (long long)y1 * a.Win + x1) * cq + c];
            a.out[e] = hy * (hx * v00 + lx * v01) + ly * (hx * v10 + lx * v11);
        }
      }
    }
}

// candidate destination range [lo, hi] whose stencil can touch source index i: scale * dst in [i - 1, i + 1), with one
// index of slack on the open end (membership is decided exactly by axis_weight)
__device__ __forceinline__ void dst_range(float scale, int i, int nout, int& lo, int& hi) {
    if (scale <= 0.f) { lo = 0; hi = nout - 1; return; }
    lo = max(0, (int)floorf((float)(i - 1) / scale));
    hi = min(nout - 1, (int)ceilf((float)(i + 1) / scale) + 1);
}
__device__ __forceinline__ float axis_weight(float scale, int dst, int nin, int i) {
    int i0, i1; float l;
    src_index(scale, dst, nin, i0, i1, l);
    return (i0 == i ? 1.f - l : 0.f) + (i1 == i ? l : 0.f);
}

// d_in[b, iy, ix, :] = sum over (oy, ox) of wy(oy, iy) * wx(ox, ix) * d_out[b, oy, ox, :]      (a.in = d_out, a.out = d_in;
// Hin/Win are the FORWARD input sizes, i.e. the sizes of d_in).  The per-axis weights of the (at most MAXR) candidate
// rows / columns are computed once per thread; wider ranges (resize ratios above ~3x) take the generic double loop.
template <bool VEC>
__global__ void __launch_bounds__(256) interp_bwd_kernel(InterpArgs a) {
    pdl_enter();
    constexpr int MAXR = 8;
    const int cq = VEC ? a.C / 4 : a.C;
    const int rowlen = a.Win * cq;
    for (int row = blockIdx.x; row < a.B * a.Hin; row += gridDim.x) {
      const int b = row / a.Hin, iy = row % a.Hin;
      int ylo, yhi;
      dst_range(a.sy, iy, a.Hout, ylo, yhi);
      for (int t = threadIdx.x; t < rowlen; t += blockDim.x) {
        const int ix = t / cq, c = t % cq;
        const long long e = (long long)row * rowlen + t;
        int xlo, xhi;
        dst_range(a.sx, ix, a.Wout, xlo, xhi);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        const long long base = (long long)b * a.Hout * a.Wout;
        const int ny = yhi - ylo + 1, nx = xhi - xlo + 1;
        if (ny <= MAXR && nx <= MAXR) {
            float wy[MAXR], wx[MAXR];
#pragma unroll
            for (int u = 0; u < MAXR; ++u) {
                wy[u] = u < ny ? axis_weight(a.sy, ylo + u, a.Hin, iy) : 0.f;
                wx[u] = u < nx ? axis_weight(a.sx, xlo + u, a.Win, ix) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < MAXR; ++u) {
                if (wy[u] == 0.f) continue;
#pragma unroll
                for (int v = 0; v < MAXR; ++v) {
                    const float w = wy[u] * wx[v];
                    if (w == 0.f) continue;
                    const long long o = (base + (long long)(ylo + u) * a.Wout + (xlo + v)) * cq + c;
                    if (VEC) {
                        const float4 g = reinterpret_cast<const float4*>(a.in)[o];
                        acc.x = fmaf(w, g.x, acc.x); acc.y = fmaf(w, g.y, acc.y);
                        acc.z = fmaf(w, g.z, acc.z); acc.w = fmaf(w, g.w, acc.w);
                    } else {
                        acc.x = fmaf(w, a.in[o], acc.x);
                    }
                }
            }
        } else {
            for (int oy = ylo; oy <= yhi; ++oy) {
                const float wyv = axis_weight(a.sy, oy, a.Hin, iy);
                if (wyv == 0.f) continue;
                for (int ox = xlo; ox <= xhi; ++ox) {
                    const float w = wyv * axis_weight(a.sx, ox, a.Win, ix);
                    if (w == 0.f) continue;
                    const long long o = (base + (long long)oy * a.Wout + ox) * cq + c;
                    if (VEC) {
                        const float4 g = reinterpret_cast<const float4*>(a.in)[o];
                        acc.x = fmaf(w, g.x, acc.x); acc.y = fmaf(w, g.y, acc.y);
                        acc.z = fmaf(w, g.z, acc.z); acc.w = fmaf(w, g.w, acc.w);
                    } else {
                        acc.x = fmaf(w, a.in[o], acc.x);
                    }
                }
            }
        }
        if (VEC) reinterpret_cast<float4*>(a.out)[e] = acc;
        else a.out[e] = acc.x;
      }
    }
}

// Table-driven backward for resize ratios up to ~3x (every shipped scaler): the per-axis candidate ranges and weights depend
// only on the pixel coordinate, so the x table (Win entries) is built once per CTA and the y weights once per row, instead of
// 16 weight evaluations + 2 range computations per THREAD (the gather above spent ~250 ALU instructions per float4 of output
// and was issue-bound at ~60-90 us for an 81 MB pass).  A warp covers one pixel's channel run, so every tap test is warp-
// uniform; the <= 8 candidate columns of a row are fetched as 8 independent predicated float4 loads.
constexpr int IB_MAXR = 8;

template <bool VEC>
__global__ void __launch_bounds__(256) interp_bwd_table_kernel(InterpArgs a) {
    pdl_enter();
    extern __shared__ __align__(16) float tab[];       // [Win][IB_MAXR] weights from the first live column on, then [Win] that column
    __shared__ float s_wy[IB_MAXR];
    __shared__ int s_ylo;
    float* wxs = tab;
    int* xlos = reinterpret_cast<int*>(tab + (size_t)a.Win * IB_MAXR);
    for (int ix = threadIdx.x; ix < a.Win; ix += blockDim.x) {
        int xlo, xhi;
        dst_range(a.sx, ix, a.Wout, xlo, xhi);
        float w[IB_MAXR];
        int first = IB_MAXR;
#pragma unroll
        for (int v = IB_MAXR - 1; v >= 0; --v) {
            w[v] = (xlo + v <= xhi) ? axis_weight(a.sx, xlo + v, a.Win, ix) : 0.f;
            if (w[v] != 0.f) first = v;
        }
        if (first == IB_MAXR) first = 0;
        xlos[ix] = xlo + first;                        // live taps are contiguous: shift them to the front
#pragma unroll
        for (int v = 0; v < IB_MAXR; ++v) {
            float t = 0.f;
#pragma unroll
            for (int q = 0; q < IB_MAXR; ++q)
                if (q == v + first) t = w[q];
            wxs[ix * IB_MAXR + v] = t;
        }
    }
    const int cq = VEC ? a.C / 4 : a.C;
    const int rowlen = a.Win * cq;
    for (int row = blockIdx.x; row < a.B * a.Hin; row += gridDim.x) {
        const int b = row / a.Hin, iy = row % a.Hin;
        __syncthreads();
        if (threadIdx.x < IB_MAXR) {
            int ylo, yhi;
            dst_range(a.sy, iy, a.Hout, ylo, yhi);
            if (threadIdx.x == 0) s_ylo = ylo;
            s_wy[threadIdx.x] = (ylo + (int)threadIdx.x <= yhi) ? axis_weight(a.sy, ylo + threadIdx.x, a.Hin, iy) : 0.f;
        }
        __syncthreads();
        const int ylo = s_ylo;
        const long long base = (long long)b * a.Hout * a.Wout;
        for (int t = threadIdx.x; t < rowlen; t += blockDim.x) {
            const int ix = t / cq, c = t % cq;
            const int xlo = xlos[ix];
            const float4 wa = *reinterpret_cast<const float4*>(wxs + ix * IB_MAXR);
            const float4 wb = *reinterpret_cast<const float4*>(wxs + ix * IB_MAXR + 4);
            const float wx[IB_MAXR] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
            const bool tail = wb.x != 0.f;                             // more than four live columns (ratios above ~2x)
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
            for (int u = 0; u < IB_MAXR; ++u) {
                const float wy = s_wy[u];
                if (wy == 0.f) continue;                               // uniform over the CTA
                const long long o = (base + (long long)(ylo + u) * a.Wout + xlo) * cq + c;
                if (VEC) {
                    float4 g[4];
#pragma unroll
                    for (int v = 0; v < 4; ++v)
                        g[v] = wx[v] != 0.f ? reinterpret_cast<const float4*>(a.in)[o + (long long)v * cq]
                                            : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int v = 0; v < 4; ++v) {
                        const float w = wy * wx[v];
                        acc.x = fmaf(w, g[v].x, acc.x); acc.y = fmaf(w, g[v].y, acc.y);
                        acc.z = fmaf(w, g[v].z, acc.z); acc.w = fmaf(w, g[v].w, acc.w);
                    }
                    if (tail) {
#pragma unroll
                        for (int v = 4; v < IB_MAXR; ++v) {
                            if (wx[v] != 0.f) {
                                const float4 gg = reinterpret_cast<const float4*>(a.in)[o + (long long)v * cq];
                                const float w = wy * wx[v];
                                acc.x = fmaf(w, gg.x, acc.x); acc.y = fmaf(w, gg.y, acc.y);
                                acc.z = fmaf(w, gg.z, acc.z); acc.w = fmaf(w, gg.w, acc.w);
                            }
                        }
                    }
                } else {
#pragma unroll
                    for (int v = 0; v < IB_MAXR; ++v)
                        if (wx[v] != 0.f) acc.x = fmaf(wy * wx[v], a.in[o + (long long)v * cq], acc.x);
                }
            }
            const long long e = (long long)row * rowlen + t;
            if (VEC) reinterpret_cast<float4*>(a.out)[e] = acc;
            else a.out[e] = acc.x;
        }
    }
}

// Forward with the same per-CTA x table (source columns and weight per output column) and per-row y weights: the per-thread
// work is four float4 loads, the blend and one float4 store.
template <bool VEC>
__global__ void __launch_bounds__(256) interp_fwd_table_kernel(InterpArgs a) {
    pdl_enter();
    extern __shared__ __align__(16) float tab[];       // [Wout] lx, then [Wout] x0, [Wout] x1 (int)
    float* lxs = tab;
    int* x0s = reinterpret_cast<int*>(tab + a.Wout);
    int* x1s = x0s + a.Wout;
    for (int ox = threadIdx.x; ox < a.Wout; ox += blockDim.x) {
        int x0, x1; float lx;
        src_index(a.sx, ox, a.Win, x0, x1, lx);
        lxs[ox] = lx; x0s[ox] = x0; x1s[ox] = x1;
    }
    __syncthreads();
    const int cq = VEC ? a.C / 4 : a.C;
    const int rowlen = a.Wout * cq;
    for (int row = blockIdx.x; row < a.B * a.Hout; row += gridDim.x) {
        const int b = row / a.Hout, oy = row % a.Hout;
        int y0, y1; float ly;
        src_index(a.sy, oy, a.Hin, y0, y1, ly);
        const float hy = 1.f - ly;
        const long long r0 = ((long long)b * a.Hin + y0) * a.Win, r1 = ((long long)b * a.Hin + y1) * a.Win;
        for (int t = threadIdx.x; t < rowlen; t += blockDim.x) {
            const int ox = t / cq, c = t % cq;
            const int x0 = x0s[ox], x1 = x1s[ox];
            const float lx = lxs[ox], hx = 1.f - lx;
            const long long e = (long long)row * rowlen + t;
            if (VEC) {
                const float4* in4 = reinterpret_cast<const float4*>(a.in);
                const float4 v00 = in4[(r0 + x0) * cq + c], v01 = in4[(r0 + x1) * cq + c];
                const float4 v10 = in4[(r1 + x0) * cq + c], v11 = in4[(r1 + x1) * cq + c];
                float4 o;
                o.x = hy * (hx * v00.x + lx * v01.x) + ly * (hx * v10.x + lx * v11.x);
                o.y = hy * (hx * v00.y + lx * v01.y) + ly * (hx * v10.y + lx * v11.y);
                o.z = hy * (hx * v00.z + lx * v01.z) + ly * (hx * v10.z + lx * v11.z);
                o.w = hy * (hx * v00.w + lx * v01.w) + ly * (hx * v10.w + lx * v11.w);
                reinterpret_cast<float4*>(a.out)[e] = o;
            } else {
                const float v00 = a.in[(r0 + x0) * cq + c], v01 = a.in[(r0 + x1) * cq + c];
                const float v10 = a.in[(r1 + x0) * cq + c], v11 = a.in[(r1 + x1) * cq + c];
                a.out[e] = hy * (hx * v00 + lx * v01) + ly * (hx * v10 + lx * v11);
            }
        }
    }
}

// widest candidate range dst_range can return for this scale (host mirror of the device arithmetic, with slack)
static int max_candidates(float scale, int nout) {
    if (scale <= 0.f) return nout;
    return (int)(2.0f / scale) + 4;
}

static int launch_interp(bool backward, const float* in, float* out, int B, int Hin, int Win, int Hout, int Wout, int C,
                         cudaStream_t st) {
    InterpArgs a;
    a.in = in; a.out = out; a.B = B; a.Hin = Hin; a.Win = Win; a.Hout = Hout; a.Wout = Wout; a.C = C;
    a.sy = Hout > 1 ? (float)(Hin - 1) / (float)(Hout - 1) : 0.f;       // same float arithmetic as ATen's
    a.sx = Wout > 1 ? (float)(Win - 1) / (float)(Wout - 1) : 0.f;       // area_pixel_compute_scale<float>(align_corners)
    const bool vec = C % 4 == 0 && ((uintptr_t)in % 16) == 0 && ((uintptr_t)out % 16) == 0;
    long long blocks = (long long)B * (backward ? Hin : Hout);      // one grid row per CTA pass
    if (blocks > 148 * 32) blocks = 148 * 32;
    if (blocks < 1) blocks = 1;
    if (backward) {
        const size_t smem = (size_t)Win * (IB_MAXR + 1) * sizeof(float);
        if (max_candidates(a.sy, Hout) <= IB_MAXR && max_candidates(a.sx, Wout) <= IB_MAXR && smem <= 40 * 1024) {
            if (vec) launch_kernel(interp_bwd_table_kernel<true>, (int)blocks, 256, smem, st, a);
            else launch_kernel(interp_bwd_table_kernel<false>, (int)blocks, 256, smem, st, a);
        } else if (vec) {
            launch_kernel(interp_bwd_kernel<true>, (int)blocks, 256, 0, st, a);
        } else {
            launch_kernel(interp_bwd_kernel<false>, (int)blocks, 256, 0, st, a);
        }
    } else {
        const size_t smem = (size_t)Wout * 3 * sizeof(float);
        if (smem <= 40 * 1024) {
            if (vec) launch_kernel(interp_fwd_table_kernel<true>, (int)blocks, 256, smem, st, a);
            else launch_kernel(interp_fwd_table_kernel<false>, (int)blocks, 256, smem, st, a);
        } else if (vec) {
            launch_kernel(interp_fwd_kernel<true>, (int)blocks, 256, 0, st, a);
        } else {
            launch_kernel(interp_fwd_kernel<false>, (int)blocks, 256, 0, st, a);
        }
    }
    return check_launch(backward ? "gb200_interp_bilinear_bwd" : "gb200_interp_bilinear_fwd");
}

}  // namespace gb200

using namespace gb200;

extern "C" int gb200_interp_bilinear_fwd(int device, const float* in, int B, int Hin, int Win, int C, float* out, int Hout,
                                         int Wout, void* stream) {
    use_device(device);
    GB_REQUIRE(in && out && B >= 1 && Hin >= 1 && Win >= 1 && Hout >= 1 && Wout >= 1 && C >= 1,
               "gb200_interp_bilinear_fwd: bad arguments");
    return launch_interp(false, in, out, B, Hin, Win, Hout, Wout, C, as_stream(stream));
}

extern "C" int gb200_interp_bilinear_bwd(int device, const float* dout, int B, int Hin, int Win, int C, float* din, int Hout,
                                         int Wout, void* stream) {
    use_device(device);
    GB_REQUIRE(dout && din && B >= 1 && Hin >= 1 && Win >= 1 && Hout >= 1 && Wout >= 1 && C >= 1,
               "gb200_interp_bilinear_bwd: bad arguments");
    return launch_interp(true, dout, din, B, Hin, Win, Hout, Wout, C, as_stream(stream));
}
