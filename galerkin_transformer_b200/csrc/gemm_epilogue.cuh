// Epilogue shared by the SIMT and tcgen05 GEMMs:
//   v = alpha*acc + bias[n];  Z = v;  v = act(v);  v *= act'(G) [gate];  v *= dropout(seed, element);
//   C = R + rscale*v  (+= C)
// The gate turns a GEMM into "input gradient of the NEXT layer times the activation/dropout derivative of THIS
// layer" (g1 = (g2 W2) * act'(z1) * mask1), i.e. the elementwise backward pass between two Linear layers fused
// into the producing GEMM.
#pragma once
#include "common.cuh"

namespace gb200 {

struct GemmEpilogue {
    float* C; int ldc; long long sC;
    float alpha;
    const float* bias;
    int act;
    float* Z; int ldz;
    float drop_p; unsigned long long seed;
    const unsigned long long* seed_off;   // device-side step counter (or null): seed += *seed_off
    const float* R; int ldr; float rscale;
    int accumulate;
    const float* G; int ldg; int gate;     // gate: ACT_RELU -> keep where G > 0; ACT_SILU -> times silu'(G); null = off

    __device__ __forceinline__ void store(int batch, int m, int n, int M, int N, float acc) const {
        float v = alpha * acc;
        if (bias) v += bias[n];
        if (Z) Z[(long long)batch * sC + (long long)m * ldz + n] = v;
        v = act_apply(act, v);
        if (G) {
            const float gv = G[(long long)batch * sC + (long long)m * ldg + n];
            v = gate == ACT_RELU ? (gv > 0.f ? v : 0.f) : v * act_grad(gate, gv);
        }
        if (drop_p > 0.f)
            v *= dropout_scale(drop_p, seed + (seed_off ? *seed_off : 0ull), ((unsigned long long)batch * M + m) * N + n);
        float* c = C + (long long)batch * sC + (long long)m * ldc + n;
        if (R) v = R[(long long)batch * sC + (long long)m * ldr + n] + rscale * v;
        else v *= rscale;
        if (accumulate) v += *c;
        *c = v;
    }
    // four consecutive columns n..n+3 of row m (n % 4 == 0; host checked 16-byte alignment of every operand and
    // N % 4 == 0, single batch): same arithmetic as store(), float4 memory operations
    __device__ __forceinline__ void store4(int m, int n, int N, float4 acc) const {
        float4 v = make_float4(alpha * acc.x, alpha * acc.y, alpha * acc.z, alpha * acc.w);
        if (bias) {
            const float4 b = *reinterpret_cast<const float4*>(bias + n);
            v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
        }
        if (Z) *reinterpret_cast<float4*>(Z + (long long)m * ldz + n) = v;
        v = make_float4(act_apply(act, v.x), act_apply(act, v.y), act_apply(act, v.z), act_apply(act, v.w));
        if (G) {
            const float4 gv = *reinterpret_cast<const float4*>(G + (long long)m * ldg + n);
            if (gate == ACT_RELU) {
                v.x = gv.x > 0.f ? v.x : 0.f; v.y = gv.y > 0.f ? v.y : 0.f;
                v.z = gv.z > 0.f ? v.z : 0.f; v.w = gv.w > 0.f ? v.w : 0.f;
            } else {
                v.x *= act_grad(gate, gv.x); v.y *= act_grad(gate, gv.y);
                v.z *= act_grad(gate, gv.z); v.w *= act_grad(gate, gv.w);
            }
        }
        if (drop_p > 0.f) {
            const float4 ds = dropout_scale4(drop_p, seed + (seed_off ? *seed_off : 0ull), (unsigned long long)m * N + n);
            v.x *= ds.x; v.y *= ds.y; v.z *= ds.z; v.w *= ds.w;
        }
        v.x *= rscale; v.y *= rscale; v.z *= rscale; v.w *= rscale;
        float4* c = reinterpret_cast<float4*>(C + (long long)m * ldc + n);
        if (R) {
            const float4 r = *reinterpret_cast<const float4*>(R + (long long)m * ldr + n);
            v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
        }
        if (accumulate) {
            const float4 o = *c;
            v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
        }
        *c = v;
    }
};

}  // namespace gb200
