// The per-vertex linears of the MPNN on vertex-major fp32 planes [V][64]: shared by the DQN gradient step (mpnn_grad.cu) and
// the forward of CSR graph sets (sparse.cu).  Each translation unit instantiates its own copy (anonymous namespace).
#pragma once
#include "eco_common.cuh"

namespace eco {
namespace {

constexpr int F = 64;

// ---- C[v][n] (+)= sum_k A[v][k] B(k, n),  n < 64,  A = [A1 | A2] (K = 64 or 128) -----------------------------------
//   FWD: B(k, n) = W[n * ldw + k]          (a Linear layer: C = A W^T), optional ReLU on the output
//   BWD: B(k, n) = W[k * ldw + koff + n]   (gradient wrt the layer's input columns koff..koff+63: C = dZ W[:, koff:])
//        with dZ = A1 masked by maskY > 0 (the ReLU of the layer that produced maskY)
constexpr int GT = 64;                 // vertices per tile
constexpr int AT_LD = 68;

template <bool BWD, int K>
__global__ void __launch_bounds__(256)
k_gemm(const float* __restrict__ A1, const float* __restrict__ A2, const float* __restrict__ maskY, const int V,
       const float* __restrict__ W, const int ldw, const int koff, float* __restrict__ C, const int relu, const int accumulate) {
    extern __shared__ __align__(16) unsigned char sm[];
    float* At = reinterpret_cast<float*>(sm);                 // [K][AT_LD]
    float* Bt = At + (size_t)K * AT_LD;                       // [K][64]
    const int tid = threadIdx.x, v0 = blockIdx.x * GT;
    // (compile-time trip counts: the independent loads of a tile are issued back to back)
#pragma unroll 8
    for (int idx = tid; idx < GT * K; idx += 256) {
        const int vv = idx / K, k = idx % K, v = v0 + vv;
        float val = 0.f;
        if (v < V) {
            val = k < 64 ? A1[(size_t)v * F + k] : A2[(size_t)v * F + k - 64];
            if (maskY != nullptr && !(maskY[(size_t)v * F + k] > 0.f)) val = 0.f;
        }
        At[k * AT_LD + vv] = val;
    }
#pragma unroll 8
    for (int idx = tid; idx < 64 * K; idx += 256) {
        if (BWD) { const int k = idx >> 6, n = idx & 63; Bt[k * 64 + n] = W[(size_t)k * ldw + koff + n]; }
        else { const int n = idx / K, k = idx % K; Bt[k * 64 + n] = W[(size_t)n * ldw + k]; }
    }
    __syncthreads();
    const int ty = tid >> 4, tx = tid & 15;
    float acc[4][4] = {};
#pragma unroll 8
    for (int k = 0; k < K; ++k) {
        const float4 a = *reinterpret_cast<const float4*>(&At[k * AT_LD + ty * 4]);
        const float4 bb = *reinterpret_cast<const float4*>(&Bt[k * 64 + tx * 4]);
        const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int v = v0 + ty * 4 + i;
        if (v >= V) continue;
        float4* dst = reinterpret_cast<float4*>(&C[(size_t)v * F + tx * 4]);
        float4 o = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        if (accumulate) { const float4 c = *dst; o.x += c.x; o.y += c.y; o.z += c.z; o.w += c.w; }
        if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
        *dst = o;
    }
}

// dynamic shared memory of k_gemm<*, K>
constexpr int gemm_smem_bytes(int K) { return (K * AT_LD + K * 64) * 4; }

}  // namespace
}  // namespace eco
