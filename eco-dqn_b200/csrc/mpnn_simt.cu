// Kernel family 2a: MPNN Q-network forward + argmax on CUDA cores (fp32).  General path: any int8
// couplings, any N <= ECO_MAX_SPINS, and the fp32 couplings of weighted graph sets (eco_wgraphs_t.Jf: the same kernel
// instantiated on float rows).  Also the on-device cross-check for the tcgen05 kernel (mpnn_tc.cu).
//
// Replaces (reference, file:line)
//   src/networks/mpnn.py:40-77    MPNN.forward
//   src/networks/mpnn.py:89-104   EdgeAndNodeEmbeddingLayer.forward -- without the [B,N,N,8]/[B,N,N,63]
//                                 intermediates: no bias + the adj!=0 mask give
//                                 ReLU(W_e [a_ij ; x_j]) = ReLU(a_ij w0 + P_j),  P = X W_x^T  (SURVEY.md section 7)
//   src/networks/mpnn.py:114-120  UpdateNodeEmbeddingLayer.forward (x3, untied)
//   src/networks/mpnn.py:143-159  ReadoutLayer.forward
//   experiments/utils.py:57-66    argmax action selection (first maximal index)
//
// One persistent CTA (8 warps) walks over episodes.  Per episode the node embeddings live in a per-CTA
// global scratch (L2 resident); neighbour aggregation scans the adjacency row 16 entries per lane (one 16-byte load
// for int8, four float4 loads for fp32) and visits only non-zeros; the 64x64 / 64x128 linears run on 8-vertex tiles per warp (16 accumulators per lane,
// weights transposed in shared memory, inputs broadcast from shared memory).
#include "eco_common.cuh"

namespace eco {

namespace {

constexpr int F = 64;
constexpr int WARPS = 8;
constexpr int TILE = 8;     // vertices per warp tile
// transposed weights staged in the scratch header (floats)
constexpr int OFF_WEF = 0;                    // [64][64]   k-major: WefT[k][f] = w_edge_feat[f][k]
constexpr int OFF_WMSG = OFF_WEF + 64 * 64;   // [3][128][64]
constexpr int OFF_WUPD = OFF_WMSG + 3 * 128 * 64;
constexpr int WT_FLOATS = OFF_WUPD + 3 * 128 * 64;

__global__ void transpose_weights_kernel(const eco_mpnn_t w, float* __restrict__ wt) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < 64 * 64) {
        const int k = idx / 64, f = idx % 64;
        wt[OFF_WEF + idx] = w.w_edge_feat[f * 64 + k];
    }
    if (idx < 128 * 64) {
        const int k = idx / 64, f = idx % 64;
        for (int l = 0; l < 3; ++l) {
            wt[OFF_WMSG + l * 128 * 64 + idx] = w.w_msg[l][f * 128 + k];
            wt[OFF_WUPD + l * 128 * 64 + idx] = w.w_upd[l][f * 128 + k];
        }
    }
}

// The graph as the kernel reads it: int8 couplings (eco_graphs_t) or fp32 ones (eco_wgraphs_t.Jf).  V is the type a
// coupling is handled in (int for int8, so the integer instantiation is the original kernel).
template <class T>
struct GView {
    const T* J;
    const float* deg;
    const int32_t* gstat;
    const float* dmax;
    int N, NP;
};
template <class T> struct CouplingVal { using type = int; };
template <> struct CouplingVal<float> { using type = float; };

// K consecutive couplings of a row, widened to V: 16 / 8 int8 (one 16- / 8-byte load) or 4 fp32 (one float4 -- wider
// chunks of fp32 rows push the kernel over its 128-register budget)
__device__ __forceinline__ void load_row(const int8_t* p, int (&v)[16]) {
    union { uint4 q; int8_t b[16]; } u;
    u.q = *reinterpret_cast<const uint4*>(p);
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = u.b[k];
}
__device__ __forceinline__ void load_row(const int8_t* p, int (&v)[8]) {
    union { uint2 q; int8_t b[8]; } u;
    u.q = *reinterpret_cast<const uint2*>(p);
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = u.b[k];
}
__device__ __forceinline__ void load_row(const float* p, float (&v)[4]) {
    const float4 f = *reinterpret_cast<const float4*>(p);
    v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
}

template <class T>
struct Smem {
    float wa[128 * F];            // current message / edge-feature weights, transposed [k][f]
    float wb[128 * F];            // current update weights
    float xs[WARPS][128 * TILE];  // per-warp input tile [k][vertex]
    uint16_t nbr_j[WARPS][256];   // per-warp compacted neighbour list of one 256-entry window: vertex ...
    T nbr_a[WARPS][256];          // ... and weight
    float w_init[64 * 7];
    float w_edge[64 * 8];
    float w_read[128];
    float pooled[F];
    float part[WARPS][F];
    float red_val[WARPS];
    int red_idx[WARPS];
    float c0;
};

// acc[0..7] (feature `lane`) and acc[8..15] (feature lane+32) for the 8 vertices of the warp's tile
__device__ __forceinline__ void tile_linear(const float* __restrict__ wt, const float* __restrict__ xs, int K,
                                            int lane, float (&acc)[16]) {
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
        const float w0 = wt[k * F + lane], w1 = wt[k * F + lane + 32];
        const float4 xa = *reinterpret_cast<const float4*>(xs + k * TILE);
        const float4 xb = *reinterpret_cast<const float4*>(xs + k * TILE + 4);
        acc[0] = fmaf(w0, xa.x, acc[0]); acc[1] = fmaf(w0, xa.y, acc[1]);
        acc[2] = fmaf(w0, xa.z, acc[2]); acc[3] = fmaf(w0, xa.w, acc[3]);
        acc[4] = fmaf(w0, xb.x, acc[4]); acc[5] = fmaf(w0, xb.y, acc[5]);
        acc[6] = fmaf(w0, xb.z, acc[6]); acc[7] = fmaf(w0, xb.w, acc[7]);
        acc[8] = fmaf(w1, xa.x, acc[8]); acc[9] = fmaf(w1, xa.y, acc[9]);
        acc[10] = fmaf(w1, xa.z, acc[10]); acc[11] = fmaf(w1, xa.w, acc[11]);
        acc[12] = fmaf(w1, xb.x, acc[12]); acc[13] = fmaf(w1, xb.y, acc[13]);
        acc[14] = fmaf(w1, xb.z, acc[14]); acc[15] = fmaf(w1, xb.w, acc[15]);
    }
}

// Visit the non-zeros of adjacency row `arow` (NP couplings) with the whole warp; fn(j, a) is warp-uniform.
template <class T, class Fn>
__device__ __forceinline__ void for_each_neighbor(const T* __restrict__ arow, int NP, int lane, Fn fn) {
    using V = typename CouplingVal<T>::type;
    constexpr int K = sizeof(T) == 1 ? 16 : 4;          // couplings per lane and chunk
    const int nchunks = NP / K;
    for (int base = 0; base < nchunks; base += 32) {
        V u[K];
#pragma unroll
        for (int k = 0; k < K; ++k) u[k] = 0;
        if (base + lane < nchunks) load_row(arow + (size_t)(base + lane) * K, u);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const V v = u[k];
            unsigned m = __ballot_sync(0xffffffffu, v != 0);
            while (m) {
                const int src = __ffs(m) - 1;
                m &= m - 1;
                const V a = __shfl_sync(0xffffffffu, v, src);
                fn((base + src) * K + k, a);
            }
        }
    }
}

// The same visit with memory-level parallelism: the non-zeros of a 256-entry window of the row are first compacted into
// a per-warp list (ballot + popc), then handed out eight at a time, so the caller issues eight independent gathers from
// the L2-resident embeddings before it uses any of them (one dependent L2 round trip per neighbour made the aggregation
// 90 % of the kernel on ER-500).  fn(j[8], a[8], cnt): entries >= cnt are (0, 0).
template <class T, class Fn>
__device__ __forceinline__ void for_each_neighbor8(const T* __restrict__ arow, int NP, int lane, uint16_t* lj, T* la, Fn fn) {
    using V = typename CouplingVal<T>::type;
    constexpr int K = sizeof(T) == 1 ? 8 : 4;           // couplings per lane and chunk: a window of 32 x K <= 256 entries
    const int nchunks = NP / K;
    for (int base = 0; base < nchunks; base += 32) {
        V u[K];
#pragma unroll
        for (int k = 0; k < K; ++k) u[k] = 0;
        if (base + lane < nchunks) load_row(arow + (size_t)(base + lane) * K, u);
        int count = 0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const V v = u[k];
            const unsigned m = __ballot_sync(0xffffffffu, v != 0);
            if (v != 0) {
                const int pos = count + __popc(m & ((1u << lane) - 1u));
                lj[pos] = (uint16_t)((base + lane) * K + k);
                la[pos] = (T)v;
            }
            count += __popc(m);
        }
        __syncwarp();
        for (int t = 0; t < count; t += 8) {
            int j[8];
            V a[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const bool in = t + e < count;
                j[e] = in ? (int)lj[t + e] : 0;
                a[e] = in ? (V)la[t + e] : (V)0;
            }
            fn(j, a, min(8, count - t));
        }
        __syncwarp();
    }
}

// (fp32 couplings: sizeof(Smem<float>) = 115 KB, so one CTA per SM fits anyway and the register budget is not halved)
template <class T>
__global__ void __launch_bounds__(WARPS * 32, sizeof(T) == 1 ? 2 : 1)
mpnn_simt_kernel(const GView<T> g, const eco_mpnn_t w, const int B, const int32_t* __restrict__ graph_idx,
                 const float* __restrict__ xn, const float* __restrict__ xg, const float norm_max,
                 float* __restrict__ q_out, int32_t* __restrict__ act_out, float* __restrict__ scratch) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using V = typename CouplingVal<T>::type;
    Smem<T>& S = *reinterpret_cast<Smem<T>*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = g.N, NP = g.NP;
    const float* wt = scratch;                                        // transposed weights (header)
    float* cta = scratch + WT_FLOATS + (size_t)blockIdx.x * 4 * NP * F;
    float* H0 = cta;                 // [NP][64] ping
    float* H1 = cta + (size_t)NP * F;     // pong
    float* E = cta + (size_t)2 * NP * F;  // edge embeddings
    float* P = cta + (size_t)3 * NP * F;  // X W_x^T (63 used)
    float* xs = S.xs[warp];
    const float dmax_set = norm_max > 0.f ? norm_max : *g.dmax;
    const int ntiles = (N + TILE - 1) / TILE;
    const bool batched = NP > 256;     // large graphs: eight neighbour gathers in flight (small rows: the serial visit is cheaper)

    for (int i = tid; i < 64 * 7; i += blockDim.x) S.w_init[i] = w.w_init[i];
    for (int i = tid; i < 64 * 8; i += blockDim.x) S.w_edge[i] = i < 63 * 8 ? w.w_edge[i] : 0.f;
    for (int i = tid; i < 128; i += blockDim.x) S.w_read[i] = w.w_read[i];

    for (int b = blockIdx.x; b < B; b += gridDim.x) {
        const int gi = graph_idx[b];
        const T* A = g.J + (size_t)gi * NP * NP;
        const float* deg = g.deg + (size_t)gi * NP;
        const float* x0 = xn + (size_t)b * 3 * NP;
        const float4 xgl = *reinterpret_cast<const float4*>(xg + (size_t)b * 4);
        const float dmax = norm_max < 0.f ? (float)max(g.gstat[(size_t)gi * 4], 1) : dmax_set;

        // edge-feature weights for phase 1
        for (int i = tid; i < 64 * F; i += blockDim.x) S.wa[i] = wt[OFF_WEF + i];
        __syncthreads();

        // ---- phase 0: h0 = ReLU(W_init x), P = W_x x --------------------------------- mpnn.py:55, :90-97
        for (int i = warp; i < N; i += WARPS) {
            const float X[7] = {x0[i], x0[NP + i], x0[2 * NP + i], xgl.x, xgl.y, xgl.z, xgl.w};
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int f = lane + 32 * half;
                float h = 0.f, p = 0.f;
#pragma unroll
                for (int c = 0; c < 7; ++c) {
                    h = fmaf(S.w_init[f * 7 + c], X[c], h);
                    p = fmaf(S.w_edge[f * 8 + 1 + c], X[c], p);
                }
                H0[(size_t)i * F + f] = fmaxf(h, 0.f);
                P[(size_t)i * F + f] = p;
            }
        }
        __syncthreads();

        // ---- phase 1: edge embeddings -------------------------------------------------- mpnn.py:89-104
        const float w0a = S.w_edge[lane * 8], w0b = S.w_edge[(lane + 32) * 8];   // column 0 multiplies a_ij
        for (int t = warp; t < ntiles; t += WARPS) {
            for (int n = 0; n < TILE; ++n) {
                const int i = t * TILE + n;
                float ga = 0.f, gb = 0.f;
                if (i < N) {
                    if (!batched) {
                        for_each_neighbor(A + (size_t)i * NP, NP, lane, [&](int j, V a) {
                            const float af = (float)a;
                            ga += fmaxf(fmaf(af, w0a, P[(size_t)j * F + lane]), 0.f);
                            gb += fmaxf(fmaf(af, w0b, P[(size_t)j * F + lane + 32]), 0.f);
                        });
                    } else
                    for_each_neighbor8(A + (size_t)i * NP, NP, lane, S.nbr_j[warp], S.nbr_a[warp], [&](const int (&j)[8], const V (&a)[8], int cnt) {
                        float pa[8], pb[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) { pa[e] = P[(size_t)j[e] * F + lane]; pb[e] = P[(size_t)j[e] * F + lane + 32]; }
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            if (e < cnt) {
                                const float af = (float)a[e];
                                ga += fmaxf(fmaf(af, w0a, pa[e]), 0.f);
                                gb += fmaxf(fmaf(af, w0b, pb[e]), 0.f);
                            }
                        }
                    });
                    const float d = deg[i];
                    ga = ga / d;
                    gb = lane == 31 ? d / dmax : gb / d;   // feature 63 = norm / norm.max()  (mpnn.py:102)
                }
                xs[lane * TILE + n] = ga;
                xs[(lane + 32) * TILE + n] = gb;
            }
            __syncwarp();
            float acc[16];
            tile_linear(S.wa, xs, 64, lane, acc);
            __syncwarp();
            for (int n = 0; n < TILE; ++n) {
                const int i = t * TILE + n;
                if (i < N) {
                    E[(size_t)i * F + lane] = fmaxf(acc[n], 0.f);
                    E[(size_t)i * F + lane + 32] = fmaxf(acc[8 + n], 0.f);
                }
            }
        }

        // ---- phase 2: three message-passing layers -------------------------------------- mpnn.py:114-120
        float* Hc = H0;
        float* Hn = H1;
        for (int l = 0; l < 3; ++l) {
            __syncthreads();   // previous layer's Hn complete; wa/wb free
            for (int i = tid; i < 128 * F; i += blockDim.x) {
                S.wa[i] = wt[OFF_WMSG + l * 128 * F + i];
                S.wb[i] = wt[OFF_WUPD + l * 128 * F + i];
            }
            __syncthreads();
            for (int t = warp; t < ntiles; t += WARPS) {
                for (int n = 0; n < TILE; ++n) {
                    const int i = t * TILE + n;
                    float aa = 0.f, ab = 0.f, ea = 0.f, eb = 0.f;
                    if (i < N) {
                        if (!batched) {
                            for_each_neighbor(A + (size_t)i * NP, NP, lane, [&](int j, V a) {
                                const float af = (float)a;
                                aa = fmaf(af, Hc[(size_t)j * F + lane], aa);
                                ab = fmaf(af, Hc[(size_t)j * F + lane + 32], ab);
                            });
                        } else
                        for_each_neighbor8(A + (size_t)i * NP, NP, lane, S.nbr_j[warp], S.nbr_a[warp], [&](const int (&j)[8], const V (&a)[8], int cnt) {
                            float ha[8], hb[8];
#pragma unroll
                            for (int e = 0; e < 8; ++e) { ha[e] = Hc[(size_t)j[e] * F + lane]; hb[e] = Hc[(size_t)j[e] * F + lane + 32]; }
#pragma unroll
                            for (int e = 0; e < 8; ++e) {           // (padding entries have a = 0; same order as the serial visit)
                                if (e < cnt) {
                                    const float af = (float)a[e];
                                    aa = fmaf(af, ha[e], aa);
                                    ab = fmaf(af, hb[e], ab);
                                }
                            }
                        });
                        const float d = deg[i];
                        aa = aa / d;
                        ab = ab / d;
                        ea = E[(size_t)i * F + lane];
                        eb = E[(size_t)i * F + lane + 32];
                    }
                    xs[lane * TILE + n] = aa;
                    xs[(lane + 32) * TILE + n] = ab;
                    xs[(64 + lane) * TILE + n] = ea;
                    xs[(96 + lane) * TILE + n] = eb;
                }
                __syncwarp();
                float acc[16];
                tile_linear(S.wa, xs, 128, lane, acc);          // message = ReLU(W_m [agg ; e])
                __syncwarp();
                for (int n = 0; n < TILE; ++n) {
                    const int i = t * TILE + n;
                    const bool ok = i < N;
                    xs[lane * TILE + n] = ok ? Hc[(size_t)i * F + lane] : 0.f;
                    xs[(lane + 32) * TILE + n] = ok ? Hc[(size_t)i * F + lane + 32] : 0.f;
                    xs[(64 + lane) * TILE + n] = fmaxf(acc[n], 0.f);
                    xs[(96 + lane) * TILE + n] = fmaxf(acc[8 + n], 0.f);
                }
                __syncwarp();
                tile_linear(S.wb, xs, 128, lane, acc);          // h' = ReLU(W_u [h ; message])
                __syncwarp();
                for (int n = 0; n < TILE; ++n) {
                    const int i = t * TILE + n;
                    if (i < N) {
                        Hn[(size_t)i * F + lane] = fmaxf(acc[n], 0.f);
                        Hn[(size_t)i * F + lane + 32] = fmaxf(acc[8 + n], 0.f);
                    }
                }
            }
            float* tmp = Hc; Hc = Hn; Hn = tmp;
        }
        __syncthreads();

        // ---- phase 3: readout + argmax --------------------------------------------------- mpnn.py:143-159
        {
            float sa = 0.f, sb = 0.f;
            for (int i = warp; i < N; i += WARPS) {
                sa += Hc[(size_t)i * F + lane];
                sb += Hc[(size_t)i * F + lane + 32];
            }
            S.part[warp][lane] = sa;
            S.part[warp][lane + 32] = sb;
        }
        __syncthreads();
        if (tid < F) {
            float s = 0.f;
            for (int ww = 0; ww < WARPS; ++ww) s += S.part[ww][tid];
            S.pooled[tid] = s / (float)N;
        }
        __syncthreads();
        if (warp == 0) {
            float c = 0.f;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int f = lane + 32 * half;
                float p = 0.f;
                for (int k = 0; k < F; ++k) p = fmaf(w.w_pool[f * F + k], S.pooled[k], p);
                c = fmaf(S.w_read[f], fmaxf(p, 0.f), c);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
            if (lane == 0) S.c0 = c + w.b_read[0];
        }
        __syncthreads();
        float best_v = -INFINITY;
        int best_i = 0x7fffffff;
        for (int i = warp; i < N; i += WARPS) {
            float v = fmaf(S.w_read[64 + lane], fmaxf(Hc[(size_t)i * F + lane], 0.f),
                           S.w_read[96 + lane] * fmaxf(Hc[(size_t)i * F + lane + 32], 0.f));
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            v += S.c0;
            if (lane == 0 && q_out) q_out[(size_t)b * NP + i] = v;
            if (v > best_v) { best_v = v; best_i = i; }   // ascending i => first maximum kept
        }
        if (lane == 0) { S.red_val[warp] = best_v; S.red_idx[warp] = best_i; }
        __syncthreads();
        if (tid == 0 && act_out) {
            float bv = S.red_val[0];
            int bi = S.red_idx[0];
            for (int ww = 1; ww < WARPS; ++ww)
                if (S.red_val[ww] > bv || (S.red_val[ww] == bv && S.red_idx[ww] < bi)) {
                    bv = S.red_val[ww];
                    bi = S.red_idx[ww];
                }
            act_out[b] = bi;
        }
        __syncthreads();
    }
}

int simt_grid(int B) {
    const int max_ctas = 148 * 2;
    return B < max_ctas ? B : max_ctas;
}

}  // namespace

size_t mpnn_simt_scratch_bytes(int B, int N) {
    const int NP = padded_n(N);
    return align256(sizeof(float) * ((size_t)WT_FLOATS + (size_t)simt_grid(B) * 4 * NP * F));
}

namespace {
template <class T>
int launch_simt(const GView<T>& g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn, const float* xg,
                float norm_max, float* q, int32_t* actions, void* scratch, cudaStream_t st) {
    static unsigned long long attr_set = 0;     // (one per instantiation)
    if (first_use_on_device(&attr_set))
        ECO_CUDA(cudaFuncSetAttribute(mpnn_simt_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)sizeof(Smem<T>)));
    transpose_weights_kernel<<<(128 * 64 + 255) / 256, 256, 0, st>>>(*w, (float*)scratch);
    ECO_LAUNCH_CHECK();
    prof_begin(ECO_PROF_MPNN, st);
    mpnn_simt_kernel<T><<<simt_grid(B), WARPS * 32, sizeof(Smem<T>), st>>>(g, *w, B, gidx, xn, xg, norm_max, q,
                                                                          actions, (float*)scratch);
    prof_end(ECO_PROF_MPNN, st);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}
}  // namespace

int launch_mpnn_simt(const eco_graphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn,
                     const float* xg, float norm_max, float* q, int32_t* actions, void* scratch,
                     cudaStream_t st) {
    const GView<int8_t> v{g->J, g->deg, g->gstat, g->dmax, g->N, g->NP};
    return launch_simt(v, w, B, gidx, xn, xg, norm_max, q, actions, scratch, st);
}

int launch_mpnn_simt_w(const eco_wgraphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn,
                       const float* xg, float norm_max, float* q, int32_t* actions, void* scratch, cudaStream_t st) {
    const GView<float> v{g->Jf, g->deg, g->gstat, g->dmax, g->N, g->NP};
    return launch_simt(v, w, B, gidx, xn, xg, norm_max, q, actions, scratch, st);
}

}  // namespace eco
