// Kernel family 3: the DQN regression step's gradients, forward + backward of the MPNN for a replay minibatch.
//
// Replaces (reference, file:line)  src/agents/dqn/dqn.py:436-447
//     q_value = self.network(states).gather(1, actions);  loss = self.loss(q_value, td_target);  loss.backward()
// i.e. MPNN.forward (src/networks/mpnn.py:38-159) and its autograd backward for a minibatch of B episodes, with the loss
// F.mse_loss / F.smooth_l1_loss (dqn.py:113-121), reduction 'mean'.  Couplings in {-1,0,1} (every training generator of
// the reference, train_eco.py:100-111).  fp32 on the CUDA cores: the minibatch is 64 x 40 vertices (C5), the step is
// launch-bound, not throughput-bound.
//
// Layout: vertex-major planes [B * NP][64] fp32 in scratch.  Forward planes are kept for the backward pass:
//   H0..H3, P (= W_x x), RP = ReLU(P + w0), RM = ReLU(P - w0), G, E, AGG0..2, M0..2;   backward: dHa/dHb (ping-pong),
//   dE (summed over the layers), dM, dAGG, dG, dRP, dRM.
// Weight gradients are reduced in two fixed-order stages (per-split partial sums, then one sum over the splits), so a
// step is bit-reproducible.  The flat gradient has the 12 tensors in state_dict order (SURVEY.md appendix A.3).
#include <cmath>

#include "eco_common.cuh"
#include "mpnn_gemm.cuh"

namespace eco {
namespace {

constexpr int NSPLIT_MAX = 64;
constexpr int N_PARAMS = 58425;
constexpr int G_WINIT = 0, G_WEDGE = 448, G_WEF = 952, G_LAYER0 = 5048, G_LAYER_STRIDE = 16384, G_WUPD_OFF = 8192;
constexpr int G_WPOOL = 54200, G_WREAD = 58296, G_BREAD = 58424;
constexpr int PART_STRIDE = N_PARAMS + 1;           // + the loss

enum { P_H0 = 0, P_H1, P_H2, P_H3, P_P, P_RP, P_RM, P_G, P_E, P_AGG0, P_AGG1, P_AGG2, P_M0, P_M1, P_M2,
       P_DHA, P_DHB, P_DE, P_DM, P_DAGG, P_DG, P_DRP, P_DRM, N_PLANES };

__device__ __forceinline__ float dmax_of(const eco_graphs_t& g, int gi, float norm_max) {
    return norm_max > 0.f ? norm_max : (norm_max < 0.f ? (float)max(g.gstat[(size_t)gi * 4], 1) : *g.dmax);
}

// ---- per-vertex input stage (mpnn.py:55, 89-100): H0, P, RP, RM; padding vertices are zero -------------------------
__global__ void __launch_bounds__(256)
k_init_fwd(const eco_graphs_t g, const eco_mpnn_t w, const int B, const float* __restrict__ xn, const float* __restrict__ xg,
           float* __restrict__ H0, float* __restrict__ P, float* __restrict__ RP, float* __restrict__ RM) {
    const int NP = g.NP, N = g.N;
    const size_t idx = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (idx >= (size_t)B * NP * F) return;
    const int f = (int)(idx & 63);
    const size_t v = idx >> 6;
    const int b = (int)(v / NP), i = (int)(v % NP);
    float h = 0.f, p = 0.f, rp = 0.f, rm = 0.f;
    if (i < N) {
        const float X[7] = {xn[((size_t)b * 3 + 0) * NP + i], xn[((size_t)b * 3 + 1) * NP + i], xn[((size_t)b * 3 + 2) * NP + i],
                            xg[b * 4 + 0], xg[b * 4 + 1], xg[b * 4 + 2], xg[b * 4 + 3]};
#pragma unroll
        for (int c = 0; c < 7; ++c) h = fmaf(w.w_init[f * 7 + c], X[c], h);
        h = fmaxf(h, 0.f);
        if (f < 63) {
#pragma unroll
            for (int c = 0; c < 7; ++c) p = fmaf(w.w_edge[f * 8 + 1 + c], X[c], p);
            const float w0 = w.w_edge[f * 8];
            rp = fmaxf(p + w0, 0.f);
            rm = fmaxf(p - w0, 0.f);
        }
    }
    H0[idx] = h; P[idx] = p; RP[idx] = rp; RM[idx] = rm;
}

// ---- signed neighbour sums over the (symmetric) adjacency ----------------------------------------------------------
//   EDGE_FWD: O1[j] = 1/deg_j * sum_i ([a=+1] X1[i] + [a=-1] X2[i]);  feature 63 = deg_j / deg_max   (mpnn.py:96-102)
//   AGG_FWD:  O1[j] = 1/deg_j * sum_i a_ij X1[i]                                                     (mpnn.py:115)
//   AGG_BWD:  O1[j] += sum_i a_ij X1[i] / deg_i                       (transpose of AGG_FWD; A is symmetric)
//   EDGE_BWD: O1[j] = sum_i [a=+1] X1[i] / deg_i,  O2[j] = sum_i [a=-1] X1[i] / deg_i   (feature 63 carries no gradient)
enum { EDGE_FWD = 0, AGG_FWD = 1, AGG_BWD = 2, EDGE_BWD = 3 };
constexpr int ADJ_ROWS = 4;

template <int MODE>
__global__ void __launch_bounds__(ADJ_ROWS * F)
k_adj(const eco_graphs_t g, const int32_t* __restrict__ graph_idx, const float* __restrict__ X1, const float* __restrict__ X2,
      float* __restrict__ O1, float* __restrict__ O2, const float norm_max) {
    extern __shared__ __align__(16) unsigned char sm[];
    const int NP = g.NP, N = g.N;
    float* rdeg = reinterpret_cast<float*>(sm);                       // [NP]
    int8_t* rows = reinterpret_cast<int8_t*>(sm + (size_t)NP * 4);      // [ADJ_ROWS][NP]
    const int b = blockIdx.y, gi = graph_idx[b];
    const int jj = threadIdx.x >> 6, f = threadIdx.x & 63, j = blockIdx.x * ADJ_ROWS + jj;
    for (int i = threadIdx.x; i < NP; i += blockDim.x) rdeg[i] = i < N ? 1.f / g.deg[(size_t)gi * NP + i] : 0.f;
    for (int t = threadIdx.x; t < ADJ_ROWS * NP; t += blockDim.x) {
        const int r = blockIdx.x * ADJ_ROWS + t / NP;
        rows[t] = r < N ? g.J[((size_t)gi * NP + r) * NP + t % NP] : (int8_t)0;
    }
    __syncthreads();
    if (j >= NP) return;
    const size_t base = (size_t)b * NP * F;
    const int8_t* row = rows + jj * NP;
    float acc = 0.f, acc2 = 0.f;
    for (int i = 0; i < N; ++i) {
        const int a = row[i];
        if (a == 0) continue;
        const size_t o = base + (size_t)i * F + f;
        if (MODE == EDGE_FWD) acc += a > 0 ? X1[o] : X2[o];
        else if (MODE == AGG_FWD) acc = fmaf((float)a, X1[o], acc);
        else if (MODE == AGG_BWD) acc = fmaf((float)a * rdeg[i], X1[o], acc);
        else { if (a > 0) acc = fmaf(rdeg[i], X1[o], acc); else acc2 = fmaf(rdeg[i], X1[o], acc2); }
    }
    const size_t o = base + (size_t)j * F + f;
    const bool valid = j < N;
    if (MODE == EDGE_FWD) {
        const float d = valid ? g.deg[(size_t)gi * NP + j] : 1.f;
        O1[o] = valid ? (f == 63 ? d / dmax_of(g, gi, norm_max) : acc / d) : 0.f;
    } else if (MODE == AGG_FWD) {
        O1[o] = valid ? acc * rdeg[j] : 0.f;
    } else if (MODE == AGG_BWD) {
        if (valid) O1[o] += acc;
    } else {
        O1[o] = (valid && f < 63) ? acc : 0.f;
        O2[o] = (valid && f < 63) ? acc2 : 0.f;
    }
}

// ---- weight gradient partial sums: part[s][o * K + k] = sum_{v in split s} dZ[v][o] X[v][k],  X = [X1 | X2] ---------
__device__ __forceinline__ void split_range(int s, int S, int ntile, int& t0, int& t1) {
    t0 = (int)((long long)s * ntile / S);
    t1 = (int)((long long)(s + 1) * ntile / S);
}

template <int K>
__global__ void __launch_bounds__(256)
k_wgrad(const float* __restrict__ dY, const float* __restrict__ maskY, const float* __restrict__ X1,
        const float* __restrict__ X2, const int V, float* __restrict__ part) {
    extern __shared__ __align__(16) unsigned char sm[];
    float* dZs = reinterpret_cast<float*>(sm);                // [GT][64]
    float* Xs = dZs + GT * 64;                                // [GT][K]
    const int tid = threadIdx.x, s = blockIdx.x, S = gridDim.x;
    int t0, t1;
    split_range(s, S, (V + GT - 1) / GT, t0, t1);
    const int to = tid >> 4, tk = tid & 15;
    float acc[4][8] = {};
    for (int t = t0; t < t1; ++t) {
        const int v0 = t * GT;
#pragma unroll 8
        for (int idx = tid; idx < GT * 64; idx += 256) {
            const int v = v0 + (idx >> 6);
            float val = 0.f;
            if (v < V) { val = dY[(size_t)v * F + (idx & 63)]; if (!(maskY[(size_t)v * F + (idx & 63)] > 0.f)) val = 0.f; }
            dZs[idx] = val;
        }
#pragma unroll 8
        for (int idx = tid; idx < GT * K; idx += 256) {
            const int vv = idx / K, k = idx % K, v = v0 + vv;
            Xs[idx] = v < V ? (k < 64 ? X1[(size_t)v * F + k] : X2[(size_t)v * F + k - 64]) : 0.f;
        }
        __syncthreads();
#pragma unroll 4
        for (int vv = 0; vv < GT; ++vv) {
            const float4 a = *reinterpret_cast<const float4*>(&dZs[vv * 64 + to * 4]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Xs[vv * K + tk * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w};
            float bv[8] = {b0.x, b0.y, b0.z, b0.w, 0.f, 0.f, 0.f, 0.f};
            if (K == 128) {
                const float4 b1 = *reinterpret_cast<const float4*>(&Xs[vv * K + 64 + tk * 4]);
                bv[4] = b1.x; bv[5] = b1.y; bv[6] = b1.z; bv[7] = b1.w;
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
    float* out = part + (size_t)s * PART_STRIDE;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int o = to * 4 + i;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            out[o * K + tk * 4 + j] = acc[i][j];
            if (K == 128) out[o * K + 64 + tk * 4 + j] = acc[i][4 + j];
        }
    }
}

// ---- readout, loss and their gradients (mpnn.py:143-159; dqn.py:436-440) --------------------------------------------
// One block per split of the episodes.  Writes dH3 (all vertices), partial sums for W_p, w_r, b and the loss.
__global__ void __launch_bounds__(256)
k_readout(const eco_graphs_t g, const eco_mpnn_t w, const int B, const float* __restrict__ H3, const int32_t* __restrict__ actions,
          const float* __restrict__ targets, const int huber, float* __restrict__ dH3, float* __restrict__ part) {
    __shared__ float red[4][64], pooled[64], pv[64], dp[64], dpool[64], s_q[2];
    const int tid = threadIdx.x, NP = g.NP, N = g.N, S = gridDim.x, s = blockIdx.x;
    const int b0 = (int)((long long)s * B / S), b1 = (int)((long long)(s + 1) * B / S);
    const int f = tid & 63, grp = tid >> 6;
    float gWp[16] = {};                                  // W_p entries tid*16 .. tid*16+15: row tid/4, columns (tid%4)*16 + j
    float gwr = 0.f, gb = 0.f, loss = 0.f;               // w_r entry tid (tid < 128)
    for (int b = b0; b < b1; ++b) {
        const float* Hb = H3 + (size_t)b * NP * F;
        float sum = 0.f;
        for (int i = grp; i < N; i += 4) sum += Hb[(size_t)i * F + f];
        red[grp][f] = sum;
        __syncthreads();
        if (tid < 64) pooled[tid] = ((red[0][tid] + red[1][tid]) + (red[2][tid] + red[3][tid])) / (float)N;
        __syncthreads();
        if (tid < 64) {
            float p = 0.f;
            for (int k = 0; k < 64; ++k) p = fmaf(w.w_pool[tid * 64 + k], pooled[k], p);
            pv[tid] = p;
        }
        __syncthreads();
        const int a = actions[b];
        if (tid < 32) {                                  // Q[b, a]
            float c = fmaf(w.w_read[tid], fmaxf(pv[tid], 0.f), w.w_read[tid + 32] * fmaxf(pv[tid + 32], 0.f));
            c += fmaf(w.w_read[64 + tid], fmaxf(Hb[(size_t)a * F + tid], 0.f),
                      w.w_read[96 + tid] * fmaxf(Hb[(size_t)a * F + tid + 32], 0.f));
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
            if (tid == 0) {
                const float diff = c + w.b_read[0] - targets[b];
                float l, dl;
                if (huber) {                             // F.smooth_l1_loss, beta = 1
                    const float ad = fabsf(diff);
                    l = ad < 1.f ? 0.5f * diff * diff : ad - 0.5f;
                    dl = ad < 1.f ? diff : (diff > 0.f ? 1.f : -1.f);
                } else { l = diff * diff; dl = 2.f * diff; }
                s_q[0] = l / (float)B;
                s_q[1] = dl / (float)B;
            }
        }
        __syncthreads();
        const float dq = s_q[1];
        if (tid == 0) { loss += s_q[0]; gb += dq; }
        if (tid < 64) dp[tid] = pv[tid] > 0.f ? dq * w.w_read[tid] : 0.f;
        if (tid < 128) gwr += tid < 64 ? dq * fmaxf(pv[tid], 0.f) : dq * fmaxf(Hb[(size_t)a * F + tid - 64], 0.f);
        __syncthreads();
        {
            const float d = dp[tid >> 2];
#pragma unroll
            for (int j = 0; j < 16; ++j) gWp[j] = fmaf(d, pooled[(tid & 3) * 16 + j], gWp[j]);
        }
        if (tid < 64) {
            float t = 0.f;
            for (int k = 0; k < 64; ++k) t = fmaf(w.w_pool[k * 64 + tid], dp[k], t);
            dpool[tid] = t / (float)N;
        }
        __syncthreads();
        float* db = dH3 + (size_t)b * NP * F;
        for (int i = grp; i < NP; i += 4) {
            float v = 0.f;
            if (i < N) {
                v = dpool[f];
                if (i == a && Hb[(size_t)a * F + f] > 0.f) v += dq * w.w_read[64 + f];
            }
            db[(size_t)i * F + f] = v;
        }
        __syncthreads();
    }
    float* out = part + (size_t)s * PART_STRIDE;
#pragma unroll
    for (int j = 0; j < 16; ++j) out[G_WPOOL + tid * 16 + j] = gWp[j];
    if (tid < 128) out[G_WREAD + tid] = gwr;
    if (tid == 0) { out[G_BREAD] = gb; out[N_PARAMS] = loss; }
}

// ---- gradients of W_init and W_e from dH0, dRP, dRM (mpnn.py:55, 89-100) ---------------------------------------------
__global__ void __launch_bounds__(256)
k_init_bwd(const eco_graphs_t g, const eco_mpnn_t w, const int B, const float* __restrict__ xn, const float* __restrict__ xg,
           const float* __restrict__ H0, const float* __restrict__ P, const float* __restrict__ dH0,
           const float* __restrict__ dRP, const float* __restrict__ dRM, float* __restrict__ part) {
    __shared__ float red[4][64][15];
    const int tid = threadIdx.x, NP = g.NP, N = g.N, S = gridDim.x, s = blockIdx.x;
    const int V = B * NP;
    int t0, t1;
    split_range(s, S, (V + GT - 1) / GT, t0, t1);
    const int f = tid & 63, grp = tid >> 6;
    const float w0 = f < 63 ? w.w_edge[f * 8] : 0.f;
    float gi[7] = {}, ge[8] = {};
    const int vend = min(t1 * GT, V);
    for (int v = t0 * GT + grp; v < vend; v += 4) {
        const int b = v / NP, i = v % NP;
        if (i >= N) continue;
        const size_t o = (size_t)v * F + f;
        const float X[7] = {xn[((size_t)b * 3 + 0) * NP + i], xn[((size_t)b * 3 + 1) * NP + i], xn[((size_t)b * 3 + 2) * NP + i],
                            xg[b * 4 + 0], xg[b * 4 + 1], xg[b * 4 + 2], xg[b * 4 + 3]};
        const float dz0 = H0[o] > 0.f ? dH0[o] : 0.f;
        float dpp = 0.f, dpm = 0.f;
        if (f < 63) {
            const float p = P[o];
            dpp = p + w0 > 0.f ? dRP[o] : 0.f;
            dpm = p - w0 > 0.f ? dRM[o] : 0.f;
        }
        const float dpv = dpp + dpm;
        ge[0] += dpp - dpm;
#pragma unroll
        for (int c = 0; c < 7; ++c) {
            gi[c] = fmaf(dz0, X[c], gi[c]);
            ge[1 + c] = fmaf(dpv, X[c], ge[1 + c]);
        }
    }
#pragma unroll
    for (int c = 0; c < 7; ++c) red[grp][f][c] = gi[c];
#pragma unroll
    for (int c = 0; c < 8; ++c) red[grp][f][7 + c] = ge[c];
    __syncthreads();
    float* out = part + (size_t)s * PART_STRIDE;
    for (int idx = tid; idx < 64 * 15; idx += 256) {
        const int ff = idx / 15, c = idx % 15;
        const float t = (red[0][ff][c] + red[1][ff][c]) + (red[2][ff][c] + red[3][ff][c]);
        if (c < 7) out[G_WINIT + ff * 7 + c] = t;
        else if (ff < 63) out[G_WEDGE + ff * 8 + c - 7] = t;
    }
}

// ---- second stage: sum over the splits in order -------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_reduce(const float* __restrict__ part, const int S, float* __restrict__ grad, float* __restrict__ loss) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i > N_PARAMS) return;
    float t = 0.f;
    for (int s = 0; s < S; ++s) t += part[(size_t)s * PART_STRIDE + i];
    if (i < N_PARAMS) grad[i] = t;
    else *loss = t;
}

// ---- Adam (torch.optim.Adam semantics: L2 weight decay added to the gradient, bias correction; dqn.py:212, 449) -----
struct AdamTable { float* p[12]; int off[13]; };

__global__ void __launch_bounds__(256)
k_adam(const AdamTable t, const float* __restrict__ grad, float* __restrict__ m, float* __restrict__ v, const float step_size,
       const float bc2_sqrt, const float beta1, const float beta2, const float eps, const float weight_decay) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= N_PARAMS) return;
    int k = 0;
#pragma unroll
    for (int j = 1; j < 12; ++j) k += i >= t.off[j];
    float* p = t.p[k] + (i - t.off[k]);
    const float w = *p;
    const float g = fmaf(weight_decay, w, grad[i]);
    const float mi = fmaf(beta1, m[i], (1.f - beta1) * g);            // exp_avg.lerp_(grad, 1 - beta1)
    const float vi = fmaf(beta2, v[i], (1.f - beta2) * g * g);        // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    *p = w - step_size * (mi / denom);
}

int n_splits(int B, int NP) {
    const int ntile = (B * NP + GT - 1) / GT;
    int S = ntile < NSPLIT_MAX ? ntile : NSPLIT_MAX;
    if (S > B) S = B;                 // the readout splits episodes
    return S < 1 ? 1 : S;
}

}  // namespace

size_t mpnn_grad_scratch_bytes(int B, int N) {
    const int NP = padded_n(N);
    return align256(sizeof(float) * ((size_t)N_PLANES * B * NP * F + (size_t)NSPLIT_MAX * PART_STRIDE));
}

// second stream + events of launch_mpnn_grad, one set per device of the process (created on first use, never destroyed)
struct SideStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
};
static SideStream& side_stream() {
    static SideStream per_dev[64];
    int dev = 0;
    cudaGetDevice(&dev);
    SideStream& s = per_dev[dev & 63];
    if (!s.stream) {
        cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking);
        for (auto& e : s.ev) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    }
    return s;
}

int launch_mpnn_grad(const eco_graphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn, const float* xg,
                     float norm_max, const int32_t* actions, const float* targets, int huber, float* loss, float* grad,
                     void* scratch, cudaEvent_t targets_ready, cudaStream_t st) {
    const int NP = g->NP, V = B * NP;
    const size_t pl = (size_t)V * F;
    float* base = (float*)scratch;
    auto P = [&](int k) { return base + (size_t)k * pl; };
    float* part = base + (size_t)N_PLANES * pl;
    const int S = n_splits(B, NP);
    const int gsm128 = (128 * AT_LD + 128 * 64) * 4, gsm64 = (64 * AT_LD + 64 * 64) * 4;
    const int wsm128 = (GT * 64 + GT * 128) * 4, wsm64 = (GT * 64 + GT * 64) * 4;
    static unsigned long long attr = 0;
    if (first_use_on_device(&attr)) {
        ECO_CUDA(cudaFuncSetAttribute(k_gemm<false, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, gsm128));
        ECO_CUDA(cudaFuncSetAttribute(k_wgrad<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, wsm128));
    }
    const int vt = (V + GT - 1) / GT;
    const dim3 agrid((NP + ADJ_ROWS - 1) / ADJ_ROWS, B);
    const int asm_bytes = NP * 4 + ADJ_ROWS * NP;
    const unsigned eblocks = (unsigned)((pl + 255) / 256);
    // the splits that a producer does not write must read as zero in k_reduce
    ECO_CUDA(cudaMemsetAsync(part, 0, sizeof(float) * (size_t)S * PART_STRIDE, st));

    // ---- forward ----
    k_init_fwd<<<eblocks, 256, 0, st>>>(*g, *w, B, xn, xg, P(P_H0), P(P_P), P(P_RP), P(P_RM));
    ECO_LAUNCH_CHECK();
    k_adj<EDGE_FWD><<<agrid, ADJ_ROWS * F, asm_bytes, st>>>(*g, gidx, P(P_RP), P(P_RM), P(P_G), nullptr, norm_max);
    ECO_LAUNCH_CHECK();
    k_gemm<false, 64><<<vt, 256, gsm64, st>>>(P(P_G), nullptr, nullptr, V, w->w_edge_feat, 64, 0, P(P_E), 1, 0);
    ECO_LAUNCH_CHECK();
    for (int l = 0; l < 3; ++l) {
        k_adj<AGG_FWD><<<agrid, ADJ_ROWS * F, asm_bytes, st>>>(*g, gidx, P(P_H0 + l), nullptr, P(P_AGG0 + l), nullptr, norm_max);
        ECO_LAUNCH_CHECK();
        k_gemm<false, 128><<<vt, 256, gsm128, st>>>(P(P_AGG0 + l), P(P_E), nullptr, V, w->w_msg[l], 128, 0, P(P_M0 + l), 1, 0);
        ECO_LAUNCH_CHECK();
        k_gemm<false, 128><<<vt, 256, gsm128, st>>>(P(P_H0 + l), P(P_M0 + l), nullptr, V, w->w_upd[l], 128, 0, P(P_H1 + l), 1, 0);
        ECO_LAUNCH_CHECK();
    }
    // ---- loss and backward ----
    // (the regression targets may still be on their way on another stream: the forward above does not need them)
    if (targets_ready) ECO_CUDA(cudaStreamWaitEvent(st, targets_ready, 0));
    k_readout<<<S, 256, 0, st>>>(*g, *w, B, P(P_H3), actions, targets, huber, P(P_DHA), part);
    ECO_LAUNCH_CHECK();
    // The weight-gradient kernels only READ the activation gradients; nothing downstream of them but the final reduction needs
    // their sums.  They run on a second stream beside the chain that carries the gradient back through the layers; what the
    // chain has to respect is that a buffer a weight gradient still reads (dcur, DM of the layer above) is not overwritten
    // yet: one event per layer.  (Inside a captured update these are parallel branches of the graph.)
    SideStream& ss = side_stream();
    cudaStream_t sw = ss.stream;
    auto after_main = [&](int k) { ECO_CUDA(cudaEventRecord(ss.ev[k], st)); ECO_CUDA(cudaStreamWaitEvent(sw, ss.ev[k], 0)); return ECO_OK; };
    float* dcur = P(P_DHA);
    float* dnext = P(P_DHB);
    for (int l = 2; l >= 0; --l) {
        float* gl = part + G_LAYER0 + l * G_LAYER_STRIDE;
        const float* Hout = P(P_H1 + l);
        if (int rc = after_main(0)) return rc;                                 // dcur of this layer is complete
        k_wgrad<128><<<S, 256, wsm128, sw>>>(dcur, Hout, P(P_H0 + l), P(P_M0 + l), V, gl + G_WUPD_OFF);
        ECO_LAUNCH_CHECK();
        if (l < 2) ECO_CUDA(cudaStreamWaitEvent(st, ss.ev[2], 0));             // the layer above no longer reads dnext / DM
        k_gemm<true, 64><<<vt, 256, gsm64, st>>>(dcur, nullptr, Hout, V, w->w_upd[l], 128, 0, dnext, 0, 0);
        ECO_LAUNCH_CHECK();
        k_gemm<true, 64><<<vt, 256, gsm64, st>>>(dcur, nullptr, Hout, V, w->w_upd[l], 128, 64, P(P_DM), 0, 0);
        ECO_LAUNCH_CHECK();
        if (int rc = after_main(1)) return rc;                                 // DM is complete
        k_wgrad<128><<<S, 256, wsm128, sw>>>(P(P_DM), P(P_M0 + l), P(P_AGG0 + l), P(P_E), V, gl);
        ECO_LAUNCH_CHECK();
        ECO_CUDA(cudaEventRecord(ss.ev[2], sw));                               // both weight gradients of this layer have read their inputs
        k_gemm<true, 64><<<vt, 256, gsm64, st>>>(P(P_DM), nullptr, P(P_M0 + l), V, w->w_msg[l], 128, 0, P(P_DAGG), 0, 0);
        ECO_LAUNCH_CHECK();
        k_gemm<true, 64><<<vt, 256, gsm64, st>>>(P(P_DM), nullptr, P(P_M0 + l), V, w->w_msg[l], 128, 64, P(P_DE), 0, l < 2 ? 1 : 0);
        ECO_LAUNCH_CHECK();
        k_adj<AGG_BWD><<<agrid, ADJ_ROWS * F, asm_bytes, st>>>(*g, gidx, P(P_DAGG), nullptr, dnext, nullptr, norm_max);
        ECO_LAUNCH_CHECK();
        float* t = dcur; dcur = dnext; dnext = t;
    }
    if (int rc = after_main(0)) return rc;                                     // DE is complete
    k_wgrad<64><<<S, 256, wsm64, sw>>>(P(P_DE), P(P_E), P(P_G), nullptr, V, part + G_WEF);
    ECO_LAUNCH_CHECK();
    ECO_CUDA(cudaEventRecord(ss.ev[3], sw));
    k_gemm<true, 64><<<vt, 256, gsm64, st>>>(P(P_DE), nullptr, P(P_E), V, w->w_edge_feat, 64, 0, P(P_DG), 0, 0);
    ECO_LAUNCH_CHECK();
    k_adj<EDGE_BWD><<<agrid, ADJ_ROWS * F, asm_bytes, st>>>(*g, gidx, P(P_DG), nullptr, P(P_DRP), P(P_DRM), norm_max);
    ECO_LAUNCH_CHECK();
    k_init_bwd<<<S, 256, 0, st>>>(*g, *w, B, xn, xg, P(P_H0), P(P_P), dcur, P(P_DRP), P(P_DRM), part);
    ECO_LAUNCH_CHECK();
    ECO_CUDA(cudaStreamWaitEvent(st, ss.ev[3], 0));                            // every weight-gradient partial sum is written
    k_reduce<<<(N_PARAMS + 1 + 255) / 256, 256, 0, st>>>(part, S, grad, loss);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

int launch_mpnn_adam(const eco_mpnn_t* w, const float* grad, float* m, float* v, int step, float lr, float beta1, float beta2,
                     float eps, float weight_decay, cudaStream_t st) {
    static const int counts[12] = {64 * 7, 63 * 8, 64 * 64, 64 * 128, 64 * 128, 64 * 128, 64 * 128, 64 * 128, 64 * 128, 64 * 64, 128, 1};
    AdamTable t;
    float* ptrs[12] = {(float*)w->w_init, (float*)w->w_edge, (float*)w->w_edge_feat, (float*)w->w_msg[0], (float*)w->w_upd[0],
                       (float*)w->w_msg[1], (float*)w->w_upd[1], (float*)w->w_msg[2], (float*)w->w_upd[2], (float*)w->w_pool,
                       (float*)w->w_read, (float*)w->b_read};
    int off = 0;
    for (int k = 0; k < 12; ++k) { t.p[k] = ptrs[k]; t.off[k] = off; off += counts[k]; }
    t.off[12] = off;
    const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
    k_adam<<<(N_PARAMS + 255) / 256, 256, 0, st>>>(t, grad, m, v, (float)((double)lr / bc1), (float)sqrt(bc2), beta1, beta2, eps,
                                                   weight_decay);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

}  // namespace eco
