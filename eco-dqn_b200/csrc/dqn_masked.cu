// The masked half of the DQN step for irreversible spins (S2V-DQN): the agent may only flip a spin that is still at -1.
//
// Replaces (reference, file:line) src/agents/dqn/dqn.py:416-428 (TD target with the flipped spins of s' masked out),
// :453-465 (epsilon-greedy acting; irreversible spins draw among the spins still at -1) and :504-512 (masked predict).
//
//   eco_dqn_masked_td_target   td = r + (1 - done) * gamma * q(s'), q(s') the masked Double-DQN (or plain max) target of a
//                              replay minibatch; the mask comes from row 0 of the replayed next-state features
//   eco_dqn_masked_argmax      argmax over the allowed vertices of feature rows (predict on replayed / snapshot states)
//   eco_dqn_masked_explore     the epsilon-greedy action of every lock-step environment, capture-safe (device epsilon,
//                              device "training ready" flag, caller-supplied uniforms)
//   eco_mpnn_grad_obs          eco_mpnn_grad_ev for a network with n_obs_in observables: the gradient of the zero-padded
//                              observable columns of W_init / W_e is written as exactly 0.0
//
// Masking rule everywhere (that of masked_argmax_kernel, env_kernels.cu): a disallowed entry compares as -1000.0, the
// lowest index wins ties, a row with no allowed vertex picks action 0.
#include <cuda_runtime.h>
#include <math.h>

#include "eco_common.cuh"

namespace eco {
namespace {

constexpr float MASKED_Q = -1000.f;
constexpr int WARPS = 8;                       // rows (episodes) per 256-thread block

// (value, index) of the masked argmax of q[0..N) on one warp; `allowed(i)` says whether vertex i may be flipped
template <typename Allowed>
__device__ __forceinline__ void warp_masked_argmax(const float* __restrict__ q, const int N, Allowed allowed, float& bv, int& bi) {
    const int lane = threadIdx.x & 31;
    bv = -INFINITY;
    bi = 0x7fffffff;
    for (int i = lane; i < N; i += 32) {
        const float v = allowed(i) ? q[i] : MASKED_Q;
        if (v > bv) { bv = v; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if (bi == 0x7fffffff) bi = 0;
}

__global__ void __launch_bounds__(WARPS * 32)
k_masked_td_target(const int B, const int N, const int NP, const float* __restrict__ q_online, const float* __restrict__ q_target,
                   const float* __restrict__ xn_next, const float* __restrict__ reward, const float* __restrict__ done,
                   const float gamma, const int double_dqn, const int clip, float* __restrict__ td, int32_t* __restrict__ chosen) {
    const int b = blockIdx.x * WARPS + (threadIdx.x >> 5);
    if (b >= B) return;
    const float* x0 = xn_next + (size_t)b * 3 * NP;           // row 0: the spins of s' as +-1.0
    auto allowed = [x0](int i) { return x0[i] == -1.f; };
    float v;
    int a;
    if (double_dqn) {
        float bv;
        warp_masked_argmax(q_online + (size_t)b * NP, N, allowed, bv, a);
        v = q_target[(size_t)b * NP + a];                    // gather from the UNMASKED target Q
    } else {
        warp_masked_argmax(q_target + (size_t)b * NP, N, allowed, v, a);   // masked max (-1000.0 if nothing is allowed)
    }
    if ((threadIdx.x & 31) == 0) {
        if (clip && v < 0.f) v = 0.f;
        // reward + (1 - done) * gamma * q, in the order torch evaluates the expression (no FMA contraction)
        td[b] = __fadd_rn(reward[b], __fmul_rn(__fmul_rn(__fsub_rn(1.f, done[b]), gamma), v));
        if (chosen) chosen[b] = a;
    }
}

__global__ void __launch_bounds__(WARPS * 32)
k_masked_argmax_rows(const int B, const int N, const int NP, const float* __restrict__ q, const float* __restrict__ xn,
                     int32_t* __restrict__ actions) {
    const int b = blockIdx.x * WARPS + (threadIdx.x >> 5);
    if (b >= B) return;
    const float* x0 = xn + (size_t)b * 3 * NP;
    float bv;
    int a;
    warp_masked_argmax(q + (size_t)b * NP, N, [x0](int i) { return x0[i] == -1.f; }, bv, a);
    if ((threadIdx.x & 31) == 0) actions[b] = a;
}

// Greedy (masked argmax) when ready && u0 >= eps, else the k-th spin still at -1 in ascending vertex order,
// k = min(floor(u1 * c), c - 1), c = number of spins still at -1 (ballot / popc over 32-vertex chunks).  c = 0: action 0.
__global__ void __launch_bounds__(WARPS * 32)
k_masked_explore(const eco_env_t env, const float* __restrict__ q, const float* __restrict__ uniforms, const float* __restrict__ eps,
                 const uint8_t* __restrict__ ready, int32_t* __restrict__ actions) {
    const int b = blockIdx.x * WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= env.B) return;
    const int N = env.N;
    const int8_t* s = env.spins + (size_t)b * env.NP;
    const float u0 = uniforms[2 * b], u1 = uniforms[2 * b + 1];
    int a = 0;
    if (*ready && u0 >= *eps) {
        float bv;
        warp_masked_argmax(q + (size_t)b * env.NP, N, [s](int i) { return s[i] < 0; }, bv, a);
    } else {
        int c = 0;
        for (int base = 0; base < N; base += 32) {
            const int i = base + lane;
            c += __popc(__ballot_sync(0xffffffffu, i < N && s[i] < 0));
        }
        if (c > 0) {
            int k = (int)floorf(__fmul_rn(u1, (float)c));
            k = k < c - 1 ? k : c - 1;
            for (int base = 0; base < N; base += 32) {
                const int i = base + lane;
                const unsigned m = __ballot_sync(0xffffffffu, i < N && s[i] < 0);
                const int cnt = __popc(m);
                if (k < cnt) {
                    // the lane holding the k-th set bit of m: k set bits below it, its own bit set
                    const bool mine = ((m >> lane) & 1u) && __popc(m & ((1u << lane) - 1u)) == k;
                    const unsigned who = __ballot_sync(0xffffffffu, mine);
                    a = base + (__ffs(who) - 1);
                    break;
                }
                k -= cnt;
            }
        }
    }
    if (lane == 0) actions[b] = a;
}

// W_init [64, 7]: columns 1..6;  W_e [63, 8]: columns 2..7 (column 0 multiplies the coupling, 1 the spin)
constexpr int G_WINIT = 0, G_WEDGE = 64 * 7;
constexpr int N_PAD_INIT = 64 * 6, N_PAD_EDGE = 63 * 6;

__global__ void __launch_bounds__(256) k_zero_padded_obs_grad(float* __restrict__ grad) {
    for (int t = threadIdx.x; t < N_PAD_INIT + N_PAD_EDGE; t += blockDim.x) {
        if (t < N_PAD_INIT) grad[G_WINIT + (t / 6) * 7 + 1 + t % 6] = 0.f;
        else grad[G_WEDGE + ((t - N_PAD_INIT) / 6) * 8 + 2 + (t - N_PAD_INIT) % 6] = 0.f;
    }
}

}  // namespace
}  // namespace eco

using namespace eco;

extern "C" {

int eco_dqn_masked_td_target(int32_t B, int32_t N, int32_t NP, const float* q_online, const float* q_target, const float* xn_next,
                             const float* reward, const float* done, float gamma, int32_t double_dqn, int32_t clip, float* td,
                             int32_t* chosen, void* stream) {
    ECO_CHECK_ARG(q_target && xn_next && reward && done && td && (q_online || !double_dqn), ECO_ERR_INVALID,
                  "eco_dqn_masked_td_target: null argument");
    ECO_CHECK_ARG(B >= 1 && N >= 1 && NP >= N, ECO_ERR_INVALID, "eco_dqn_masked_td_target: need B >= 1 and 1 <= N <= NP");
    k_masked_td_target<<<(B + WARPS - 1) / WARPS, WARPS * 32, 0, (cudaStream_t)stream>>>(
        B, N, NP, q_online, q_target, xn_next, reward, done, gamma, double_dqn, clip, td, chosen);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

int eco_dqn_masked_argmax(int32_t B, int32_t N, int32_t NP, const float* q, const float* xn, int32_t* actions, void* stream) {
    ECO_CHECK_ARG(q && xn && actions, ECO_ERR_INVALID, "eco_dqn_masked_argmax: null argument");
    ECO_CHECK_ARG(B >= 1 && N >= 1 && NP >= N, ECO_ERR_INVALID, "eco_dqn_masked_argmax: need B >= 1 and 1 <= N <= NP");
    k_masked_argmax_rows<<<(B + WARPS - 1) / WARPS, WARPS * 32, 0, (cudaStream_t)stream>>>(B, N, NP, q, xn, actions);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

int eco_dqn_masked_explore(const eco_env_t* env, const float* q, const float* uniforms, const float* eps, const uint8_t* ready,
                           int32_t* actions, void* stream) {
    ECO_CHECK_ARG(env && env->spins && q && uniforms && eps && ready && actions, ECO_ERR_INVALID,
                  "eco_dqn_masked_explore: null argument");
    ECO_CHECK_ARG(env->B >= 1, ECO_ERR_INVALID, "eco_dqn_masked_explore: empty environment batch");
    k_masked_explore<<<(env->B + WARPS - 1) / WARPS, WARPS * 32, 0, (cudaStream_t)stream>>>(*env, q, uniforms, eps, ready, actions);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

int eco_mpnn_grad_obs(const eco_graphs_t* g, const eco_mpnn_t* w, int32_t B, const int32_t* gidx, const float* xn, const float* xg,
                      float norm_max, const int32_t* actions, const float* targets, int32_t loss_kind, int32_t n_obs_in,
                      float* loss, float* grad, void* scratch, void* targets_ready_event, void* stream) {
    ECO_CHECK_ARG(n_obs_in == 1 || n_obs_in == ECO_N_OBS, ECO_ERR_INVALID, "eco_mpnn_grad_obs: n_obs_in must be 1 or %d, got %d",
                  ECO_N_OBS, n_obs_in);
    const int rc = eco_mpnn_grad_ev(g, w, B, gidx, xn, xg, norm_max, actions, targets, loss_kind, loss, grad, scratch,
                                    targets_ready_event, stream);
    if (rc != ECO_OK || n_obs_in == ECO_N_OBS) return rc;
    k_zero_padded_obs_grad<<<1, 256, 0, (cudaStream_t)stream>>>(grad);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

}  // extern "C"
