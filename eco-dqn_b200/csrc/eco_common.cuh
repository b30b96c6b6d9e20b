// Shared device/host helpers for the ECO-DQN B200 engine (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "ecodqn_b200.h"

namespace eco {

// row stride of the per-graph lookup tables gain_tab / dn_tab: entries k = -NP..NP at [NP + k], padded to a multiple of 4
// entries so that every row (and the window around k = 0) is 16-byte aligned for bulk copies
__host__ __device__ inline int tab_stride(int NP) { return 2 * NP + 4; }


// ---- error plumbing -------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);
void prof_begin(int kind, cudaStream_t st, int units = 1);   // no-ops unless eco_profile_enable(1)
void prof_end(int kind, cudaStream_t st);

#define ECO_CHECK_ARG(cond, code, ...)            \
    do {                                          \
        if (!(cond)) {                            \
            eco::set_error(__VA_ARGS__);          \
            return (code);                        \
        }                                         \
    } while (0)

#define ECO_CUDA(call)                                                                        \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            eco::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, \
                           __LINE__);                                                         \
            return ECO_ERR_CUDA;                                                              \
        }                                                                                     \
    } while (0)

#define ECO_LAUNCH_CHECK()                                                                        \
    do {                                                                                          \
        cudaError_t e__ = cudaGetLastError();                                                     \
        if (e__ != cudaSuccess) {                                                                 \
            eco::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), __FILE__, \
                           __LINE__);                                                             \
            return ECO_ERR_CUDA;                                                                  \
        }                                                                                         \
        eco::count_launch();                                                                      \
    } while (0)

// Function attributes (opt-in dynamic shared memory) and the SM count belong to a DEVICE, not to the process: a
// `static bool` guard would leave the second GPU of a process unconfigured.  `mask` is the caller's static bit set of
// devices already configured; true on the first call per device.  (Entry points are not re-entrant: no locking.)
static inline bool first_use_on_device(unsigned long long* mask) {
    int dev = 0;
    cudaGetDevice(&dev);
    const unsigned long long bit = 1ull << (dev & 63);
    if (*mask & bit) return false;
    *mask |= bit;
    return true;
}
static inline int device_sm_count() {
    static int n_sm[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    int& n = n_sm[dev & 63];
    if (!n && cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) n = 148;
    return n;
}

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
static inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }
static inline int padded_n(int n) { return round_up(n, 16); }

// Byte offset of core matrix (cb = K group, rb = column group; 8 x 8 bf16 = 128 bytes) in a graph's bf16 operand image
// (eco_graphs_t.tc_ops, built by graph_prepare.cu; NB = NP / 8 groups per side).  Column groups are stored in slabs of
// 32 (256 columns) and, inside a slab, K group after K group: a (K panel x slab) block is one contiguous run for the
// bulk copies of the large-graph kernels, and for NP <= 256 this is the plain (cb * NB + rb) order that the resident
// kernel (mpnn_tc.cu) uses as its shared-memory layout.
__host__ __device__ inline size_t tc_image_core(int NB, int cb, int rb) {
    const int s = rb >> 5, left = NB - 32 * s, wg = left < 32 ? left : 32;
    return ((size_t)s * NB * 32 + (size_t)cb * wg + (rb & 31)) * 128;
}

// ---- episode flags --------------------------------------------------------------------------------------
constexpr int FLAG_DONE = 1;
constexpr int FLAG_STOPPED = 2;
constexpr uint64_t VISITED_SALT0 = 0x9E3779B97F4A7C15ull;  // stored key = key ^ salt, so 0 means "empty slot"
constexpr uint64_t VISITED_SALT1 = 0xC2B2AE3D27D4EB4Full;

// one 32-byte sector in ONE store (STG.E.256, sm_100): two 16-byte stores of a lane each fill half a sector
__device__ __forceinline__ void st_f32x8(float* p, const float (&v)[8]) {
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
                 "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]) : "memory");
}

// ---- sub-warp group reductions (TPE lanes per episode, TPE <= 32 handled with shuffles) -------------------
template <int W>
__device__ __forceinline__ int group_sum(int v) {
#pragma unroll
    for (int o = W / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o, W);
    return v;
}
template <int W>
__device__ __forceinline__ int group_max(int v) {
#pragma unroll
    for (int o = W / 2; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o, W));
    return v;
}

// ---- internal launchers (one translation unit each) -------------------------------------------------------
int launch_graph_scatter_edges(const eco_graphs_t* g, int first, int count, const int64_t* offsets, const int32_t* rows,
                               const int32_t* cols, const int8_t* wts, long long n_entries, int symmetric, int* err_dev,
                               cudaStream_t st);
int launch_graph_prepare(const eco_graphs_t* g, int first, int count, cudaStream_t st);
int launch_graph_pad(const eco_graphs_t* g, const int8_t* dense_dev, int first, int count, cudaStream_t st);
int launch_env_reset(const eco_graphs_t* g, eco_env_t* env, const int32_t* gidx, const int8_t* spins, cudaStream_t st);
int launch_env_step(const eco_graphs_t* g, eco_env_t* env, int policy, const int32_t* actions, double* reward,
                    uint8_t* done, int32_t* ha, double* hr, double* hs, cudaStream_t st);
int launch_env_observation(const eco_env_t* env, float* obs7, cudaStream_t st);
int launch_masked_argmax(const eco_env_t* env, const float* q, int32_t* actions, cudaStream_t st);
int launch_env_results(const eco_env_t* env, int32_t* best_cut, int8_t* best_spins, int32_t* steps, cudaStream_t st);
int launch_mpnn_simt(const eco_graphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn,
                     const float* xg, float norm_max, float* q, int32_t* actions, void* scratch, cudaStream_t st);
int launch_wgraph_prepare(const eco_wgraphs_t* g, const double* dense, cudaStream_t st);
int launch_wenv_reset(const eco_wgraphs_t* g, eco_wenv_t* we, const int32_t* gidx, const int8_t* spins, cudaStream_t st);
int launch_wenv_step(const eco_wgraphs_t* g, eco_wenv_t* we, int policy, const int32_t* actions, double* reward, uint8_t* done,
                     int32_t* ha, double* hr, double* hs, cudaStream_t st);
int launch_wenv_results(const eco_wenv_t* we, double* best_cut, int8_t* best_spins, int32_t* steps, cudaStream_t st);
int launch_mpnn_simt_w(const eco_wgraphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn,
                       const float* xg, float norm_max, float* q, int32_t* actions, void* scratch, cudaStream_t st);
size_t mpnn_simt_scratch_bytes(int B, int N);
int launch_sgraph_prepare(const eco_sgraphs_t* g, cudaStream_t st);
int launch_senv_reset(const eco_sgraphs_t* g, eco_env_t* env, const int32_t* gidx, const int8_t* spins, cudaStream_t st);
int launch_senv_step(const eco_sgraphs_t* g, eco_env_t* env, int policy, const int32_t* actions, double* reward, uint8_t* done,
                     int32_t* ha, double* hr, double* hs, cudaStream_t st);
size_t smpnn_scratch_bytes(int B, int N);
int launch_smpnn(const eco_sgraphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn, const float* xg,
                 float norm_max, float* q, int32_t* actions, void* scratch, cudaStream_t st);
int launch_smpnn_tc(const eco_sgraphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn, const float* xg,
                    float norm_max, float* q, int32_t* actions, void* scratch, cudaStream_t st);
int launch_sparse_linear_tc(const float* A1, const float* A2, int K, long long V, const void* w_packed, float* C,
                            cudaStream_t st);
int launch_mpnn_tc(const eco_graphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn,
                   const float* xg, float norm_max, float* q, int32_t* actions, void* scratch, cudaStream_t st);
bool mpnn_tc_can_fuse(const eco_graphs_t* g, const eco_env_t* env);
int launch_mpnn_tc_fused(const eco_graphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn,
                         const float* xg, float norm_max, float* q, int32_t* actions, void* scratch, const eco_env_t* fused,
                         int n_steps, int32_t* ha, double* hr, double* hs, cudaStream_t st);
size_t mpnn_tc_scratch_bytes(int B, int N);
size_t mpnn_tc_packed_bytes();
int launch_mpnn_pack(const eco_mpnn_t* w, void* packed, cudaStream_t st);
bool mpnn_tc_supported(const eco_graphs_t* g);
size_t mpnn_grad_scratch_bytes(int B, int N);
int launch_mpnn_grad(const eco_graphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn, const float* xg,
                     float norm_max, const int32_t* actions, const float* targets, int huber, float* loss, float* grad,
                     void* scratch, cudaEvent_t targets_ready, cudaStream_t st);
int launch_mpnn_adam(const eco_mpnn_t* w, const float* grad, float* m, float* v, int step, float lr, float beta1, float beta2,
                     float eps, float weight_decay, cudaStream_t st);
bool mpnn_tcl_supported(const eco_graphs_t* g);
size_t mpnn_tcl_scratch_bytes(int B, int N);
int launch_mpnn_tcl(const eco_graphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn,
                    const float* xg, float norm_max, float* q, int32_t* actions, void* scratch, cudaStream_t st);
int launch_tcl_contract(const eco_graphs_t* g, const int32_t* gidx, int B, const float* X1, int which1, const float* X2,
                        int which2, size_t x_stride, float* out, size_t out_stride, float scale, int edge,
                        float norm_max, cudaStream_t st);

}  // namespace eco
