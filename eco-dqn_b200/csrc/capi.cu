// C ABI (include/ecodqn_b200.h): argument checking, workspace carving, the rollout loop and the host-buffer
// session.  No compute lives here; every entry point enqueues kernels from the other translation units.
#include <stdarg.h>

#include <atomic>
#include <vector>

#include <stdlib.h>

#include "eco_common.cuh"

namespace eco {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(int n) { g_launches += n; }

struct Prof {
    bool on = false;
    int stride = 1;
    long long count[3] = {0, 0, 0};
    long long units[3] = {0, 0, 0};    // what eco_profile_read reports as `launches`: recorded launches (kinds 0, 1), rollout steps (2)
    bool sampled[3] = {false, false, false};
    std::vector<cudaEvent_t> pool;
    std::vector<cudaEvent_t> rec[3];   // start/stop pairs per kind
    cudaEvent_t get() {
        cudaEvent_t e;
        if (!pool.empty()) { e = pool.back(); pool.pop_back(); return e; }
        cudaEventCreate(&e);
        return e;
    }
};
static Prof g_prof;
// every `stride`-th launch of a kind is bracketed by two events (an event record between two kernels costs about as much
// as a small kernel: bracketing every launch of a 400-step rollout adds ~4 % to it)
void prof_begin(int kind, cudaStream_t st, int units) {
    if (!g_prof.on) return;
    g_prof.sampled[kind] = kind == ECO_PROF_ROLLOUT || (g_prof.count[kind]++ % g_prof.stride) == 0;
    if (!g_prof.sampled[kind]) return;
    g_prof.units[kind] += units;
    cudaEvent_t e = g_prof.get();
    cudaEventRecord(e, st);
    g_prof.rec[kind].push_back(e);
}
void prof_end(int kind, cudaStream_t st) {
    if (!g_prof.on || !g_prof.sampled[kind]) return;
    cudaEvent_t e = g_prof.get();
    cudaEventRecord(e, st);
    g_prof.rec[kind].push_back(e);
}

struct Carver {
    unsigned char* base;
    size_t off = 0;
    explicit Carver(void* p) : base(static_cast<unsigned char*>(p)) {}
    template <class T>
    T* take(size_t count) {
        T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off = align256(off + count * sizeof(T));
        return p;
    }
};

static void carve_graphs(eco_graphs_t* g, Carver& c, int G, int N) {
    const int NP = padded_n(N);
    g->G = G; g->N = N; g->NP = NP; g->reserved = 0;
    g->J = c.take<int8_t>((size_t)G * NP * NP);
    g->gscal = c.take<double>((size_t)G * 4);
    g->deg = c.take<float>((size_t)G * NP);
    g->gstat = c.take<int32_t>((size_t)G * 4);
    g->dmax = c.take<float>(64);
    g->gain_tab = c.take<float>((size_t)G * tab_stride(NP));
    g->dn_tab = c.take<double>((size_t)G * tab_stride(NP));
    g->tc_ops = c.take<uint16_t>((size_t)G * 2 * NP * NP);   // (N > 208: used panel by panel by the aggregation kernel)
}

static int hcap_for(int T) {
    int c = 64;
    while (c < 2 * (T + 1)) c <<= 1;
    return c;
}

static void carve_env(eco_env_t* e, Carver& c, int B, int N, int T, double basin) {
    const int NP = padded_n(N);
    e->B = B; e->N = N; e->NP = NP; e->NW = (NP + 31) / 32;
    e->T = T; e->HCAP = hcap_for(T); e->use_basin = basin >= 0.0 ? 1 : 0; e->reserved = 0;
    e->basin_reward = basin >= 0.0 ? basin : 0.0;
    e->spins = c.take<int8_t>((size_t)B * NP);
    e->hfield = c.take<int16_t>((size_t)B * NP);
    e->last_flip = c.take<uint16_t>((size_t)B * NP);
    e->diff_bits = c.take<uint32_t>((size_t)B * e->NW);
    e->graph_idx = c.take<int32_t>((size_t)B);
    e->ep = c.take<eco_episode_t>((size_t)B);
    e->visited = c.take<uint64_t>(e->use_basin ? (size_t)B * e->HCAP * 2 : 2);
    e->zobrist = c.take<uint64_t>((size_t)NP * 2);
    e->tsf_tab = c.take<float>((size_t)T + 1);
    e->imm_tab = c.take<float>((size_t)T + 1);
    e->xn = c.take<float>((size_t)B * 3 * NP);
    e->xg = c.take<float>((size_t)B * 4);
    e->frac_tab = c.take<float>((size_t)N + 1);
}

static void carve_wgraphs(eco_wgraphs_t* g, Carver& c, int G, int N) {
    const int NP = padded_n(N);
    g->G = G; g->N = N; g->NP = NP; g->reserved = 0;
    g->J = c.take<double>((size_t)G * NP * NP);
    g->Jf = c.take<float>((size_t)G * NP * NP);
    g->gscal = c.take<double>((size_t)G * 4);
    g->deg = c.take<float>((size_t)G * NP);
    g->gstat = c.take<int32_t>((size_t)G * 4);
    g->dmax = c.take<float>(64);
}

static void carve_wenv(eco_wenv_t* e, Carver& c, int B, int N, int T, double basin) {
    carve_env(&e->base, c, B, N, T, basin);
    e->h = c.take<double>((size_t)B * e->base.NP);
    e->cut = c.take<double>((size_t)B * 2);
}

static void carve_sgraphs(eco_sgraphs_t* g, Carver& c, int G, int N, int64_t nnz) {
    const int NP = padded_n(N);
    g->G = G; g->N = N; g->NP = NP; g->reserved = 0; g->nnz = nnz;
    g->row_ptr = c.take<int64_t>((size_t)G * N + 1);
    g->col = c.take<int32_t>((size_t)nnz);
    g->val = c.take<int8_t>((size_t)nnz);
    g->gscal = c.take<double>((size_t)G * 4);
    g->deg = c.take<float>((size_t)G * NP);
    g->gstat = c.take<int32_t>((size_t)G * 4);
    g->dmax = c.take<float>(64);
}

static bool shape_ok(int N) { return N >= 1 && N <= ECO_MAX_SPINS; }
static bool sparse_shape_ok(int N) { return N >= 1 && N <= ECO_MAX_SPINS_SPARSE; }

__global__ void frac_tab_kernel(float* tab, int N) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k <= N) tab[k] = (float)__ddiv_rn((double)k, (double)N);     // np.sum(gains > 0) / n_spins, then the fp32 cast
}

__global__ void dmax_kernel(const eco_graphs_t g) {
    // single warp: max degree over all graphs of the set -> g.dmax[0]
    int m = 1;
    for (int i = threadIdx.x; i < g.G; i += 32) m = max(m, g.gstat[(size_t)i * 4]);
    m = group_max<32>(m);
    if (threadIdx.x == 0) g.dmax[0] = (float)m;
}

static int prepare(const eco_graphs_t* g, cudaStream_t st, int first = 0, int count = -1) {
    int rc = launch_graph_prepare(g, first, count < 0 ? g->G : count, st);
    if (rc != ECO_OK) return rc;
    dmax_kernel<<<1, 32, 0, st>>>(*g);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

static int pick_impl(const eco_graphs_t* g, const eco_mpnn_t* w, int impl) {
    // tensor cores: the resident kernel for N <= 208, the operand-tile pipeline (mpnn_large.cu) above
    if (impl == ECO_MPNN_AUTO) {
        if (w->packed && mpnn_tc_supported(g)) return ECO_MPNN_TCGEN05;
        if (w->packed && g->N > 208 && mpnn_tcl_supported(g)) return ECO_MPNN_TCGEN05;
        return ECO_MPNN_SIMT;
    }
    return impl;
}

}  // namespace eco

using namespace eco;

extern "C" {

const char* eco_last_error(void) { return g_err; }
int eco_abi_version(void) { return ECO_ABI_VERSION; }
int64_t eco_launch_count(int reset) {
    long long v = g_launches.load();
    if (reset) g_launches = 0;
    return v;
}

int eco_profile_enable(int on) {
    for (int k = 0; k < 3; ++k) {
        for (cudaEvent_t e : g_prof.rec[k]) g_prof.pool.push_back(e);
        g_prof.rec[k].clear();
        g_prof.count[k] = g_prof.units[k] = 0;
    }
    g_prof.on = on != 0;
    g_prof.stride = on > 1 ? on : 1;
    return ECO_OK;
}

int eco_profile_read(int kind, double* total_ms, int64_t* launches) {
    ECO_CHECK_ARG(kind >= 0 && kind < 3 && total_ms && launches, ECO_ERR_INVALID, "eco_profile_read: bad argument");
    ECO_CUDA(cudaDeviceSynchronize());
    double tot = 0.0;
    const auto& r = g_prof.rec[kind];
    for (size_t i = 0; i + 1 < r.size(); i += 2) {
        float ms = 0.f;
        ECO_CUDA(cudaEventElapsedTime(&ms, r[i], r[i + 1]));
        tot += ms;
    }
    *total_ms = tot;
    *launches = (int64_t)g_prof.units[kind];
    return ECO_OK;
}

// ------------------------------------------------------------------------------------------------ graphs
size_t eco_graphs_workspace_bytes(int32_t G, int32_t N) {
    if (G < 1 || !shape_ok(N)) return 0;
    eco_graphs_t g;
    Carver c(nullptr);
    carve_graphs(&g, c, G, N);
    return c.off;
}

int eco_graphs_bind(eco_graphs_t* g, void* ws, int32_t G, int32_t N) {
    ECO_CHECK_ARG(g && ws, ECO_ERR_INVALID, "eco_graphs_bind: null argument");
    ECO_CHECK_ARG(G >= 1 && shape_ok(N), ECO_ERR_INVALID, "eco_graphs_bind: need G >= 1 and 1 <= N <= %d (got G=%d N=%d)",
                  ECO_MAX_SPINS, G, N);
    ECO_CHECK_ARG(((uintptr_t)ws & 255) == 0, ECO_ERR_INVALID, "eco_graphs_bind: workspace must be 256-byte aligned");
    Carver c(ws);
    carve_graphs(g, c, G, N);
    return ECO_OK;
}

int eco_graphs_upload(eco_graphs_t* g, const int8_t* J_host, void* stream) {
    ECO_CHECK_ARG(g && J_host && g->J, ECO_ERR_INVALID, "eco_graphs_upload: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int G = g->G, N = g->N, NP = g->NP;
    if (N == NP) {
        ECO_CUDA(cudaMemcpyAsync(g->J, J_host, (size_t)G * N * N, cudaMemcpyHostToDevice, st));
    } else {
        ECO_CUDA(cudaMemsetAsync(g->J, 0, (size_t)G * NP * NP, st));
        cudaMemcpy3DParms p;
        memset(&p, 0, sizeof(p));
        p.srcPtr = make_cudaPitchedPtr((void*)J_host, N, N, N);
        p.dstPtr = make_cudaPitchedPtr((void*)g->J, NP, NP, NP);
        p.extent = make_cudaExtent(N, N, G);
        p.kind = cudaMemcpyHostToDevice;
        ECO_CUDA(cudaMemcpy3DAsync(&p, st));
    }
    return prepare(g, st);
}

int eco_graphs_load_dev(eco_graphs_t* g, const int8_t* J_dev, void* stream) {
    ECO_CHECK_ARG(g && J_dev && g->J, ECO_ERR_INVALID, "eco_graphs_load_dev: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = launch_graph_pad(g, J_dev, 0, g->G, st);
    if (rc != ECO_OK) return rc;
    return prepare(g, st);
}

int eco_graphs_update(eco_graphs_t* g, int32_t first, int32_t count, const int8_t* J_dev, void* stream) {
    ECO_CHECK_ARG(g && J_dev && g->J, ECO_ERR_INVALID, "eco_graphs_update: null argument");
    ECO_CHECK_ARG(first >= 0 && count >= 1 && first + count <= g->G, ECO_ERR_INVALID,
                  "eco_graphs_update: slots [%d, %d) outside the set of %d graphs", first, first + count, g->G);
    cudaStream_t st = (cudaStream_t)stream;
    int rc = launch_graph_pad(g, J_dev, first, count, st);
    if (rc != ECO_OK) return rc;
    return prepare(g, st, first, count);
}

int eco_graphs_load_edges_dev(eco_graphs_t* g, int32_t first, int32_t count, const int64_t* offsets_dev, const int32_t* rows_dev,
                              const int32_t* cols_dev, const int8_t* weights_dev, int64_t n_entries, int32_t symmetric,
                              void* stream) {
    ECO_CHECK_ARG(g && g->J && offsets_dev, ECO_ERR_INVALID, "eco_graphs_load_edges_dev: null argument");
    ECO_CHECK_ARG(first >= 0 && count >= 1 && first + count <= g->G, ECO_ERR_INVALID,
                  "eco_graphs_load_edges_dev: slots [%d, %d) outside the set of %d graphs", first, first + count, g->G);
    ECO_CHECK_ARG(n_entries >= 0 && (n_entries == 0 || (rows_dev && cols_dev && weights_dev)), ECO_ERR_INVALID,
                  "eco_graphs_load_edges_dev: %lld entries without edge arrays", (long long)n_entries);
    cudaStream_t st = (cudaStream_t)stream;
    ECO_CUDA(cudaMemsetAsync(g->J + (size_t)first * g->NP * g->NP, 0, (size_t)count * g->NP * g->NP, st));
    static int* err_words[64] = {nullptr};               // one device word per GPU of the process, allocated on first use
    int dev = 0;
    ECO_CUDA(cudaGetDevice(&dev));
    ECO_CHECK_ARG(dev >= 0 && dev < 64, ECO_ERR_UNSUPPORTED, "eco_graphs_load_edges_dev: device ordinal %d", dev);
    if (!err_words[dev]) ECO_CUDA(cudaMalloc(&err_words[dev], sizeof(int)));
    int* err_dev = err_words[dev];
    ECO_CUDA(cudaMemsetAsync(err_dev, 0, sizeof(int), st));
    int rc = launch_graph_scatter_edges(g, first, count, offsets_dev, rows_dev, cols_dev, weights_dev, n_entries, symmetric,
                                        err_dev, st);
    if (rc != ECO_OK) return rc;
    int err = 0;
    ECO_CUDA(cudaMemcpyAsync(&err, err_dev, sizeof(int), cudaMemcpyDeviceToHost, st));
    ECO_CUDA(cudaStreamSynchronize(st));
    ECO_CHECK_ARG(err == 0, ECO_ERR_INVALID, "eco_graphs_load_edges_dev: an entry names a vertex outside [0, %d)", g->N);
    return prepare(g, st, first, count);
}

// ------------------------------------------------------------------------------------------------ env
size_t eco_env_workspace_bytes(int32_t B, int32_t N, int32_t T) {
    if (B < 1 || !shape_ok(N) || T < 1 || T > 65535) return 0;
    eco_env_t e;
    Carver c(nullptr);
    carve_env(&e, c, B, N, T, 1.0);
    return c.off;
}

int eco_env_bind(eco_env_t* env, void* ws, int32_t B, int32_t N, int32_t T, double basin_reward) {
    ECO_CHECK_ARG(env && ws, ECO_ERR_INVALID, "eco_env_bind: null argument");
    ECO_CHECK_ARG(B >= 1 && shape_ok(N), ECO_ERR_INVALID, "eco_env_bind: need B >= 1 and 1 <= N <= %d", ECO_MAX_SPINS);
    ECO_CHECK_ARG(T >= 1 && T <= 65535, ECO_ERR_INVALID, "eco_env_bind: max_steps must be in [1, 65535] (got %d)", T);
    ECO_CHECK_ARG(((uintptr_t)ws & 255) == 0, ECO_ERR_INVALID, "eco_env_bind: workspace must be 256-byte aligned");
    Carver c(ws);
    carve_env(env, c, B, N, T, basin_reward);
    return ECO_OK;
}

int eco_env_set_tables(eco_env_t* env, const uint64_t* zob, const float* tsf, const float* imm, void* stream) {
    ECO_CHECK_ARG(env && zob && tsf && imm, ECO_ERR_INVALID, "eco_env_set_tables: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    ECO_CUDA(cudaMemcpyAsync(env->zobrist, zob, (size_t)env->NP * 16, cudaMemcpyHostToDevice, st));
    ECO_CUDA(cudaMemcpyAsync(env->tsf_tab, tsf, ((size_t)env->T + 1) * 4, cudaMemcpyHostToDevice, st));
    ECO_CUDA(cudaMemcpyAsync(env->imm_tab, imm, ((size_t)env->T + 1) * 4, cudaMemcpyHostToDevice, st));
    frac_tab_kernel<<<(env->N + 256) / 256, 256, 0, st>>>(env->frac_tab, env->N);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

static int check_pair(const eco_graphs_t* g, const eco_env_t* env, const char* who) {
    ECO_CHECK_ARG(g && env, ECO_ERR_INVALID, "%s: null argument", who);
    ECO_CHECK_ARG(g->N == env->N && g->NP == env->NP, ECO_ERR_INVALID, "%s: graph set has N=%d but env has N=%d", who,
                  g->N, env->N);
    return ECO_OK;
}

int eco_env_reset(const eco_graphs_t* g, eco_env_t* env, const int32_t* gidx, const int8_t* spins, void* stream) {
    int rc = check_pair(g, env, "eco_env_reset");
    if (rc) return rc;
    ECO_CHECK_ARG(gidx && spins, ECO_ERR_INVALID, "eco_env_reset: null argument");
    return launch_env_reset(g, env, gidx, spins, (cudaStream_t)stream);
}

int eco_env_step(const eco_graphs_t* g, eco_env_t* env, int32_t policy, const int32_t* actions, double* reward,
                 uint8_t* done, int32_t* ha, double* hr, double* hs, void* stream) {
    int rc = check_pair(g, env, "eco_env_step");
    if (rc) return rc;
    ECO_CHECK_ARG(policy == ECO_POLICY_ACTIONS || policy == ECO_POLICY_GREEDY, ECO_ERR_INVALID,
                  "eco_env_step: policy must be ECO_POLICY_ACTIONS or ECO_POLICY_GREEDY");
    ECO_CHECK_ARG(policy != ECO_POLICY_ACTIONS || actions, ECO_ERR_INVALID, "eco_env_step: actions_dev is NULL");
    return launch_env_step(g, env, policy, actions, reward, done, ha, hr, hs, (cudaStream_t)stream);
}

int eco_env_observation(const eco_env_t* env, float* obs7, void* stream) {
    ECO_CHECK_ARG(env && obs7, ECO_ERR_INVALID, "eco_env_observation: null argument");
    return launch_env_observation(env, obs7, (cudaStream_t)stream);
}

int eco_env_best_spins(const eco_env_t* env, int8_t* best_spins, void* stream) {
    ECO_CHECK_ARG(env && best_spins, ECO_ERR_INVALID, "eco_env_best_spins: null argument");
    return launch_env_results(env, nullptr, best_spins, nullptr, (cudaStream_t)stream);
}

int eco_env_results(const eco_env_t* env, int32_t* best_cut, int8_t* best_spins, int32_t* steps, void* stream) {
    ECO_CHECK_ARG(env, ECO_ERR_INVALID, "eco_env_results: null argument");
    return launch_env_results(env, best_cut, best_spins, steps, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ mpnn
// kernel scratch, followed by a [B, NP] fp32 Q buffer (eco_rollout needs the Q-values themselves when the argmax is
// masked: irreversible spins)
static size_t mpnn_kernel_scratch_bytes(int32_t B, int32_t N, int32_t impl) {
    size_t a = mpnn_simt_scratch_bytes(B, N);
    size_t b = (impl == ECO_MPNN_SIMT) ? 0 : (N <= 208 ? mpnn_tc_scratch_bytes(B, N) : mpnn_tcl_scratch_bytes(B, N));
    return align256(a > b ? a : b);
}
size_t eco_mpnn_scratch_bytes(int32_t B, int32_t N, int32_t impl) {
    if (B < 1 || !shape_ok(N)) return 0;
    return mpnn_kernel_scratch_bytes(B, N, impl) + align256((size_t)B * padded_n(N) * sizeof(float));
}

size_t eco_mpnn_packed_bytes(void) { return mpnn_tc_packed_bytes(); }

int eco_mpnn_pack(const eco_mpnn_t* w, void* packed, void* stream) {
    ECO_CHECK_ARG(w && packed, ECO_ERR_INVALID, "eco_mpnn_pack: null argument");
    return launch_mpnn_pack(w, packed, (cudaStream_t)stream);
}

static int check_weights(const eco_mpnn_t* w, const char* who) {
    ECO_CHECK_ARG(w && w->w_init && w->w_edge && w->w_edge_feat && w->w_pool && w->w_read && w->b_read,
                  ECO_ERR_INVALID, "%s: weight pointer is NULL", who);
    for (int l = 0; l < 3; ++l)
        ECO_CHECK_ARG(w->w_msg[l] && w->w_upd[l], ECO_ERR_INVALID, "%s: layer %d weight pointer is NULL", who, l);
    return ECO_OK;
}

int eco_mpnn_forward(const eco_graphs_t* g, const eco_mpnn_t* w, int32_t B, const int32_t* gidx, const float* xn,
                     const float* xg, float norm_max, float* q, int32_t* actions, void* scratch, int32_t impl,
                     void* stream) {
    ECO_CHECK_ARG(g && gidx && xn && xg && scratch, ECO_ERR_INVALID, "eco_mpnn_forward: null argument");
    ECO_CHECK_ARG(B >= 1, ECO_ERR_INVALID, "eco_mpnn_forward: B must be >= 1");
    int rc = check_weights(w, "eco_mpnn_forward");
    if (rc) return rc;
    const int use = pick_impl(g, w, impl);
    if (use == ECO_MPNN_TCGEN05 && g->N > 208) {
        ECO_CHECK_ARG(w->packed, ECO_ERR_INVALID, "eco_mpnn_forward: tcgen05 path needs eco_mpnn_pack() output");
        ECO_CHECK_ARG((((uintptr_t)xn | (uintptr_t)xg | (uintptr_t)scratch) & 15) == 0, ECO_ERR_INVALID,
                      "eco_mpnn_forward: xn, xg and scratch must be 16-byte aligned");
        ECO_CHECK_ARG(mpnn_tcl_supported(g), ECO_ERR_UNSUPPORTED,
                      "eco_mpnn_forward: the tensor-core paths need couplings in {-1,0,1}; use ECO_MPNN_SIMT");
        return launch_mpnn_tcl(g, w, B, gidx, xn, xg, norm_max, q, actions, scratch, (cudaStream_t)stream);
    }
    if (use == ECO_MPNN_TCGEN05) {
        ECO_CHECK_ARG(w->packed, ECO_ERR_INVALID, "eco_mpnn_forward: tcgen05 path needs eco_mpnn_pack() output");
        ECO_CHECK_ARG(mpnn_tc_supported(g), ECO_ERR_UNSUPPORTED,
                      "eco_mpnn_forward: the tensor-core paths need couplings in {-1,0,1}; use ECO_MPNN_SIMT");
        return launch_mpnn_tc(g, w, B, gidx, xn, xg, norm_max, q, actions, scratch, (cudaStream_t)stream);
    }
    ECO_CHECK_ARG(use == ECO_MPNN_SIMT, ECO_ERR_INVALID, "eco_mpnn_forward: unknown impl %d", impl);
    return launch_mpnn_simt(g, w, B, gidx, xn, xg, norm_max, q, actions, scratch, (cudaStream_t)stream);
}

size_t eco_mpnn_grad_scratch_bytes(int32_t B, int32_t N) { return (B >= 1 && N >= 1) ? mpnn_grad_scratch_bytes(B, N) : 0; }

int eco_mpnn_grad_ev(const eco_graphs_t* g, const eco_mpnn_t* w, int32_t B, const int32_t* gidx, const float* xn, const float* xg,
                     float norm_max, const int32_t* actions, const float* targets, int32_t loss_kind, float* loss, float* grad,
                     void* scratch, void* targets_ready_event, void* stream) {
    ECO_CHECK_ARG(g && gidx && xn && xg && actions && targets && loss && grad && scratch, ECO_ERR_INVALID,
                  "eco_mpnn_grad: null argument");
    ECO_CHECK_ARG(B >= 1 && B <= 65535, ECO_ERR_INVALID, "eco_mpnn_grad: B must be in 1..65535 (minibatch), got %d", B);
    ECO_CHECK_ARG(loss_kind == ECO_LOSS_MSE || loss_kind == ECO_LOSS_HUBER, ECO_ERR_INVALID, "eco_mpnn_grad: unknown loss %d",
                  loss_kind);
    ECO_CHECK_ARG(g->reserved & ECO_GRAPHS_PM1, ECO_ERR_UNSUPPORTED, "eco_mpnn_grad: needs couplings in {-1,0,1}");
    ECO_CHECK_ARG((((uintptr_t)scratch | (uintptr_t)grad) & 15) == 0, ECO_ERR_INVALID, "eco_mpnn_grad: scratch and grad must be 16-byte aligned");
    int rc = check_weights(w, "eco_mpnn_grad");
    if (rc) return rc;
    return launch_mpnn_grad(g, w, B, gidx, xn, xg, norm_max, actions, targets, loss_kind == ECO_LOSS_HUBER, loss, grad, scratch,
                            (cudaEvent_t)targets_ready_event, (cudaStream_t)stream);
}

int eco_mpnn_grad(const eco_graphs_t* g, const eco_mpnn_t* w, int32_t B, const int32_t* gidx, const float* xn, const float* xg,
                  float norm_max, const int32_t* actions, const float* targets, int32_t loss_kind, float* loss, float* grad,
                  void* scratch, void* stream) {
    return eco_mpnn_grad_ev(g, w, B, gidx, xn, xg, norm_max, actions, targets, loss_kind, loss, grad, scratch, nullptr, stream);
}

int eco_mpnn_adam(const eco_mpnn_t* w, const float* grad, float* exp_avg, float* exp_avg_sq, int32_t step, float lr, float beta1,
                  float beta2, float eps, float weight_decay, void* stream) {
    ECO_CHECK_ARG(grad && exp_avg && exp_avg_sq, ECO_ERR_INVALID, "eco_mpnn_adam: null argument");
    ECO_CHECK_ARG(step >= 1, ECO_ERR_INVALID, "eco_mpnn_adam: step counts from 1");
    int rc = check_weights(w, "eco_mpnn_adam");
    if (rc) return rc;
    return launch_mpnn_adam(w, grad, exp_avg, exp_avg_sq, step, lr, beta1, beta2, eps, weight_decay, (cudaStream_t)stream);
}

int eco_graph_aggregate(const eco_graphs_t* g, int32_t B, const int32_t* gidx, const float* x, int32_t use_abs,
                        float scale, float* out, void* stream) {
    ECO_CHECK_ARG(g && gidx && x && out && B >= 1, ECO_ERR_INVALID, "eco_graph_aggregate: bad argument");
    ECO_CHECK_ARG(mpnn_tcl_supported(g), ECO_ERR_UNSUPPORTED, "eco_graph_aggregate: needs couplings in {-1,0,1}");
    return launch_tcl_contract(g, gidx, B, x, use_abs ? 1 : 0, nullptr, 0, (size_t)g->N * 64, out, (size_t)g->N * 64, scale,
                               0, 0.f, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ rollout
int eco_env_masked_argmax(const eco_env_t* env, const float* q, int32_t* actions, void* stream) {
    ECO_CHECK_ARG(env && q && actions && env->spins, ECO_ERR_INVALID, "eco_env_masked_argmax: null argument");
    return launch_masked_argmax(env, q, actions, (cudaStream_t)stream);
}

int eco_rollout(const eco_graphs_t* g, eco_env_t* env, const eco_mpnn_t* w, int32_t n_steps, int32_t policy,
                float norm_max, int32_t* act, void* scratch, int32_t impl, int32_t* ha, double* hr, double* hs,
                void* stream) {
    int rc = check_pair(g, env, "eco_rollout");
    if (rc) return rc;
    ECO_CHECK_ARG(n_steps >= 0, ECO_ERR_INVALID, "eco_rollout: n_steps < 0");
    ECO_CHECK_ARG(policy == ECO_POLICY_NETWORK || policy == ECO_POLICY_GREEDY, ECO_ERR_INVALID,
                  "eco_rollout: policy must be ECO_POLICY_NETWORK or ECO_POLICY_GREEDY");
    cudaStream_t st = (cudaStream_t)stream;
    if (policy == ECO_POLICY_GREEDY) {
        for (int t = 0; t < n_steps; ++t) {
            rc = launch_env_step(g, env, ECO_POLICY_GREEDY, nullptr, nullptr, nullptr, ha, hr, hs, st);
            if (rc) return rc;
        }
        return ECO_OK;
    }
    ECO_CHECK_ARG(act && scratch, ECO_ERR_INVALID, "eco_rollout: network policy needs actions and mpnn scratch buffers");
    rc = check_weights(w, "eco_rollout");
    if (rc) return rc;
    const bool masked = (env->reserved & ECO_ENV_IRREVERSIBLE) != 0;   // argmax over the spins still at -1 only
    float* qbuf = masked ? (float*)((char*)scratch + mpnn_kernel_scratch_bytes(env->B, env->N, impl)) : nullptr;
    // The ECO-DQN configuration on the resident tensor-core kernel (N <= 208, >= 2 episodes per SM): the WHOLE rollout is one
    // launch -- the kernel's tail warp applies each flip itself and every CTA takes its own episodes through all n_steps steps
    // (mpnn_tc.cu, FUSED; episodes never interact, so there is nothing to synchronise between steps).  Bit-identical to the
    // two-launches-per-step path below (tests/test_gpu_round2.py), which ECO_FUSED_STEP=0 selects.
    static const bool fuse = !(getenv("ECO_FUSED_STEP") && atoi(getenv("ECO_FUSED_STEP")) == 0);
    if (fuse && n_steps > 0 && !masked && pick_impl(g, w, impl) == ECO_MPNN_TCGEN05 && g->N <= 208 && w->packed &&
        mpnn_tc_can_fuse(g, env))
        return launch_mpnn_tc_fused(g, w, env->B, env->graph_idx, env->xn, env->xg, norm_max, nullptr, act, scratch, env, n_steps,
                                    ha, hr, hs, st);
    for (int t = 0; t < n_steps; ++t) {
        rc = eco_mpnn_forward(g, w, env->B, env->graph_idx, env->xn, env->xg, norm_max, qbuf, masked ? nullptr : act,
                              scratch, impl, stream);
        if (rc) return rc;
        if (masked) {
            rc = launch_masked_argmax(env, qbuf, act, st);
            if (rc) return rc;
        }
        rc = launch_env_step(g, env, ECO_POLICY_ACTIONS, act, nullptr, nullptr, ha, hr, hs, st);
        if (rc) return rc;
    }
    return ECO_OK;
}

// ------------------------------------------------------------------------------------------------ weighted graphs
size_t eco_wgraphs_workspace_bytes(int32_t G, int32_t N) {
    if (G < 1 || !shape_ok(N)) return 0;
    eco_wgraphs_t g;
    Carver c(nullptr);
    carve_wgraphs(&g, c, G, N);
    return c.off;
}

int eco_wgraphs_bind(eco_wgraphs_t* g, void* ws, int32_t G, int32_t N) {
    ECO_CHECK_ARG(g && ws, ECO_ERR_INVALID, "eco_wgraphs_bind: null argument");
    ECO_CHECK_ARG(G >= 1 && shape_ok(N), ECO_ERR_INVALID, "eco_wgraphs_bind: need G >= 1 and 1 <= N <= %d (got G=%d N=%d)",
                  ECO_MAX_SPINS, G, N);
    ECO_CHECK_ARG(((uintptr_t)ws & 255) == 0, ECO_ERR_INVALID, "eco_wgraphs_bind: workspace must be 256-byte aligned");
    Carver c(ws);
    carve_wgraphs(g, c, G, N);
    return ECO_OK;
}

int eco_wgraphs_load_dev(eco_wgraphs_t* g, const double* J_dev, void* stream) {
    ECO_CHECK_ARG(g && J_dev && g->J, ECO_ERR_INVALID, "eco_wgraphs_load_dev: null argument");
    ECO_CHECK_ARG(g->reserved == 0, ECO_ERR_UNSUPPORTED, "eco_wgraphs_load_dev: weighted graph sets support OptimisationTarget.CUT only");
    return launch_wgraph_prepare(g, J_dev, (cudaStream_t)stream);
}

size_t eco_wenv_workspace_bytes(int32_t B, int32_t N, int32_t T) {
    if (B < 1 || !shape_ok(N) || T < 1 || T > 65535) return 0;
    eco_wenv_t e;
    Carver c(nullptr);
    carve_wenv(&e, c, B, N, T, 1.0);
    return c.off;
}

int eco_wenv_bind(eco_wenv_t* env, void* ws, int32_t B, int32_t N, int32_t T, double basin_reward) {
    ECO_CHECK_ARG(env && ws, ECO_ERR_INVALID, "eco_wenv_bind: null argument");
    ECO_CHECK_ARG(B >= 1 && shape_ok(N), ECO_ERR_INVALID, "eco_wenv_bind: need B >= 1 and 1 <= N <= %d", ECO_MAX_SPINS);
    ECO_CHECK_ARG(T >= 1 && T <= 65535, ECO_ERR_INVALID, "eco_wenv_bind: max_steps must be in [1, 65535] (got %d)", T);
    ECO_CHECK_ARG(((uintptr_t)ws & 255) == 0, ECO_ERR_INVALID, "eco_wenv_bind: workspace must be 256-byte aligned");
    Carver c(ws);
    carve_wenv(env, c, B, N, T, basin_reward);
    return ECO_OK;
}

static int check_wpair(const eco_wgraphs_t* g, const eco_wenv_t* env, const char* who) {
    ECO_CHECK_ARG(g && env, ECO_ERR_INVALID, "%s: null argument", who);
    ECO_CHECK_ARG(g->N == env->base.N && g->NP == env->base.NP, ECO_ERR_INVALID, "%s: graph set has N=%d but env has N=%d",
                  who, g->N, env->base.N);
    ECO_CHECK_ARG(env->base.reserved == 0 && g->reserved == 0, ECO_ERR_UNSUPPORTED,
                  "%s: weighted graphs support the ECO-DQN configuration only (CUT target, BLS reward, reversible spins)", who);
    return ECO_OK;
}

int eco_wenv_reset(const eco_wgraphs_t* g, eco_wenv_t* env, const int32_t* gidx, const int8_t* spins, void* stream) {
    int rc = check_wpair(g, env, "eco_wenv_reset");
    if (rc) return rc;
    ECO_CHECK_ARG(gidx && spins, ECO_ERR_INVALID, "eco_wenv_reset: null argument");
    return launch_wenv_reset(g, env, gidx, spins, (cudaStream_t)stream);
}

int eco_wenv_step(const eco_wgraphs_t* g, eco_wenv_t* env, int32_t policy, const int32_t* actions, double* reward,
                  uint8_t* done, int32_t* ha, double* hr, double* hs, void* stream) {
    int rc = check_wpair(g, env, "eco_wenv_step");
    if (rc) return rc;
    ECO_CHECK_ARG(policy == ECO_POLICY_ACTIONS || policy == ECO_POLICY_GREEDY, ECO_ERR_INVALID,
                  "eco_wenv_step: policy must be ECO_POLICY_ACTIONS or ECO_POLICY_GREEDY");
    ECO_CHECK_ARG(policy != ECO_POLICY_ACTIONS || actions, ECO_ERR_INVALID, "eco_wenv_step: actions_dev is NULL");
    return launch_wenv_step(g, env, policy, actions, reward, done, ha, hr, hs, (cudaStream_t)stream);
}

int eco_wmpnn_forward(const eco_wgraphs_t* g, const eco_mpnn_t* w, int32_t B, const int32_t* gidx, const float* xn,
                      const float* xg, float norm_max, float* q, int32_t* actions, void* scratch, int32_t impl,
                      void* stream) {
    ECO_CHECK_ARG(g && gidx && xn && xg && scratch, ECO_ERR_INVALID, "eco_wmpnn_forward: null argument");
    ECO_CHECK_ARG(B >= 1, ECO_ERR_INVALID, "eco_wmpnn_forward: B must be >= 1");
    int rc = check_weights(w, "eco_wmpnn_forward");
    if (rc) return rc;
    // the tensor-core kernels factor the edge stage into contractions with J and |J| in {-1,0,1} (DESIGN.md section 4.2);
    // a real a_ij does not factor that way
    ECO_CHECK_ARG(impl != ECO_MPNN_TCGEN05, ECO_ERR_UNSUPPORTED,
                  "eco_wmpnn_forward: the tensor-core MPNN needs couplings in {-1,0,1}; weighted graphs run on ECO_MPNN_SIMT");
    ECO_CHECK_ARG(impl == ECO_MPNN_AUTO || impl == ECO_MPNN_SIMT, ECO_ERR_INVALID, "eco_wmpnn_forward: unknown impl %d", impl);
    return launch_mpnn_simt_w(g, w, B, gidx, xn, xg, norm_max, q, actions, scratch, (cudaStream_t)stream);
}

int eco_wrollout(const eco_wgraphs_t* g, eco_wenv_t* env, const eco_mpnn_t* w, int32_t n_steps, int32_t policy,
                 float norm_max, int32_t* act, void* scratch, int32_t impl, int32_t* ha, double* hr, double* hs,
                 void* stream) {
    int rc = check_wpair(g, env, "eco_wrollout");
    if (rc) return rc;
    ECO_CHECK_ARG(n_steps >= 0, ECO_ERR_INVALID, "eco_wrollout: n_steps < 0");
    ECO_CHECK_ARG(policy == ECO_POLICY_NETWORK || policy == ECO_POLICY_GREEDY, ECO_ERR_INVALID,
                  "eco_wrollout: policy must be ECO_POLICY_NETWORK or ECO_POLICY_GREEDY");
    cudaStream_t st = (cudaStream_t)stream;
    if (policy == ECO_POLICY_GREEDY) {
        for (int t = 0; t < n_steps; ++t) {
            rc = launch_wenv_step(g, env, ECO_POLICY_GREEDY, nullptr, nullptr, nullptr, ha, hr, hs, st);
            if (rc) return rc;
        }
        return ECO_OK;
    }
    ECO_CHECK_ARG(act && scratch, ECO_ERR_INVALID, "eco_wrollout: network policy needs actions and mpnn scratch buffers");
    for (int t = 0; t < n_steps; ++t) {
        rc = eco_wmpnn_forward(g, w, env->base.B, env->base.graph_idx, env->base.xn, env->base.xg, norm_max, nullptr, act,
                               scratch, impl, stream);
        if (rc) return rc;
        rc = launch_wenv_step(g, env, ECO_POLICY_ACTIONS, act, nullptr, nullptr, ha, hr, hs, st);
        if (rc) return rc;
    }
    return ECO_OK;
}

int eco_wenv_results(const eco_wenv_t* env, double* best_cut, int8_t* best_spins, int32_t* steps, void* stream) {
    ECO_CHECK_ARG(env, ECO_ERR_INVALID, "eco_wenv_results: null argument");
    return launch_wenv_results(env, best_cut, best_spins, steps, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ sparse (CSR) graphs
size_t eco_sgraphs_workspace_bytes(int32_t G, int32_t N, int64_t nnz) {
    if (G < 1 || !sparse_shape_ok(N) || nnz < 0) return 0;
    eco_sgraphs_t g;
    Carver c(nullptr);
    carve_sgraphs(&g, c, G, N, nnz);
    return c.off;
}

int eco_sgraphs_bind(eco_sgraphs_t* g, void* ws, int32_t G, int32_t N, int64_t nnz) {
    ECO_CHECK_ARG(g && ws, ECO_ERR_INVALID, "eco_sgraphs_bind: null argument");
    ECO_CHECK_ARG(G >= 1 && sparse_shape_ok(N) && nnz >= 0, ECO_ERR_INVALID,
                  "eco_sgraphs_bind: need G >= 1, 1 <= N <= %d and nnz >= 0 (got G=%d N=%d nnz=%lld)", ECO_MAX_SPINS_SPARSE, G, N,
                  (long long)nnz);
    ECO_CHECK_ARG(((uintptr_t)ws & 255) == 0, ECO_ERR_INVALID, "eco_sgraphs_bind: workspace must be 256-byte aligned");
    Carver c(ws);
    carve_sgraphs(g, c, G, N, nnz);
    return ECO_OK;
}

int eco_sgraphs_load_dev(eco_sgraphs_t* g, const int64_t* row_ptr, const int32_t* col, const int8_t* val, void* stream) {
    ECO_CHECK_ARG(g && g->row_ptr && row_ptr && (g->nnz == 0 || (col && val)), ECO_ERR_INVALID, "eco_sgraphs_load_dev: null argument");
    ECO_CHECK_ARG(!(g->reserved & ECO_GRAPHS_MIN_CUT), ECO_ERR_UNSUPPORTED,
                  "eco_sgraphs_load_dev: sparse graph sets support OptimisationTarget.CUT only");
    cudaStream_t st = (cudaStream_t)stream;
    ECO_CUDA(cudaMemcpyAsync(g->row_ptr, row_ptr, ((size_t)g->G * g->N + 1) * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    if (g->nnz > 0) {
        ECO_CUDA(cudaMemcpyAsync(g->col, col, (size_t)g->nnz * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        ECO_CUDA(cudaMemcpyAsync(g->val, val, (size_t)g->nnz, cudaMemcpyDeviceToDevice, st));
    }
    return launch_sgraph_prepare(g, st);
}

size_t eco_senv_workspace_bytes(int32_t B, int32_t N, int32_t T) {
    if (B < 1 || !sparse_shape_ok(N) || T < 1 || T > 65535) return 0;
    eco_env_t e;
    Carver c(nullptr);
    carve_env(&e, c, B, N, T, 1.0);
    return c.off;
}

int eco_senv_bind(eco_env_t* env, void* ws, int32_t B, int32_t N, int32_t T, double basin_reward) {
    ECO_CHECK_ARG(env && ws, ECO_ERR_INVALID, "eco_senv_bind: null argument");
    ECO_CHECK_ARG(B >= 1 && sparse_shape_ok(N), ECO_ERR_INVALID, "eco_senv_bind: need B >= 1 and 1 <= N <= %d",
                  ECO_MAX_SPINS_SPARSE);
    ECO_CHECK_ARG(T >= 1 && T <= 65535, ECO_ERR_INVALID, "eco_senv_bind: max_steps must be in [1, 65535] (got %d)", T);
    ECO_CHECK_ARG(((uintptr_t)ws & 255) == 0, ECO_ERR_INVALID, "eco_senv_bind: workspace must be 256-byte aligned");
    Carver c(ws);
    carve_env(env, c, B, N, T, basin_reward);
    return ECO_OK;
}

static int check_spair(const eco_sgraphs_t* g, const eco_env_t* env, const char* who) {
    ECO_CHECK_ARG(g && env, ECO_ERR_INVALID, "%s: null argument", who);
    ECO_CHECK_ARG(g->N == env->N && g->NP == env->NP, ECO_ERR_INVALID, "%s: graph set has N=%d but env has N=%d", who, g->N,
                  env->N);
    ECO_CHECK_ARG(env->reserved == 0 && !(g->reserved & ECO_GRAPHS_MIN_CUT), ECO_ERR_UNSUPPORTED,
                  "%s: sparse graph sets support the ECO-DQN configuration only (CUT target, BLS reward, reversible spins)", who);
    return ECO_OK;
}

int eco_senv_reset(const eco_sgraphs_t* g, eco_env_t* env, const int32_t* gidx, const int8_t* spins, void* stream) {
    int rc = check_spair(g, env, "eco_senv_reset");
    if (rc) return rc;
    ECO_CHECK_ARG(gidx && spins, ECO_ERR_INVALID, "eco_senv_reset: null argument");
    return launch_senv_reset(g, env, gidx, spins, (cudaStream_t)stream);
}

int eco_senv_step(const eco_sgraphs_t* g, eco_env_t* env, int32_t policy, const int32_t* actions, double* reward, uint8_t* done,
                  int32_t* ha, double* hr, double* hs, void* stream) {
    int rc = check_spair(g, env, "eco_senv_step");
    if (rc) return rc;
    ECO_CHECK_ARG(policy == ECO_POLICY_ACTIONS || policy == ECO_POLICY_GREEDY, ECO_ERR_INVALID,
                  "eco_senv_step: policy must be ECO_POLICY_ACTIONS or ECO_POLICY_GREEDY");
    ECO_CHECK_ARG(policy != ECO_POLICY_ACTIONS || actions, ECO_ERR_INVALID, "eco_senv_step: actions_dev is NULL");
    return launch_senv_step(g, env, policy, actions, reward, done, ha, hr, hs, (cudaStream_t)stream);
}

size_t eco_smpnn_scratch_bytes(int32_t B, int32_t N) {
    if (B < 1 || !sparse_shape_ok(N)) return 0;
    return smpnn_scratch_bytes(B, N);
}

int eco_smpnn_forward(const eco_sgraphs_t* g, const eco_mpnn_t* w, int32_t B, const int32_t* gidx, const float* xn,
                      const float* xg, float norm_max, float* q, int32_t* actions, void* scratch, void* stream) {
    ECO_CHECK_ARG(g && gidx && xn && xg && scratch, ECO_ERR_INVALID, "eco_smpnn_forward: null argument");
    ECO_CHECK_ARG(B >= 1, ECO_ERR_INVALID, "eco_smpnn_forward: B must be >= 1");
    ECO_CHECK_ARG(((uintptr_t)scratch & 15) == 0, ECO_ERR_INVALID, "eco_smpnn_forward: scratch must be 16-byte aligned");
    int rc = check_weights(w, "eco_smpnn_forward");
    if (rc) return rc;
    return launch_smpnn(g, w, B, gidx, xn, xg, norm_max, q, actions, scratch, (cudaStream_t)stream);
}

int eco_srollout(const eco_sgraphs_t* g, eco_env_t* env, const eco_mpnn_t* w, int32_t n_steps, int32_t policy, float norm_max,
                 int32_t* act, void* scratch, int32_t* ha, double* hr, double* hs, void* stream) {
    int rc = check_spair(g, env, "eco_srollout");
    if (rc) return rc;
    ECO_CHECK_ARG(n_steps >= 0, ECO_ERR_INVALID, "eco_srollout: n_steps < 0");
    ECO_CHECK_ARG(policy == ECO_POLICY_NETWORK || policy == ECO_POLICY_GREEDY, ECO_ERR_INVALID,
                  "eco_srollout: policy must be ECO_POLICY_NETWORK or ECO_POLICY_GREEDY");
    cudaStream_t st = (cudaStream_t)stream;
    if (policy == ECO_POLICY_GREEDY) {
        for (int t = 0; t < n_steps; ++t) {
            rc = launch_senv_step(g, env, ECO_POLICY_GREEDY, nullptr, nullptr, nullptr, ha, hr, hs, st);
            if (rc) return rc;
        }
        return ECO_OK;
    }
    ECO_CHECK_ARG(act && scratch, ECO_ERR_INVALID, "eco_srollout: network policy needs actions and mpnn scratch buffers");
    for (int t = 0; t < n_steps; ++t) {
        rc = eco_smpnn_forward(g, w, env->B, env->graph_idx, env->xn, env->xg, norm_max, nullptr, act, scratch, stream);
        if (rc) return rc;
        rc = launch_senv_step(g, env, ECO_POLICY_ACTIONS, act, nullptr, nullptr, ha, hr, hs, st);
        if (rc) return rc;
    }
    return ECO_OK;
}

// ------------------------------------------------------------------------------------------------ session
struct eco_session {
    int G, N, B, T, impl;
    eco_graphs_t graphs;
    eco_env_t env;
    eco_mpnn_t w;
    void *ws_graphs = nullptr, *ws_env = nullptr, *ws_w = nullptr, *ws_scratch = nullptr, *ws_io = nullptr;
    void* packed_buf = nullptr;
    int8_t *d_Jdense, *d_spins, *d_best_spins;
    int32_t *d_gidx, *d_act, *d_best_cut;
};

static const int kWeightCounts[12] = {64 * 7, 63 * 8, 64 * 64, 64 * 128, 64 * 128, 64 * 128,
                                      64 * 128, 64 * 128, 64 * 128, 64 * 64, 128, 1};

void eco_session_destroy(eco_session_t* s) {
    if (!s) return;
    cudaFree(s->ws_graphs); cudaFree(s->ws_env); cudaFree(s->ws_w); cudaFree(s->ws_scratch); cudaFree(s->ws_io);
    delete s;
}

int eco_session_create(eco_session_t** out, int32_t G, int32_t N, int32_t B, int32_t T, double basin,
                       const float* const weights_host[12], int32_t impl) {
    ECO_CHECK_ARG(out && weights_host, ECO_ERR_INVALID, "eco_session_create: null argument");
    ECO_CHECK_ARG(G >= 1 && B >= 1 && shape_ok(N) && T >= 1 && T <= 65535, ECO_ERR_INVALID,
                  "eco_session_create: bad shape G=%d N=%d B=%d T=%d", G, N, B, T);
    eco_session* s = new eco_session();
    s->G = G; s->N = N; s->B = B; s->T = T; s->impl = impl;
#define SESSION_CUDA(call)                                                        \
    do {                                                                          \
        cudaError_t e__ = (call);                                                 \
        if (e__ != cudaSuccess) {                                                 \
            set_error("%s failed: %s", #call, cudaGetErrorString(e__));           \
            eco_session_destroy(s);                                               \
            return ECO_ERR_CUDA;                                                  \
        }                                                                         \
    } while (0)
    SESSION_CUDA(cudaMalloc(&s->ws_graphs, eco_graphs_workspace_bytes(G, N)));
    SESSION_CUDA(cudaMalloc(&s->ws_env, eco_env_workspace_bytes(B, N, T)));
    SESSION_CUDA(cudaMalloc(&s->ws_scratch, eco_mpnn_scratch_bytes(B, N, impl)));
    size_t wfloats = 0;
    for (int i = 0; i < 12; ++i) wfloats += (size_t)((kWeightCounts[i] + 63) / 64 * 64);
    SESSION_CUDA(cudaMalloc(&s->ws_w, wfloats * 4 + align256(eco_mpnn_packed_bytes()) + 256));
    Carver io(nullptr);
    io.take<int8_t>((size_t)G * N * N); io.take<int8_t>((size_t)B * N); io.take<int8_t>((size_t)B * N);
    io.take<int32_t>(B); io.take<int32_t>(B); io.take<int32_t>(B);
    SESSION_CUDA(cudaMalloc(&s->ws_io, io.off));
    Carver io2(s->ws_io);
    s->d_Jdense = io2.take<int8_t>((size_t)G * N * N);
    s->d_spins = io2.take<int8_t>((size_t)B * N);
    s->d_best_spins = io2.take<int8_t>((size_t)B * N);
    s->d_gidx = io2.take<int32_t>(B);
    s->d_act = io2.take<int32_t>(B);
    s->d_best_cut = io2.take<int32_t>(B);

    int rc = eco_graphs_bind(&s->graphs, s->ws_graphs, G, N);
    if (!rc) rc = eco_env_bind(&s->env, s->ws_env, B, N, T, basin);
    if (rc) { eco_session_destroy(s); return rc; }

    // weights: host fp32 (state_dict order) -> device
    float* wd = (float*)s->ws_w;
    const float* ptrs[12];
    for (int i = 0; i < 12; ++i) {
        ptrs[i] = wd;
        SESSION_CUDA(cudaMemcpy(wd, weights_host[i], (size_t)kWeightCounts[i] * 4, cudaMemcpyHostToDevice));
        wd += (kWeightCounts[i] + 63) / 64 * 64;
    }
    s->w.w_init = ptrs[0]; s->w.w_edge = ptrs[1]; s->w.w_edge_feat = ptrs[2];
    for (int l = 0; l < 3; ++l) { s->w.w_msg[l] = ptrs[3 + 2 * l]; s->w.w_upd[l] = ptrs[4 + 2 * l]; }
    s->w.w_pool = ptrs[9]; s->w.w_read = ptrs[10]; s->w.b_read = ptrs[11];
    s->w.packed = nullptr;
    s->packed_buf = (void*)(((uintptr_t)wd + 255) & ~(uintptr_t)255);

    // tables: Zobrist keys (splitmix64), time-since-flip and immanency tables in the reference's fp64 arithmetic
    std::vector<uint64_t> zob((size_t)s->env.NP * 2);
    uint64_t x = 0x243F6A8885A308D3ull;
    for (auto& z : zob) {
        x += 0x9E3779B97F4A7C15ull;
        uint64_t v = x;
        v = (v ^ (v >> 30)) * 0xBF58476D1CE4E5B9ull;
        v = (v ^ (v >> 27)) * 0x94D049BB133111EBull;
        z = v ^ (v >> 31);
    }
    std::vector<float> tsf(T + 1), imm(T + 1);
    double acc = 0.0;
    const double inc = 1.0 / (double)T;
    tsf[0] = 0.f; imm[0] = 0.f;
    for (int k = 1; k <= T; ++k) {
        acc = acc + inc;                                            // spinsystem.py:493
        tsf[k] = (float)acc;
        const double v = ((double)(k - T) / (double)T) + 1.0;        // spinsystem.py:511
        imm[k] = (float)(v > 0.0 ? v : 0.0);
    }
    rc = eco_env_set_tables(&s->env, zob.data(), tsf.data(), imm.data(), nullptr);
    if (rc) { eco_session_destroy(s); return rc; }
    SESSION_CUDA(cudaDeviceSynchronize());
#undef SESSION_CUDA
    *out = s;
    return ECO_OK;
}

int eco_session_rollout(eco_session_t* s, const int8_t* J_host, const int32_t* gidx_host, const int8_t* spins_host,
                        int32_t policy, float norm_max, int32_t* best_cut_host, int8_t* best_spins_host,
                        void* stream) {
    ECO_CHECK_ARG(s && gidx_host && spins_host && best_cut_host, ECO_ERR_INVALID, "eco_session_rollout: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if (J_host) {  // NULL: keep the graphs of the previous call
        ECO_CUDA(cudaMemcpyAsync(s->d_Jdense, J_host, (size_t)s->G * s->N * s->N, cudaMemcpyHostToDevice, st));
        rc = eco_graphs_load_dev(&s->graphs, s->d_Jdense, stream);
        if (rc) return rc;
        // graph flags decide whether the tcgen05 path (couplings in {-1,0,1}) may be used
        std::vector<int32_t> stat((size_t)s->G * 4);
        ECO_CUDA(cudaMemcpyAsync(stat.data(), s->graphs.gstat, stat.size() * 4, cudaMemcpyDeviceToHost, st));
        ECO_CUDA(cudaStreamSynchronize(st));
        int flags = 0;
        for (int i = 0; i < s->G; ++i) flags |= stat[(size_t)i * 4 + 3];
        ECO_CHECK_ARG(!(flags & 6), ECO_ERR_INVALID,
                      "eco_session_rollout: a graph is not symmetric with zero diagonal, or has no non-zero degree");
        s->graphs.reserved = (flags & 1) ? 0 : ECO_GRAPHS_PM1;
        if (s->impl != ECO_MPNN_SIMT && !s->w.packed && eco_mpnn_packed_bytes() > 0) {
            rc = eco_mpnn_pack(&s->w, s->packed_buf, stream);
            if (rc) return rc;
            s->w.packed = s->packed_buf;
        }
    }
    ECO_CUDA(cudaMemcpyAsync(s->d_gidx, gidx_host, (size_t)s->B * 4, cudaMemcpyHostToDevice, st));
    ECO_CUDA(cudaMemcpyAsync(s->d_spins, spins_host, (size_t)s->B * s->N, cudaMemcpyHostToDevice, st));
    rc = eco_env_reset(&s->graphs, &s->env, s->d_gidx, s->d_spins, stream);
    if (rc) return rc;
    rc = eco_rollout(&s->graphs, &s->env, &s->w, s->T, policy, norm_max, s->d_act, s->ws_scratch, s->impl, nullptr,
                     nullptr, nullptr, stream);
    if (rc) return rc;
    rc = eco_env_results(&s->env, s->d_best_cut, best_spins_host ? s->d_best_spins : nullptr, nullptr, stream);
    if (rc) return rc;
    ECO_CUDA(cudaMemcpyAsync(best_cut_host, s->d_best_cut, (size_t)s->B * 4, cudaMemcpyDeviceToHost, st));
    if (best_spins_host)
        ECO_CUDA(cudaMemcpyAsync(best_spins_host, s->d_best_spins, (size_t)s->B * s->N, cudaMemcpyDeviceToHost, st));
    ECO_CUDA(cudaStreamSynchronize(st));
    return ECO_OK;
}

}  // extern "C"
