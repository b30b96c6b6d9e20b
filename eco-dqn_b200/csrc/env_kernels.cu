// Kernel family 1: the fused, batched environment step (and reset) for Max-Cut ECO-DQN episodes.
//
// Replaces (reference, file:line)
//   src/envs/spinsystem.py:355-559   SpinSystemBase.step      -> env_step_kernel
//   src/envs/spinsystem.py:183-259   SpinSystemBase.reset     -> env_reset_kernel
//   src/envs/spinsystem.py:283-330   _reset_state             -> env_reset_kernel
//   src/envs/spinsystem.py:561-574   get_observation          -> env_observation_kernel (rows 0..6 only)
//   src/envs/score_solver.py:377-419 MaximumCutUnbiasedScorer masks  -> O(N) incremental local fields
//   src/envs/utils.py:97-102         calculate_cut_changes    -> s_i * h_i with h updated from row a of J
//   src/envs/utils.py:438-464        HistoryBuffer            -> 128-bit Zobrist key + open-addressed set
//   src/agents/solver.py:105-131     Greedy.step              -> ECO_POLICY_GREEDY inside env_step_kernel
//
// One flip touches, per episode: row a of the int8 adjacency (N B), the spins (N B), the int16 local
// fields (2N B read + 2N B write), the uint16 last-flip steps (2N B), the best-diff bitmask, the three fp32
// per-vertex observable rows (12N B written) and a 96-byte scalar block: 20.25 N + 96 bytes, all in
// 8-vertex (8/16/32-byte) vector accesses, TPE lanes per episode.  The fp64 bookkeeping reproduces the
// reference's operation order (SURVEY.md appendix A.2) with explicit round-to-nearest intrinsics so the
// compiler cannot contract it.
#include "eco_common.cuh"
#include "env_step_device.cuh"

namespace eco {

namespace {

template <int TPE, bool BLOCK>
struct Grp {
    // BLOCK == false: TPE <= 32 lanes of one warp own an episode; BLOCK == true: the whole CTA (TPE threads).
    __device__ static int lane() { return BLOCK ? threadIdx.x : (threadIdx.x % TPE); }
    __device__ static long long episode() {
        return BLOCK ? (long long)blockIdx.x : ((long long)blockIdx.x * blockDim.x + threadIdx.x) / TPE;
    }
    __device__ static void sync() {
        if (BLOCK) __syncthreads(); else __syncwarp();
    }
    __device__ static int sum(int v, int* sm) {
        if constexpr (!BLOCK) {
            return group_sum<TPE>(v);
        } else {
            v = group_sum<32>(v);
            __syncthreads();
            if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
            __syncthreads();
            int t = 0;
            for (int w = 0; w < TPE / 32; ++w) t += sm[w];
            return t;
        }
    }
    __device__ static int maxv(int v, int* sm) {
        if constexpr (!BLOCK) {
            return group_max<TPE>(v);
        } else {
            v = group_max<32>(v);
            __syncthreads();
            if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
            __syncthreads();
            int t = INT_MIN;
            for (int w = 0; w < TPE / 32; ++w) t = max(t, sm[w]);
            return t;
        }
    }
    __device__ static int bcast(int v, int* sm) {  // value of lane 0
        if constexpr (!BLOCK) {
            return __shfl_sync(0xffffffffu, v, 0, TPE);
        } else {
            __syncthreads();
            if (threadIdx.x == 0) sm[0] = v;
            __syncthreads();
            return sm[0];
        }
    }
};

// ------------------------------------------------------------------------------------------------ step
template <int TPE, bool BLOCK>
__global__ void __launch_bounds__(BLOCK ? TPE : 128)
env_step_kernel(const eco_graphs_t g, const eco_env_t env, const int policy, const int32_t* __restrict__ actions,
                double* __restrict__ reward_out, uint8_t* __restrict__ done_out, int32_t* __restrict__ hist_a,
                double* __restrict__ hist_r, double* __restrict__ hist_s) {
    using G = Grp<TPE, BLOCK>;
    __shared__ int sm[8];
    const int lane = G::lane();
    long long b = G::episode();
    const bool in_range = b < env.B;
    if (!in_range) b = env.B - 1;  // keep every lane alive for the group shuffles
    const int N = env.N, NP = env.NP, NCH = NP / 8;
    const int sgn = (g.reserved & ECO_GRAPHS_MIN_CUT) ? -1 : 1;             // Min-Cut: every mask is the negated cut change
    const bool irreversible = (env.reserved & ECO_ENV_IRREVERSIBLE) != 0;   // S2V-DQN: spins are flipped at most once
    const bool dense_reward = (env.reserved & ECO_ENV_DENSE_REWARD) != 0;   // reward = normalised score change

    eco_episode_t* ep = env.ep + b;
    const int flags = ep->flags;
    bool active = in_range && !(flags & (FLAG_DONE | FLAG_STOPPED));
    const int step_new = ep->step + 1;
    if (active && step_new > env.T) active = false;  // reference raises here (spinsystem.py:365-367)

    const int gi = env.graph_idx[b];
    const int8_t* Jg = g.J + (size_t)gi * NP * NP;
    int8_t* spins = env.spins + (size_t)b * NP;
    int16_t* hf = env.hfield + (size_t)b * NP;
    uint16_t* lf = env.last_flip + (size_t)b * NP;
    const double mlr = g.gscal[(size_t)gi * 4 + 0];

    // ---- choose the action ----------------------------------------------------------------------------
    int a;
    if (policy == ECO_POLICY_GREEDY) {
        // argmax_i s_i h_i, first maximal index (numpy argmax, solver.py:116)
        int best = INT_MIN;
        for (int c = lane; c < NCH; c += TPE) {
            V8s s; V8h h;
            s.v = *reinterpret_cast<const uint2*>(spins + c * 8);
            h.v = *reinterpret_cast<const uint4*>(hf + c * 8);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int i = c * 8 + k;
                // key = (gain + 32768) : (65535 - i) as an unsigned pair, biased so that signed max orders it
                if (i < N && (!irreversible || s.b[k] < 0))      // solver.py:116-121: irreversible -> only spins still at -1
                    best = max(best, (int)((((uint32_t)(sgn * s.b[k] * h.h[k] + 32768) << 16) | (uint32_t)(0xFFFF - i)) ^ 0x80000000u));
            }
        }
        best = G::maxv(best, sm);
        const uint32_t ukey = (uint32_t)best ^ 0x80000000u;
        a = 0xFFFF - (int)(ukey & 0xFFFFu);
        if (active && (best == INT_MIN || ((int)(ukey >> 16) - 32768) < 0)) {  // solver.py:124: stop only if the best gain is < 0
            active = false;
            if (lane == 0) ep->flags = flags | FLAG_STOPPED;
        }
    } else {
        a = actions[b];
    }
    if (a < 0 || a >= N) { a = 0; active = false; }

    const int s_a_old = spins[a];
    const int h_a_old = hf[a];
    const int s_a_new = -s_a_old;
    const uint32_t old_word = env.diff_bits[(size_t)b * env.NW + (a >> 5)];
    G::sync();  // everyone has read the pre-flip values before anyone writes

    // ---- O(N) local-field update + per-vertex observables ------------------------------------------
    int nimp = 0, nneg = 0;
    if (active) {
        const int8_t* Jrow = Jg + (size_t)a * NP;
        float* x0 = env.xn + (size_t)b * 3 * NP;
        float* x1 = x0 + NP;
        float* x2 = x1 + NP;
        for (int c = lane; c < NCH; c += TPE) {
            V8s s, j; V8h h; V8u l;
            s.v = *reinterpret_cast<const uint2*>(spins + c * 8);
            j.v = *reinterpret_cast<const uint2*>(Jrow + c * 8);
            h.v = *reinterpret_cast<const uint4*>(hf + c * 8);
            l.v = *reinterpret_cast<const uint4*>(lf + c * 8);
            float f0[8], f1[8], f2[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int i = c * 8 + k;
                int si = s.b[k];
                if (i == a) { si = s_a_new; s.b[k] = (int8_t)si; l.h[k] = (uint16_t)step_new; }
                const int hi = h.h[k] + 2 * j.b[k] * s_a_new;  // J_aa == 0, so h_a is unchanged
                h.h[k] = (int16_t)hi;
                const int gain = sgn * si * hi;
                nimp += gain > 0;
                nneg += (i < N && si < 0);
                f0[k] = (float)si;
                f1[k] = feat_gain(gain, mlr);
                f2[k] = env.tsf_tab[step_new - l.h[k]];
            }
            *reinterpret_cast<uint4*>(hf + c * 8) = h.v;
            if ((a >> 3) == c) {
                *reinterpret_cast<uint2*>(spins + c * 8) = s.v;
                *reinterpret_cast<uint4*>(lf + c * 8) = l.v;
            }
            st_f32x8(x0 + c * 8, f0);             // one 32-byte sector per lane and row: 256-bit stores
            st_f32x8(x1 + c * 8, f1);
            st_f32x8(x2 + c * 8, f2);
        }
    }
    nimp = G::sum(nimp, sm);
    if (irreversible) nneg = G::sum(nneg, sm);          // spins that can still be flipped (spinsystem.py:552-556)

    // ---- scalar bookkeeping, lane 0, in the reference's fp64 operation order (appendix A.2) ---------
    int new_best = 0;
    if (lane == 0 && active) {
        const double qn = g.gscal[(size_t)gi * 4 + 1];
        const int dcut = s_a_old * h_a_old;                             // change of the cut value
        const int delta = sgn * dcut;                                   // spinsystem.py:393 (score mask at the action)
        // the reference multiplies in fp64: a zero field times a spin of -1 is -0.0 (visible in the dense reward);
        // the Min-Cut scorer negates it once more
        const double delta_d = (delta == 0 && (s_a_old < 0) == (sgn > 0)) ? -0.0 : (double)delta;
        const double delta_n = __ddiv_rn(delta_d, qn);                  // :394
        const double score = __dadd_rn(ep->score, (double)delta);       // :399
        const double nscore = __dadd_rn(ep->nscore, delta_n);           // :400
        const double best_score = ep->best_score, best_nscore = ep->best_nscore;
        const int cut = ep->cut + dcut;
        double rew = 0.0;
        if (dense_reward) rew = delta_n;                                // :435-436 (DENSE, normalised)
        else if (score > best_score) rew = __dsub_rn(nscore, best_nscore);   // :418-424 (BLS, normalised)

        uint64_t k0 = ep->key[0] ^ env.zobrist[2 * a], k1 = ep->key[1] ^ env.zobrist[2 * a + 1];
        int n_visited = ep->n_visited;
        if (env.use_basin) {                                            // :443-457
            const uint64_t e0 = k0 ^ VISITED_SALT0, e1 = k1 ^ VISITED_SALT1;
            uint64_t* tab = env.visited + (size_t)b * env.HCAP * 2;
            uint32_t slot = (uint32_t)(k0 ^ (k0 >> 29)) & (env.HCAP - 1);
            bool is_new = false;
            for (int probe = 0; probe < env.HCAP; ++probe) {
                const uint64_t t0 = tab[2 * slot], t1 = tab[2 * slot + 1];
                if (t0 == 0 && t1 == 0) { tab[2 * slot] = e0; tab[2 * slot + 1] = e1; is_new = true; ++n_visited; break; }
                if (t0 == e0 && t1 == e1) break;
                slot = (slot + 1) & (env.HCAP - 1);
            }
            if (nimp == 0 && is_new) rew = __dadd_rn(rew, env.basin_reward);
        }
        int dist = ep->dist + (((old_word >> (a & 31)) & 1u) ? -1 : 1);
        int best_cut = ep->best_cut;
        double nbs = best_score, nbn = best_nscore;
        if (score > best_score) {                                       // :459-463
            nbs = score; nbn = nscore; best_cut = cut; dist = 0; new_best = 1;
        }
        const int done = step_new == env.T || (irreversible && nneg == 0);   // :541-544, :552-556
        ep->step = step_new; ep->cut = cut; ep->best_cut = best_cut; ep->dist = dist;
        ep->n_improving = nimp; ep->flags = flags | (done ? FLAG_DONE : 0); ep->n_visited = n_visited;
        ep->score = score; ep->nscore = nscore; ep->best_score = nbs; ep->best_nscore = nbn;
        ep->key[0] = k0; ep->key[1] = k1;
        ep->total_reward = __dadd_rn(ep->total_reward, rew); ep->last_reward = rew;

        // global observables rows 3..6 (spinsystem.py:509-527), fp64 then the driver's fp32 cast
        float4 xg;
        xg.x = (float)__ddiv_rn(fabs(__dsub_rn(score, nbs)), mlr);
        xg.y = (float)dist;
        xg.z = (float)__ddiv_rn((double)nimp, (double)N);
        xg.w = env.imm_tab[step_new];
        *reinterpret_cast<float4*>(env.xg + (size_t)b * 4) = xg;

        if (reward_out) reward_out[b] = rew;
        if (done_out) done_out[b] = (uint8_t)done;
        const size_t hidx = (size_t)b * env.T + (step_new - 1);
        if (hist_a) hist_a[hidx] = a;
        if (hist_r) hist_r[hidx] = rew;
        if (hist_s) hist_s[hidx] = score;
    } else if (lane == 0 && in_range) {
        if (reward_out) reward_out[b] = 0.0;
        if (done_out) done_out[b] = 1;
    }
    new_best = G::bcast(new_best, sm);

    // ---- best-diff bitmask: toggle bit a, or clear everything when this state is the new best --------
    if (active) {
        uint32_t* diff = env.diff_bits + (size_t)b * env.NW;
        for (int w = lane; w < env.NW; w += TPE) {
            if (new_best) diff[w] = 0u;
            else if (w == (a >> 5)) diff[w] = old_word ^ (1u << (a & 31));
        }
    }
}

// ------------------------------------------------------------------------------------------------ step, N <= 256
// Latency-optimised variant for the common case (one sub-warp group per episode, at most one 8-vertex chunk per lane).
// Same arithmetic as env_step_kernel; the difference is the load schedule: everything that does not depend on the
// action is requested first (scalar block, graph index, the lane's spins / fields / last-flip chunk), then everything
// that depends on it (adjacency row chunk, Zobrist key, scorer constants), then the visited-set slot -- three
// dependent memory round trips per step instead of six -- and the flipped vertex's old spin / field come from a
// shuffle instead of extra loads.  Few registers, so many episodes are in flight per SM.
template <int TPE>
__global__ void __launch_bounds__(128, 8)
env_step_sw_kernel(const eco_graphs_t g, const eco_env_t env, const int policy, const int32_t* __restrict__ actions,
                   double* __restrict__ reward_out, uint8_t* __restrict__ done_out, int32_t* __restrict__ hist_a,
                   double* __restrict__ hist_r, double* __restrict__ hist_s) {
    const int lane = threadIdx.x % TPE;
    long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / TPE;
    const bool in_range = b < env.B;
    if (!in_range) b = env.B - 1;
    env_step_group<TPE>(g, env, b, lane, in_range, policy, policy == ECO_POLICY_GREEDY ? 0 : actions[b], reward_out, done_out,
                        hist_a, hist_r, hist_s);
}

// ------------------------------------------------------------------------------------------------ step, 128 < N <= 256
// Staged variant: persistent warps, two episode streams per warp (one per half-warp), a 3-deep shared-memory ring per
// stream filled with 16-byte asynchronous copies (cp.async, one commit group per episode).  While episode e is processed
// from shared memory, the copies of episode e+2 -- spins, local fields, last-flip steps, the scalar block and row `a` of
// its adjacency -- are already in flight, so no global-load latency sits on the per-episode path.
// Same arithmetic as env_step_kernel (bit-exact; the fp64 bookkeeping is bls_step_scalars); caller-supplied actions only
// (the greedy policy needs the fields to pick the row).
namespace tma {
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
}  // namespace tma

constexpr int TMA_TSF_MAX = 1024;   // time-since-flip table entries kept in shared memory (T + 1 <= this, else read from global)
constexpr int TMA_WARPS = 4;
// Two episodes per warp: each half-warp (16 lanes, 16 vertices per lane in four 4-vertex quads) runs its own episode
// stream with its own ring, so the scalar bookkeeping of two episodes -- done by lanes 0 and 16 -- issues ONCE.
// TPE lanes per episode stream (16 or 8): 32 / TPE streams per warp.  The ring lives in dynamic shared memory, one stage =
// [spins NP | h 2NP | last_flip 2NP | J row NP | scalar block 96] bytes.
// FAST: the rollout configuration proper -- couplings in {-1,0,1} and T + 1 <= TMA_TSF_MAX -- with a vertex loop stripped to
// what it has to do (end of round 2: the general loop spent ~35 instructions per vertex, a third of them on `is this the
// flipped vertex?`, 64-bit address arithmetic for the per-graph gain table and generic loads of the time-since-flip table):
// the flip is applied to the packed words of the one quad that holds it BEFORE the loop, row 1 is gain / mlr by reciprocal
// and two FMAs (small_div: bit-identical to the table, no memory access), the time-since-flip table is read with
// shared-memory loads, every field is extracted with one PRMT.
template <int TPE, int STAGES, bool FAST>
__global__ void __launch_bounds__(TMA_WARPS * 32, 4)
env_step_ring_kernel(const eco_graphs_t g, const eco_env_t env, const int32_t* __restrict__ actions,
                    double* __restrict__ reward_out, uint8_t* __restrict__ done_out, int32_t* __restrict__ hist_a,
                    double* __restrict__ hist_r, double* __restrict__ hist_s) {
    extern __shared__ __align__(16) unsigned char ring_raw[];
    constexpr int SPW = 32 / TPE, NSTREAMS = TMA_WARPS * SPW;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int l16 = lane % TPE, stream = warp * SPW + lane / TPE;
    const long long sglobal = (long long)blockIdx.x * NSTREAMS + stream;
    const long long stotal = (long long)gridDim.x * NSTREAMS;
    const int N = env.N, NP = env.NP, NCH = NP >> 3;
    const int stage_bytes = 6 * NP + (int)sizeof(eco_episode_t);
    unsigned char* my_ring = ring_raw + (size_t)stream * STAGES * stage_bytes;
    const bool use_tab = (g.reserved & ECO_GRAPHS_PM1) != 0;
    // the two tables every episode indexes with data-dependent addresses live in shared memory (L2 latency otherwise
    // sits between the loads and the first feature store / the visited-set probe)
    __shared__ __align__(16) uint64_t s_zob[2 * 256];
    __shared__ float s_tsf[TMA_TSF_MAX];
    for (int i = threadIdx.x; i < 2 * NP; i += blockDim.x) s_zob[i] = env.zobrist[i];
    const bool tsf_shared = env.T + 1 <= TMA_TSF_MAX;
    if (tsf_shared)
        for (int i = threadIdx.x; i <= env.T; i += blockDim.x) s_tsf[i] = env.tsf_tab[i];
    const float* tsf = tsf_shared ? s_tsf : env.tsf_tab;
    __syncthreads();

    // all 16 lanes of the stream: 16-byte asynchronous copies (cp.async) of episode b into stage st, one commit group.
    // (Five small bulk copies per episode kept the SM's single TMA unit busy ~70 cycles each -- that, not HBM or the
    //  issue slots, bounded the first version of this kernel.)
    const int p1 = NP >> 4, p2 = 3 * p1, p3 = 5 * p1, p4 = 6 * p1, p5 = p4 + (int)(sizeof(eco_episode_t) >> 4);
    auto issue = [&](long long b, int a, int gi, int st, bool go) {
        char* S = (char*)my_ring + (size_t)st * stage_bytes;      // the stage is laid out in copy order
        if (go) {
            for (int p = l16; p < p5; p += TPE) {
                const char* src;
                if (p < p1) src = (const char*)(env.spins + (size_t)b * NP) + 16 * p;
                else if (p < p2) src = (const char*)(env.hfield + (size_t)b * NP) + 16 * (p - p1);
                else if (p < p3) src = (const char*)(env.last_flip + (size_t)b * NP) + 16 * (p - p2);
                else if (p < p4) src = (const char*)(g.J + ((size_t)gi * NP + a) * NP) + 16 * (p - p3);
                else src = (const char*)(env.ep + b) + 16 * (p - p4);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(tma::smem_addr(S + 16 * p)), "l"(src) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");     // (an empty group keeps the group count uniform)
    };
    auto clamp_action = [&](int a) { return (a < 0 || a >= N) ? 0 : a; };

    // prologue: the first D = TMA_STAGES - 1 episodes of this stream in flight; action / graph of the next one in registers
    constexpr int D = STAGES - 1;
    const long long b0 = sglobal;
    int an[D + 1], gn[D + 1];       // action / graph index of episodes b, b + stotal, ..., b + D * stotal
    double mlrn[D];                 // max local reward of the graphs of episodes b, ..., b + (D - 1) * stotal: requested one
                                    // iteration after the graph index arrived, consumed D iterations later (the dependent
                                    // load graph_idx -> gscal sat on the critical path: 27 % of the kernel's stall samples)
#pragma unroll
    for (int k = 0; k <= D; ++k) {
        an[k] = 0; gn[k] = 0;
        if (b0 + k * stotal < env.B) { an[k] = actions[b0 + k * stotal]; gn[k] = env.graph_idx[b0 + k * stotal]; }
    }
#pragma unroll
    for (int k = 0; k < D; ++k) mlrn[k] = g.gscal[(size_t)gn[k] * 4 + 0];
    // word of the best-configuration bitmask that holds the flipped vertex, also requested one iteration ahead (FAST)
    uint32_t old_word_next = 0;
    if (FAST && b0 < env.B) old_word_next = env.diff_bits[(size_t)b0 * env.NW + (clamp_action(an[0]) >> 5)];
#pragma unroll
    for (int k = 0; k < D; ++k) issue(b0 + k * stotal, clamp_action(an[k]), gn[k], k, b0 + k * stotal < env.B);
    int st = 0;

    for (long long b = b0; __any_sync(0xffffffffu, b < env.B); b += stotal) {
        const bool valid = b < env.B;                 // (the two streams of a warp may differ by one episode at the end)
        const unsigned char* Sb = my_ring + (size_t)st * stage_bytes;
        const int8_t* S_spins = reinterpret_cast<const int8_t*>(Sb);
        const int16_t* S_h = reinterpret_cast<const int16_t*>(Sb + NP);
        const uint16_t* S_lf = reinterpret_cast<const uint16_t*>(Sb + 3 * NP);
        const int8_t* S_jrow = reinterpret_cast<const int8_t*>(Sb + 5 * NP);
        const eco_episode_t* S_ep = reinterpret_cast<const eco_episode_t*>(Sb + 6 * NP);
        // ---- keep the pipeline full: bulk copies of episode b + D*stotal, action / graph of b + (D+1)*stotal ----
        const long long bD = b + D * stotal, bN = b + (D + 1) * stotal;
        int a_new = 0, gi_new = 0;
        if (bN < env.B) { a_new = actions[bN]; gi_new = env.graph_idx[bN]; }
        const double mlr_new = g.gscal[(size_t)gn[D] * 4 + 0];
        const uint32_t old_word_cur = old_word_next;
        if (FAST && b + stotal < env.B) old_word_next = env.diff_bits[(size_t)(b + stotal) * env.NW + (clamp_action(an[1]) >> 5)];
        issue(bD, clamp_action(an[D]), gn[D], (st + D) % STAGES, bD < env.B);
        const int a_cur = an[0], gi_cur = gn[0];

        asm volatile("cp.async.wait_group %0;" ::"n"(D) : "memory");   // this episode's group (D newer ones may be in flight)
        __syncwarp();                                                  // ... of every lane of the stream

        // ---- episode b from shared memory ---------------------------------------------------------------------
        const int gi = gi_cur;
        int a = a_cur;
        int4 e0 = make_int4(0, 0, 0, 0), e1 = make_int4(0, FLAG_DONE, 0, 0);
        if (valid) {
            e0 = *reinterpret_cast<const int4*>(S_ep);
            e1 = *(reinterpret_cast<const int4*>(S_ep) + 1);
        }
        const int flags = e1.y;
        const int step_new = e0.x + 1;
        bool active = valid && !(flags & (FLAG_DONE | FLAG_STOPPED)) && step_new <= env.T;
        if (a < 0 || a >= N) { a = 0; active = false; }
        const int s_a_old = valid ? S_spins[a] : 1;
        const int h_a_old = valid ? S_h[a] : 0;
        const int s_a_new = -s_a_old;
        const int delta = s_a_old * h_a_old;                            // spinsystem.py:393
        const double mlr = mlrn[0];
        const float* gtab = g.gain_tab + (size_t)gi * tab_stride(NP) + NP;

        // lanes 0 / 16: scalar state, dependent lookups requested now, used after the vertex loop
        double sc[4] = {0, 0, 0, 0}, total_reward = 0, delta_n = 0, qn = 1.0;
        ulonglong2 key = make_ulonglong2(0, 0), zob = make_ulonglong2(0, 0);
        uint32_t old_word = 0;
        if (l16 == 0 && valid) {
            sc[0] = S_ep->score; sc[1] = S_ep->nscore; sc[2] = S_ep->best_score; sc[3] = S_ep->best_nscore;
            key = make_ulonglong2(S_ep->key[0], S_ep->key[1]);
            total_reward = S_ep->total_reward;
            zob = *reinterpret_cast<const ulonglong2*>(s_zob + 2 * a);
            old_word = FAST ? old_word_cur : env.diff_bits[(size_t)b * env.NW + (a >> 5)];
            // (the normalised score change stays a table gather: an inline fp64 division on this chain costs 160 us per launch)
            if (use_tab) delta_n = __ldg(g.dn_tab + (size_t)gi * tab_stride(NP) + NP + delta);
            else qn = g.gscal[(size_t)gi * 4 + 1];
        }
        const uint64_t k0 = key.x ^ zob.x, k1 = key.y ^ zob.y;
        uint64_t* tab = env.visited + (size_t)(valid ? b : 0) * env.HCAP * 2;
        uint32_t slot = (uint32_t)(k0 ^ (k0 >> 29)) & (env.HCAP - 1);
        ulonglong2 tv = make_ulonglong2(0, 0);
        if (l16 == 0 && active && env.use_basin) tv = *reinterpret_cast<const ulonglong2*>(tab + 2 * slot);

        int nimp = 0;
        // FAST: gd.ok always holds (couplings in {-1,0,1} give |mlr| <= 255; graph_prepare_kernel sets mlr = 1 when no row sum
        // is non-zero), so FAST never reaches the general loop below.  It stays compiled in on purpose: without it ptxas
        // rebuilds the shared-memory window base in every pass of the FAST loop, 3 us (1.3 %) per launch at B = 262 144.
        const SmallDiv gd = small_div_setup(mlr, FAST);
        // Vertex loop: a lane takes FOUR consecutive vertices per pass (quad qd = l16 + TPE * pass), so the 16 lanes of a stream
        // write 256 contiguous bytes of every feature row with one store instruction -- whole 32-byte sectors.  (With eight
        // vertices per lane the two float4 stores of a row each filled HALF of every sector they touched: twice the write
        // transactions for 58 % of the kernel's bytes; 309 -> 241 us per launch at B = 262 144, bit-identical.)
        const int NQ = NP >> 2, qa = a >> 2, ka = a & 3;
        if (FAST && active && gd.ok) {
            const int two_sa = 2 * s_a_new;
            const float* tsf_now = s_tsf + step_new;       // time-since-flip of vertex k: tsf_now[-last_flip[k]]
#pragma unroll
            for (int pass = 0; pass < 64 / TPE; ++pass) {
                const int qd = l16 + TPE * pass;
                if (qd >= NQ) continue;
                uint32_t sw = *reinterpret_cast<const uint32_t*>(S_spins + qd * 4);
                const uint32_t jw = *reinterpret_cast<const uint32_t*>(S_jrow + qd * 4);
                const uint2 hw = *reinterpret_cast<const uint2*>(S_h + qd * 4);
                uint2 lw = *reinterpret_cast<const uint2*>(S_lf + qd * 4);
                if (qd == qa) {                            // the flipped vertex: new spin (a +-1 byte negated), last-flip step
                    sw ^= 0xFEu << (8 * ka);
                    const uint32_t sh = 16 * (ka & 1), keep = ~(0xFFFFu << sh), val = ((uint32_t)step_new & 0xFFFFu) << sh;
                    if ((ka >> 1) == 0) lw.x = (lw.x & keep) | val;
                    else lw.y = (lw.y & keep) | val;
                }
                const uint32_t hws[2] = {hw.x, hw.y}, lws[2] = {lw.x, lw.y};
                float* x0 = env.xn + (size_t)b * 3 * NP + qd * 4;
                float f0[4], f1[4], f2[4];
                int hv[4];
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const int si = sx8(sw, kk);
                    const int hi = sx16(hws[kk >> 1], kk & 1) + sx8(jw, kk) * two_sa;
                    hv[kk] = hi;
                    const int gain = si * hi;
                    nimp += gain > 0;
                    f0[kk] = (float)si;
                    f1[kk] = small_div((float)gain, gd);
                    f2[kk] = tsf_now[-zx16(lws[kk >> 1], kk & 1)];
                }
                *reinterpret_cast<float4*>(x0) = make_float4(f0[0], f0[1], f0[2], f0[3]);
                *reinterpret_cast<float4*>(x0 + NP) = make_float4(f1[0], f1[1], f1[2], f1[3]);
                *reinterpret_cast<float4*>(x0 + 2 * NP) = make_float4(f2[0], f2[1], f2[2], f2[3]);
                *reinterpret_cast<uint2*>(env.hfield + (size_t)b * NP + qd * 4) =
                    make_uint2(__byte_perm((uint32_t)hv[0], (uint32_t)hv[1], 0x5410), __byte_perm((uint32_t)hv[2], (uint32_t)hv[3], 0x5410));
                if (qd == qa) {
                    *reinterpret_cast<uint32_t*>(env.spins + (size_t)b * NP + qd * 4) = sw;
                    *reinterpret_cast<uint2*>(env.last_flip + (size_t)b * NP + qd * 4) = lw;
                }
            }
        } else if (active) {
#pragma unroll
            for (int pass = 0; pass < 64 / TPE; ++pass) {  // NP <= 256: at most 64 quads
                const int qd = l16 + TPE * pass;
                if (qd >= NQ) continue;
                V4s sv, jv; V4h hv; V4u lv;
                sv.v = *reinterpret_cast<const uint32_t*>(S_spins + qd * 4);
                jv.v = *reinterpret_cast<const uint32_t*>(S_jrow + qd * 4);
                hv.v = *reinterpret_cast<const uint2*>(S_h + qd * 4);
                lv.v = *reinterpret_cast<const uint2*>(S_lf + qd * 4);
                float* x0 = env.xn + (size_t)b * 3 * NP + qd * 4;
                float f0[4], f1[4], f2[4];
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    int si = sv.b[kk];
                    if (qd == qa && kk == ka) { si = s_a_new; sv.b[kk] = (int8_t)si; lv.h[kk] = (uint16_t)step_new; }
                    const int hi = hv.h[kk] + 2 * jv.b[kk] * s_a_new;
                    hv.h[kk] = (int16_t)hi;
                    const int gain = si * hi;
                    nimp += gain > 0;
                    f0[kk] = (float)si;
                    f1[kk] = use_tab ? __ldg(gtab + gain) : feat_gain(gain, mlr);
                    f2[kk] = tsf[step_new - lv.h[kk]];
                }
                *reinterpret_cast<float4*>(x0) = make_float4(f0[0], f0[1], f0[2], f0[3]);
                *reinterpret_cast<float4*>(x0 + NP) = make_float4(f1[0], f1[1], f1[2], f1[3]);
                *reinterpret_cast<float4*>(x0 + 2 * NP) = make_float4(f2[0], f2[1], f2[2], f2[3]);
                *reinterpret_cast<uint2*>(env.hfield + (size_t)b * NP + qd * 4) = hv.v;
                if (qd == qa) {
                    *reinterpret_cast<uint32_t*>(env.spins + (size_t)b * NP + qd * 4) = sv.v;
                    *reinterpret_cast<uint2*>(env.last_flip + (size_t)b * NP + qd * 4) = lv.v;
                }
            }
        }
        nimp = group_sum<TPE>(nimp);

        int new_best = 0;
        eco_episode_t* ep = env.ep + (valid ? b : 0);
        if (l16 == 0 && active) {
            if (!use_tab) delta_n = __ddiv_rn((double)delta, qn);           // :394
            const int cut = e0.y + delta;
            const StepScalars r = bls_step_scalars(env, sc, (double)delta, delta_n, nimp, e1.z, tab, slot, tv, k0, k1);
            const double score = r.score, nscore = r.nscore, rew = r.rew;
            int dist = e0.w + (((old_word >> (a & 31)) & 1u) ? -1 : 1);
            int best_cut = e0.z;
            double nbs = sc[2], nbn = sc[3];
            // (a rarely taken branch instead of r.best_score / r.best_nscore: compiled as selects, this tail made the general
            // instantiation 0.8 % slower on a B200)
            if (__builtin_expect(r.new_best, 0)) { nbs = score; nbn = nscore; best_cut = cut; dist = 0; new_best = 1; }
            const int done = step_new == env.T;                             // :541-544
            int4* epw = reinterpret_cast<int4*>(ep);
            epw[0] = make_int4(step_new, cut, best_cut, dist);
            epw[1] = make_int4(nimp, flags | (done ? FLAG_DONE : 0), r.n_visited, 0);
            *reinterpret_cast<double2*>(&ep->score) = make_double2(score, nscore);
            *reinterpret_cast<double2*>(&ep->best_score) = make_double2(nbs, nbn);
            *reinterpret_cast<ulonglong2*>(&ep->key[0]) = make_ulonglong2(k0, k1);
            *reinterpret_cast<double2*>(&ep->total_reward) = make_double2(__dadd_rn(total_reward, rew), rew);
            float4 xg;                                                      // rows 3..6 (spinsystem.py:509-527)
            const double gap = fabs(__dsub_rn(score, nbs));                 // integer-valued for integer couplings
            xg.x = (gd.ok && gap <= 65536.0) ? small_div((float)gap, gd) : (float)__ddiv_rn(gap, mlr);
            xg.y = (float)dist;
            xg.z = __ldg(env.frac_tab + nimp);
            xg.w = __ldg(env.imm_tab + step_new);
            *reinterpret_cast<float4*>(env.xg + (size_t)b * 4) = xg;
            if (reward_out) reward_out[b] = rew;
            if (done_out) done_out[b] = (uint8_t)done;
            const size_t hidx = (size_t)b * env.T + (step_new - 1);
            if (hist_a) hist_a[hidx] = a;
            if (hist_r) hist_r[hidx] = rew;
            if (hist_s) hist_s[hidx] = score;
            if (!new_best) env.diff_bits[(size_t)b * env.NW + (a >> 5)] = old_word ^ (1u << (a & 31));
        } else if (l16 == 0 && valid) {
            if (reward_out) reward_out[b] = 0.0;
            if (done_out) done_out[b] = 1;
        }
        new_best = __shfl_sync(0xffffffffu, new_best, 0, TPE);
        if (new_best && active && l16 < env.NW) env.diff_bits[(size_t)b * env.NW + l16] = 0u;

        __syncwarp();                 // every lane is done with this stage before it is refilled two iterations on
        st = (st + 1) % STAGES;
#pragma unroll
        for (int k = 0; k < D; ++k) { an[k] = an[k + 1]; gn[k] = gn[k + 1]; }
        an[D] = a_new; gn[D] = gi_new;
#pragma unroll
        for (int k = 0; k + 1 < D; ++k) mlrn[k] = mlrn[k + 1];
        mlrn[D - 1] = mlr_new;
    }
}

// ------------------------------------------------------------------------------------------------ reset
template <int TPE, bool BLOCK>
__global__ void __launch_bounds__(BLOCK ? TPE : 128)
env_reset_kernel(const eco_graphs_t g, const eco_env_t env, const int32_t* __restrict__ graph_idx,
                 const int8_t* __restrict__ init_spins) {
    using G = Grp<TPE, BLOCK>;
    __shared__ int sm[8];
    const int lane = G::lane();
    long long b = G::episode();
    const bool in_range = b < env.B;
    if (!in_range) b = env.B - 1;
    const int N = env.N, NP = env.NP;
    const int gi = graph_idx[b];
    const int8_t* Jg = g.J + (size_t)gi * NP * NP;
    int8_t* spins = env.spins + (size_t)b * NP;
    int16_t* hf = env.hfield + (size_t)b * NP;
    const double mlr = g.gscal[(size_t)gi * 4 + 0];

    if (in_range) {
        for (int i = lane; i < NP; i += TPE) {
            spins[i] = i < N ? init_spins[(size_t)b * N + i] : (int8_t)0;
            env.last_flip[(size_t)b * NP + i] = 0;
        }
        for (int w = lane; w < env.NW; w += TPE) env.diff_bits[(size_t)b * env.NW + w] = 0u;
        if (lane == 0) env.graph_idx[b] = gi;
    }
    G::sync();
    __threadfence_block();

    const bool min_cut = (g.reserved & ECO_GRAPHS_MIN_CUT) != 0;
    int nimp = 0, ssh = 0;
    if (in_range) {
        float* x0 = env.xn + (size_t)b * 3 * NP;
        const int* sw = reinterpret_cast<const int*>(spins);
        for (int i = lane; i < NP; i += TPE) {
            const int* jw = reinterpret_cast<const int*>(Jg + (size_t)i * NP);
            int acc = 0;
            for (int w = 0; w < NP / 4; ++w) acc = __dp4a(jw[w], sw[w], acc);  // h_i = sum_j J_ij s_j
            hf[i] = (int16_t)acc;
            const int si = spins[i];
            ssh += si * acc;
            const int gain = min_cut ? -(si * acc) : si * acc;         // score mask (score_solver.py:409-413 / :486-490)
            nimp += gain > 0;
            x0[i] = (float)si;                                         // spinsystem.py:294/299
            x0[NP + i] = i < N ? feat_gain(gain, mlr) : 0.f;           // :311-312
            x0[2 * NP + i] = 0.f;
        }
    }
    nimp = G::sum(nimp, sm);
    ssh = G::sum(ssh, sm);
    if (lane == 0 && in_range) {
        const double qn = g.gscal[(size_t)gi * 4 + 1], lb = g.gscal[(size_t)gi * 4 + 2];
        const int sumJ = (int)g.gscal[(size_t)gi * 4 + 3];
        const int cut = (sumJ - ssh) / 4;                              // utils.py:90-94, exact in integers
        // quality: cut + |min(0, lb)| (score_solver.py:196-200) or, minimising, max(0, qn) - cut (:219-222)
        const double score = min_cut ? __dsub_rn(fmax(0.0, qn), (double)cut) : __dadd_rn((double)cut, fabs(fmin(0.0, lb)));
        const double nscore = __ddiv_rn(score, qn);                    // :190-194
        eco_episode_t e;
        e.step = 0; e.cut = cut; e.best_cut = cut; e.dist = 0; e.n_improving = nimp; e.flags = 0;
        e.n_visited = 0; e.reserved = 0;
        e.score = score; e.nscore = nscore; e.best_score = score; e.best_nscore = nscore;
        e.key[0] = 0; e.key[1] = 0; e.total_reward = 0.0; e.last_reward = 0.0;
        env.ep[b] = e;
        float4 xg = make_float4(0.f, 0.f, (float)__ddiv_rn((double)nimp, (double)N), 0.f);  // :321-322
        *reinterpret_cast<float4*>(env.xg + (size_t)b * 4) = xg;
    }
}

// ------------------------------------------------------------------------------------------------ views
__global__ void env_observation_kernel(const eco_env_t env, float* __restrict__ obs7) {
    const size_t total = (size_t)env.B * 7 * env.N;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        const int i = idx % env.N;
        const int r = (idx / env.N) % 7;
        const size_t b = idx / ((size_t)7 * env.N);
        obs7[idx] = r < 3 ? env.xn[(b * 3 + r) * env.NP + i] : env.xg[b * 4 + (r - 3)];
    }
}

__global__ void env_results_kernel(const eco_env_t env, int32_t* __restrict__ best_cut,
                                   int8_t* __restrict__ best_spins, int32_t* __restrict__ steps) {
    const size_t total = (size_t)env.B * env.N;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total;
         idx += (size_t)gridDim.x * blockDim.x) {
        const int i = idx % env.N;
        const size_t b = idx / env.N;
        if (best_spins) {
            const int s = env.spins[b * env.NP + i];
            const uint32_t w = env.diff_bits[b * env.NW + (i >> 5)];
            best_spins[idx] = (int8_t)(((w >> (i & 31)) & 1u) ? -s : s);
        }
        if (i == 0) {
            if (best_cut) best_cut[b] = env.ep[b].best_cut;
            if (steps) steps[b] = env.ep[b].step;
        }
    }
}

}  // namespace

#define ECO_ENV_DISPATCH(KERNEL, ...)                                                                       \
    do {                                                                                                    \
        const int NP_ = env->NP;                                                                            \
        const long long B_ = env->B;                                                                        \
        if (NP_ <= 32) {                                                                                    \
            KERNEL<4, false><<<(unsigned)((B_ * 4 + 127) / 128), 128, 0, st>>>(__VA_ARGS__);                \
        } else if (NP_ <= 64) {                                                                             \
            KERNEL<8, false><<<(unsigned)((B_ * 8 + 127) / 128), 128, 0, st>>>(__VA_ARGS__);                \
        } else if (NP_ <= 128) {                                                                            \
            KERNEL<16, false><<<(unsigned)((B_ * 16 + 127) / 128), 128, 0, st>>>(__VA_ARGS__);              \
        } else if (NP_ <= 256) {                                                                            \
            KERNEL<32, false><<<(unsigned)((B_ * 32 + 127) / 128), 128, 0, st>>>(__VA_ARGS__);              \
        } else if (NP_ <= 1024) {                                                                           \
            KERNEL<128, true><<<(unsigned)B_, 128, 0, st>>>(__VA_ARGS__);                                   \
        } else {                                                                                            \
            KERNEL<256, true><<<(unsigned)B_, 256, 0, st>>>(__VA_ARGS__);                                   \
        }                                                                                                   \
    } while (0)

int launch_env_step(const eco_graphs_t* g, eco_env_t* env, int policy, const int32_t* actions, double* reward,
                    uint8_t* done, int32_t* ha, double* hr, double* hs, cudaStream_t st) {
    prof_begin(ECO_PROF_ENV_STEP, st);
    if (env->reserved != 0 || (g->reserved & ECO_GRAPHS_MIN_CUT)) {   // S2V-DQN modes, Min-Cut: the general kernel
        ECO_ENV_DISPATCH(env_step_kernel, *g, *env, policy, actions, reward, done, ha, hr, hs);
    } else {
        const int NP_ = env->NP;
        const long long B_ = env->B;
#define ECO_SW(TPE) env_step_sw_kernel<TPE><<<(unsigned)((B_ * TPE + 127) / 128), 128, 0, st>>>(*g, *env, policy, actions, reward, done, ha, hr, hs)
        if (NP_ <= 32) ECO_SW(4);
        else if (NP_ <= 64) ECO_SW(8);
        else if (NP_ <= 128) ECO_SW(16);
        else if (NP_ <= 256) {
            if (policy == ECO_POLICY_ACTIONS && B_ >= 4096) {      // bulk-copy staged, persistent warps
                const int n_sm = device_sm_count();
                // 16 lanes per stream (two streams per warp), 3-deep ring.  (8 lanes per stream with a 2-deep ring -- 64
                // streams per SM -- was measured slower: 377 us vs 327 us.)
                constexpr int TPE = 16, STAGES = 3, NSTREAMS = TMA_WARPS * (32 / TPE);
                const size_t ring_bytes = (size_t)NSTREAMS * STAGES * (6 * NP_ + sizeof(eco_episode_t));
                static unsigned long long attr = 0;
                if (first_use_on_device(&attr)) {
                    ECO_CUDA((cudaFuncSetAttribute(env_step_ring_kernel<TPE, STAGES, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024)));
                    ECO_CUDA((cudaFuncSetAttribute(env_step_ring_kernel<TPE, STAGES, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024)));
                }
                long long blocks = (B_ + NSTREAMS - 1) / NSTREAMS;
                if (blocks > (long long)n_sm * 4) blocks = (long long)n_sm * 4;
                // the stripped vertex loop: +-1 couplings (|gain| <= 255, |mlr| <= 255: small_div is exact), table in shared memory
                const bool fast = (g->reserved & ECO_GRAPHS_PM1) && env->T + 1 <= TMA_TSF_MAX;
                if (fast) env_step_ring_kernel<TPE, STAGES, true><<<(unsigned)blocks, TMA_WARPS * 32, ring_bytes, st>>>(*g, *env, actions, reward, done, ha, hr, hs);
                else env_step_ring_kernel<TPE, STAGES, false><<<(unsigned)blocks, TMA_WARPS * 32, ring_bytes, st>>>(*g, *env, actions, reward, done, ha, hr, hs);
            } else ECO_SW(32);
        }
        else if (NP_ <= 1024) env_step_kernel<128, true><<<(unsigned)B_, 128, 0, st>>>(*g, *env, policy, actions, reward, done, ha, hr, hs);
        else env_step_kernel<256, true><<<(unsigned)B_, 256, 0, st>>>(*g, *env, policy, actions, reward, done, ha, hr, hs);
#undef ECO_SW
    }
    prof_end(ECO_PROF_ENV_STEP, st);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

int launch_env_reset(const eco_graphs_t* g, eco_env_t* env, const int32_t* gidx, const int8_t* spins,
                     cudaStream_t st) {
    if (env->use_basin)
        ECO_CUDA(cudaMemsetAsync(env->visited, 0, (size_t)env->B * env->HCAP * 16, st));
    ECO_ENV_DISPATCH(env_reset_kernel, *g, *env, gidx, spins);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

// argmax_i Q_i over the spins still at -1, lowest index on ties (experiments/utils.py:67-74, irreversible spins: the
// reference fills the others with -1000 before its argmax); one warp per episode.  No spin left: action 0.
__global__ void masked_argmax_kernel(const eco_env_t env, const float* __restrict__ q, int32_t* __restrict__ actions) {
    const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= env.B) return;
    const int8_t* s = env.spins + (size_t)b * env.NP;
    const float* qb = q + (size_t)b * env.NP;
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = lane; i < env.N; i += 32) {
        const float v = s[i] < 0 ? qb[i] : -1000.f;
        if (v > bv) { bv = v; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) actions[b] = bi == 0x7fffffff ? 0 : bi;
}

int launch_masked_argmax(const eco_env_t* env, const float* q, int32_t* actions, cudaStream_t st) {
    masked_argmax_kernel<<<(env->B + 7) / 8, 256, 0, st>>>(*env, q, actions);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

int launch_env_observation(const eco_env_t* env, float* obs7, cudaStream_t st) {
    const size_t total = (size_t)env->B * 7 * env->N;
    const int blocks = (int)((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
    env_observation_kernel<<<blocks, 256, 0, st>>>(*env, obs7);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

int launch_env_results(const eco_env_t* env, int32_t* best_cut, int8_t* best_spins, int32_t* steps,
                       cudaStream_t st) {
    const size_t total = (size_t)env->B * env->N;
    const int blocks = (int)((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
    env_results_kernel<<<blocks, 256, 0, st>>>(*env, best_cut, best_spins, steps);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

}  // namespace eco
