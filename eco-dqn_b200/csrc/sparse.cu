// Kernel family 5: graph sets stored as CSR (eco_sgraphs_t), N <= ECO_MAX_SPINS_SPARSE -- graph preparation, environment
// reset / step in O(degree) + one O(N) feature row, and the MPNN forward as neighbour gathers plus per-vertex linears.
//
// Replaces (reference, file:line)
//   src/envs/score_solver.py:353-375 MaximumCutUnbiasedScorer constants  -> sgraph_prepare_kernel
//   src/networks/mpnn.py:34-38       get_normalisation                   -> sgraph_prepare_kernel (deg = nnz of the row)
//   src/envs/spinsystem.py:183-330   reset / _reset_state                -> senv_reset_kernel
//   src/envs/spinsystem.py:355-559   step                                -> senv_step_kernel
//   src/agents/solver.py:105-131     Greedy.step                         -> ECO_POLICY_GREEDY inside senv_step_kernel
//   src/networks/mpnn.py:40-159      MPNN.forward                        -> k_sinit, k_sgather, k_gemm, k_sreadout
//                                                                          (linears on the tensor cores: sparse_tc.cu)
//
// The environment keeps the int8 path's state (eco_env_t: int16 fields, uint16 last-flip steps, the best-diff bitmask, the
// 96-byte episode block) and its integer / fp64 rules, so for N <= ECO_MAX_SPINS every array equals the dense path's bit for
// bit.  A flip of vertex a changes the fields of a's neighbours only, so the step touches row a of the CSR and, per
// neighbour, its spin, field and observable row 1; observable row 2 (time since flip) changes for every vertex and is written
// in full.  The scalar bookkeeping is bls_step_scalars (env_step_device.cuh), shared with the int8 and fp64 steps.
//
// Bytes per episode-step of senv_step_kernel (algorithmic, ACTIONS policy, d = degree of the flipped vertex):
//   row 2: last-flip steps read 2N + fp32 row written 4N                                       6N
//   row a: column 4d + coupling d;  per neighbour: spin 1, field read + write 4, row 1 written 4  14d
//   the flipped vertex: spin, last-flip step, rows 0 / 1, field, best-diff word                 ~20
//   scalar block 96, xg 16, visited-set probe 16 (basin reward)                                128
//   = 6N + 14d + ~150 bytes; a new best clears the best-diff words, + N/8.  ECO_POLICY_GREEDY reads the spins and the fields
//   of every vertex first: + 3N.
#include <limits.h>

#include "eco_common.cuh"
#include "env_step_device.cuh"
#include "mpnn_gemm.cuh"
#include "mpnn_pack.cuh"

namespace eco {

namespace {

constexpr int SENV_THREADS = 256;

__device__ __forceinline__ long long block_sum_ll(long long v, long long* sm) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
    __syncthreads();
    long long t = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sm[w];     // fixed order: every thread gets the same sum
    return t;
}

// ------------------------------------------------------------------------------------------------ prepare
// one CTA per graph, one warp per row (strided).  Every entry (i, j, v) is checked: j in [0, N), columns strictly ascending,
// v != 0, v == J_ji (binary search for i in row j), j != i.
__global__ void __launch_bounds__(256) sgraph_prepare_kernel(const eco_sgraphs_t g) {
    const int gi = blockIdx.x;
    const int N = g.N, NP = g.NP;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    const int64_t* rp = g.row_ptr + (size_t)gi * N;

    __shared__ long long s_sum[8], s_pos[8], s_neg[8], s_nnz[8];
    __shared__ int s_mlr[8], s_maxdeg[8], s_maxabs[8], s_flags[8];
    long long t_sum = 0, t_pos = 0, t_neg = 0, t_nnz = 0;
    int t_mlr = INT_MIN, t_maxdeg = 0, t_maxabs = 0, t_flags = 0;

    for (int i = warp; i < NP; i += nwarp) {
        int rs = 0, ra = 0, rpos = 0, rneg = 0, cnt = 0, bad = 0;
        if (i < N) {
            const int64_t s = rp[i], e = rp[i + 1];
            if (s < 0 || e < s || e > g.nnz) {
                bad = ECO_SGRAPH_NONCANONICAL;
            } else {
                for (int64_t k = s + lane; k < e; k += 32) {
                    const int j = g.col[k], v = g.val[k];
                    if (j < 0 || j >= N || (k > s && g.col[k - 1] >= j) || v == 0) { bad |= ECO_SGRAPH_NONCANONICAL; continue; }
                    rs += v;
                    ra += abs(v);
                    rpos += v > 0 ? v : 0;
                    rneg += v < 0 ? v : 0;
                    ++cnt;
                    if (v > 1 || v < -1) bad |= 1;
                    if (j == i) bad |= 4;
                    // J_ji: binary search for column i in row j
                    int64_t lo = rp[j], hi = rp[j + 1];
                    if (lo < 0 || hi < lo || hi > g.nnz) { bad |= ECO_SGRAPH_NONCANONICAL; continue; }
                    while (lo < hi) {
                        const int64_t mid = (lo + hi) >> 1;
                        if (g.col[mid] < i) lo = mid + 1; else hi = mid;
                    }
                    if (lo >= rp[j + 1] || g.col[lo] != i || g.val[lo] != v) bad |= 4;
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            rs += __shfl_xor_sync(0xffffffffu, rs, o);
            ra += __shfl_xor_sync(0xffffffffu, ra, o);
            rpos += __shfl_xor_sync(0xffffffffu, rpos, o);
            rneg += __shfl_xor_sync(0xffffffffu, rneg, o);
            cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
            bad |= __shfl_xor_sync(0xffffffffu, bad, o);
        }
        if (lane == 0) g.deg[(size_t)gi * NP + i] = (float)max(cnt, 1);
        t_sum += rs; t_pos += rpos; t_neg += rneg; t_nnz += cnt;
        t_flags |= bad;
        t_maxdeg = max(t_maxdeg, cnt);
        t_maxabs = max(t_maxabs, ra);
        if (i < N && rs != 0) t_mlr = max(t_mlr, rs);                    // max non-zero weighted degree (:367-375)
    }
    if (lane == 0) {
        s_sum[warp] = t_sum; s_pos[warp] = t_pos; s_neg[warp] = t_neg; s_nnz[warp] = t_nnz;
        s_mlr[warp] = t_mlr; s_maxdeg[warp] = t_maxdeg; s_maxabs[warp] = t_maxabs; s_flags[warp] = t_flags;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        long long sum = 0, pos = 0, neg = 0, nnz = 0;
        int mlr = INT_MIN, maxdeg = 0, maxabs = 0, flags = 0;
        for (int w = 0; w < nwarp; ++w) {
            sum += s_sum[w]; pos += s_pos[w]; neg += s_neg[w]; nnz += s_nnz[w];
            mlr = max(mlr, s_mlr[w]); maxdeg = max(maxdeg, s_maxdeg[w]); maxabs = max(maxabs, s_maxabs[w]); flags |= s_flags[w];
        }
        if (mlr == INT_MIN) { flags |= 2; mlr = 1; }
        if (maxabs > 32767) flags |= ECO_SGRAPH_FIELD_RANGE;
        double* gs = g.gscal + (size_t)gi * 4;
        gs[0] = (double)mlr;
        gs[1] = fmax(1.0, (double)pos / 2.0);                              // :353-357
        gs[2] = fmin(0.0, (double)neg / 2.0);                              // :359-365
        gs[3] = (double)sum;
        int32_t* st = g.gstat + (size_t)gi * 4;
        st[0] = maxdeg; st[1] = (int32_t)min(nnz, (long long)INT_MAX); st[2] = maxabs; st[3] = flags;
    }
}

__global__ void sgraph_dmax_kernel(const eco_sgraphs_t g) {
    int m = 1;
    for (int i = threadIdx.x; i < g.G; i += 32) m = max(m, g.gstat[(size_t)i * 4]);
    m = group_max<32>(m);
    if (threadIdx.x == 0) g.dmax[0] = (float)m;
}

// ------------------------------------------------------------------------------------------------ reset
// one CTA per episode: h = J s over the CSR rows, then env_reset_kernel's integer formulas
__global__ void __launch_bounds__(SENV_THREADS) senv_reset_kernel(const eco_sgraphs_t g, const eco_env_t env,
                                                                  const int32_t* __restrict__ graph_idx,
                                                                  const int8_t* __restrict__ init_spins) {
    __shared__ long long sm[SENV_THREADS / 32];
    const long long b = blockIdx.x;
    const int N = env.N, NP = env.NP;
    const int gi = graph_idx[b];
    int8_t* spins = env.spins + (size_t)b * NP;
    int16_t* hf = env.hfield + (size_t)b * NP;
    const int64_t* rp = g.row_ptr + (size_t)gi * N;
    const double mlr = g.gscal[(size_t)gi * 4 + 0];

    for (int i = threadIdx.x; i < NP; i += blockDim.x) {
        spins[i] = i < N ? init_spins[(size_t)b * N + i] : (int8_t)0;
        env.last_flip[(size_t)b * NP + i] = 0;
    }
    for (int w = threadIdx.x; w < env.NW; w += blockDim.x) env.diff_bits[(size_t)b * env.NW + w] = 0u;
    if (threadIdx.x == 0) env.graph_idx[b] = gi;
    __syncthreads();

    long long nimp = 0, ssh = 0;
    float* x0 = env.xn + (size_t)b * 3 * NP;
    for (int i = threadIdx.x; i < NP; i += blockDim.x) {
        int acc = 0;                                                       // h_i = sum_j J_ij s_j
        if (i < N)
            for (int64_t k = rp[i]; k < rp[i + 1]; ++k) acc += (int)g.val[k] * (int)spins[g.col[k]];
        hf[i] = (int16_t)acc;
        const int si = spins[i];
        const int gain = si * acc;
        ssh += gain;
        nimp += gain > 0;
        x0[i] = (float)si;                                                 // spinsystem.py:294/299
        x0[NP + i] = i < N ? feat_gain(gain, mlr) : 0.f;                   // :311-312
        x0[2 * NP + i] = 0.f;
    }
    nimp = block_sum_ll(nimp, sm);
    ssh = block_sum_ll(ssh, sm);
    if (threadIdx.x == 0) {
        const double qn = g.gscal[(size_t)gi * 4 + 1], lb = g.gscal[(size_t)gi * 4 + 2];
        const long long sumJ = (long long)g.gscal[(size_t)gi * 4 + 3];
        const int cut = (int)((sumJ - ssh) / 4);                           // utils.py:90-94, exact in integers
        const double score = __dadd_rn((double)cut, fabs(fmin(0.0, lb)));  // score_solver.py:196-200
        const double nscore = __ddiv_rn(score, qn);                        // :190-194
        eco_episode_t e;
        e.step = 0; e.cut = cut; e.best_cut = cut; e.dist = 0; e.n_improving = (int)nimp; e.flags = 0;
        e.n_visited = 0; e.reserved = 0;
        e.score = score; e.nscore = nscore; e.best_score = score; e.best_nscore = nscore;
        e.key[0] = 0; e.key[1] = 0; e.total_reward = 0.0; e.last_reward = 0.0;
        env.ep[b] = e;
        *reinterpret_cast<float4*>(env.xg + (size_t)b * 4) = make_float4(0.f, 0.f, (float)__ddiv_rn((double)nimp, (double)N), 0.f);
    }
}

// ------------------------------------------------------------------------------------------------ step
// one CTA per episode
__global__ void __launch_bounds__(SENV_THREADS) senv_step_kernel(const eco_sgraphs_t g, const eco_env_t env, const int policy,
                                                                 const int32_t* __restrict__ actions,
                                                                 double* __restrict__ reward_out, uint8_t* __restrict__ done_out,
                                                                 int32_t* __restrict__ hist_a, double* __restrict__ hist_r,
                                                                 double* __restrict__ hist_s) {
    __shared__ long long sm[SENV_THREADS / 32];
    __shared__ int s_key[SENV_THREADS / 32];
    __shared__ int s_new_best;
    const int tid = threadIdx.x;
    const long long b = blockIdx.x;
    const int N = env.N, NP = env.NP;
    eco_episode_t* ep = env.ep + b;
    const int4 e0 = *reinterpret_cast<const int4*>(ep);                 // step, cut, best_cut, dist
    const int4 e1 = *(reinterpret_cast<const int4*>(ep) + 1);           // n_improving, flags, n_visited, reserved
    const int flags = e1.y;
    const int step_new = e0.x + 1;
    bool active = !(flags & (FLAG_DONE | FLAG_STOPPED)) && step_new <= env.T;   // :365-367
    const int gi = env.graph_idx[b];
    int8_t* spins = env.spins + (size_t)b * NP;
    int16_t* hf = env.hfield + (size_t)b * NP;
    uint16_t* lf = env.last_flip + (size_t)b * NP;
    const double mlr = g.gscal[(size_t)gi * 4 + 0];

    int a;
    if (policy == ECO_POLICY_GREEDY) {
        // argmax_i s_i h_i, first maximal index (numpy argmax, solver.py:116): key (gain + 32768) : (65535 - i), as the int8 step
        int best = INT_MIN;
        for (int i = tid; i < N; i += blockDim.x)
            best = max(best, (int)((((uint32_t)(spins[i] * hf[i] + 32768) << 16) | (uint32_t)(0xFFFF - i)) ^ 0x80000000u));
        best = group_max<32>(best);
        if ((tid & 31) == 0) s_key[tid >> 5] = best;
        __syncthreads();
        best = INT_MIN;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) best = max(best, s_key[w]);
        const uint32_t ukey = (uint32_t)best ^ 0x80000000u;
        a = 0xFFFF - (int)(ukey & 0xFFFFu);
        if (active && (best == INT_MIN || ((int)(ukey >> 16) - 32768) < 0)) {   // solver.py:124: stop only if the best gain is < 0
            active = false;
            if (tid == 0) ep->flags = flags | FLAG_STOPPED;
        }
    } else {
        a = actions[b];
    }
    if (a < 0 || a >= N) { a = 0; active = false; }

    const int s_a_old = spins[a];
    const int h_a_old = hf[a];
    const int s_a_new = -s_a_old;
    const uint32_t old_word = env.diff_bits[(size_t)b * env.NW + (a >> 5)];
    __syncthreads();                                                     // pre-flip values read before anyone writes

    long long dn = 0;                                                    // change of n_improving
    float* x0 = env.xn + (size_t)b * 3 * NP;
    if (active) {
        // neighbours of a: h_j += 2 J_ja s_a (J symmetric: J_ja is the entry of row a), their gains and row 1
        const int64_t* rp = g.row_ptr + (size_t)gi * N;
        const int64_t ks = rp[a], ke = rp[a + 1];
        for (int64_t k = ks + tid; k < ke; k += blockDim.x) {
            const int j = g.col[k];
            const int sj = spins[j], ho = hf[j];
            const int hn = ho + 2 * (int)g.val[k] * s_a_new;
            hf[j] = (int16_t)hn;
            const int gn = sj * hn;
            dn += (gn > 0) - (sj * ho > 0);
            x0[NP + j] = feat_gain(gn, mlr);                              // :490
        }
        if (tid == 0) {                                                   // the flipped vertex (J_aa = 0: h_a is unchanged)
            const int gn = s_a_new * h_a_old;
            dn += (gn > 0) - (s_a_old * h_a_old > 0);
            spins[a] = (int8_t)s_a_new;
            x0[a] = (float)s_a_new;
            x0[NP + a] = feat_gain(gn, mlr);
        }
        // row 2, time since flip, for every vertex (:493-495); the thread that owns a's quad records a's flip
        const float* tsf_now = env.tsf_tab + step_new;
        const int qa = a >> 2, ka = a & 3;
        for (int q = tid; q < (NP >> 2); q += blockDim.x) {
            uint2 lw = *reinterpret_cast<const uint2*>(lf + 4 * q);
            if (q == qa) {
                const uint32_t sh = 16 * (ka & 1), keep = ~(0xFFFFu << sh), val = ((uint32_t)step_new & 0xFFFFu) << sh;
                if ((ka >> 1) == 0) lw.x = (lw.x & keep) | val;
                else lw.y = (lw.y & keep) | val;
                *reinterpret_cast<uint2*>(lf + 4 * q) = lw;
            }
            *reinterpret_cast<float4*>(x0 + 2 * NP + 4 * q) =
                make_float4(tsf_now[-zx16(lw.x, 0)], tsf_now[-zx16(lw.x, 1)], tsf_now[-zx16(lw.y, 0)], tsf_now[-zx16(lw.y, 1)]);
        }
    }
    const int nimp = e1.x + (int)block_sum_ll(dn, sm);

    if (tid == 0) {
        int new_best = 0;
        if (active) {
            const double qn = g.gscal[(size_t)gi * 4 + 1];
            const int delta = s_a_old * h_a_old;                               // spinsystem.py:393
            // the reference multiplies in fp64: a zero field times a spin of -1 is -0.0 (as env_step_kernel)
            const double delta_n = __ddiv_rn((delta == 0 && s_a_old < 0) ? -0.0 : (double)delta, qn);   // :394
            const double sc[4] = {ep->score, ep->nscore, ep->best_score, ep->best_nscore};
            const uint64_t k0 = ep->key[0] ^ env.zobrist[2 * a], k1 = ep->key[1] ^ env.zobrist[2 * a + 1];
            uint64_t* tab = env.visited + (size_t)b * env.HCAP * 2;
            const uint32_t slot = (uint32_t)(k0 ^ (k0 >> 29)) & (env.HCAP - 1);
            ulonglong2 tv = make_ulonglong2(0, 0);
            if (env.use_basin) tv = *reinterpret_cast<const ulonglong2*>(tab + 2 * slot);
            const StepScalars r = bls_step_scalars(env, sc, (double)delta, delta_n, nimp, e1.z, tab, slot, tv, k0, k1);
            const int cut = e0.y + delta;
            int dist = e0.w + (((old_word >> (a & 31)) & 1u) ? -1 : 1);
            int best_cut = e0.z;
            if (r.new_best) { best_cut = cut; dist = 0; new_best = 1; }
            const int done = step_new == env.T;                                // :541-544
            int4* epw = reinterpret_cast<int4*>(ep);
            epw[0] = make_int4(step_new, cut, best_cut, dist);
            epw[1] = make_int4(nimp, flags | (done ? FLAG_DONE : 0), r.n_visited, 0);
            *reinterpret_cast<double2*>(&ep->score) = make_double2(r.score, r.nscore);
            *reinterpret_cast<double2*>(&ep->best_score) = make_double2(r.best_score, r.best_nscore);
            *reinterpret_cast<ulonglong2*>(&ep->key[0]) = make_ulonglong2(k0, k1);
            *reinterpret_cast<double2*>(&ep->total_reward) = make_double2(__dadd_rn(ep->total_reward, r.rew), r.rew);
            float4 xg;                                                         // rows 3..6 (spinsystem.py:509-527)
            xg.x = (float)__ddiv_rn(fabs(__dsub_rn(r.score, r.best_score)), mlr);
            xg.y = (float)dist;
            xg.z = env.frac_tab[nimp];
            xg.w = env.imm_tab[step_new];
            *reinterpret_cast<float4*>(env.xg + (size_t)b * 4) = xg;
            if (reward_out) reward_out[b] = r.rew;
            if (done_out) done_out[b] = (uint8_t)done;
            const size_t hidx = (size_t)b * env.T + (step_new - 1);
            if (hist_a) hist_a[hidx] = a;
            if (hist_r) hist_r[hidx] = r.rew;
            if (hist_s) hist_s[hidx] = r.score;
            if (!new_best) env.diff_bits[(size_t)b * env.NW + (a >> 5)] = old_word ^ (1u << (a & 31));
        } else {
            if (reward_out) reward_out[b] = 0.0;
            if (done_out) done_out[b] = 1;
        }
        s_new_best = new_best;
    }
    __syncthreads();
    if (s_new_best)                                                      // the new best: every spin equals its best value
        for (int w = tid; w < env.NW; w += blockDim.x) env.diff_bits[(size_t)b * env.NW + w] = 0u;
}

// ------------------------------------------------------------------------------------------------ MPNN
// Vertex-major planes [B * NP][64] fp32; padding vertices are zero in every plane.
__device__ __forceinline__ float sdmax_of(const eco_sgraphs_t& g, int gi, float norm_max) {
    return norm_max > 0.f ? norm_max : (norm_max < 0.f ? (float)max(g.gstat[(size_t)gi * 4], 1) : *g.dmax);
}

// input stage (mpnn.py:55, :90-97): H0 = ReLU(W_init x), P = W_e[:, 1:8] x (feature 63: 0)
__global__ void __launch_bounds__(256)
k_sinit(const int N, const int NP, const eco_mpnn_t w, const long long V, const float* __restrict__ xn, const float* __restrict__ xg,
        float* __restrict__ H0, float* __restrict__ P) {
    const size_t idx = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (idx >= (size_t)V * F) return;
    const int f = (int)(idx & 63);
    const size_t v = idx >> 6;
    const size_t b = v / NP;
    const int i = (int)(v % NP);
    float h = 0.f, p = 0.f;
    if (i < N) {
        const float X[7] = {xn[(b * 3 + 0) * NP + i], xn[(b * 3 + 1) * NP + i], xn[(b * 3 + 2) * NP + i],
                            xg[b * 4 + 0], xg[b * 4 + 1], xg[b * 4 + 2], xg[b * 4 + 3]};
#pragma unroll
        for (int c = 0; c < 7; ++c) h = fmaf(w.w_init[f * 7 + c], X[c], h);
        h = fmaxf(h, 0.f);
        if (f < 63) {
#pragma unroll
            for (int c = 0; c < 7; ++c) p = fmaf(w.w_edge[f * 8 + 1 + c], X[c], p);
        }
    }
    H0[idx] = h;
    P[idx] = p;
}

// Neighbour gathers over the CSR rows, ascending column order, 64 threads (one per feature) per vertex:
//   EDGE: O[i] = 1/d_i sum_j ReLU(a_ij w0 + X[j]), feature 63 = d_i / d_max          (mpnn.py:89-104, any int8 a_ij)
//   AGG:  O[i] = 1/d_i sum_j a_ij X[j]                                                (mpnn.py:114-116)
template <bool EDGE>
__global__ void __launch_bounds__(256)
k_sgather(const eco_sgraphs_t g, const int32_t* __restrict__ graph_idx, const eco_mpnn_t w, const long long V,
          const float* __restrict__ X, float* __restrict__ O, const float norm_max) {
    const size_t idx = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (idx >= (size_t)V * F) return;
    const int N = g.N, NP = g.NP;
    const int f = (int)(idx & 63);
    const size_t v = idx >> 6;
    const size_t b = v / NP;
    const int i = (int)(v % NP);
    float out = 0.f;
    if (i < N) {
        const int gi = graph_idx[b];
        const int64_t* rp = g.row_ptr + (size_t)gi * N + i;
        const int64_t ks = rp[0], ke = rp[1];
        const float* Xb = X + b * NP * F + f;
        const float w0 = (EDGE && f < 63) ? w.w_edge[f * 8] : 0.f;
        float acc = 0.f;
        for (int64_t k = ks; k < ke; ++k) {
            const float a = (float)g.val[k];
            const float x = Xb[(size_t)g.col[k] * F];
            if (EDGE) acc += fmaxf(fmaf(a, w0, x), 0.f);
            else acc = fmaf(a, x, acc);
        }
        const float d = g.deg[(size_t)gi * NP + i];
        out = (EDGE && f == 63) ? d / sdmax_of(g, gi, norm_max) : acc / d;
    }
    O[idx] = out;
}

// readout (mpnn.py:143-159) + argmax, one CTA (8 warps) per episode: pooled mean in a fixed order, Q_i, lowest index on ties
__global__ void __launch_bounds__(256)
k_sreadout(const int N, const int NP, const eco_mpnn_t w, const float* __restrict__ H, float* __restrict__ q_out,
           int32_t* __restrict__ act_out) {
    __shared__ float part[8][F], pooled[F], red_val[8], c0s;
    __shared__ int red_idx[8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t b = blockIdx.x;
    const float* Hb = H + b * NP * F;
    {
        float sa = 0.f, sb = 0.f;
        for (int i = warp; i < N; i += 8) {
            sa += Hb[(size_t)i * F + lane];
            sb += Hb[(size_t)i * F + lane + 32];
        }
        part[warp][lane] = sa;
        part[warp][lane + 32] = sb;
    }
    __syncthreads();
    if (tid < F) {
        float s = 0.f;
        for (int ww = 0; ww < 8; ++ww) s += part[ww][tid];
        pooled[tid] = s / (float)N;
    }
    __syncthreads();
    if (warp == 0) {
        float c = 0.f;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int f = lane + 32 * half;
            float p = 0.f;
            for (int k = 0; k < F; ++k) p = fmaf(w.w_pool[f * F + k], pooled[k], p);
            c = fmaf(w.w_read[f], fmaxf(p, 0.f), c);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (lane == 0) c0s = c + w.b_read[0];
    }
    __syncthreads();
    const float c0 = c0s, wr0 = w.w_read[64 + lane], wr1 = w.w_read[96 + lane];
    float best_v = -INFINITY;
    int best_i = 0x7fffffff;
    for (int i = warp; i < N; i += 8) {
        float v = fmaf(wr0, fmaxf(Hb[(size_t)i * F + lane], 0.f), wr1 * fmaxf(Hb[(size_t)i * F + lane + 32], 0.f));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        v += c0;
        if (lane == 0 && q_out) q_out[b * NP + i] = v;
        if (v > best_v) { best_v = v; best_i = i; }                       // ascending i => first maximum kept
    }
    if (lane == 0) { red_val[warp] = best_v; red_idx[warp] = best_i; }
    __syncthreads();
    if (tid == 0 && act_out) {
        float bv = red_val[0];
        int bi = red_idx[0];
        for (int ww = 1; ww < 8; ++ww)
            if (red_val[ww] > bv || (red_val[ww] == bv && red_idx[ww] < bi)) { bv = red_val[ww]; bi = red_idx[ww]; }
        act_out[b] = bi == 0x7fffffff ? 0 : bi;
    }
}

constexpr int SMPNN_PLANES = 5;

}  // namespace

size_t smpnn_scratch_bytes(int B, int N) {
    return align256(sizeof(float) * (size_t)SMPNN_PLANES * B * padded_n(N) * F);
}

int launch_sgraph_prepare(const eco_sgraphs_t* g, cudaStream_t st) {
    sgraph_prepare_kernel<<<g->G, 256, 0, st>>>(*g);
    ECO_LAUNCH_CHECK();
    sgraph_dmax_kernel<<<1, 32, 0, st>>>(*g);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

int launch_senv_reset(const eco_sgraphs_t* g, eco_env_t* env, const int32_t* gidx, const int8_t* spins, cudaStream_t st) {
    if (env->use_basin) ECO_CUDA(cudaMemsetAsync(env->visited, 0, (size_t)env->B * env->HCAP * 16, st));
    senv_reset_kernel<<<(unsigned)env->B, SENV_THREADS, 0, st>>>(*g, *env, gidx, spins);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

int launch_senv_step(const eco_sgraphs_t* g, eco_env_t* env, int policy, const int32_t* actions, double* reward, uint8_t* done,
                     int32_t* ha, double* hr, double* hs, cudaStream_t st) {
    prof_begin(ECO_PROF_ENV_STEP, st);
    senv_step_kernel<<<(unsigned)env->B, SENV_THREADS, 0, st>>>(*g, *env, policy, actions, reward, done, ha, hr, hs);
    prof_end(ECO_PROF_ENV_STEP, st);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

// Planes: H ping / pong, E, and two planes that hold P then the aggregate (X) and G then the message (Y).  The seven
// per-vertex linears run as k_gemm (fp32 CUDA cores) or, with `tc`, as sparse_linear_tc_kernel (sparse_tc.cu, tensor
// cores, bf16 hi/lo operands from eco_mpnn_pack); every other launch is the same.
static int smpnn_sequence(const eco_sgraphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn,
                          const float* xg, float norm_max, float* q, int32_t* actions, void* scratch, bool tc, cudaStream_t st) {
    const int N = g->N, NP = g->NP;
    const long long V = (long long)B * NP;
    const size_t pl = (size_t)V * F;
    float* base = (float*)scratch;
    float *Ha = base, *Hb = base + pl, *E = base + 2 * pl, *X = base + 3 * pl, *Y = base + 4 * pl;
    static unsigned long long attr = 0;
    if (!tc && first_use_on_device(&attr))
        ECO_CUDA(cudaFuncSetAttribute(k_gemm<false, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm_smem_bytes(128)));
    const unsigned eblocks = (unsigned)((pl + 255) / 256);
    const unsigned vt = (unsigned)((V + GT - 1) / GT);
    const uint32_t* pk = static_cast<const uint32_t*>(w->packed);
    prof_begin(ECO_PROF_MPNN, st);
    k_sinit<<<eblocks, 256, 0, st>>>(N, NP, *w, V, xn, xg, Ha, X);
    ECO_LAUNCH_CHECK();
    k_sgather<true><<<eblocks, 256, 0, st>>>(*g, gidx, *w, V, X, Y, norm_max);
    ECO_LAUNCH_CHECK();
    int rc;
    if (tc) {
        if ((rc = launch_sparse_linear_tc(Y, nullptr, 64, V, pk + PK_WEF, E, st))) return rc;
    } else {
        k_gemm<false, 64><<<vt, 256, gemm_smem_bytes(64), st>>>(Y, nullptr, nullptr, (int)V, w->w_edge_feat, 64, 0, E, 1, 0);
        ECO_LAUNCH_CHECK();
    }
    float *Hc = Ha, *Hn = Hb;
    for (int l = 0; l < 3; ++l) {
        k_sgather<false><<<eblocks, 256, 0, st>>>(*g, gidx, *w, V, Hc, X, norm_max);
        ECO_LAUNCH_CHECK();
        if (tc) {
            if ((rc = launch_sparse_linear_tc(X, E, 128, V, pk + PK_WM + l * 128 * 64, Y, st))) return rc;
            if ((rc = launch_sparse_linear_tc(Hc, Y, 128, V, pk + PK_WU + l * 128 * 64, Hn, st))) return rc;
        } else {
            k_gemm<false, 128><<<vt, 256, gemm_smem_bytes(128), st>>>(X, E, nullptr, (int)V, w->w_msg[l], 128, 0, Y, 1, 0);
            ECO_LAUNCH_CHECK();
            k_gemm<false, 128><<<vt, 256, gemm_smem_bytes(128), st>>>(Hc, Y, nullptr, (int)V, w->w_upd[l], 128, 0, Hn, 1, 0);
            ECO_LAUNCH_CHECK();
        }
        float* t = Hc; Hc = Hn; Hn = t;
    }
    k_sreadout<<<(unsigned)B, 256, 0, st>>>(N, NP, *w, Hc, q, actions);
    prof_end(ECO_PROF_MPNN, st);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

int launch_smpnn(const eco_sgraphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn, const float* xg,
                 float norm_max, float* q, int32_t* actions, void* scratch, cudaStream_t st) {
    return smpnn_sequence(g, w, B, gidx, xn, xg, norm_max, q, actions, scratch, false, st);
}

int launch_smpnn_tc(const eco_sgraphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn, const float* xg,
                    float norm_max, float* q, int32_t* actions, void* scratch, cudaStream_t st) {
    return smpnn_sequence(g, w, B, gidx, xn, xg, norm_max, q, actions, scratch, true, st);
}

}  // namespace eco
