// Kernel family 4: real-valued couplings (EdgeType.RANDOM) -- graph preparation, environment reset / step / results with
// fp64 local fields.  The MPNN of these graphs is mpnn_simt_kernel<float> (mpnn_simt.cu) on the fp32 copy of J.
//
// Replaces (reference, file:line)
//   src/envs/score_solver.py:353-375 MaximumCutUnbiasedScorer constants  -> wgraph_prepare_kernel (fp64 sums)
//   src/networks/mpnn.py:34-38       get_normalisation (on the fp32 obs) -> wgraph_prepare_kernel (deg from fp32(J))
//   src/envs/spinsystem.py:183-330   reset / _reset_state                -> wenv_reset_kernel
//   src/envs/spinsystem.py:355-559   step                                -> wenv_step_kernel
//   src/agents/solver.py:105-131     Greedy.step                         -> ECO_POLICY_GREEDY inside wenv_step_kernel
//
// Precision: everything the environment computes is fp64, as the reference's fp64 `matrix` makes it -- couplings, local
// fields, gains, score, normalised score, cut, rewards.  The local fields are updated incrementally, h_i += 2 J_ia s_a
// (the product is exact, so one rounding per step), where the reference recomputes J s; for integer couplings both are
// exact and every result equals the int8 path bit for bit.  The scalar bookkeeping is bls_step_scalars
// (env_step_device.cuh), shared with the int8 kernels.  Observable row 1 is (float)(gain / mlr) with a real fp64
// division; the normalised score change is gain / qn in fp64.
//
// Bytes per episode-step of wenv_step_kernel (algorithmic, ACTIONS policy): row a of the fp64 couplings 8N, spins N, fp64
// fields read + write 16N, last-flip steps 2N, best-diff bits 2*ceil(N/8), the three fp32 feature rows 12N, scalar block
// 96:  39.25 N + 96 bytes (N = 200: 7 946 B).  HBM-bound like the int8 kernel (20.25 N + 96, DESIGN.md section 4.1).
#include <limits.h>

#include "eco_common.cuh"
#include "env_step_device.cuh"

namespace eco {

namespace {

template <int W>
__device__ __forceinline__ double group_sum_d(double v) {
#pragma unroll
    for (int o = W / 2; o > 0; o >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o, W));
    return v;
}

// ------------------------------------------------------------------------------------------------ prepare
// one CTA per graph, one warp per row (strided).  `dense` [G, N, N] fp64.
__global__ void __launch_bounds__(256) wgraph_prepare_kernel(eco_wgraphs_t g, const double* __restrict__ dense) {
    const int gi = blockIdx.x;
    const int N = g.N, NP = g.NP;
    const double* src = dense + (size_t)gi * N * N;
    double* J = g.J + (size_t)gi * NP * NP;
    float* Jf = g.Jf + (size_t)gi * NP * NP;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;

    __shared__ double s_sum[8], s_pos[8], s_neg[8], s_mlr[8];
    __shared__ int s_maxdeg[8], s_nnz[8], s_flags[8], s_has[8];
    double t_sum = 0.0, t_pos = 0.0, t_neg = 0.0, t_mlr = -INFINITY;
    int t_maxdeg = 0, t_nnz = 0, t_flags = 0, t_has = 0;

    for (int i = warp; i < NP; i += nwarp) {
        double rs = 0.0, rp = 0.0, rn = 0.0;
        int cnt = 0, bad = 0;
        for (int j = lane; j < NP; j += 32) {
            const double v = (i < N && j < N) ? src[(size_t)i * N + j] : 0.0;
            const float vf = (float)v;
            J[(size_t)i * NP + j] = v;
            Jf[(size_t)i * NP + j] = vf;
            rs = __dadd_rn(rs, v);
            if (v > 0.0) rp = __dadd_rn(rp, v);
            if (v < 0.0) rn = __dadd_rn(rn, v);
            cnt += vf != 0.f;                                       // the MPNN's degree counts fp32 non-zeros
            if (!isfinite(v)) bad |= ECO_WGRAPH_NONFINITE;
            if (i < N && j < N && src[(size_t)j * N + i] != v) bad |= ECO_WGRAPH_ASYMMETRIC;
            if (i == j && v != 0.0) bad |= ECO_WGRAPH_ASYMMETRIC;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            rs = __dadd_rn(rs, __shfl_xor_sync(0xffffffffu, rs, o));
            rp = __dadd_rn(rp, __shfl_xor_sync(0xffffffffu, rp, o));
            rn = __dadd_rn(rn, __shfl_xor_sync(0xffffffffu, rn, o));
            cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
            bad |= __shfl_xor_sync(0xffffffffu, bad, o);
        }
        if (lane == 0) g.deg[(size_t)gi * NP + i] = (float)max(cnt, 1);
        t_sum = __dadd_rn(t_sum, rs);
        t_pos = __dadd_rn(t_pos, rp);
        t_neg = __dadd_rn(t_neg, rn);
        t_nnz += cnt;
        t_flags |= bad;
        t_maxdeg = max(t_maxdeg, cnt);
        if (i < N && rs != 0.0) { t_mlr = fmax(t_mlr, rs); t_has = 1; }   // max non-zero gain of the all -1 state (:367-375)
    }
    if (lane == 0) {
        s_sum[warp] = t_sum; s_pos[warp] = t_pos; s_neg[warp] = t_neg; s_mlr[warp] = t_mlr;
        s_maxdeg[warp] = t_maxdeg; s_nnz[warp] = t_nnz; s_flags[warp] = t_flags; s_has[warp] = t_has;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double sum = 0.0, pos = 0.0, neg = 0.0, mlr = -INFINITY;
        int maxdeg = 0, nnz = 0, flags = 0, has = 0;
        for (int w = 0; w < nwarp; ++w) {
            sum = __dadd_rn(sum, s_sum[w]); pos = __dadd_rn(pos, s_pos[w]); neg = __dadd_rn(neg, s_neg[w]);
            mlr = fmax(mlr, s_mlr[w]);
            maxdeg = max(maxdeg, s_maxdeg[w]); nnz += s_nnz[w]; flags |= s_flags[w]; has |= s_has[w];
        }
        if (!has) { flags |= ECO_WGRAPH_NO_DEGREE; mlr = 1.0; }
        double* gs = g.gscal + (size_t)gi * 4;
        gs[0] = mlr;
        gs[1] = fmax(1.0, __ddiv_rn(pos, 2.0));                          // :353-357
        gs[2] = fmin(0.0, __ddiv_rn(neg, 2.0));                          // :359-365
        gs[3] = sum;
        int32_t* st = g.gstat + (size_t)gi * 4;
        st[0] = maxdeg; st[1] = nnz; st[2] = 0; st[3] = flags;
    }
}

__global__ void wgraph_dmax_kernel(const eco_wgraphs_t g) {
    int m = 1;
    for (int i = threadIdx.x; i < g.G; i += 32) m = max(m, g.gstat[(size_t)i * 4]);
    m = group_max<32>(m);
    if (threadIdx.x == 0) g.dmax[0] = (float)m;
}

// ------------------------------------------------------------------------------------------------ reset
// one warp per episode (not on the per-step path: O(N^2) per episode, once)
__global__ void __launch_bounds__(128) wenv_reset_kernel(const eco_wgraphs_t g, const eco_wenv_t we,
                                                         const int32_t* __restrict__ graph_idx,
                                                         const int8_t* __restrict__ init_spins) {
    const eco_env_t& env = we.base;
    const int lane = threadIdx.x & 31;
    long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= env.B) return;                                             // whole warps leave together
    const int N = env.N, NP = env.NP;
    const int gi = graph_idx[b];
    const double* Jg = g.J + (size_t)gi * NP * NP;
    int8_t* spins = env.spins + (size_t)b * NP;
    double* hf = we.h + (size_t)b * NP;
    const double mlr = g.gscal[(size_t)gi * 4 + 0];

    for (int i = lane; i < NP; i += 32) {
        spins[i] = i < N ? init_spins[(size_t)b * N + i] : (int8_t)0;
        env.last_flip[(size_t)b * NP + i] = 0;
    }
    for (int w = lane; w < env.NW; w += 32) env.diff_bits[(size_t)b * env.NW + w] = 0u;
    if (lane == 0) env.graph_idx[b] = gi;
    __syncwarp();

    int nimp = 0;
    double ssh = 0.0;
    float* x0 = env.xn + (size_t)b * 3 * NP;
    for (int i = lane; i < NP; i += 32) {
        double acc = 0.0;                                               // h_i = sum_j J_ij s_j
        for (int j = 0; j < N; ++j) acc = __dadd_rn(acc, __dmul_rn(Jg[(size_t)i * NP + j], (double)spins[j]));
        hf[i] = acc;
        const int si = spins[i];
        const double gain = __dmul_rn((double)si, acc);                 // calculate_cut_changes (utils.py:97-102)
        ssh = __dadd_rn(ssh, gain);
        nimp += gain > 0.0;
        x0[i] = (float)si;                                              // spinsystem.py:294/299
        x0[NP + i] = i < N ? (float)__ddiv_rn(gain, mlr) : 0.f;        // :311-312
        x0[2 * NP + i] = 0.f;
    }
    nimp = group_sum<32>(nimp);
    ssh = group_sum_d<32>(ssh);
    if (lane == 0) {
        const double qn = g.gscal[(size_t)gi * 4 + 1], lb = g.gscal[(size_t)gi * 4 + 2], sumJ = g.gscal[(size_t)gi * 4 + 3];
        // utils.py:90-94: 1/4 sum_ij J_ij (1 - s_i s_j) = (sum J - s.h) / 4 (exact for integer couplings)
        const double cut = __dmul_rn(__dsub_rn(sumJ, ssh), 0.25);
        const double score = __dadd_rn(cut, fabs(fmin(0.0, lb)));      // score_solver.py:196-200
        const double nscore = __ddiv_rn(score, qn);                    // :190-194
        eco_episode_t e;
        e.step = 0; e.cut = 0; e.best_cut = 0; e.dist = 0; e.n_improving = nimp; e.flags = 0;
        e.n_visited = 0; e.reserved = 0;
        e.score = score; e.nscore = nscore; e.best_score = score; e.best_nscore = nscore;
        e.key[0] = 0; e.key[1] = 0; e.total_reward = 0.0; e.last_reward = 0.0;
        env.ep[b] = e;
        *reinterpret_cast<double2*>(we.cut + 2 * b) = make_double2(cut, cut);
        *reinterpret_cast<float4*>(env.xg + (size_t)b * 4) = make_float4(0.f, 0.f, env.frac_tab[nimp], 0.f);   // :321-322
    }
}

// ------------------------------------------------------------------------------------------------ step
// TPE lanes per episode, four vertices per lane and pass (16-byte spin / 32-byte field and coupling / 16-byte feature
// accesses).  Same structure as env_step_kernel (env_kernels.cu) with fp64 fields.
template <int TPE>
__global__ void __launch_bounds__(128) wenv_step_kernel(const eco_wgraphs_t g, const eco_wenv_t we, const int policy,
                                                        const int32_t* __restrict__ actions, double* __restrict__ reward_out,
                                                        uint8_t* __restrict__ done_out, int32_t* __restrict__ hist_a,
                                                        double* __restrict__ hist_r, double* __restrict__ hist_s) {
    const eco_env_t& env = we.base;
    const int lane = threadIdx.x % TPE;
    long long b = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / TPE;
    const bool in_range = b < env.B;
    if (!in_range) b = env.B - 1;                                       // keep every lane alive for the group shuffles
    const int N = env.N, NP = env.NP, NQ = NP >> 2;

    eco_episode_t* ep = env.ep + b;
    const int4 e0 = *reinterpret_cast<const int4*>(ep);                 // step, cut (unused), best_cut (unused), dist
    const int4 e1 = *(reinterpret_cast<const int4*>(ep) + 1);           // n_improving, flags, n_visited, reserved
    const int flags = e1.y;
    const int step_new = e0.x + 1;
    bool active = in_range && !(flags & (FLAG_DONE | FLAG_STOPPED)) && step_new <= env.T;   // :365-367
    const int gi = env.graph_idx[b];
    int8_t* spins = env.spins + (size_t)b * NP;
    double* hf = we.h + (size_t)b * NP;
    uint16_t* lf = env.last_flip + (size_t)b * NP;

    int a;
    if (policy == ECO_POLICY_GREEDY) {
        // argmax_i s_i h_i in fp64, first maximal index (numpy argmax, solver.py:116)
        double bv = -INFINITY;
        int bi = INT_MAX;
        for (int q = lane; q < NQ; q += TPE) {
            const uint32_t sw = *reinterpret_cast<const uint32_t*>(spins + 4 * q);
            const double2 h01 = *reinterpret_cast<const double2*>(hf + 4 * q);
            const double2 h23 = *reinterpret_cast<const double2*>(hf + 4 * q + 2);
            const double hv[4] = {h01.x, h01.y, h23.x, h23.y};
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const double gain = __dmul_rn((double)sx8(sw, kk), hv[kk]);
                if (4 * q + kk < N && gain > bv) { bv = gain; bi = 4 * q + kk; }
            }
        }
#pragma unroll
        for (int o = TPE / 2; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, o, TPE);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o, TPE);
            if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
        a = bi;
        if (active && !(bv >= 0.0)) {                                   // solver.py:124: stop only if the best gain is < 0
            active = false;
            if (lane == 0) ep->flags = flags | FLAG_STOPPED;
        }
    } else {
        a = actions[b];
    }
    if (a < 0 || a >= N) { a = 0; active = false; }

    const int s_a_old = spins[a];
    const double h_a_old = hf[a];
    const uint32_t old_word = env.diff_bits[(size_t)b * env.NW + (a >> 5)];
    __syncwarp();                                                       // pre-flip values read before anyone writes

    const double mlr = g.gscal[(size_t)gi * 4 + 0];
    int nimp = 0;
    if (active) {
        const double* Jrow = g.J + ((size_t)gi * NP + a) * NP;
        const double two_sa = -2.0 * (double)s_a_old;                   // 2 s_a (new spin)
        const float* tsf_now = env.tsf_tab + step_new;                  // time since flip of vertex k: tsf_now[-last_flip[k]]
        const int qa = a >> 2, ka = a & 3;
        for (int q = lane; q < NQ; q += TPE) {
            uint32_t sw = *reinterpret_cast<const uint32_t*>(spins + 4 * q);
            const double2 j01 = *reinterpret_cast<const double2*>(Jrow + 4 * q);
            const double2 j23 = *reinterpret_cast<const double2*>(Jrow + 4 * q + 2);
            const double2 h01 = *reinterpret_cast<const double2*>(hf + 4 * q);
            const double2 h23 = *reinterpret_cast<const double2*>(hf + 4 * q + 2);
            uint2 lw = *reinterpret_cast<const uint2*>(lf + 4 * q);
            if (q == qa) {                                              // the flipped vertex: new spin, last-flip step
                sw ^= 0xFEu << (8 * ka);
                const uint32_t sh = 16 * (ka & 1), keep = ~(0xFFFFu << sh), val = ((uint32_t)step_new & 0xFFFFu) << sh;
                if ((ka >> 1) == 0) lw.x = (lw.x & keep) | val;
                else lw.y = (lw.y & keep) | val;
            }
            const double jv[4] = {j01.x, j01.y, j23.x, j23.y};
            double hv[4] = {h01.x, h01.y, h23.x, h23.y};
            const uint32_t lws[2] = {lw.x, lw.y};
            float f0[4], f1[4], f2[4];
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const int si = sx8(sw, kk);
                hv[kk] = __dadd_rn(hv[kk], __dmul_rn(jv[kk], two_sa));    // J_aa == 0: h_a is unchanged
                const double gain = __dmul_rn((double)si, hv[kk]);       // spinsystem.py:414-416
                nimp += gain > 0.0;
                f0[kk] = (float)si;
                f1[kk] = (float)__ddiv_rn(gain, mlr);                    // :490
                f2[kk] = tsf_now[-zx16(lws[kk >> 1], kk & 1)];           // :493-495
            }
            float* x0 = env.xn + (size_t)b * 3 * NP + 4 * q;
            *reinterpret_cast<float4*>(x0) = make_float4(f0[0], f0[1], f0[2], f0[3]);
            *reinterpret_cast<float4*>(x0 + NP) = make_float4(f1[0], f1[1], f1[2], f1[3]);
            *reinterpret_cast<float4*>(x0 + 2 * NP) = make_float4(f2[0], f2[1], f2[2], f2[3]);
            *reinterpret_cast<double2*>(hf + 4 * q) = make_double2(hv[0], hv[1]);
            *reinterpret_cast<double2*>(hf + 4 * q + 2) = make_double2(hv[2], hv[3]);
            if (q == qa) {
                *reinterpret_cast<uint32_t*>(spins + 4 * q) = sw;
                *reinterpret_cast<uint2*>(lf + 4 * q) = lw;
            }
        }
    }
    nimp = group_sum<TPE>(nimp);

    int new_best = 0;
    if (lane == 0 && active) {
        const double qn = g.gscal[(size_t)gi * 4 + 1];
        const double delta = __dmul_rn((double)s_a_old, h_a_old);          // :393 (a zero field gives -0.0, as in numpy)
        const double delta_n = __ddiv_rn(delta, qn);                      // :394
        const double sc[4] = {ep->score, ep->nscore, ep->best_score, ep->best_nscore};
        const uint64_t k0 = ep->key[0] ^ env.zobrist[2 * a], k1 = ep->key[1] ^ env.zobrist[2 * a + 1];
        uint64_t* tab = env.visited + (size_t)b * env.HCAP * 2;
        const uint32_t slot = (uint32_t)(k0 ^ (k0 >> 29)) & (env.HCAP - 1);
        ulonglong2 tv = make_ulonglong2(0, 0);
        if (env.use_basin) tv = *reinterpret_cast<const ulonglong2*>(tab + 2 * slot);
        const StepScalars r = bls_step_scalars(env, sc, delta, delta_n, nimp, e1.z, tab, slot, tv, k0, k1);
        const double2 cuts = *reinterpret_cast<const double2*>(we.cut + 2 * b);
        const double cut = __dadd_rn(cuts.x, delta);                      // CUT target: the score mask is the cut change
        int dist = e0.w + (((old_word >> (a & 31)) & 1u) ? -1 : 1);
        if (r.new_best) { dist = 0; new_best = 1; }
        const int done = step_new == env.T;                               // :541-544
        int4* epw = reinterpret_cast<int4*>(ep);
        epw[0] = make_int4(step_new, 0, 0, dist);
        epw[1] = make_int4(nimp, flags | (done ? FLAG_DONE : 0), r.n_visited, 0);
        *reinterpret_cast<double2*>(&ep->score) = make_double2(r.score, r.nscore);
        *reinterpret_cast<double2*>(&ep->best_score) = make_double2(r.best_score, r.best_nscore);
        *reinterpret_cast<ulonglong2*>(&ep->key[0]) = make_ulonglong2(k0, k1);
        *reinterpret_cast<double2*>(&ep->total_reward) = make_double2(__dadd_rn(ep->total_reward, r.rew), r.rew);
        *reinterpret_cast<double2*>(we.cut + 2 * b) = make_double2(cut, r.new_best ? cut : cuts.y);
        float4 xg;                                                        // rows 3..6 (spinsystem.py:509-527)
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
    } else if (lane == 0 && in_range) {
        if (reward_out) reward_out[b] = 0.0;
        if (done_out) done_out[b] = 1;
    }
    new_best = __shfl_sync(0xffffffffu, new_best, 0, TPE);
    if (new_best && active)
        for (int w = lane; w < env.NW; w += TPE) env.diff_bits[(size_t)b * env.NW + w] = 0u;
}

// ------------------------------------------------------------------------------------------------ results
__global__ void wenv_results_kernel(const eco_wenv_t we, double* __restrict__ best_cut, int8_t* __restrict__ best_spins,
                                    int32_t* __restrict__ steps) {
    const eco_env_t& env = we.base;
    const size_t total = (size_t)env.B * env.N;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int i = idx % env.N;
        const size_t b = idx / env.N;
        if (best_spins) {
            const int s = env.spins[b * env.NP + i];
            const uint32_t w = env.diff_bits[b * env.NW + (i >> 5)];
            best_spins[idx] = (int8_t)(((w >> (i & 31)) & 1u) ? -s : s);
        }
        if (i == 0) {
            if (best_cut) best_cut[b] = we.cut[2 * b + 1];
            if (steps) steps[b] = env.ep[b].step;
        }
    }
}

}  // namespace

int launch_wgraph_prepare(const eco_wgraphs_t* g, const double* dense, cudaStream_t st) {
    wgraph_prepare_kernel<<<g->G, 256, 0, st>>>(*g, dense);
    ECO_LAUNCH_CHECK();
    wgraph_dmax_kernel<<<1, 32, 0, st>>>(*g);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

int launch_wenv_reset(const eco_wgraphs_t* g, eco_wenv_t* we, const int32_t* gidx, const int8_t* spins, cudaStream_t st) {
    const eco_env_t& env = we->base;
    if (env.use_basin) ECO_CUDA(cudaMemsetAsync(env.visited, 0, (size_t)env.B * env.HCAP * 16, st));
    wenv_reset_kernel<<<(unsigned)(((long long)env.B * 32 + 127) / 128), 128, 0, st>>>(*g, *we, gidx, spins);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

int launch_wenv_step(const eco_wgraphs_t* g, eco_wenv_t* we, int policy, const int32_t* actions, double* reward, uint8_t* done,
                     int32_t* ha, double* hr, double* hs, cudaStream_t st) {
    const int NP = we->base.NP;
    const long long B = we->base.B;
    prof_begin(ECO_PROF_ENV_STEP, st);
#define ECO_WSTEP(TPE) \
    wenv_step_kernel<TPE><<<(unsigned)((B * TPE + 127) / 128), 128, 0, st>>>(*g, *we, policy, actions, reward, done, ha, hr, hs)
    if (NP <= 32) ECO_WSTEP(8);
    else if (NP <= 64) ECO_WSTEP(16);
    else ECO_WSTEP(32);
#undef ECO_WSTEP
    prof_end(ECO_PROF_ENV_STEP, st);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

int launch_wenv_results(const eco_wenv_t* we, double* best_cut, int8_t* best_spins, int32_t* steps, cudaStream_t st) {
    const size_t total = (size_t)we->base.B * we->base.N;
    const int blocks = (int)((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
    wenv_results_kernel<<<blocks, 256, 0, st>>>(*we, best_cut, best_spins, steps);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

}  // namespace eco
