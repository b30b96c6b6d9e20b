// The environment step of ONE episode by a group of TPE <= 32 lanes of a warp (8 vertices per lane), as a device function:
// the body of env_step_sw_kernel (env_kernels.cu), shared with the MPNN kernel (mpnn_tc.cu), whose readout warp applies the
// flip it has just chosen instead of leaving it to a second launch.
//
// Replaces (reference, file:line) src/envs/spinsystem.py:355-559 SpinSystemBase.step for the ECO-DQN Max-Cut configuration
// (reversible spins, BLS reward, CUT target: `env.reserved == 0`, no ECO_GRAPHS_MIN_CUT); see env_kernels.cu for the
// layout and the fp64 bookkeeping rules.
#pragma once
#include <limits.h>

#include "eco_common.cuh"

namespace eco {

union V8s { uint2 v; int8_t b[8]; };
union V8h { uint4 v; int16_t h[8]; };
union V8u { uint4 v; uint16_t h[8]; };
union V4s { uint32_t v; int8_t b[4]; };      // four vertices: env_step_ring_kernel
union V4h { uint2 v; int16_t h[4]; };
union V4u { uint2 v; uint16_t h[4]; };

__device__ __forceinline__ float feat_gain(int gain, double mlr) {
    // row 1: immediate_quality_changes / max_local_reward in fp64, then the driver's fp32 cast
    return (float)__ddiv_rn((double)gain, mlr);
}
// (An exact fp32 alternative exists -- __fdiv_rn((float)gain, (float)mlr) equals the fp64-then-fp32 result because double
// rounding is innocuous for a division when 53 >= 2*24+2 -- but it costs more issue slots than the table lookup: measured
// 448 us vs 330 us per launch in env_step_ring_kernel.)

// a / m for small integers by one multiplication with the correctly rounded reciprocal y = RN(1 / m) and two FMAs
// (Markstein's correction step):  q0 = RN(a y),  r = a - q0 m (exact in one FMA),  q = RN(q0 + r y)  ==  RN(a / m)  ==
// (float)((double)a / (double)m).  Checked exhaustively against the fp64-then-fp32 expression for every |m| <= 2048,
// |a| <= 70000, signed zeros included (tests/test_capi_cpu.py::test_small_int_division_identity restates the check in C).
struct SmallDiv {
    float m, y;      // divisor and its correctly rounded reciprocal
    bool ok;         // integer divisor, non-zero, in the checked range (otherwise the caller divides in fp64)
};
__device__ __forceinline__ SmallDiv small_div_setup(double mlr, bool integer_couplings) {
    SmallDiv d;
    d.m = (float)mlr;
    d.ok = integer_couplings && mlr != 0.0 && fabs(mlr) <= 2048.0;
    d.y = __frcp_rn(d.ok ? d.m : 1.f);
    return d;
}
__device__ __forceinline__ float small_div(float a, const SmallDiv& d) {     // |a| <= 70000, integer-valued
    const float q0 = __fmul_rn(a, d.y);
    const float r = __fmaf_rn(-q0, d.m, a);
    return __fmaf_rn(r, d.y, q0);
}
// byte / half-word extraction in one PRMT each (selector bit 3 replicates the sign of the selected byte; __byte_perm ignores
// that bit, hence the PTX form)
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}
__device__ __forceinline__ int sx8(uint32_t w, int k) { return (int)prmt(w, 0, k | ((8 | k) << 4) | ((8 | k) << 8) | ((8 | k) << 12)); }
__device__ __forceinline__ int sx16(uint32_t w, int hh) {
    return (int)prmt(w, 0, (2 * hh) | ((2 * hh + 1) << 4) | ((8 | (2 * hh + 1)) << 8) | ((8 | (2 * hh + 1)) << 12));
}
__device__ __forceinline__ int zx16(uint32_t w, int hh) { return (int)prmt(w, 0, (2 * hh) | ((2 * hh + 1) << 4) | 0x4400); }

// The scalar part of one ECO-DQN step (lane 0 of an episode), in the reference's fp64 operation order (appendix A.2):
// score / normalised score (spinsystem.py:399-400), BLS reward (:418-424), basin reward through the visited set (:443-457),
// best tracking (:459-463).  delta / delta_n: the score mask and normalised score mask at the action (:393-394).  The
// visited-set slot `tv` at `slot` of `tab` was requested by the caller (k0 / k1: the Zobrist key after the flip).  Shared
// by the int8 steps (env_step_group below, env_step_ring_kernel) and the fp64-field kernel of weighted graphs (weighted.cu).
struct StepScalars {
    double score, nscore, best_score, best_nscore, rew;
    int n_visited;
    bool new_best;
};
__device__ __forceinline__ StepScalars bls_step_scalars(const eco_env_t& env, const double (&sc)[4], double delta,
                                                        double delta_n, int nimp, int n_visited, uint64_t* tab, uint32_t slot,
                                                        ulonglong2 tv, uint64_t k0, uint64_t k1) {
    StepScalars r;
    r.score = __dadd_rn(sc[0], delta);                                 // :399
    r.nscore = __dadd_rn(sc[1], delta_n);                              // :400
    r.rew = 0.0;
    if (r.score > sc[2]) r.rew = __dsub_rn(r.nscore, sc[3]);           // :418-424
    if (env.use_basin) {                                               // :443-457
        const uint64_t w0 = k0 ^ VISITED_SALT0, w1 = k1 ^ VISITED_SALT1;
        bool is_new = false;
        for (int probe = 0; probe < env.HCAP; ++probe) {
            if (tv.x == 0 && tv.y == 0) {
                *reinterpret_cast<ulonglong2*>(tab + 2 * slot) = make_ulonglong2(w0, w1);
                is_new = true; ++n_visited;
                break;
            }
            if (tv.x == w0 && tv.y == w1) break;
            slot = (slot + 1) & (env.HCAP - 1);
            tv = *reinterpret_cast<const ulonglong2*>(tab + 2 * slot);
        }
        if (nimp == 0 && is_new) r.rew = __dadd_rn(r.rew, env.basin_reward);
    }
    r.n_visited = n_visited;
    r.new_best = r.score > sc[2];                                      // :459-463
    r.best_score = r.new_best ? r.score : sc[2];
    r.best_nscore = r.new_best ? r.nscore : sc[3];
    return r;
}

// Latency-optimised form for NP <= 256: everything that does not depend on the action is requested first, the flipped
// vertex's old spin / field come from a shuffle, the visited-set slot is prefetched, observable row 1 and the normalised
// score change come from per-graph tables.  All TPE lanes of the group must call it (group shuffles); lanes of an episode
// out of range pass in_range = false with b clamped.
// WIDE: a lane's eight values of a feature row -- one 32-byte sector -- leave in ONE 256-bit store (two 16-byte stores each
// fill half a sector: twice the write transactions, measured on env_step_ring_kernel).  The tail warp of mpnn_tc_kernel
// instantiates the narrow form: 12 live feature registers instead of 24 inside the resident kernel's 96-register budget.
template <int TPE, bool WIDE = true>
__device__ __forceinline__ void env_step_group(const eco_graphs_t& g, const eco_env_t& env, long long b, const int lane,
                                               const bool in_range, const int policy, const int action,
                                               double* __restrict__ reward_out, uint8_t* __restrict__ done_out,
                                               int32_t* __restrict__ hist_a, double* __restrict__ hist_r,
                                               double* __restrict__ hist_s) {
    const int N = env.N, NP = env.NP, NCH = NP >> 3;
    const bool has = lane < NCH;

    // ---- round 1: loads that do not depend on the action ------------------------------------------------
    eco_episode_t* ep = env.ep + b;
    const int4 e0 = *reinterpret_cast<const int4*>(ep);            // step, cut, best_cut, dist
    const int4 e1 = *(reinterpret_cast<const int4*>(ep) + 1);      // n_improving, flags, n_visited, reserved
    const int gi = env.graph_idx[b];
    int a = policy == ECO_POLICY_GREEDY ? 0 : action;
    int8_t* spins = env.spins + (size_t)b * NP;
    int16_t* hf = env.hfield + (size_t)b * NP;
    uint16_t* lf = env.last_flip + (size_t)b * NP;
    V8s s; V8h h; V8u l;
    s.v = make_uint2(0, 0); h.v = make_uint4(0, 0, 0, 0); l.v = make_uint4(0, 0, 0, 0);
    if (has) {
        s.v = *reinterpret_cast<const uint2*>(spins + lane * 8);
        h.v = *reinterpret_cast<const uint4*>(hf + lane * 8);
        l.v = *reinterpret_cast<const uint4*>(lf + lane * 8);
    }
    double sc[4] = {0, 0, 0, 0};
    ulonglong2 key = make_ulonglong2(0, 0);
    double total_reward = 0.0;
    if (lane == 0) {
        const double2 d0 = *reinterpret_cast<const double2*>(&ep->score);
        const double2 d1 = *reinterpret_cast<const double2*>(&ep->best_score);
        sc[0] = d0.x; sc[1] = d0.y; sc[2] = d1.x; sc[3] = d1.y;
        key = *reinterpret_cast<const ulonglong2*>(&ep->key[0]);
        total_reward = ep->total_reward;
    }
    const int flags = e1.y;
    const int step_new = e0.x + 1;
    bool active = in_range && !(flags & (FLAG_DONE | FLAG_STOPPED)) && step_new <= env.T;

    if (policy == ECO_POLICY_GREEDY) {
        int best = INT_MIN;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int i = lane * 8 + k;
            if (has && i < N)
                best = max(best, (int)((((uint32_t)(s.b[k] * h.h[k] + 32768) << 16) | (uint32_t)(0xFFFF - i)) ^ 0x80000000u));
        }
        best = group_max<TPE>(best);
        const uint32_t ukey = (uint32_t)best ^ 0x80000000u;
        a = 0xFFFF - (int)(ukey & 0xFFFFu);
        if (active && ((int)(ukey >> 16) - 32768) < 0) {
            active = false;
            if (lane == 0) ep->flags = flags | FLAG_STOPPED;
        }
    }
    if (a < 0 || a >= N) { a = 0; active = false; }

    // ---- round 2: loads that depend on the action / graph -----------------------------------------------
    V8s j;
    j.v = make_uint2(0, 0);
    if (has && active) j.v = *reinterpret_cast<const uint2*>(g.J + ((size_t)gi * NP + a) * NP + lane * 8);
    const double mlr = g.gscal[(size_t)gi * 4 + 0];
    const bool use_tab = (g.reserved & ECO_GRAPHS_PM1) != 0;       // couplings in {-1,0,1}: |gain| <= degree < NP
    const float* gtab = g.gain_tab + (size_t)gi * tab_stride(NP) + NP;
    double qn = 1.0;
    ulonglong2 zob = make_ulonglong2(0, 0);
    uint32_t old_word = 0;
    if (lane == 0) {
        if (!use_tab) qn = g.gscal[(size_t)gi * 4 + 1];
        zob = *reinterpret_cast<const ulonglong2*>(env.zobrist + 2 * a);
        old_word = env.diff_bits[(size_t)b * env.NW + (a >> 5)];
    }
    // the flipped vertex's current spin and field: element a&7 of lane a>>3
    const int ka = a & 7;
    const uint32_t sw = ka < 4 ? s.v.x : s.v.y;
    const int my_s = (int)(int8_t)(sw >> (8 * (ka & 3)));
    const uint32_t hw = ka < 2 ? h.v.x : (ka < 4 ? h.v.y : (ka < 6 ? h.v.z : h.v.w));
    const int my_h = (int)(int16_t)(hw >> (16 * (ka & 1)));
    const int s_a_old = __shfl_sync(0xffffffffu, my_s, a >> 3, TPE);
    const int h_a_old = __shfl_sync(0xffffffffu, my_h, a >> 3, TPE);
    const int s_a_new = -s_a_old;

    // ---- round 3: the visited-set slot (lane 0) -----------------------------------------------------------
    const uint64_t k0 = key.x ^ zob.x, k1 = key.y ^ zob.y;
    uint64_t* tab = env.visited + (size_t)b * env.HCAP * 2;
    uint32_t slot = (uint32_t)(k0 ^ (k0 >> 29)) & (env.HCAP - 1);
    ulonglong2 tv = make_ulonglong2(0, 0);
    const int delta = s_a_old * h_a_old;                                // spinsystem.py:393
    double delta_n = 0.0;
    if (lane == 0 && active) {
        if (env.use_basin) tv = *reinterpret_cast<const ulonglong2*>(tab + 2 * slot);
        if (use_tab) delta_n = __ldg(g.dn_tab + (size_t)gi * tab_stride(NP) + NP + delta);   // requested early, used late
    }

    // ---- O(N) local-field update + per-vertex observables ----------------------------------------------
    int nimp = 0;
    if (has && active) {
        float* x0 = env.xn + (size_t)b * 3 * NP + lane * 8;
        auto vertex = [&](int k, float& o0, float& o1, float& o2) {
            const int i = lane * 8 + k;
            int si = s.b[k];
            if (i == a) { si = s_a_new; s.b[k] = (int8_t)si; l.h[k] = (uint16_t)step_new; }
            const int hi = h.h[k] + 2 * j.b[k] * s_a_new;
            h.h[k] = (int16_t)hi;
            const int gain = si * hi;
            nimp += gain > 0;
            o0 = (float)si;
            o1 = use_tab ? __ldg(gtab + gain) : feat_gain(gain, mlr);
            o2 = __ldg(env.tsf_tab + (step_new - l.h[k]));
        };
        if (WIDE) {
            float f0[8], f1[8], f2[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) vertex(k, f0[k], f1[k], f2[k]);
            st_f32x8(x0, f0);
            st_f32x8(x0 + NP, f1);
            st_f32x8(x0 + 2 * NP, f2);
        } else {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                float f0[4], f1[4], f2[4];
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) vertex(half * 4 + kk, f0[kk], f1[kk], f2[kk]);
                *reinterpret_cast<float4*>(x0 + 4 * half) = make_float4(f0[0], f0[1], f0[2], f0[3]);
                *reinterpret_cast<float4*>(x0 + NP + 4 * half) = make_float4(f1[0], f1[1], f1[2], f1[3]);
                *reinterpret_cast<float4*>(x0 + 2 * NP + 4 * half) = make_float4(f2[0], f2[1], f2[2], f2[3]);
            }
        }
        *reinterpret_cast<uint4*>(hf + lane * 8) = h.v;
        if ((a >> 3) == lane) {
            *reinterpret_cast<uint2*>(spins + lane * 8) = s.v;
            *reinterpret_cast<uint4*>(lf + lane * 8) = l.v;
        }
    }
    nimp = group_sum<TPE>(nimp);

    // ---- scalar bookkeeping, lane 0, in the reference's fp64 operation order (appendix A.2) ---------------
    int new_best = 0;
    if (lane == 0 && active) {
        if (!use_tab) delta_n = __ddiv_rn((double)delta, qn);           // :394
        const int cut = e0.y + delta;
        const StepScalars r = bls_step_scalars(env, sc, (double)delta, delta_n, nimp, e1.z, tab, slot, tv, k0, k1);
        const double score = r.score, nscore = r.nscore, rew = r.rew, nbs = r.best_score, nbn = r.best_nscore;
        const int n_visited = r.n_visited;
        int dist = e0.w + (((old_word >> (a & 31)) & 1u) ? -1 : 1);
        int best_cut = e0.z;
        if (r.new_best) { best_cut = cut; dist = 0; new_best = 1; }
        const int done = step_new == env.T;                             // :541-544
        int4* epw = reinterpret_cast<int4*>(ep);
        epw[0] = make_int4(step_new, cut, best_cut, dist);
        epw[1] = make_int4(nimp, flags | (done ? FLAG_DONE : 0), n_visited, 0);
        *reinterpret_cast<double2*>(&ep->score) = make_double2(score, nscore);
        *reinterpret_cast<double2*>(&ep->best_score) = make_double2(nbs, nbn);
        *reinterpret_cast<ulonglong2*>(&ep->key[0]) = make_ulonglong2(k0, k1);
        *reinterpret_cast<double2*>(&ep->total_reward) = make_double2(__dadd_rn(total_reward, rew), rew);
        float4 xg;                                                      // rows 3..6 (spinsystem.py:509-527)
        const double gap = fabs(__dsub_rn(score, nbs));                 // integer-valued for integer couplings
        xg.x = (float)__ddiv_rn(gap, mlr);
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
    } else if (lane == 0 && in_range) {
        if (reward_out) reward_out[b] = 0.0;
        if (done_out) done_out[b] = 1;
    }
    new_best = __shfl_sync(0xffffffffu, new_best, 0, TPE);
    if (new_best && active && lane < env.NW) env.diff_bits[(size_t)b * env.NW + lane] = 0u;   // NW <= 8 <= TPE... see launch
}

}  // namespace eco
