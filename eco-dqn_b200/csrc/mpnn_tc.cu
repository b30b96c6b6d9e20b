// Kernel family 2b: MPNN Q-network forward + argmax on the 5th-gen tensor cores (tcgen05 + TMEM), sm_100a.
//
// Replaces (reference, file:line) src/networks/mpnn.py:40-159 (MPNN.forward and its three layer classes) and
// the argmax of experiments/utils.py:57-66, for graphs with couplings in {-1,0,+1} and N <= 208.
//
// One persistent CTA per SM runs whole episodes; every activation stays on chip between the layers:
//
//   orientation   D^T[feature, vertex] = W[feature, k] * X^T[k, vertex]   (linears:   A-operand = weights, TMEM)
//                 D^T[feature, vertex] = H^T[feature, j] * A[j, vertex]   (aggregate: B-operand = adjacency, smem)
//   precision     every activation / weight x is stored as hi = bf16(x), lo = bf16(x - hi): two bf16 terms, about 16
//                 mantissa bits per operand, fp32 accumulation (measured against the reference's fp32 Q-values: at most
//                 0.03 of the parity tolerance 1e-3 |q| + 1e-4 max|q|; one fp16 / tf32 term per operand measured 10-20x
//                 OVER it, tools/precision_study.py).  hi and lo rows are STACKED in the M dimension (128 = 64 features x
//                 {hi,lo}), so one M=128 MMA chain yields both partial products and the split costs no extra
//                 instructions for the aggregation (A in {-1,0,1} is exact) and 2 chains for the linears: W_hi X_hi, W_lo X_hi
//                 (M = 128) and W_hi X_lo (M = 64, the hi rows only: lo x lo is never computed -- issue_part()).
//                 Stacked row order r = 32q + 16s + t  <->  feature 16q + t, s in {hi, lo}: the two halves of a
//                 feature sit in the same TMEM lane quadrant, so one warp adds them after two 16x256b loads.
//   smem          adjacency bf16 (N x N, K-major core matrices), H^T and E^T stacked hi/lo (one copy serves as
//                 K-major A-operand of the aggregation AND MN-major B-operand of the linears), one 64-vertex chunk
//                 buffer per warp group.  No swizzle: 8x16-byte core matrices, written conflict-free by the epilogues.
//   TMEM          cols 0..207 aggregation accumulator (the linears of a chunk accumulate in place in its consumed
//                 columns), 208..335 one 64-column accumulator per group, 336.. weight A-operands (tcgen05.st from
//                 registers, straight from L2); the edge-stage A-operands S = R+ + R-, D = R+ - R- live in TMEM too
//                 (g = (|A| S + A D) / (2 deg), SURVEY.md section 7 identity).
//   edge stage    ReLU(W_e [a_ij ; x_j]) = ReLU(a_ij w0 + P_j): two dense N x N contractions instead of the
//                 reference's [B,N,N,63] intermediate; the MMAs of k-step block r are issued as soon as the workers have
//                 stored S / D of round r, so the contraction runs behind the CUDA-core stage that feeds it.
//   schedule      20 warps.  Warps 0-15 only ever run epilogues (TMEM -> registers -> split -> smem): two groups of 8
//                 (2 warps per TMEM lane quadrant), each owning up to two column chunks (208 vertices: 64, 48 | 48, 48)
//                 that it processes interleaved -- the MMAs of one chunk run under the epilogue of the other.  Warp 16
//                 issues the N x N contractions (edge stage, aggregation per column half).  Warps 17 / 18 issue the
//                 linear-layer MMAs of group 0 / 1: a worker warp that has written its part of a batch's operands fences
//                 and arrives on the issuer's mbarrier (no CTA or group barrier inside a layer); the issuer commits every
//                 batch to one of the group's three mbarriers (B1, B2, B3) that the workers wait on before they touch
//                 its results.  Warp 19 works through the tail of the PREVIOUS episode (pooling, W_p, Q, argmax and, in a
//                 rollout, SpinSystemBase.step for that episode; packed mode: the K episodes of the previous pack) while
//                 the others are on the next one.
//   rollout       FUSED: one launch per rollout -- every CTA takes its own episodes through all steps, two or three
//                 episodes at a time (see FusedEnv).
#include <cuda_bf16.h>
#include <stdlib.h>

#include "eco_common.cuh"
#include "tc_prims.cuh"
#include "mpnn_pack.cuh"
#include "env_step_device.cuh"

namespace eco {
namespace {

using namespace tc;

constexpr int NPMAX = 208;
constexpr int PACK_NPMAX = 192;   // packed mode: K graphs of NP <= 96 vertices, K * NP <= 192 (leaves room behind the image)
constexpr int CHUNK = 64;        // max vertices per linear-layer chunk (accumulator columns)
constexpr int SUBS = 2;            // warps per (group, TMEM lane quadrant): they split the 16-column blocks of every epilogue
constexpr int THREADS = 256 * SUBS;
constexpr int GROUP_THREADS = 128 * SUBS;
constexpr int NWARPS = THREADS / 32;
constexpr int ISSUERS = 4;                     // warp 16: the N x N contractions; warps 17, 18: the linear layers of group 0 / 1;
                                               // warp 19: the tail of every episode (readout, argmax, fused env step)
constexpr int LAUNCH_THREADS = THREADS + 32 * ISSUERS;   // (tcgen05.mma issue blocks while the tensor queue is full, which
                                                         //  must not hold up an epilogue warp: the workers never issue)

// ---- TMEM column map -------------------------------------------------------------------------------------
constexpr uint32_t T_ACC0 = 0;       // 208 cols: aggregation / edge accumulator
constexpr uint32_t T_ACC1 = 208;     // 2 x 64 cols: linear accumulators of group 0 / group 1 (chunk relative)
constexpr uint32_t T_WM = 336;       // 64 cols: message weights (128 stacked rows x 128 k, bf16 pairs)
constexpr uint32_t T_WU = 400;       // 64 cols: update weights
constexpr uint32_t T_WEF = 464;      // 32 cols: edge-feature weights (k = 64)
constexpr uint32_t T_S = 208;        // 104 cols: edge-stage A-operand S   (dead before ACC1 / WM / WU are live)
constexpr uint32_t T_D = 312;        // 104 cols: edge-stage A-operand D

// ---- shared memory map (bytes) -----------------------------------------------------------------------------
constexpr int SM_A = 0;                                  // adjacency, bf16, up to 208 x 208
constexpr int SM_H = SM_A + NPMAX * NPMAX * 2;           // H^T stacked [128][208]
constexpr int SM_E = SM_H + 128 * NPMAX * 2;             // E^T stacked
constexpr int SM_T = SM_E + 128 * NPMAX * 2;             // chunk buffers [2 groups][128][48]
constexpr int SM_ABS = SM_H;                             // |A| overlays H and E during the edge stage
constexpr int SM_XF = SM_T + 128 * CHUNK * 2;            // float xf[7][208] overlays group 1's chunk buffer (dead by then)
constexpr int SM_DEG = SM_T + 2 * 128 * CHUNK * 2;       // float rdeg[208] = 1/deg
constexpr int SM_QP = SM_DEG + NPMAX * 4;                // float qpart[4][208]
constexpr int MAXCHUNKS = (NPMAX + CHUNK - 1) / CHUNK;
constexpr int SM_PP = SM_QP + 4 * NPMAX * 4;             // float ppart[MAXCHUNKS][SUBS][64]: per-chunk pooled partial sums
constexpr int SM_MISC = SM_PP + MAXCHUNKS * SUBS * 64 * 4;   // c0, cross-warp reductions (pooled[64] overlays rdeg)
constexpr int SM_TOTAL = SM_MISC + 64 + 16 * 4 + 16 * 4;
static_assert(NPMAX * NPMAX * 2 <= 2 * 128 * NPMAX * 2, "|A| must fit in the H+E region");
static_assert(7 * NPMAX * 4 <= 128 * CHUNK * 2, "xf must fit in a chunk buffer");
static_assert(SM_TOTAL + 256 <= 227 * 1024, "shared memory budget (dynamic + static)");

__global__ void mpnn_pack_kernel(const eco_mpnn_t w, uint32_t* __restrict__ out) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= PK_WORDS) return;
    if (idx >= PK_WPT) {                 // W_p^T, plain fp32
        const int k = (idx - PK_WPT) >> 6, f = (idx - PK_WPT) & 63;
        out[idx] = __float_as_uint(w.w_pool[f * 64 + k]);
        return;
    }
    const float* src;
    int kw, rel, base;   // words per row, index within the matrix, matrix offset
    if (idx < PK_WM) { src = w.w_edge_feat; kw = 32; rel = idx; base = PK_WEF; }
    else if (idx < PK_WU) { const int l = (idx - PK_WM) / (128 * 64); src = w.w_msg[l]; kw = 64; rel = (idx - PK_WM) % (128 * 64); base = PK_WM + l * 128 * 64; }
    else { const int l = (idx - PK_WU) / (128 * 64); src = w.w_upd[l]; kw = 64; rel = (idx - PK_WU) % (128 * 64); base = PK_WU + l * 128 * 64; }
    const int r = rel / kw, c = rel % kw;
    const int f = 16 * (r >> 5) + (r & 15), s = (r >> 4) & 1;
    const float a = src[f * (2 * kw) + 2 * c], b = src[f * (2 * kw) + 2 * c + 1];
    uint32_t hi, lo;
    split2(a, b, hi, lo);
    out[base + packed_index(r, c, kw)] = s ? lo : hi;
}

struct Ctx {
    unsigned char* smem;
    uint32_t tmem;
    uint64_t* bar_all;     // completion of CTA-wide MMA batches (edge contraction, aggregation)
    uint64_t* bar_grp;     // completion of this group's linear MMAs (B1)
    uint64_t* bar_g2;      // second / third per-group MMA barrier (B2, B3): several batches of a group in flight at once
    uint64_t* bar_g3;
    uint32_t phase_all, phase_grp, phase_g2, phase_g3;
    int tid, warp, lane, q, grp, sub;
    int N, NP, NB;
};

// Linear-layer chunks.  The NP/16 column blocks are shared out between the two warp groups (group 0 takes the extra block:
// its aggregation columns are ready first), then each group's blocks are split into (at most) two chunks of <= CHUNK/16
// blocks, processed interleaved (208 vertices: 7 + 6 blocks -> chunks 64, 48 | 48, 48).  A larger share for group 0
// (8 + 5 blocks) was measured slower: 0.596 ms against 0.589 ms per launch.
__device__ __forceinline__ int group0_blocks(int nblocks) { return min((nblocks + 1) / 2, 2 * (CHUNK / 16)); }
__device__ __forceinline__ void workers_sync() { asm volatile("bar.sync 3, %0;" ::"n"(THREADS) : "memory"); }
__device__ __forceinline__ void cta_stage_sync() {   // operands written by every worker (smem: generic proxy; TMEM: st/ld retired)
    fence_proxy_async();
    tc_fence_before();
    workers_sync();
}
__device__ __forceinline__ void wait_all(Ctx& c) {
    mbar_wait(c.bar_all, c.phase_all);
    c.phase_all ^= 1;
    tc_fence_after();
}
__device__ __forceinline__ void wait_grp(Ctx& c) {
    mbar_wait(c.bar_grp, c.phase_grp);
    c.phase_grp ^= 1;
    tc_fence_after();
}
__device__ __forceinline__ void wait_g2(Ctx& c) {
    mbar_wait(c.bar_g2, c.phase_g2);
    c.phase_g2 ^= 1;
    tc_fence_after();
}
__device__ __forceinline__ void wait_g3(Ctx& c) {
    mbar_wait(c.bar_g3, c.phase_g3);
    c.phase_g3 ^= 1;
    tc_fence_after();
}

// weights: global packed [128][KW] words -> registers -> TMEM columns [tcol, tcol + KW); the two warps that share a
// lane quadrant split the columns.  Split in two so the L2 latency can be hidden behind a barrier / MMA wait.
template <int KW>
__device__ __forceinline__ void ldg_weights(const Ctx& c, const uint32_t* __restrict__ pk, uint4 (&buf)[KW / (8 * SUBS)]) {
    // this warp: quadrant q, 8-column groups [part * CGP, (part + 1) * CGP); buf[2i], buf[2i+1] = the two 4-word halves
    constexpr int CGP = KW / (16 * SUBS);
    const int part = c.grp * SUBS + c.sub;
    const uint4* src = reinterpret_cast<const uint4*>(pk) + ((c.q * (KW / 8) + part * CGP) * 2) * 32 + c.lane;
#pragma unroll
    for (int i = 0; i < 2 * CGP; ++i) buf[i] = __ldg(src + i * 32);
}
template <int KW>
__device__ __forceinline__ void sttm_weights(const Ctx& c, const uint4 (&buf)[KW / (8 * SUBS)], uint32_t tcol) {
    constexpr int CGP = KW / (16 * SUBS);
    const int part = c.grp * SUBS + c.sub;
#pragma unroll
    for (int i = 0; i < CGP; ++i) {
        const uint4 a = buf[2 * i], b = buf[2 * i + 1];
        const uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        tmem_st_32x32b_x8(tmem_addr(c.tmem, 32 * c.q, tcol + (part * CGP + i) * 8), v);
    }
}

// Epilogue over accumulator columns [col0, col0 + width) of `acc` (width % 16 == 0) by the warp owning quadrant q of
// one group: loads the hi-row and lo-row halves, adds them and calls fn(blk_col, v[8]) where v[i] belongs to feature
// 16q + lane/4 + 8*((i>>1)&1) and column blk_col + 8*(i>>2) + 2*(lane&3) + (i&1)  (blk_col relative to col0).
template <class Fn>
__device__ __forceinline__ void epilogue(const Ctx& c, uint32_t acc, int col0, int width, Fn fn) {
    for (int blk = c.sub; blk < width / 16; blk += SUBS) {
        uint32_t vh[8], vl[8];
        tmem_ld_16x256b_x2(tmem_addr(c.tmem, 32 * c.q, acc + col0 + 16 * blk), vh);
        tmem_ld_16x256b_x2(tmem_addr(c.tmem, 32 * c.q + 16, acc + col0 + 16 * blk), vl);
        tmem_ld_wait();
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; i += 2)
            add2(v[i], v[i + 1], __uint_as_float(vh[i]), __uint_as_float(vh[i + 1]), __uint_as_float(vl[i]), __uint_as_float(vl[i + 1]));
        fn(16 * blk, v);
    }
}

// Store the 8 epilogue values of a 16-column block into a stacked hi/lo buffer (core(rb, cb) at (cb*16 + rb)*128).
// `node0` = buffer-relative vertex index of the block's first column.
__device__ __forceinline__ void store_block(const Ctx& c, unsigned char* buf, int node0, const float (&v)[8]) {
    const int rowoff = 16 * (c.lane >> 2) + 4 * (c.lane & 3);
#pragma unroll
    for (int half = 0; half < 2; ++half) {          // columns +0 / +8
        const int cb = (node0 >> 3) + half;
#pragma unroll
        for (int fr = 0; fr < 2; ++fr) {            // feature rows lane/4 and lane/4 + 8
            uint32_t hi, lo;
            split2(v[4 * half + 2 * fr], v[4 * half + 2 * fr + 1], hi, lo);
            unsigned char* p = buf + ((cb * 16 + 4 * c.q + fr) * 128) + rowoff;
            *reinterpret_cast<uint32_t*>(p) = hi;             // rb = 4q + fr      (hi rows)
            *reinterpret_cast<uint32_t*>(p + 2 * 128) = lo;   // rb = 4q + 2 + fr  (lo rows)
        }
    }
}

// Half of a linear layer on a chunk (single issuing thread): acc (+)= W[:, 64*part .. 64*part+63] * X, X a stacked buffer
// used MN-major: k-step kq covers features 16kq..16kq+15, split s selects the hi / lo rows (256-byte steps).
__device__ __forceinline__ void issue_part(const Ctx& c, uint32_t acc_col, uint32_t tw, const unsigned char* x, int cb0,
                                           int width /* the MMAs' N */, bool accumulate) {
    // The lo x lo product is not computed: the MMAs that read the lo rows of X are issued with M = 64, whose 64 A / D rows are
    // TMEM lanes 32q + 0..15 -- exactly the hi rows of the stacked order -- so they add W_hi X_lo to the hi rows and leave the lo
    // rows (W_lo X_hi) alone.  Same cycles as M = 128, a quarter fewer MACs in every linear: the kernel runs against the
    // board's power cap, and this alone took the SM clock from ~1.90 back to 1.965 GHz (+1.3 % env-steps/s).
    const uint32_t idesc = instr_desc_bf16(128, width, false, true);
    const uint32_t idesc_lo = instr_desc_bf16(64, width, false, true);
    const uint64_t d = smem_desc(smem_u32(x) + cb0 * 2048, /*LBO (k groups)*/ 128, /*SBO (vertex groups)*/ 2048);
#pragma unroll
    for (int i = 0; i < 8; ++i)     // i = 2*kq + s
        mma_ts(c.tmem + acc_col, c.tmem + tw + 8 * (i >> 1), d + (uint64_t)(16 * i), (i & 1) ? idesc_lo : idesc, accumulate || i > 0);
}

// PACKED: K = packK >= 2 small graphs (NP <= 96) are processed side by side as ONE block-diagonal graph of K * NP <= 192
// vertices ("pack"): the tensor part below does not know about it; only the inputs (per-vertex episode), the operand
// images (diagonal blocks: fetched by the 32 lanes of the contraction issuer), feature 63 and the readout (pooling / argmax
// per episode: the tail warp, readout_packed_warp) are per episode.
// FUSED (rollouts of the ECO-DQN configuration): the warp that has just taken an episode's argmax also applies the flip --
// SpinSystemBase.step for that episode (env_step_device.cuh), state and next observations written back -- and, because
// episodes never interact, the CTA then simply carries on: it takes ITS episodes through all `n_steps` steps of the rollout
// in one launch, with no grid-wide synchronisation at all.  Its episode list is cut into windows of two consecutive entries
// (the last window takes a third when the count is odd); a window goes through all steps, its members taking turns, before
// the next window starts: item = (window, step, member).  So only the operand images of 2 - 3 episodes per CTA are live at
// a time (148 CTAs x 3 x 173 kB <= 77 MB at N = 200: they stay in L2, and each is read from HBM once per rollout rather
// than once per step, which a step-major order over 4096 distinct graphs = 708 MB of images would need).  An episode's next
// observations are read (cp.async.cg: L2, never a stale L1 line) at least one whole item after the tail warp wrote and
// fenced them, which needs >= 2 members per window, i.e. >= 2 episodes per CTA (checked by the launcher).  A rollout is ONE
// launch instead of 2 T.
struct FusedEnv {
    eco_env_t env;
    int32_t* hist_a;
    double* hist_r;
    double* hist_s;
    int n_steps;
};

template <bool PACKED, bool TLINE, bool FUSED = false>
__global__ void __launch_bounds__(LAUNCH_THREADS, 1)
mpnn_tc_kernel(const eco_graphs_t g, const eco_mpnn_t w, const int B, const int32_t* __restrict__ graph_idx,
               const float* __restrict__ xn, const float* __restrict__ xg, const float norm_max,
               float* __restrict__ q_out, int32_t* __restrict__ act_out, unsigned long long* __restrict__ dbg,
               const int packK, const FusedEnv fe) {
    extern __shared__ __align__(128) unsigned char smem[];
    // optional timeline (tools/tc_timeline.py): CTA 0, lane 0 of every warp records (event id << 48 | clock)
    int dbg_n = 0;
#define TL(id)                                                                                           \
    do {                                                                                                 \
        if (TLINE && dbg != nullptr && blockIdx.x == 0 && (threadIdx.x & 31) == 0 && dbg_n < 1024)       \
            dbg[(threadIdx.x >> 5) * 1024 + dbg_n++] = ((unsigned long long)(id) << 48) | (clock64() & 0xFFFFFFFFFFFFull); \
    } while (0)
    __shared__ uint64_t bars[9];      // 0: edge contraction; 1, 2: linear MMAs of group 0 / 1 (B1); 3, 4: aggregation columns of
                                      // group 0 / 1; 5, 6: B2 of group 0 / 1; 7, 8: B3 of group 0 / 1
    __shared__ uint64_t sig[2];       // workers -> contraction issuer: [1] layer inputs ready; [0] PACKED: |A| region cleared, fetch the next pack
    __shared__ uint64_t sdbar[4];     // worker warps -> contraction issuer: blocks 4r .. 4r+3 of the edge operands S, D are in TMEM
    __shared__ uint64_t tail_sig, tail_done;   // workers -> tail warp: an episode's readout partials are complete; and back
    __shared__ uint64_t gsig[2][2];   // the warps of group g -> its linear-layer issuer: operands of the next MMA batch are
                                      // written (one arrival per warp; consecutive batches alternate between the two)
    __shared__ uint64_t bar_ops[2];   // arrival of the bulk copies of the adjacency operand images: 0 = A, 1 = |A|
    __shared__ uint32_t tmem_base_s;
    Ctx c;
    c.smem = smem; c.phase_all = 0; c.phase_grp = 0; c.phase_g2 = 0; c.phase_g3 = 0;
    c.tid = threadIdx.x; c.lane = c.tid & 31;
    c.warp = __shfl_sync(0xffffffffu, c.tid >> 5, 0);     // warp-uniform: MMA issue code stays on the uniform datapath
    c.q = c.warp & 3; c.sub = (c.warp >> 2) % SUBS;
    c.grp = c.warp < NWARPS ? c.warp / (4 * SUBS) : (c.warp == NWARPS + 2 ? 1 : 0);
    const bool linear_issuer = c.warp == NWARPS + 1 || c.warp == NWARPS + 2;
    c.bar_all = &bars[0]; c.bar_grp = &bars[1 + c.grp]; c.bar_g2 = &bars[5 + c.grp]; c.bar_g3 = &bars[7 + c.grp];
    const int K = PACKED ? packK : 1;                     // episodes per pack
    const int NPs = g.NP, Ns = g.N;                       // per-episode sizes; NP / N below are the pack's
    c.NP = K * NPs; c.NB = c.NP >> 3; c.N = PACKED ? c.NP : g.N;
    const int N = c.N, NP = c.NP, NB = c.NB;
    // vertex columns the MMAs produce: NP is a multiple of 16 (block granularity of the epilogues), the instruction's N only
    // has to be a multiple of 8 -- when N <= NP - 8 the last eight (all-padding) columns are left out of every MMA (N = 200:
    // 3.8 % of the MACs).  Those accumulator columns are zeroed once per launch, so whatever the epilogues carry through the
    // padding columns of H^T / E^T stays finite (0 x NaN in an aggregation would poison real vertices).
    const int N8 = PACKED ? NP : ((N + 7) & ~7);
    const int npacks = (B + K - 1) / K;
    // this CTA's work: episodes (packs) blockIdx.x, + gridDim.x, ...; FUSED: every entry of that list once per rollout step,
    // window by window (see FusedEnv): item = (window, step, member)
    const int n_e = (int)blockIdx.x < npacks ? (npacks - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int n_items = n_e * (FUSED ? fe.n_steps : 1);
    auto item_ep = [&](int it) {
        if (!FUSED) return (int)blockIdx.x + it * (int)gridDim.x;
        const int nw = n_e >> 1, span = 2 * fe.n_steps;          // windows; items of a two-entry window
        const int wi = min(it / span, nw - 1);                    // (the last window takes the odd entry: three members)
        const int members = wi == nw - 1 ? n_e - 2 * wi : 2;
        return (int)blockIdx.x + (2 * wi + (it - wi * span) % members) * (int)gridDim.x;
    };
    auto vertex_ok = [&](int n) { return PACKED ? (n % NPs) < Ns : n < N; };     // not a padding vertex
    // PACKED extras live behind the (at most 192 x 192) adjacency image
    float* rdmaxv = reinterpret_cast<float*>(smem + SM_A + PACK_NPMAX * PACK_NPMAX * 2);   // [192] 1 / deg_max of the vertex's graph
    float* pp_blk = rdmaxv + PACK_NPMAX;                  // [12][64] pooled partial sums per 16-vertex block
    float* pooled_e = pp_blk + (PACK_NPMAX / 16) * 64;    // [K][64]
    float* tef = pooled_e + (PACK_NPMAX / 16) * 64;       // [K][64] w_r[f] ReLU(p_f) per episode

    float* xf = reinterpret_cast<float*>(smem + SM_XF);
    float* rdeg = reinterpret_cast<float*>(smem + SM_DEG);      // 1 / deg
    float* qpart = reinterpret_cast<float*>(smem + SM_QP);
    float* ppart = reinterpret_cast<float*>(smem + SM_PP);
    float* pooled = ppart;                                        // readout only: in place over the first 64 partial sums
    float* s_c0 = reinterpret_cast<float*>(smem + SM_MISC);
    float* red_val = s_c0 + 16;
    int* red_idx = reinterpret_cast<int*>(s_c0 + 32);
    unsigned char* sA = smem + SM_A;
    unsigned char* sAbs = smem + SM_ABS;
    unsigned char* sH = smem + SM_H;
    unsigned char* sE = smem + SM_E;
    unsigned char* sT = smem + SM_T + c.grp * (128 * CHUNK * 2);     // this group's chunk buffer
    const uint32_t acc1 = T_ACC1 + 64 * c.grp;                       // this group's linear accumulator
    const uint32_t* pk = reinterpret_cast<const uint32_t*>(w.packed);

    if (c.warp == 0) tmem_alloc(&tmem_base_s, 512);
    if (c.tid == 0) {
        for (int i = 0; i < 9; ++i) mbar_init(&bars[i], 1);
        mbar_init(&bar_ops[0], 1); mbar_init(&bar_ops[1], 1);
        mbar_init(&sig[0], 1); mbar_init(&sig[1], 1);
        for (int i = 0; i < 4; ++i) mbar_init(&gsig[i >> 1][i & 1], 4 * SUBS);
        for (int i = 0; i < 4; ++i) mbar_init(&sdbar[i], NWARPS);
        mbar_init(&tail_sig, 1); mbar_init(&tail_done, 1);
        fence_mbar_init();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    c.tmem = tmem_base_s;
    if (c.warp < 4 && N8 < NP) {                           // ACC0 columns N8 .. NP-1, all 128 lanes: zero, once
        const uint32_t z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        tmem_st_32x32b_x8(tmem_addr(c.tmem, 32 * c.q, T_ACC0 + N8), z);
        tmem_st_wait();
        tc_fence_before();
    }
    const float dmax_set = norm_max > 0.f ? norm_max : *g.dmax;
    const int nsteps_A = NP >> 4;                         // k-steps over vertices
    const int nblocks = NP >> 4;
    const int nb0 = group0_blocks(nblocks), nb1 = nblocks - nb0;       // blocks of group 0 / group 1
    const int nch0 = nb0 >= 2 ? 2 : nb0, nch1 = nb1 >= 2 ? 2 : nb1;     // chunks of group 0 / group 1
    const int nchunks = nch0 + nch1;
    // group 0 owns the first half of the chunks, group 1 the rest: the aggregation is issued (and committed) per half, so
    // group 0 starts its epilogues while group 1's columns are still being computed -- the two groups stay out of phase
    // and one's MMAs run under the other's epilogue
    const int chunk_split = nch0;                          // global index of group 1's first chunk
    const int cs = c.grp == 0 ? 0 : nch0;
    const int ncols0 = 16 * nb0;                           // columns of group 0's chunks
    uint32_t phase_half = 0, phase_other = 0, phase_tail = 0;
    // this group's (at most two) chunks: first column and width, fixed for the whole launch
    const int nmine = (c.warp < NWARPS || linear_issuer) ? (c.grp == 0 ? nch0 : nch1) : 0;
    const int nbm = c.grp == 0 ? nb0 : nb1;                // this group's blocks: chunk a = the first ceil(nbm / 2) of them
    const int cA0 = c.grp == 0 ? 0 : ncols0, cAw = nmine > 1 ? 16 * ((nbm + 1) / 2) : 16 * nbm;
    const int cB0 = cA0 + cAw, cBw = 16 * nbm - cAw;
    const int cAm = min(cAw, N8 - cA0), cBm = min(cBw, N8 - cB0);      // the MMAs' N of the two chunks (>= 8)
    // worker warp -> its group's issuer: "my part of the operands of batch k is written" (smem: generic proxy, fenced for
    // the async proxy; TMEM loads of the accumulator the batch overwrites have completed)
    auto signal_issuer = [&](int k) {
        fence_proxy_async();
        tc_fence_before();
        __syncwarp();
        if (c.lane == 0) mbar_arrive(&gsig[c.grp][k & 1]);
    };

    // The adjacency operands come ready-made (graph_prepare.cu: bf16 images of J and |J| in this kernel's core-matrix
    // layout): one bulk copy each, issued as soon as the previous episode's last reader of the destination retired, so
    // the transfer of episode e+1 runs under the layers / readout of episode e.
    // PACKED: graph j of the pack goes to diagonal block j of the image: its NP/8 column-block runs (NP/8 core matrices
    // = NP * 16 bytes each, contiguous in both layouts) are copied one by one; the off-diagonal blocks stay zero.
    auto fetch_ops = [&](int which, int pack) {             // one thread
        unsigned char* dst = which ? smem + SM_ABS : smem + SM_A;
        if (!PACKED) {
            const uint32_t ops_bytes = (uint32_t)NP * NP * 2;
            const uint16_t* src = g.tc_ops + ((size_t)graph_idx[pack] * 2 + which) * NP * NP;
            mbar_expect_tx(&bar_ops[which], ops_bytes);
            bulk_g2s(dst, src, ops_bytes, &bar_ops[which]);
        } else {
            const int kk = min(K, B - pack * K), NBs = NPs >> 3;
            mbar_expect_tx(&bar_ops[which], (uint32_t)kk * NPs * NPs * 2);
            for (int j = 0; j < kk; ++j) {
                const uint16_t* src = g.tc_ops + ((size_t)graph_idx[pack * K + j] * 2 + which) * NPs * NPs;
                for (int cb = 0; cb < NBs; ++cb)
                    bulk_g2s(dst + ((size_t)(j * NBs + cb) * NB + j * NBs) * 128, src + (size_t)cb * NBs * 64, NBs * 128,
                             &bar_ops[which]);
            }
        }
    };
    // PACKED, all 32 lanes of one warp (the contraction issuer): one run per lane instead of kk * NP/8 serial issues by a worker
    // thread (a pack of nine ER-20 graphs: 27 runs per image, ~4 k cycles of one thread on the workers' critical path, twice)
    auto fetch_ops_warp = [&](int which, int pack) {
        unsigned char* dst = which ? smem + SM_ABS : smem + SM_A;
        const int kk = min(K, B - pack * K), NBs = NPs >> 3;
        if (c.lane == 0) mbar_expect_tx(&bar_ops[which], (uint32_t)kk * NPs * NPs * 2);
        __syncwarp();
        for (int idx = c.lane; idx < kk * NBs; idx += 32) {
            const int j = idx / NBs, cb = idx % NBs;
            const uint16_t* src = g.tc_ops + ((size_t)graph_idx[pack * K + j] * 2 + which) * NPs * NPs;
            bulk_g2s(dst + ((size_t)(j * NBs + cb) * NB + j * NBs) * 128, src + (size_t)cb * NBs * 64, NBs * 128, &bar_ops[which]);
        }
        __syncwarp();
    };
    auto zero_image = [&](unsigned char* dst) {             // all worker threads; generic proxy, fenced for the bulk copies
        for (int off = c.tid * 16; off < NP * NP * 2; off += THREADS * 16)
            *reinterpret_cast<uint4*>(dst + off) = make_uint4(0, 0, 0, 0);
        fence_proxy_async();
    };
    if (PACKED) {
        if (c.warp < NWARPS) { zero_image(smem + SM_A); zero_image(smem + SM_ABS); }
        __syncthreads();
    }
    if (c.tid == 0 && n_items > 0) { fetch_ops(0, blockIdx.x); fetch_ops(1, blockIdx.x); }

    // per-episode inputs, requested one episode ahead (during the previous readout): this thread's vertex observations
    // and degree, the four graph-level observations, the graph's maximum degree
    const bool has_v = c.tid < NP;                 // NP <= 208 < THREADS: one vertex per thread
    float xin0 = 0.f, xin1 = 0.f, xin2 = 0.f, degv = 1.f;
    float4 gl = make_float4(0.f, 0.f, 0.f, 0.f);
    int gmaxdeg = 1;
    auto load_inputs = [&](int e) {                         // e: episode, or pack of K episodes
        if (!PACKED) {
            const int ge = graph_idx[e];
            if (has_v) {
                xin0 = xn[((size_t)e * 3 + 0) * NP + c.tid];
                xin1 = xn[((size_t)e * 3 + 1) * NP + c.tid];
                xin2 = xn[((size_t)e * 3 + 2) * NP + c.tid];
                degv = g.deg[(size_t)ge * NP + c.tid];
            }
            gl = *reinterpret_cast<const float4*>(xg + (size_t)e * 4);
            gmaxdeg = g.gstat[(size_t)ge * 4];
        } else {                                            // this thread's vertex belongs to episode e * K + tid / NPs
            const int be = e * K + c.tid / NPs, v = c.tid % NPs;
            xin0 = xin1 = xin2 = 0.f; degv = 1.f; gmaxdeg = 1;
            gl = make_float4(0.f, 0.f, 0.f, 0.f);
            if (has_v && be < B) {
                const int ge = graph_idx[be];
                xin0 = xn[((size_t)be * 3 + 0) * NPs + v];
                xin1 = xn[((size_t)be * 3 + 1) * NPs + v];
                xin2 = xn[((size_t)be * 3 + 2) * NPs + v];
                degv = g.deg[(size_t)ge * NPs + v];
                gl = *reinterpret_cast<const float4*>(xg + (size_t)be * 4);
                gmaxdeg = g.gstat[(size_t)ge * 4];
            }
        }
    };
    // ================= readout + argmax of one episode by ONE warp (mpnn.py:143-159; experiments/utils.py:57-66) ==========
    // Not PACKED.  Reads only the pooled partial sums and the per-vertex partial dot products that the last layer's
    // epilogues left in shared memory, which the next episode does not touch before ITS last layer: warp 19 does nothing
    // else -- it is woken at the end of every episode and works through the tail (pooling, W_p, Q, argmax and, FUSED, the
    // environment step with its chains of dependent global loads) while the other 19 warps are already on the next
    // episode, so the tail costs the epilogue warps nothing and never delays an MMA issue.
    const float bread = __ldg(w.b_read);
    auto readout_warp_a = [&]() -> float {            // c0 = w_r[0:64] . ReLU(W_p mean_i h_i) + b
        TL(60);
        float pa = 0.f, pb = 0.f;
        for (int k = 0; k < nchunks * SUBS; ++k) { pa += ppart[k * 64 + c.lane]; pb += ppart[k * 64 + 32 + c.lane]; }
        pooled[c.lane] = pa / (float)N;               // (in place: a lane only ever read its own two columns)
        pooled[32 + c.lane] = pb / (float)N;
        __syncwarp();
        // p = W_p pooled from the transposed copy (rows k, k + 1 of W_p^T per 512-byte warp load): this lane accumulates
        // outputs f = 4 (lane % 16) .. + 3 over the k of its parity, the two parities are added at the end
        const float4* wt = reinterpret_cast<const float4*>(pk + PK_WPT) + c.lane;
        const int f4 = 4 * (c.lane & 15), kpar = c.lane >> 4;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
        for (int k0 = 0; k0 < 64; k0 += 32) {         // 16 x 16 bytes in flight per lane
            float4 a[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) a[j] = __ldg(wt + (k0 / 2 + j) * 32);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float pv = pooled[k0 + 2 * j + kpar];
                acc.x = fmaf(a[j].x, pv, acc.x); acc.y = fmaf(a[j].y, pv, acc.y);
                acc.z = fmaf(a[j].z, pv, acc.z); acc.w = fmaf(a[j].w, pv, acc.w);
            }
        }
        acc.x += __shfl_xor_sync(0xffffffffu, acc.x, 16); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, 16);
        acc.z += __shfl_xor_sync(0xffffffffu, acc.z, 16); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, 16);
        const float4 wr = __ldg(reinterpret_cast<const float4*>(w.w_read + f4));
        float t = kpar == 0 ? fmaf(wr.x, fmaxf(acc.x, 0.f), fmaf(wr.y, fmaxf(acc.y, 0.f),
                              fmaf(wr.z, fmaxf(acc.z, 0.f), wr.w * fmaxf(acc.w, 0.f)))) : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        TL(62);
        return bread + t;
    };
    auto readout_warp_b = [&](const int be, const float c0v) {    // Q of every vertex, argmax (lowest index on ties)
        TL(63);
        float bv = -INFINITY;
        int bi = 0x7fffffff;
        for (int i = c.lane; i < N; i += 32) {
            const float qv = c0v + ((qpart[i] + qpart[NPMAX + i]) + (qpart[2 * NPMAX + i] + qpart[3 * NPMAX + i]));
            if (q_out) q_out[(size_t)be * NP + i] = qv;
            if (qv > bv) { bv = qv; bi = i; }         // (i ascending: the first maximum stays)
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
        if (c.lane == 0 && act_out) act_out[be] = bi;
        if (FUSED)        // every lane holds the same (bv, bi) after the butterfly: the warp steps the episode it has just decided
            env_step_group<32, false>(g, fe.env, be, c.lane, true, ECO_POLICY_ACTIONS, bi, nullptr, nullptr, fe.hist_a, fe.hist_r, fe.hist_s);
        TL(64);
    };
    // Not PACKED: the next episode's inputs do not pass through registers.  The threads of group 1 copy them with cp.async
    // (16 bytes each, no register, no wait) into the rows of `xf` -- their own chunk buffer, free once the group's last
    // W_m agg batch of the episode retired -- well before the episode ends: vertex observations [3][NP], the degrees,
    // the four graph-level observations and the graph's maximum degree.  Consumed after one cp.async.wait + CTA barrier at
    // the top of the next episode.  (Padding vertices keep whatever the env kernels wrote for them: finite values that
    // only ever reach padding columns -- the adjacency rows of padding vertices are zero.)
    constexpr int XF_DEG = 4, XF_GL = 5, XF_GMAX = 6;      // rows of xf used by the staging (rows 0..2: the observations)
    // ... and the two small input weights W_e [63][8], W_init [64][7] behind them (3.8 KB from L2 every episode: 30 values
    // per thread that would otherwise be 30 dependent-latency global loads at the top of the episode, or 30 registers)
    float* wsm_e = xf + 7 * NPMAX;
    float* wsm_i = wsm_e + 63 * 8;
    auto stage_inputs = [&](int e) {                        // threads 256 .. 511
        const int i = c.tid - GROUP_THREADS, per_row = NP >> 2;
        const int ge = graph_idx[e];
        if (i < 4 * per_row) {
            const int row = i / per_row, col = 4 * (i % per_row);
            const float* src = row < 3 ? xn + ((size_t)e * 3 + row) * NP + col : g.deg + (size_t)ge * NP + col;
            float* dst = xf + (row < 3 ? row : XF_DEG) * NPMAX + col;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
        } else if (i == 4 * per_row) {
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(xf + XF_GL * NPMAX)), "l"(xg + (size_t)e * 4) : "memory");
        } else if (i == 4 * per_row + 1) {
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(xf + XF_GMAX * NPMAX)), "l"(g.gstat + (size_t)ge * 4) : "memory");
        }
        if (i < (63 * 8) / 4)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_u32(wsm_e + 4 * i)), "l"(w.w_edge + 4 * i) : "memory");
        if (i < (64 * 7) / 4)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_u32(wsm_i + 4 * i)), "l"(w.w_init + 4 * i) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // PACKED: readout + argmax of the K episodes of a pack by ONE warp (the tail warp, like readout_warp_a / _b): the same sums
    // in the same order as the all-worker readout it replaces (four CTA barriers and ~9 k cycles of all sixteen epilogue warps
    // per pack, exposed under an edge contraction of ~2.7 k), now beside the next pack's stages.
    auto readout_packed_warp = [&](const int be) {
        TL(60);
        const int bpe = NPs >> 4;                         // 16-vertex blocks per episode
        for (int idx = c.lane; idx < K * 64; idx += 32) {                  // pooled[e][f] = mean_i h_i[f]
            const int e = idx >> 6, f = idx & 63;
            float t = 0.f;
            for (int j = 0; j < bpe; ++j) t += pp_blk[(e * bpe + j) * 64 + f];
            pooled_e[idx] = t / (float)Ns;
        }
        __syncwarp();
        TL(61);
        // p[e][f] = W_p[f, :] pooled[e], k ascending; this lane: f = lane, lane + 32.  Rows of W_p^T: coalesced 128-byte loads,
        // 32 of them in flight per lane
        constexpr int KMAX = PACK_NPMAX / 16;
        float p0[KMAX], p1[KMAX];
#pragma unroll
        for (int e = 0; e < KMAX; ++e) { p0[e] = 0.f; p1[e] = 0.f; }
        const float* wt = reinterpret_cast<const float*>(pk + PK_WPT) + c.lane;
#pragma unroll 1
        for (int k0 = 0; k0 < 64; k0 += 16) {
            float wa[16], wb[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) { wa[j] = __ldg(wt + (k0 + j) * 64); wb[j] = __ldg(wt + (k0 + j) * 64 + 32); }
#pragma unroll
            for (int j = 0; j < 16; ++j) {
#pragma unroll
                for (int e = 0; e < KMAX; ++e) {
                    if (e < K) {
                        const float pv = pooled_e[e * 64 + k0 + j];
                        p0[e] = fmaf(wa[j], pv, p0[e]);
                        p1[e] = fmaf(wb[j], pv, p1[e]);
                    }
                }
            }
        }
        TL(62);
        const float wr0 = __ldg(w.w_read + c.lane), wr1 = __ldg(w.w_read + 32 + c.lane);
        __syncwarp();                                      // pooled_e is dead: c0 goes to its first K entries
#pragma unroll
        for (int e = 0; e < KMAX; ++e) {
            if (e < K) {                                   // tef[e][f] = w_r[f] ReLU(p[e][f])
                tef[e * 64 + c.lane] = wr0 * fmaxf(p0[e], 0.f);
                tef[e * 64 + 32 + c.lane] = wr1 * fmaxf(p1[e], 0.f);
            }
        }
        __syncwarp();
        if (c.lane < K) {                                  // c0[e] = b + sum_f tef[e][f], f ascending
            float c0v = bread;
            for (int f = 0; f < 64; ++f) c0v += tef[c.lane * 64 + f];
            pooled_e[c.lane] = c0v;
        }
        __syncwarp();
        TL(63);
        for (int e = 0, i0 = 0; e < K; ++e, i0 += NPs) {   // Q of every vertex; the final value goes to qpart row 0
            const int ep = be * K + e;
            const float c0v = pooled_e[e];
            for (int v = c.lane; v < NPs; v += 32) {
                const int i = i0 + v;
                const float qv = c0v + ((qpart[i] + qpart[NPMAX + i]) + (qpart[2 * NPMAX + i] + qpart[3 * NPMAX + i]));
                const bool ok = v < Ns && ep < B;
                if (ok && q_out) q_out[(size_t)ep * NPs + v] = qv;
                qpart[i] = ok ? qv : -INFINITY;
            }
        }
        __syncwarp();
        TL(65);
        for (int e = 0; e < K; ++e) {                      // argmax per episode, lowest index on ties
            const int ep = be * K + e;
            float bv = -INFINITY;
            int bi = 0x7fffffff;
            for (int v = c.lane; v < Ns; v += 32) {
                const float qv = qpart[e * NPs + v];
                if (qv > bv) { bv = qv; bi = v; }          // (v ascending: the first maximum stays)
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
            }
            if (c.lane == 0 && ep < B && act_out) act_out[ep] = bi;
        }
        TL(64);
    };
    if (c.warp == NWARPS) {
        // ================= contraction issuer ===============================================================

        uint32_t sp0 = 0, sp1 = 0, sp2 = 0, op = 0;
        for (int it = 0; it < n_items; ++it) {
            mbar_wait(&bar_ops[0], op);               // A and |A| of this episode have landed (async proxy -> async proxy)
            mbar_wait(&bar_ops[1], op); op ^= 1u;
            TL(51);
            // edge contraction  S |A| + D A, k-step by k-step behind the workers that produce S and D: the MMAs of the
            // blocks of round r run while round r + 1 is being computed
            for (int r = 0; 4 * r < nsteps_A; ++r) {
                mbar_wait(&sdbar[r], sp0);
                tc_fence_after();
                if (r == 0) TL(50);
                if (elect_one()) {
                    const uint32_t idesc = instr_desc_bf16(128, N8, false, false);
                    const uint64_t bd_abs = smem_desc(smem_u32(sAbs), NB * 128, 128);
                    const uint64_t bd_a = smem_desc(smem_u32(sA), NB * 128, 128);
                    const uint64_t kstep = (uint64_t)((2 * NB * 128) >> 4);
                    for (int ks = 4 * r; ks < min(4 * r + 4, nsteps_A); ++ks) {
                        mma_ts(c.tmem + T_ACC0, c.tmem + T_S + 8 * ks, bd_abs + ks * kstep, idesc, ks > 0);
                        mma_ts(c.tmem + T_ACC0, c.tmem + T_D + 8 * ks, bd_a + ks * kstep, idesc, true);
                    }
                    if (4 * r + 4 >= nsteps_A) mma_commit(c.bar_all);
                }
                __syncwarp();
            }
            sp0 ^= 1u;
            TL(52);
            for (int l = 0; l < 3; ++l) {
                mbar_wait(&sig[1], sp1); sp1 ^= 1u;
                tc_fence_after();
                TL(53);
                if (elect_one()) {                    // agg^T = H^T A  (both hi and lo rows in one M=128 chain), per half
                    const uint64_t ad = smem_desc(smem_u32(sH), 2048, 128);
                    const uint64_t bstep = (uint64_t)((2 * NB * 128) >> 4);
                    for (int half = 0; half < 2; ++half) {
                        const int n0 = half ? ncols0 : 0, ncols = half ? N8 - ncols0 : min(ncols0, N8);
                        if (ncols == 0) break;
                        const uint32_t idesc = instr_desc_bf16(128, ncols, false, false);
                        const uint64_t bd = smem_desc(smem_u32(sA) + (n0 >> 3) * 128, NB * 128, 128);
                        for (int ks = 0; ks < nsteps_A; ++ks)
                            mma_ss(c.tmem + T_ACC0 + n0, ad + (uint64_t)ks * (4096 >> 4), bd + ks * bstep, idesc, ks > 0);
                        mma_commit(&bars[3 + half]);
                    }
                }
                __syncwarp();
                TL(54);
            }
            if (PACKED && it + 1 < n_items) {
                // the next pack's operand images.  A has no reader left once the last aggregation of layer 2 retired (the halves
                // retire in order; completion 3 it + 2 of that half's barrier); |A| overlays H / E: free once the workers have
                // finished the pack and cleared the off-diagonal blocks (sig[0])
                mbar_wait(&bars[N8 > ncols0 ? 4 : 3], (uint32_t)((3 * it + 2) & 1));
                fetch_ops_warp(0, item_ep(it + 1));
                mbar_wait(&sig[0], sp2); sp2 ^= 1u;
                fetch_ops_warp(1, item_ep(it + 1));
            }
        }
    }
    if (c.warp == NWARPS + 3) {
        // ================= episode tail ====================================================================
        uint32_t ph = 0;
        for (int it = 0; it < n_items - (PACKED ? 1 : 0); ++it) {    // (PACKED: the last pack is read out by all workers)
            mbar_wait(&tail_sig, ph);
            ph ^= 1u;
            if (PACKED) readout_packed_warp(item_ep(it));
            else readout_warp_b(item_ep(it), readout_warp_a());
            if (FUSED) __threadfence();                    // the episode's new state / observations, before the arrival below
            __syncwarp();
            if (c.lane == 0) mbar_arrive(&tail_done);      // the partial sums may be overwritten (next episode's last layer)
        }
    }
    if (linear_issuer && nmine > 0) {
        // ================= linear-layer issuer of group c.grp ================================================
        // Follows the group's schedule (see stage 1 / stage 2 below): waits for the group's k-th signal, issues the batch,
        // commits it to B1 / B2 / B3.  Signals alternate between gsig[g][0] and gsig[g][1]; a signal is never raised
        // before the batch two signals earlier was committed and waited for, so one phase bit per barrier is enough.
        uint32_t ph[2] = {0, 0};
        auto wait_sig = [&](int k) {
            mbar_wait(&gsig[c.grp][k & 1], ph[k & 1]);
            ph[k & 1] ^= 1u;
            tc_fence_after();
        };
        for (int it = 0; it < n_items; ++it) {
            wait_sig(0);                                                                 // g(a) is in E^T[a]
            if (elect_one()) { issue_part(c, T_ACC0 + cA0, T_WEF, sE, cA0 >> 3, cAm, false); mma_commit(c.bar_grp); }
            __syncwarp();
            if (nmine > 1) {
                wait_sig(1);
                // (chunk b accumulates in ACC1, which is free until the first layer: its epilogue runs under layer 0's aggregation,
                //  which overwrites every column of ACC0)
                if (elect_one()) { issue_part(c, acc1, T_WEF, sE, cB0 >> 3, cBm, false); mma_commit(c.bar_g2); }
                __syncwarp();
            }
            for (int l = 0; l < 3; ++l) {
                wait_sig(0);                                                             // S0: layer weights in TMEM
                if (elect_one()) issue_part(c, acc1, T_WM + 32, sE, cA0 >> 3, cAm, false);   // M1e(a), ahead
                __syncwarp();
                wait_sig(1);                                                             // S1: agg(a) in the chunk buffer
                if (elect_one()) {
                    issue_part(c, acc1, T_WM, sT, 0, cAm, true);                         // M1a(a): += W_m[:, :64] agg
                    mma_commit(c.bar_grp);                                               //   -> B1
                    issue_part(c, T_ACC0 + cA0, T_WU, sH, cA0 >> 3, cAm, false);         // M2h(a): W_u[:, :64] h, ahead
                    mma_commit(c.bar_g2);                                                //   -> B2
                }
                __syncwarp();
                if (nmine > 1) {
                    wait_sig(0);                                                         // S2: agg(b) in the chunk buffer
                    if (elect_one()) {
                        issue_part(c, T_ACC0 + cB0, T_WU, sH, cB0 >> 3, cBm, false);     // M2h(b), ahead
                        mma_commit(c.bar_g3);                                            //   -> B3
                    }
                    __syncwarp();
                }
                wait_sig(1);                                                             // S3: m(a) in H^T[a]
                if (elect_one()) {
                    issue_part(c, T_ACC0 + cA0, T_WU + 32, sH, cA0 >> 3, cAm, true);     // M2m(a): += W_u[:, 64:] m
                    mma_commit(c.bar_grp);                                               //   -> B1
                    if (nmine > 1) {
                        issue_part(c, acc1, T_WM + 32, sE, cB0 >> 3, cBm, false);        // M1(b) = W_m [agg ; e]
                        issue_part(c, acc1, T_WM, sT, 0, cBm, true);
                        mma_commit(c.bar_g2);                                            //   -> B2
                    }
                }
                __syncwarp();
                if (nmine > 1) {
                    wait_sig(0);                                                         // S4: m(b) in H^T[b]
                    if (elect_one()) {
                        issue_part(c, T_ACC0 + cB0, T_WU + 32, sH, cB0 >> 3, cBm, true); // M2m(b)
                        mma_commit(c.bar_grp);                                           //   -> B1
                    }
                    __syncwarp();
                }
            }
        }
    }
    if (c.warp < NWARPS && n_items > 0) {
        {   // W_ef is the same for every item and its columns overlap no other TMEM range: stored once per launch
            uint4 wef[32 / (8 * SUBS)];
            ldg_weights<32>(c, pk + PK_WEF, wef);
            sttm_weights<32>(c, wef, T_WEF);
            tmem_st_wait();
            tc_fence_before();
            workers_sync();           // complete (all 16 warps' columns) before either group signals its issuer
        }
        if (PACKED) load_inputs(blockIdx.x);
        else if (c.grp == 1) stage_inputs(blockIdx.x);
    }

    // PACKED: the same readout by all sixteen epilogue warps -- for the CTA's LAST pack only, whose tail nothing runs beside
    // (~9 k cycles instead of the ~30 k one warp takes; identical sums in identical order)
    auto readout_packed_all = [&](const int be) {
        if (PACKED) {
            // be = pack.  All K episodes at once, every sum in a fixed order.
            const int bpe = NPs >> 4;                     // 16-vertex blocks per episode
            for (int idx = c.tid; idx < K * 64; idx += THREADS) {          // pooled[e][f] = mean_i h_i[f]
                const int e = idx >> 6, f = idx & 63;
                float t = 0.f;
                for (int j = 0; j < bpe; ++j) t += pp_blk[(e * bpe + j) * 64 + f];
                pooled_e[idx] = t / (float)Ns;
            }
            workers_sync();
            for (int idx = c.tid; idx < K * 64; idx += THREADS) {          // tef[e][f] = w_r[f] ReLU(W_p[f,:] pooled[e])
                const int e = idx >> 6, f = idx & 63;
                const float4* wp = reinterpret_cast<const float4*>(w.w_pool + f * 64);
                const float* pv = pooled_e + e * 64;
                float p = 0.f;
#pragma unroll 4
                for (int k4 = 0; k4 < 16; ++k4) {
                    const float4 wv = __ldg(wp + k4);
                    p = fmaf(wv.x, pv[4 * k4], p); p = fmaf(wv.y, pv[4 * k4 + 1], p);
                    p = fmaf(wv.z, pv[4 * k4 + 2], p); p = fmaf(wv.w, pv[4 * k4 + 3], p);
                }
                tef[idx] = __ldg(w.w_read + f) * fmaxf(p, 0.f);
            }
            workers_sync();
            if (c.tid < NP) {                             // Q of this thread's vertex; the final value goes to qpart row 0
                const int i = c.tid, e = i / NPs, v = i % NPs, ep = be * K + e;
                float c0v = bread;
                for (int f = 0; f < 64; ++f) c0v += tef[e * 64 + f];
                const float qv = c0v + ((qpart[i] + qpart[NPMAX + i]) + (qpart[2 * NPMAX + i] + qpart[3 * NPMAX + i]));
                const bool ok = v < Ns && ep < B;
                if (ok && q_out) q_out[(size_t)ep * NPs + v] = qv;
                qpart[i] = ok ? qv : -INFINITY;
            }
            workers_sync();
            for (int e = c.warp; e < K; e += NWARPS) {    // argmax of episode e by one warp, lowest index on ties
                const int ep = be * K + e;
                float bv = -INFINITY;
                int bi = 0x7fffffff;
                for (int v = c.lane; v < Ns; v += 32) {
                    const float qv = qpart[e * NPs + v];
                    if (qv > bv) { bv = qv; bi = v; }     // (v ascending: the first maximum stays)
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
                    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
                }
                if (c.lane == 0 && ep < B && act_out) act_out[ep] = bi;
            }
            workers_sync();               // qpart / pp_blk / tef may be reused
            return;
        }
        // (not PACKED: readout_warp_a / readout_warp_b above)
    };
    int last_b = -1;

    for (int it = 0; it < n_items && c.warp < NWARPS; ++it) {
        const int b = item_ep(it);
        const bool has_next = it + 1 < n_items;
        const int b_next = has_next ? item_ep(it + 1) : 0;
        TL(1);
        if (!PACKED) {                                      // the staged inputs of this episode have landed
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            TL(70);
            workers_sync();
            TL(71);
            gl = *reinterpret_cast<const float4*>(xf + XF_GL * NPMAX);
            gmaxdeg = *reinterpret_cast<const int*>(xf + XF_GMAX * NPMAX);
            if (has_v) rdeg[c.tid] = __fdividef(1.f, xf[XF_DEG * NPMAX + c.tid]);
        }
        // (fast reciprocal: a correctly rounded 1.f / x is a subroutine call of several hundred cycles at the top of every episode)
        const float rdmax = __fdividef(1.f, norm_max < 0.f ? (float)max(gmaxdeg, 1) : dmax_set);

        // ================= stage 0: operands of the edge contraction ======================================
        // this thread's rows of the two small input weights (features fa, fb), issued early so the latency is hidden
        const int fa = 16 * c.q + (c.lane >> 2), fb = fa + 8;
        float wxa[8], wxb[8], wia[7], wib[7];
        {
            const float* we = PACKED ? w.w_edge : wsm_e;      // (not PACKED: staged in shared memory with the inputs)
            const float* wi = PACKED ? w.w_init : wsm_i;
#pragma unroll
            for (int k = 0; k < 8; ++k) {   // row 63 of the 63 x 8 edge weight does not exist: zero
                wxa[k] = we[fa * 8 + k];
                wxb[k] = fb < 63 ? we[fb * 8 + k] : 0.f;
            }
#pragma unroll
            for (int k = 0; k < 7; ++k) { wia[k] = wi[fa * 7 + k]; wib[k] = wi[fb * 7 + k]; }
        }
        if (PACKED && has_v) {
            const int i = c.tid;
            const bool ok = vertex_ok(i);
            xf[0 * NPMAX + i] = ok ? xin0 : 0.f;
            xf[1 * NPMAX + i] = ok ? xin1 : 0.f;
            xf[2 * NPMAX + i] = ok ? xin2 : 0.f;
            rdeg[i] = __fdividef(1.f, degv);
            {                                  // the graph-level observations and deg_max differ from vertex to vertex
                xf[3 * NPMAX + i] = ok ? gl.x : 0.f;
                xf[4 * NPMAX + i] = ok ? gl.y : 0.f;
                xf[5 * NPMAX + i] = ok ? gl.z : 0.f;
                xf[6 * NPMAX + i] = ok ? gl.w : 0.f;
                rdmaxv[i] = 1.f / (norm_max < 0.f ? (float)max(gmaxdeg, 1) : dmax_set);
            }
        }
        // observations 3..6 are the same for every vertex: their share of W_x x and W_init x is one constant per feature
        // (padded vertices get it too; nothing reads their columns: no edges, masked out of the pooling and the argmax)
        float cxa = wxa[4] * gl.x, cxb = wxb[4] * gl.x, cia = wia[3] * gl.x, cib = wib[3] * gl.x;
        cxa = fmaf(wxa[5], gl.y, cxa); cxb = fmaf(wxb[5], gl.y, cxb); cia = fmaf(wia[4], gl.y, cia); cib = fmaf(wib[4], gl.y, cib);
        cxa = fmaf(wxa[6], gl.z, cxa); cxb = fmaf(wxb[6], gl.z, cxb); cia = fmaf(wia[5], gl.z, cia); cib = fmaf(wib[5], gl.z, cib);
        cxa = fmaf(wxa[7], gl.w, cxa); cxb = fmaf(wxb[7], gl.w, cxb); cia = fmaf(wia[6], gl.w, cia); cib = fmaf(wib[6], gl.w, cib);
        if (PACKED) { cxa = 0.f; cxb = 0.f; cia = 0.f; cib = 0.f; }      // (all 7 observations come from xf)
        constexpr int NOBS = PACKED ? 7 : 3;
        TL(2);
        if (PACKED) workers_sync();                       // xf visible
        TL(3);
        // S = R+ + R-, D = R+ - R- with R+- = ReLU(P +- w0), P = W_x x  -> TMEM A operands (mpnn.py:89-100 factorised)
        {
            for (int r = 0; 4 * r < nsteps_A; ++r) {
                const int blk = 4 * r + c.grp * SUBS + c.sub;
                if (blk < nsteps_A) {
                uint32_t sh[4], sl[4], dh[4], dl[4];
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const int n0 = 16 * blk + 8 * half + 2 * (c.lane & 3);
                    float pa0 = cxa, pa1 = cxa, pb0 = cxb, pb1 = cxb;
#pragma unroll
                    for (int k = 0; k < NOBS; ++k) {
                        const float2 x = *reinterpret_cast<const float2*>(xf + k * NPMAX + n0);
                        fma2(pa0, pa1, wxa[1 + k], wxa[1 + k], x.x, x.y, pa0, pa1);
                        fma2(pb0, pb1, wxb[1 + k], wxb[1 + k], x.x, x.y, pb0, pb1);
                    }
                    float rpa0, rpa1, rma0, rma1, rpb0, rpb1, rmb0, rmb1;
                    add2(rpa0, rpa1, pa0, pa1, wxa[0], wxa[0]); sub2(rma0, rma1, pa0, pa1, wxa[0], wxa[0]);
                    add2(rpb0, rpb1, pb0, pb1, wxb[0], wxb[0]); sub2(rmb0, rmb1, pb0, pb1, wxb[0], wxb[0]);
                    rpa0 = fmaxf(rpa0, 0.f); rpa1 = fmaxf(rpa1, 0.f); rma0 = fmaxf(rma0, 0.f); rma1 = fmaxf(rma1, 0.f);
                    rpb0 = fmaxf(rpb0, 0.f); rpb1 = fmaxf(rpb1, 0.f); rmb0 = fmaxf(rmb0, 0.f); rmb1 = fmaxf(rmb1, 0.f);
                    float sa0, sa1, sb0, sb1, da0, da1, db0, db1;
                    add2(sa0, sa1, rpa0, rpa1, rma0, rma1); add2(sb0, sb1, rpb0, rpb1, rmb0, rmb1);
                    sub2(da0, da1, rpa0, rpa1, rma0, rma1); sub2(db0, db1, rpb0, rpb1, rmb0, rmb1);
                    split2(sa0, sa1, sh[2 * half + 0], sl[2 * half + 0]);
                    split2(sb0, sb1, sh[2 * half + 1], sl[2 * half + 1]);
                    split2(da0, da1, dh[2 * half + 0], dl[2 * half + 0]);
                    split2(db0, db1, dh[2 * half + 1], dl[2 * half + 1]);
                }
                tmem_st_16x128b_x2(tmem_addr(c.tmem, 32 * c.q, T_S + 8 * blk), sh);
                tmem_st_16x128b_x2(tmem_addr(c.tmem, 32 * c.q + 16, T_S + 8 * blk), sl);
                tmem_st_16x128b_x2(tmem_addr(c.tmem, 32 * c.q, T_D + 8 * blk), dh);
                tmem_st_16x128b_x2(tmem_addr(c.tmem, 32 * c.q + 16, T_D + 8 * blk), dl);
                }
                tmem_st_wait();                       // -> issuer: this warp's share of round r is in TMEM
                tc_fence_before();
                __syncwarp();
                if (c.lane == 0) mbar_arrive(&sdbar[r]);
            }
        }
        TL(4);
        {   // layer-0 weights: L2 -> registers while the edge contraction runs, registers -> TMEM once S / D are dead
            uint4 wm[64 / (8 * SUBS)], wu[64 / (8 * SUBS)];
            ldg_weights<64>(c, pk + PK_WM, wm);
            ldg_weights<64>(c, pk + PK_WU, wu);
            wait_all(c);
            TL(7);
            sttm_weights<64>(c, wm, T_WM);
            sttm_weights<64>(c, wu, T_WU);
        }

        // ================= stage 1: edge embeddings e, h0 (CUDA cores) =====================================
        // g = (S|A| + D A) / (2 deg) goes straight into the chunk's own columns of E^T (e overwrites it once W_ef g has
        // retired) and W_ef g accumulates in the chunk's own -- just consumed -- columns of ACC0: no chunk buffer, no
        // second accumulator, so both chunks of a group are in flight and h0 is computed under their MMAs.
        {
            for (int k = 0; k < nmine; ++k) {
                const int c0 = k ? cB0 : cA0, width = k ? cBw : cAw;
                // feature 63 = deg / deg_max   (mpnn.py:100-102)
                const bool has63 = c.q == 3 && (c.lane >> 2) == 7;     // feature 63 = 16 q + lane/4 + 8: this thread's second row
                epilogue(c, T_ACC0, c0, width, [&](int bc, float (&v)[8]) {
                    const int n0 = c0 + bc + 2 * (c.lane & 3);
                    const float2 r0 = *reinterpret_cast<const float2*>(rdeg + n0), r1 = *reinterpret_cast<const float2*>(rdeg + n0 + 8);
                    const float rd[4] = {r0.x, r0.y, r1.x, r1.y};
#pragma unroll
                    for (int i = 0; i < 8; i += 2) {
                        mul2(v[i], v[i + 1], v[i], v[i + 1], 0.5f, 0.5f);
                        mul2(v[i], v[i + 1], v[i], v[i + 1], rd[2 * (i >> 2)], rd[2 * (i >> 2) + 1]);
                    }
                    if (has63) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) {                   // v[2], v[3], v[6], v[7]: columns n0 + {0, 1, 8, 9}
                            const int n = n0 + 8 * (j >> 1) + (j & 1);
                            v[2 + 4 * (j >> 1) + (j & 1)] = __fdividef(PACKED ? rdmaxv[n] : rdmax, rd[j]);
                        }
                    }
                    store_block(c, sE, c0 + bc, v);
                });
                signal_issuer(k);                   // -> W_ef g of this chunk (B1 / B2)
                TL(10);
            }
        }
        {   // h0 = ReLU(W_init x): thread owns features fa, fb and 4 vertices of every 16-vertex block (epilogue mapping)
            for (int blk = c.grp * SUBS + c.sub; blk < nsteps_A; blk += 2 * SUBS) {
                float v[8];
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const int n0 = 16 * blk + 8 * half + 2 * (c.lane & 3);
                    float a0 = cia, a1 = cia, b0 = cib, b1 = cib;
#pragma unroll
                    for (int k = 0; k < NOBS; ++k) {
                        const float2 x = *reinterpret_cast<const float2*>(xf + k * NPMAX + n0);
                        fma2(a0, a1, wia[k], wia[k], x.x, x.y, a0, a1);
                        fma2(b0, b1, wib[k], wib[k], x.x, x.y, b0, b1);
                    }
                    v[4 * half + 0] = fmaxf(a0, 0.f); v[4 * half + 1] = fmaxf(a1, 0.f);
                    v[4 * half + 2] = fmaxf(b0, 0.f); v[4 * half + 3] = fmaxf(b1, 0.f);
                }
                store_block(c, sH, 16 * blk, v);
            }
        }
        tmem_st_wait();              // layer-0 weights (visible to the MMAs after the layer's first barrier)
        TL(8);
        // e = ReLU(W_ef g): chunk a here; chunk b at the top of layer 0, in the wait for the aggregation (nothing reads e(b)
        // before the group's second batch of that layer)
        auto epi_e = [&](uint32_t acc, int acc_col, int c0, int width) {
            epilogue(c, acc, acc_col, width, [&](int bc, float (&v)[8]) {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = fmaxf(v[i], 0.f);
                store_block(c, sE, c0 + bc, v);
            });
        };
        if (nmine > 0) {
            TL(15);
            wait_grp(c);
            TL(12);
            epi_e(T_ACC0, cA0, cA0, cAw);
            TL(13);
        }

        // ================= stage 2: three message-passing layers (mpnn.py:114-120) ==========================
        // per chunk:  m = ReLU(W_m [agg ; e]) accumulates in the group's ACC1, h' = ReLU(W_u [h ; m]) accumulates in the
        // chunk's own (already consumed) columns of ACC0; m is written over the chunk's columns of H^T once W_u h and
        // every aggregation MMA that reads them retired, so the chunk buffer only ever holds agg.  A group's two chunks
        // a, b are interleaved -- the MMAs of one run under the epilogue of the other:
        //   E1 agg(a)->T | M1a(a) M2h(a) | E2 agg(b)->T | M2h(b) | E3 m(a)->H[a] | M2m(a) M1(b) | E4 h'(a) | E5 m(b)->H[b]
        //   | M2m(b) | E6 h'(b);   B1 / B2 / B3 = the group's three MMA barriers.
        // The halves that do not depend on the running epilogue (W_m e, W_u h) are issued ahead.
        auto epi_agg = [&](int c0, int width, bool wait_b1) {          // agg = (H^T A) / deg -> chunk buffer
            bool waited = !wait_b1;
            epilogue(c, T_ACC0, c0, width, [&](int bc, float (&v)[8]) {
                const int n0 = c0 + bc + 2 * (c.lane & 3);
                const float2 r0 = *reinterpret_cast<const float2*>(rdeg + n0), r1 = *reinterpret_cast<const float2*>(rdeg + n0 + 8);
                const float rd[4] = {r0.x, r0.y, r1.x, r1.y};
#pragma unroll
                for (int i = 0; i < 8; i += 2) mul2(v[i], v[i + 1], v[i], v[i + 1], rd[2 * (i >> 2)], rd[2 * (i >> 2) + 1]);
                if (!waited) { wait_grp(c); waited = true; }           // the previous reader of the chunk buffer retired
                store_block(c, sT, bc, v);
            });
            if (!waited) wait_grp(c);
        };
        auto epi_m = [&](int c0, int width) {                           // m = ReLU(acc1) -> the chunk's columns of H^T
            epilogue(c, acc1, 0, width, [&](int bc, float (&v)[8]) {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = fmaxf(v[i], 0.f);
                store_block(c, sH, c0 + bc, v);
            });
        };
        for (int l = 0; l < 3; ++l) {
            TL(20);
            cta_stage_sync();                   // every h / e column of the previous stage is written
            TL(21);
            if (c.tid == 0) mbar_arrive(&sig[1]);   // -> issuer: agg^T = H^T A, per half
            if (l > 0) {                        // the previous layer's MMAs all retired (barrier above): overwrite weights
                uint4 wm[64 / (8 * SUBS)], wu[64 / (8 * SUBS)];   // (loaded after the barrier: before it, the global loads would contend
                ldg_weights<64>(c, pk + PK_WM + l * 128 * 64, wm);   //  with the slower group's shared-memory stores)
                ldg_weights<64>(c, pk + PK_WU + l * 128 * 64, wu);
                sttm_weights<64>(c, wm, T_WM);
                sttm_weights<64>(c, wu, T_WU);
                tmem_st_wait();
                tc_fence_before();
                workers_sync();
            }
            if (l == 0 && nmine > 1) {                      // e(b), from the group's ACC1 (see stage 1)
                wait_g2(c);
                epi_e(acc1, 0, cB0, cBw);
                TL(13);
            }
            if (nmine > 0) signal_issuer(0);                // S0 -> M1e(a): the W_m e-half of the first chunk, ahead
            TL(22);
            // readout weights of this thread's two features: requested before the wait (last layer only)
            float wa = 0.f, wb = 0.f;
            if (l == 2) { wa = __ldg(w.w_read + 64 + fa); wb = __ldg(w.w_read + 64 + fa + 8); }
            if (l == 2 && last_b >= 0) {                    // the tail warp has read the previous episode's (pack's) partial sums
                mbar_wait(&tail_done, phase_tail);
                phase_tail ^= 1u;
            }
            if (nmine > 0) {                                  // this group's aggregation columns
                mbar_wait(&bars[3 + c.grp], phase_half);
                phase_half ^= 1u;
                tc_fence_after();
            }
            TL(23);
            // A has no reader left once the LAST half retired (the halves retire in order)
            if (!PACKED && l == 2 && c.tid == (chunk_split < nchunks ? THREADS / 2 : 0) && has_next) fetch_ops(0, b_next);   // (PACKED: warp 16)
            // h' of a chunk: next layer's H^T, or (last layer) the readout partials straight from the fp32 registers
            auto epi_h = [&](int ci, int c0, int width) {
                if (l < 2) {
                    epilogue(c, T_ACC0, c0, width, [&](int bc, float (&v)[8]) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) v[i] = fmaxf(v[i], 0.f);
                        store_block(c, sH, c0 + bc, v);
                    });
                    return;
                }
                // (mpnn.py:143-159; pooled sums are kept per chunk and added in chunk order, so the result does not
                //  depend on which group happened to process which chunk)
                float pool_a = 0.f, pool_b = 0.f;
                epilogue(c, T_ACC0, c0, width, [&](int bc, float (&v)[8]) {
                    float qv[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {     // j: columns {0,1,8,9} + 2(lane&3)
                        const int ia = 4 * (j >> 1) + (j & 1), ib = ia + 2;
                        const int n = c0 + bc + 8 * (j >> 1) + 2 * (c.lane & 3) + (j & 1);
                        const float ha = fmaxf(v[ia], 0.f), hb = fmaxf(v[ib], 0.f);
                        if (vertex_ok(n)) { pool_a += ha; pool_b += hb; }
                        qv[j] = fmaf(wa, ha, wb * hb);
                    }
                    if (PACKED) {             // a 16-vertex block lies inside one graph: its pooled partial on its own
                        pool_a += __shfl_xor_sync(0xffffffffu, pool_a, 1); pool_a += __shfl_xor_sync(0xffffffffu, pool_a, 2);
                        pool_b += __shfl_xor_sync(0xffffffffu, pool_b, 1); pool_b += __shfl_xor_sync(0xffffffffu, pool_b, 2);
                        if ((c.lane & 3) == 0) {
                            pp_blk[((c0 + bc) >> 4) * 64 + fa] = pool_a;
                            pp_blk[((c0 + bc) >> 4) * 64 + fa + 8] = pool_b;
                        }
                        pool_a = 0.f; pool_b = 0.f;
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        qv[j] += __shfl_xor_sync(0xffffffffu, qv[j], 4);
                        qv[j] += __shfl_xor_sync(0xffffffffu, qv[j], 8);
                        qv[j] += __shfl_xor_sync(0xffffffffu, qv[j], 16);
                    }
                    if ((c.lane >> 2) == 0) {
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            qpart[c.q * NPMAX + c0 + bc + 8 * (j >> 1) + 2 * (c.lane & 3) + (j & 1)] = qv[j];
                    }
                });
                pool_a += __shfl_xor_sync(0xffffffffu, pool_a, 1); pool_a += __shfl_xor_sync(0xffffffffu, pool_a, 2);
                pool_b += __shfl_xor_sync(0xffffffffu, pool_b, 1); pool_b += __shfl_xor_sync(0xffffffffu, pool_b, 2);
                if (!PACKED && (c.lane & 3) == 0) {
                    ppart[(ci * SUBS + c.sub) * 64 + fa] = pool_a;
                    ppart[(ci * SUBS + c.sub) * 64 + fa + 8] = pool_b;
                }
            };
            if (nmine > 0) {
                // ---- E1: agg(a) -> chunk buffer
                epi_agg(cA0, cAw, false);
                signal_issuer(1);                           // S1 -> M1a(a) (B1), M2h(a) (B2)
                TL(30);
                if (nmine > 1) {
                    // ---- E2: agg(b) -> chunk buffer, once M1a(a) has read it (B1)
                    epi_agg(cB0, cBw, true);
                    signal_issuer(0);                       // S2 -> M2h(b) (B3)
                    TL(31);
                } else {
                    wait_grp(c);                                                            // B1
                }
                // ---- E3: m(a) -> H^T[a]: W_u h (a) retired (B2) and so did every aggregation MMA (they read all of H^T)
                wait_g2(c);
                if (c.grp == 0 && chunk_split < nchunks) {
                    mbar_wait(&bars[4], phase_other);
                    phase_other ^= 1u;
                }
                TL(33);
                epi_m(cA0, cAw);
                signal_issuer(1);                           // S3 -> M2m(a) (B1), M1(b) (B2)
                TL(34);
                // ---- E4: h'(a)
                wait_grp(c);                                                                // B1: M2m(a)
                TL(37);
                epi_h(cs, cA0, cAw);
                TL(38);
                if (nmine > 1) {
                    // ---- E5: m(b) -> H^T[b]
                    wait_g2(c);                                                             // B2: M1(b)
                    wait_g3(c);                                                             // B3: M2h(b)
                    // the chunk buffer has no reader left in this episode: the next episode's inputs go there
                    if (!PACKED && l == 2 && c.grp == 1 && has_next) stage_inputs(b_next);
                    TL(33);
                    epi_m(cB0, cBw);
                    signal_issuer(0);                       // S4 -> M2m(b) (B1)
                    TL(35);
                    // ---- E6: h'(b)
                    wait_grp(c);
                    TL(37);
                    epi_h(cs + 1, cB0, cBw);
                    TL(38);
                }
            }
        }
        TL(40);

        // ================= end of the episode's tensor work ==================================================
        // (its readout runs later, under the next episode's edge contraction)
        if (has_next) {                                   // next episode's inputs: in flight from here (or earlier, above)
            if (PACKED) load_inputs(b_next);
            else if (c.grp == 1 && nmine < 2) stage_inputs(b_next);
        }
        workers_sync();
        if (PACKED && has_next) {                         // the off-diagonal blocks of |A| were overwritten by H / E: clear
            TL(42);
            zero_image(smem + SM_ABS);
            workers_sync();
            TL(43);
        }
        if (c.tid == 0 && has_next) {                     // H / E (which |A| overlays) have no reader left
            if (PACKED) mbar_arrive(&sig[0]);             // -> contraction issuer: fetches the pack's |A| blocks with all its lanes
            else fetch_ops(1, b_next);
        }
        if (c.tid == 0 && (!PACKED || has_next)) mbar_arrive(&tail_sig);   // -> tail warp: this episode's (pack's) partial sums are complete
        last_b = b;
        TL(41);
    }
    if (PACKED && c.warp < NWARPS && last_b >= 0) readout_packed_all(last_b);
#undef TL

    tc_fence_before();
    __syncthreads();
    if (c.warp == 0) tmem_dealloc(c.tmem, 512);
}

}  // namespace

bool mpnn_tc_supported(const eco_graphs_t* g) { return g->N <= NPMAX && (g->reserved & ECO_GRAPHS_PM1) && g->tc_ops != nullptr; }
size_t mpnn_tc_scratch_bytes(int, int) { return (NWARPS + ISSUERS) * 1024 * 8 + 256; }   // room for the optional debug timeline
size_t mpnn_tc_packed_bytes() { return (size_t)PK_WORDS * 4; }

int launch_mpnn_pack(const eco_mpnn_t* w, void* packed, cudaStream_t st) {
    mpnn_pack_kernel<<<(PK_WORDS + 255) / 256, 256, 0, st>>>(*w, (uint32_t*)packed);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

// Can a rollout step of this (graph set, environment) pair run as one fused launch?  The resident kernel must take the batch
// unpacked (one episode per CTA iteration) and the environment must be the plain ECO-DQN configuration the sub-warp env step
// implements (reversible spins, BLS reward, Max-Cut).
bool mpnn_tc_can_fuse(const eco_graphs_t* g, const eco_env_t* env) {
    const bool packed = PACK_NPMAX / g->NP >= 2 && env->B >= 2;
    // (>= 2 episodes per CTA: an episode's next observations are staged one item after its tail wrote them)
    return mpnn_tc_supported(g) && !packed && env->reserved == 0 && !(g->reserved & ECO_GRAPHS_MIN_CUT) && env->N == g->N &&
           env->B >= 2 * device_sm_count();
}

int launch_mpnn_tc(const eco_graphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn,
                   const float* xg, float norm_max, float* q, int32_t* actions, void* scratch, cudaStream_t st) {
    return launch_mpnn_tc_fused(g, w, B, gidx, xn, xg, norm_max, q, actions, scratch, nullptr, 1, nullptr, nullptr, nullptr, st);
}

int launch_mpnn_tc_fused(const eco_graphs_t* g, const eco_mpnn_t* w, int B, const int32_t* gidx, const float* xn,
                         const float* xg, float norm_max, float* q, int32_t* actions, void* scratch, const eco_env_t* fused,
                         int n_steps, int32_t* ha, double* hr, double* hs, cudaStream_t st) {
    static unsigned long long attr_set = 0;
    const int n_sm = device_sm_count();
    if (first_use_on_device(&attr_set)) {
        ECO_CUDA((cudaFuncSetAttribute(mpnn_tc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL)));
        ECO_CUDA((cudaFuncSetAttribute(mpnn_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL)));
        ECO_CUDA((cudaFuncSetAttribute(mpnn_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL)));
        ECO_CUDA((cudaFuncSetAttribute(mpnn_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL)));
        ECO_CUDA((cudaFuncSetAttribute(mpnn_tc_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL)));
    }
    const int packK = PACK_NPMAX / g->NP;                  // small graphs: several per CTA iteration
    const bool packed = packK >= 2 && B >= 2;
    if (fused && packed) { set_error("launch_mpnn_tc_fused: packed batches cannot be fused"); return ECO_ERR_INVALID; }
    const int units = packed ? (B + packK - 1) / packK : B;
    const int grid = units < n_sm ? units : n_sm;
    const int prof_kind = fused ? ECO_PROF_ROLLOUT : ECO_PROF_MPNN;
    prof_begin(prof_kind, st, fused ? n_steps : 1);
    static const bool timeline = getenv("ECO_TC_TIMELINE") != nullptr;
    if (timeline) ECO_CUDA(cudaMemsetAsync(scratch, 0, (NWARPS + ISSUERS) * 1024 * 8, st));
    unsigned long long* dbg = timeline ? (unsigned long long*)scratch : nullptr;
    // (the clock trace of tools/tc_timeline.py is its own instantiation: the production kernels carry no trace code)
    FusedEnv fe{};
    fe.n_steps = 1;
    if (fused) {
        if (n_steps < 1 || B < 2 * grid) { set_error("launch_mpnn_tc_fused: needs n_steps >= 1 and two episodes per CTA"); return ECO_ERR_INVALID; }
        fe.env = *fused; fe.hist_a = ha; fe.hist_r = hr; fe.hist_s = hs; fe.n_steps = n_steps;
    }
    if (packed && dbg) mpnn_tc_kernel<true, true><<<grid, LAUNCH_THREADS, SM_TOTAL, st>>>(*g, *w, B, gidx, xn, xg, norm_max, q, actions, dbg, packK, fe);
    else if (packed) mpnn_tc_kernel<true, false><<<grid, LAUNCH_THREADS, SM_TOTAL, st>>>(*g, *w, B, gidx, xn, xg, norm_max, q, actions, nullptr, packK, fe);
    else if (dbg) mpnn_tc_kernel<false, true><<<grid, LAUNCH_THREADS, SM_TOTAL, st>>>(*g, *w, B, gidx, xn, xg, norm_max, q, actions, dbg, 1, fe);
    else if (fused) mpnn_tc_kernel<false, false, true><<<grid, LAUNCH_THREADS, SM_TOTAL, st>>>(*g, *w, B, gidx, xn, xg, norm_max, q, actions, nullptr, 1, fe);
    else mpnn_tc_kernel<false, false><<<grid, LAUNCH_THREADS, SM_TOTAL, st>>>(*g, *w, B, gidx, xn, xg, norm_max, q, actions, nullptr, 1, fe);
    prof_end(prof_kind, st);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

}  // namespace eco
