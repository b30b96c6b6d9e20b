// Kernel family 2c: stand-alone tensor-core neighbour aggregation on fp32 rows (eco_graph_aggregate), couplings in
// {-1,0,1}, any N <= 2048.
//
// Replaces (reference, file:line) the N x N product of the MPNN layers:
//   src/networks/mpnn.py:114-116  UpdateNodeEmbeddingLayer: torch.matmul(adj, node_features) / norm
//   src/networks/mpnn.py:89-102   EdgeAndNodeEmbeddingLayer: sum_j ReLU(W_e [a_ij ; x_j]) [a_ij != 0] / norm, in the
//                                 factorised form 1/2 (|A| S + A D) of mpnn_tc.cu (S = R+ + R-, D = R+ - R-)
// for callers that hold [N][64] fp32 features.  (The MPNN forward for large graphs, mpnn_large.cu, keeps its
// activations as operand tiles and has its own bulk-copy-fed contraction.)
//
//   OUT[b][i][f] = scale / deg_i * sum_j ( X1[b][j][f] * IMG1_g[j][i]  (+ X2[b][j][f] * IMG2_g[j][i]) )
//
// One CTA per (episode, 128-column slab).  K is walked in 64-vertex panels: the fp32 rows X[j][0..63] are split into
// bf16 hi/lo, stacked along M (128 rows, same row order as mpnn_tc.cu) and written as a K-major A-operand; the matching
// panel of the graph's bf16 operand image (graph_prepare.cu: tc_ops) arrives by bulk copies; tcgen05.mma accumulates the
// slab in TMEM (128 columns, so four CTAs share an SM and overlap each other's load / convert / MMA phases -- there is
// no pipeline inside a CTA).
#include <cuda_bf16.h>

#include "eco_common.cuh"
#include "tc_prims.cuh"

namespace eco {
namespace {

using namespace tc;

constexpr int SLAB = 128;        // accumulator columns (vertices i) per CTA
constexpr int PANEL = 64;        // vertices j per K panel
constexpr int TCL_THREADS = 128;
constexpr int XF_BYTES = 64 * 65 * 4 + 256;                 // fp32 staging [64][65], padded to a multiple of 128 bytes
static_assert(XF_BYTES % 128 == 0, "staging size");
constexpr int OP_BYTES = 128 * PANEL * 2;                   // one operand panel (A: 128 rows x 64 k; B: 64 k x 128 cols)

template <int PAIRS>
__global__ void __launch_bounds__(TCL_THREADS)
graph_aggregate_kernel(const eco_graphs_t g, const int32_t* __restrict__ graph_idx, const int B,
                    const float* __restrict__ X1, const int which1, const float* __restrict__ X2, const int which2,
                    const size_t x_stride, float* __restrict__ out, const size_t out_stride, const float scale,
                    const int edge, const float norm_max) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bar_b, bar_mma;
    __shared__ uint32_t tmem_base_s;
    float* sXf = reinterpret_cast<float*>(smem);
    unsigned char* sX[2] = {smem + XF_BYTES, smem + XF_BYTES + 2 * OP_BYTES};
    unsigned char* sB[2] = {smem + XF_BYTES + OP_BYTES, smem + XF_BYTES + 3 * OP_BYTES};
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int N = g.N, NP = g.NP, NB = NP >> 3;
    const int nslabs = (NP + SLAB - 1) / SLAB;
    const int b = blockIdx.x / nslabs, slab = blockIdx.x % nslabs;
    const int n0 = slab * SLAB, w = min(SLAB, NP - n0);      // NP is a multiple of 16, so is w
    const int gi = graph_idx[b];
    const float* Xp[2] = {X1 + (size_t)b * x_stride, PAIRS == 2 ? X2 + (size_t)b * x_stride : nullptr};
    const uint16_t* img[2] = {g.tc_ops + ((size_t)gi * 2 + which1) * NP * NP,
                              g.tc_ops + ((size_t)gi * 2 + (PAIRS == 2 ? which2 : which1)) * NP * NP};

    if (warp == 0) tmem_alloc(&tmem_base_s, 128);
    if (tid == 0) { mbar_init(&bar_b, 1); mbar_init(&bar_mma, 1); fence_mbar_init(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;
    uint32_t phase_b = 0, phase_m = 0;
    // this thread's stacked operand row: r = 32q + 16s + t  <->  feature 16q + t, split s (hi / lo)
    const int r = tid, f = 16 * (r >> 5) + (r & 15), split = (r >> 4) & 1;
    const int npanels = (NP + PANEL - 1) / PANEL;
    const int run = (w >> 3) * 128;                            // bytes of one 8-vertex K group of the B panel

    for (int kp = 0; kp < npanels; ++kp) {
        const int k0 = kp * PANEL, kw = min(PANEL, NP - k0);
        if (kp > 0) { mbar_wait(&bar_mma, phase_m); phase_m ^= 1u; }       // the previous panel's MMAs have read smem
        if (tid == 0) {
            mbar_expect_tx(&bar_b, (uint32_t)(PAIRS * (kw >> 3) * run));
            for (int p = 0; p < PAIRS; ++p)
                for (int cb = 0; cb < (kw >> 3); ++cb)
                    bulk_g2s(sB[p] + cb * run, reinterpret_cast<const unsigned char*>(img[p]) + tc_image_core(NB, (k0 >> 3) + cb, n0 >> 3), run, &bar_b);
        }
        for (int p = 0; p < PAIRS; ++p) {
            if (p > 0) __syncthreads();                                     // sXf is reused
            for (int idx = tid; idx < kw * 64; idx += TCL_THREADS) {        // coalesced fp32 rows of the panel
                const int jj = idx >> 6, ff = idx & 63;
                sXf[jj * 65 + ff] = (k0 + jj < N) ? Xp[p][(size_t)(k0 + jj) * 64 + ff] : 0.f;
            }
            __syncthreads();
            for (int jj = 0; jj < kw; jj += 2) {
                uint32_t hi, lo;
                split2(sXf[jj * 65 + f], sXf[(jj + 1) * 65 + f], hi, lo);
                *reinterpret_cast<uint32_t*>(sX[p] + (((jj >> 3) * 16 + (r >> 3)) * 128 + (r & 7) * 16 + (jj & 7) * 2)) =
                    split ? lo : hi;
            }
        }
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (warp == 0) {
            mbar_wait(&bar_b, phase_b);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t idesc = instr_desc_bf16(128, w, false, false);
                for (int p = 0; p < PAIRS; ++p) {
                    const uint64_t ad = smem_desc(smem_u32(sX[p]), 2048, 128);
                    const uint64_t bd = smem_desc(smem_u32(sB[p]), run, 128);
                    for (int ks = 0; ks < (kw >> 4); ++ks)
                        mma_ss(tmem, ad + (uint64_t)ks * (4096 >> 4), bd + (uint64_t)ks * ((2 * run) >> 4), idesc,
                               kp > 0 || p > 0 || ks > 0);
                }
                mma_commit(&bar_mma);
            }
            __syncwarp();
        }
        phase_b ^= 1u;
    }
    mbar_wait(&bar_mma, phase_m);
    tc_fence_after();

    // epilogue: hi + lo rows, scale, 1 / deg; feature 63 of the edge stage = deg / deg_max (mpnn.py:102)
    const float dmax = norm_max > 0.f ? norm_max : (norm_max < 0.f ? (float)max(g.gstat[(size_t)gi * 4], 1) : *g.dmax);
    float* ob = out + (size_t)b * out_stride;
    for (int blk = 0; blk < (w >> 4); ++blk) {
        uint32_t vh[8], vl[8];
        tmem_ld_16x256b_x2(tmem_addr(tmem, 32 * warp, 16 * blk), vh);
        tmem_ld_16x256b_x2(tmem_addr(tmem, 32 * warp + 16, 16 * blk), vl);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int n = n0 + 16 * blk + 8 * (i >> 2) + 2 * (lane & 3) + (i & 1);
            const int ff = 16 * warp + (lane >> 2) + 8 * ((i >> 1) & 1);
            if (n < N) {
                const float d = g.deg[(size_t)gi * NP + n];
                const float v = (__uint_as_float(vh[i]) + __uint_as_float(vl[i])) * scale;
                ob[(size_t)n * 64 + ff] = (edge && ff == 63) ? d / dmax : v / d;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 128);
}

}  // namespace

bool mpnn_tcl_supported(const eco_graphs_t* g) { return (g->reserved & ECO_GRAPHS_PM1) && g->tc_ops != nullptr; }

// OUT = scale / deg * (X1 * IMG[which1] (+ X2 * IMG[which2]));  X*, OUT: [B][*][64] fp32 with the given episode strides
int launch_tcl_contract(const eco_graphs_t* g, const int32_t* gidx, int B, const float* X1, int which1, const float* X2,
                        int which2, size_t x_stride, float* out, size_t out_stride, float scale, int edge,
                        float norm_max, cudaStream_t st) {
    static unsigned long long attr = 0;
    const int smem1 = XF_BYTES + 2 * OP_BYTES, smem2 = XF_BYTES + 4 * OP_BYTES;
    if (first_use_on_device(&attr)) {
        ECO_CUDA(cudaFuncSetAttribute(graph_aggregate_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem1));
        ECO_CUDA(cudaFuncSetAttribute(graph_aggregate_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2));
    }
    const int nslabs = (g->NP + SLAB - 1) / SLAB;
    const unsigned grid = (unsigned)((size_t)B * nslabs);
    if (X2)
        graph_aggregate_kernel<2><<<grid, TCL_THREADS, smem2, st>>>(*g, gidx, B, X1, which1, X2, which2, x_stride, out,
                                                                 out_stride, scale, edge, norm_max);
    else
        graph_aggregate_kernel<1><<<grid, TCL_THREADS, smem1, st>>>(*g, gidx, B, X1, which1, nullptr, which1, x_stride, out,
                                                                 out_stride, scale, edge, norm_max);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

}  // namespace eco
