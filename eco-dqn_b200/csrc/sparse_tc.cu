// Kernel family 5b: the per-vertex linears of the CSR-set MPNN forward on the tensor cores.
//
// Replaces (reference, file:line)  src/networks/mpnn.py:40-159 MPNN.forward, its Linear layers
//   :99 edge_feature_NN (W_ef, K = 64),  :117 message_layer (W_m, K = 128),  :119 update_layer (W_u, K = 128)
// in the gather forward of sparse.cu (launch_smpnn_tc): the same contract as k_gemm<false, K> there,
//   C[v][0:64] = ReLU([A1 | A2][v][0:K] . W^T),   planes [V][64] fp32, vertex-major,
// so the gathers, the input stage and the readout run unchanged around it.
//
// Precision (as the operand-tile pipeline, mpnn_large.cu, DESIGN.md section 4.2): W and the inputs are each split into bf16
// hi + lo; the product sums W_hi X_hi + W_lo X_hi + W_hi X_lo with fp32 accumulation (W_lo X_lo is never computed).
//
// Persistent CTAs of 128 threads over 64-vertex items.  The packed weights (eco_mpnn_pack) sit in TMEM for the whole
// launch.  Per item: one thread fetches the next item's fp32 rows into the other staging buffer by bulk copy (each row is
// read once, by one CTA); all threads split the staged rows into bf16 hi / lo operand tiles (the tile format of
// mpnn_large.cu: 128 stacked rows x 64 vertices, core matrices of 8 rows x 8 vertices); one thread issues the MMAs
// (D^T[stacked feature row][vertex] in TMEM); the epilogue adds the hi and lo rows, applies ReLU, transposes through the
// staging buffer just consumed and stores whole [v][64] rows, one 32-byte sector per store.
// Bytes per vertex: K * 4 read, 256 written (the algorithmic minimum, as k_gemm).
#include "eco_common.cuh"
#include "tc_prims.cuh"
#include "mpnn_pack.cuh"

namespace eco {
namespace {

using namespace tc;

constexpr int SV = 64;                          // vertices per item
constexpr int STILE = 128 * SV * 2;             // 16 KB: one bf16 hi/lo operand tile (64 features)
constexpr int SROWS = SV * 64 * 4;              // 16 KB: 64 fp32 rows of one input plane
constexpr uint32_t ST_W = 0, ST_ACC = 64;       // TMEM columns: weights (K / 2), accumulator (64 vertices)

template <int K>
constexpr int stc_smem() { return 2 * (K / 64) * SROWS + (K / 64) * STILE; }

// 8 MMAs: acc (+)= W[:, 64-feature group at TMEM column tw] * X, X an operand tile used as MN-major B operand; the lo
// rows of X meet W_hi only (M = 64 covers TMEM lanes 32q + 0..15, the hi rows of the stacked order), as mpnn_large.cu
__device__ __forceinline__ void issue_tile(uint32_t tmem, uint32_t tw, const unsigned char* x, int width, bool accumulate) {
    const uint32_t idesc = instr_desc_bf16(128, width, false, true);
    const uint32_t idesc_lo = instr_desc_bf16(64, width, false, true);
    const uint64_t d = smem_desc(smem_u32(x), /*LBO (k groups)*/ 128, /*SBO (vertex groups)*/ 2048);
#pragma unroll
    for (int i = 0; i < 8; ++i)     // i = 2*kq + s: features 16kq..16kq+15, split s
        mma_ts(tmem + ST_ACC, tmem + tw + 8 * (i >> 1), d + (uint64_t)(16 * i), (i & 1) ? idesc_lo : idesc, accumulate || i > 0);
}

template <int K>
__global__ void __launch_bounds__(128, 2)
sparse_linear_tc_kernel(const float* __restrict__ A1, const float* __restrict__ A2, const long long V,
                        const uint32_t* __restrict__ pk, float* __restrict__ Cout) {
    constexpr int NIN = K / 64;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t full[2], bar;
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const long long nitems = (V + SV - 1) / SV;
    unsigned char* tiles = smem + 2 * NIN * SROWS;

    if (warp == 0) tmem_alloc(&tmem_base_s, 128);
    if (tid == 0) { mbar_init(&full[0], 1); mbar_init(&full[1], 1); mbar_init(&bar, 1); fence_mbar_init(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;

    auto fetch = [&](long long item, int s) {              // one thread: the item's rows of every input plane -> stage s
        const long long v0 = item * SV;
        const uint32_t bytes = (uint32_t)min((long long)SV, V - v0) * 256u;
        mbar_expect_tx(&full[s], NIN * bytes);
        bulk_g2s(smem + (s * NIN + 0) * SROWS, A1 + v0 * 64, bytes, &full[s]);
        if (NIN == 2) bulk_g2s(smem + (s * NIN + 1) * SROWS, A2 + v0 * 64, bytes, &full[s]);
    };
    if (tid == 0 && (long long)blockIdx.x < nitems) fetch(blockIdx.x, 0);
    {   // the weights: packed global -> registers -> TMEM (warp q owns lane quadrant q), as tcl_linear_kernel
        constexpr int KW = K / 2;                          // words per stacked row
        const uint4* src = reinterpret_cast<const uint4*>(pk) + (size_t)(warp * (KW / 8) * 2) * 32 + lane;
        for (int cg = 0; cg < KW / 8; ++cg) {
            const uint4 x = __ldg(src + (2 * cg) * 32), y = __ldg(src + (2 * cg + 1) * 32);
            const uint32_t v[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
            tmem_st_32x32b_x8(tmem_addr(tmem, 32 * warp, ST_W + cg * 8), v);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncthreads();
    }
    uint32_t phase = 0;
    int it = 0;
    for (long long item = blockIdx.x; item < nitems; item += gridDim.x, ++it) {
        const int s = it & 1;
        const long long v0 = item * SV;
        const int wdt = (int)min((long long)SV, V - v0);   // V = B * NP, NP % 16 == 0: so is wdt
        if (tid == 0 && item + (long long)gridDim.x < nitems) fetch(item + gridDim.x, s ^ 1);   // idle since the last item
        mbar_wait(&full[s], (uint32_t)((it >> 1) & 1));
        // split: thread (feature f, 8-vertex group cb) -> 16 bytes of hi and of lo, core (cb, stacked row of f)
        const float* rows = reinterpret_cast<const float*>(smem + s * NIN * SROWS);
        for (int task = tid; task < NIN * 64 * (wdt >> 3); task += 128) {
            const int f = task & 63, p = (task >> 6) % NIN, cb = (task >> 6) / NIN;
            const float* r = rows + p * (SROWS / 4) + (cb * 8) * 64 + f;
            float x[8];
#pragma unroll
            for (int v = 0; v < 8; ++v) x[v] = r[v * 64];
            uint4 hi, lo;
            split2(x[0], x[1], hi.x, lo.x);
            split2(x[2], x[3], hi.y, lo.y);
            split2(x[4], x[5], hi.z, lo.z);
            split2(x[6], x[7], hi.w, lo.w);
            const int hr = 32 * (f >> 4) + (f & 15);       // stacked hi row of feature f; the lo row is 2 core rows further
            unsigned char* t = tiles + p * STILE + (cb * 16 + (hr >> 3)) * 128 + (hr & 7) * 16;
            *reinterpret_cast<uint4*>(t) = hi;
            *reinterpret_cast<uint4*>(t + 256) = lo;
        }
        fence_proxy_async();                               // the tiles are read by the tensor cores (async proxy)
        tc_fence_before();
        __syncthreads();
        if (warp == 0) {
            tc_fence_after();
            if (elect_one()) {
                issue_tile(tmem, ST_W, tiles, wdt, false);
                if (NIN == 2) issue_tile(tmem, ST_W + 32, tiles + STILE, wdt, true);
                mma_commit(&bar);
            }
            __syncwarp();
        }
        mbar_wait(&bar, phase);
        phase ^= 1u;
        tc_fence_after();
        // epilogue: hi + lo rows, ReLU -> out[v][f] over the staged rows of this item (consumed), swizzled: float4 group
        // g of row v at g ^ (v & 7) -- conflict-free for the TMEM fragment writes and for the row reads below
        float* out = reinterpret_cast<float*>(smem + s * NIN * SROWS);
        for (int blk = 0; blk < (wdt >> 4); ++blk) {
            uint32_t vh[8], vl[8];
            tmem_ld_16x256b_x2(tmem_addr(tmem, 32 * warp, ST_ACC + 16 * blk), vh);
            tmem_ld_16x256b_x2(tmem_addr(tmem, 32 * warp + 16, ST_ACC + 16 * blk), vl);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 8; ++i) {                  // (row lane/4 + 8 ((i >> 1) & 1), col 2 (lane & 3) + (i & 1) + 8 (i >> 2))
                const int f = 16 * warp + (lane >> 2) + 8 * ((i >> 1) & 1);
                const int v = 16 * blk + 2 * (lane & 3) + (i & 1) + 8 * (i >> 2);
                out[v * 64 + (f ^ ((v & 7) << 2))] = fmaxf(__uint_as_float(vh[i]) + __uint_as_float(vl[i]), 0.f);
            }
        }
        __syncthreads();
        // rows out: thread (vertex v, sector j) stores features 8j..8j+7 in one 32-byte store; lanes j >= 4 read their
        // upper float4 first (no bank conflict between the two halves of a quarter warp)
        for (int idx = tid; idx < wdt * 8; idx += 128) {
            const int v = idx >> 3, j = idx & 7, sw = v & 7, h = (j >> 2) & 1;
            const float4 a = *reinterpret_cast<const float4*>(&out[v * 64 + 4 * ((2 * j + h) ^ sw)]);
            const float4 b = *reinterpret_cast<const float4*>(&out[v * 64 + 4 * ((2 * j + (h ^ 1)) ^ sw)]);
            const float4 lo4 = h ? b : a, hi4 = h ? a : b;
            const float o[8] = {lo4.x, lo4.y, lo4.z, lo4.w, hi4.x, hi4.y, hi4.z, hi4.w};
            st_f32x8(Cout + (v0 + v) * 64 + 8 * j, o);
        }
        fence_proxy_async();                               // this stage is refilled by a bulk copy (async proxy)
        tc_fence_before();
        __syncthreads();                                   // the stage, the tiles and the accumulator are reused
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 128);
}

}  // namespace

// C = ReLU([A1 | A2] W^T) on V vertex rows; w_packed: the matrix's words of eco_mpnn_pack output (PK_WEF for K = 64,
// PK_WM / PK_WU + layer * 128 * 64 for K = 128).  A1, A2, C 16-byte aligned, V a multiple of 16.
int launch_sparse_linear_tc(const float* A1, const float* A2, int K, long long V, const void* w_packed, float* C,
                            cudaStream_t st) {
    static unsigned long long attr = 0;
    if (first_use_on_device(&attr)) {
        ECO_CUDA(cudaFuncSetAttribute(sparse_linear_tc_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, stc_smem<64>()));
        ECO_CUDA(cudaFuncSetAttribute(sparse_linear_tc_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, stc_smem<128>()));
    }
    const long long items = (V + SV - 1) / SV, cap = 2LL * device_sm_count();
    const unsigned grid = (unsigned)(items < cap ? items : cap);
    const uint32_t* pk = static_cast<const uint32_t*>(w_packed);
    if (K == 64) sparse_linear_tc_kernel<64><<<grid, 128, stc_smem<64>(), st>>>(A1, nullptr, V, pk, C);
    else sparse_linear_tc_kernel<128><<<grid, 128, stc_smem<128>(), st>>>(A1, A2, V, pk, C);
    ECO_LAUNCH_CHECK();
    return ECO_OK;
}

}  // namespace eco
