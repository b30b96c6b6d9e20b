/*
 * ecodqn_b200.h -- C ABI of the B200-native batched ECO-DQN Max-Cut rollout engine.
 *
 * This is the drop-in boundary for ONE hot path of BetterBelle/eco-dqn: batched environment stepping +
 * MPNN Q-evaluation + greedy action selection (SURVEY.md section 8).  The reference is pure Python and has
 * no FFI of its own; each entry point below names the reference interface it replaces (file:line under the
 * reference tree) and INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  Pointers named *_dev are CUDA device pointers on the
 *     current device; *_host are host pointers (pinned memory recommended).  `stream` is a cudaStream_t
 *     passed as void* (NULL = legacy default stream).  Nothing here allocates device memory except
 *     eco_host_session_*; callers own every buffer (PyTorch's caching allocator in the Python host).
 *   - Every function returns ECO_OK (0) or a negative error code; eco_last_error() gives the message of the
 *     last failure on the calling thread.  Shape / configuration violations are rejected before any launch.
 *   - All work is enqueued asynchronously on `stream`; no entry point synchronises unless it says so.
 *   - Vertices are padded to NP = 16*ceil(N/16) per row; padded entries are zero and never selected.
 *   - Integer-weight graphs (int8 couplings; the reference's EdgeType.UNIFORM / DISCRETE) through eco_graphs_t, and
 *     real-valued graphs (fp64 couplings; EdgeType.RANDOM) through the eco_wgraphs_t / eco_wenv_t entry points at the
 *     end of this header, and integer-weight graphs of up to ECO_MAX_SPINS_SPARSE vertices stored as CSR through the
 *     eco_sgraphs_t entry points after them.  There is no CPU fallback anywhere in this library.
 */
#ifndef ECODQN_B200_H
#define ECODQN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ECO_OK                 0
#define ECO_ERR_INVALID       -1   /* bad argument / shape / alignment                                    */
#define ECO_ERR_UNSUPPORTED   -2   /* configuration outside the accelerated path (NotImplementedError)    */
#define ECO_ERR_CUDA          -3   /* a CUDA runtime call failed (message has the cudaError string)       */
#define ECO_ERR_STATE         -4   /* e.g. stepping an environment that already returned done             */

#define ECO_ABI_VERSION        1
#define ECO_N_FEATURES         64  /* MPNN width, reference src/networks/mpnn.py:9                         */
#define ECO_N_OBS              7   /* DEFAULT_OBSERVABLES, reference src/envs/utils.py:68-74               */
#define ECO_MAX_SPINS          2048

/* policies for eco_env_step / eco_rollout */
#define ECO_POLICY_ACTIONS     0   /* actions supplied by the caller (teacher forcing, epsilon-greedy)     */
#define ECO_POLICY_NETWORK     1   /* argmax_i Q_i, lowest index on ties (experiments/utils.py:57-66)      */
#define ECO_POLICY_GREEDY      2   /* argmax_i s_i h_i, stop when the best gain < 0 (src/agents/solver.py:105-131) */

/* eco_graphs_t.reserved bits: every coupling is in {-1,0,1} (asserted by the caller, see gstat flags); OptimisationTarget.MIN_CUT
 * instead of CUT (quality = qn - cut, qn = |sum of negative weights|, masks = negated cut changes) */
#define ECO_GRAPHS_PM1         1
#define ECO_GRAPHS_MIN_CUT     2

/* eco_env_t.reserved mode bits: the S2V-DQN configuration of the reference (experiments/pretrained_agent/test_s2v.py) is
 * ECO_ENV_IRREVERSIBLE | ECO_ENV_DENSE_REWARD with use_basin = 0 */
#define ECO_ENV_IRREVERSIBLE   1   /* reversible_spins=False: done when no spin is left at -1 (spinsystem.py:552-556);
                                      ECO_POLICY_GREEDY / ECO_POLICY_NETWORK choose among the spins still at -1
                                      (solver.py:116-121, experiments/utils.py:67-74)                       */
#define ECO_ENV_DENSE_REWARD   2   /* RewardSignal.DENSE: reward = normalised score change (spinsystem.py:435-436) */

/* MPNN implementations */
#define ECO_MPNN_AUTO          0
#define ECO_MPNN_SIMT          1   /* fp32 CUDA-core kernel: any int8 weights, any N <= ECO_MAX_SPINS      */
#define ECO_MPNN_TCGEN05       2   /* tcgen05/TMEM tensor-core kernels: weights in {-1,0,1}                  */

const char* eco_last_error(void);
int         eco_abi_version(void);

/* ---------------------------------------------------------------------------------------------------------
 * Graph set: G dense symmetric int8 adjacency matrices of N vertices, shared read-only by all episodes.
 * Replaces the per-env `self.matrix` (reference src/envs/spinsystem.py:151-155,196) supplied by
 * SingleGraphGenerator / SetGraphGenerator (src/envs/utils.py:337-345, 376-382), and the scorer constants
 * of MaximumCutUnbiasedScorer (src/envs/score_solver.py:347-375): mlr, qn, lb.
 * --------------------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t  G, N, NP, reserved;   /* ECO_GRAPHS_PM1: caller asserts every coupling is in {-1,0,1} (see gstat flags);
                                      ECO_GRAPHS_MIN_CUT: set BEFORE upload/load/update -- the constants below are the
                                      Min-Cut scorer's (score_solver.py:423-505) and every env kernel negates its masks */
    int8_t*  J;          /* [G, NP, NP]  couplings, zero padded                                              */
    double*  gscal;      /* [G, 4]       mlr (max non-zero weighted degree), qn, lb, sum_ij J_ij             */
    float*   deg;        /* [G, NP]      max(1, #non-zeros in row i)  (mpnn.py:34-38)                        */
    int32_t* gstat;      /* [G, 4]       max degree, nnz, max |row abs sum|, flags (bit0: weights outside {-1,0,1},
                                         bit1: all weighted degrees zero, bit2: not symmetric / non-zero diagonal)  */
    float*   dmax;       /* [1]          max degree over the whole set (default norm.max(), mpnn.py:102)     */
    float*   gain_tab;   /* [G, 2*NP+4]  entry [NP + k] = (float)((double)k / mlr) for k = -NP..NP: observable row 1 of a vertex whose
                                         flip changes the cut by k (valid for couplings in {-1,0,1}; spinsystem.py:490) */
    double*  dn_tab;     /* [G, 2*NP+4]  entry [NP + k] = (double)k / qn: the normalised score change of such a flip (spinsystem.py:394) */
    uint16_t* tc_ops;    /* [G, 2, NP*NP] bf16 images of J and |J| in the tensor-core kernels' shared-memory operand
                                         layout (8x8 core matrices; slabs of 256 columns for NP > 256), fetched with one
                                         bulk copy per episode (N <= 208) or per 64-row panel (larger graphs)     */
} eco_graphs_t;

size_t eco_graphs_workspace_bytes(int32_t G, int32_t N);
/* carve `workspace_dev` (>= eco_graphs_workspace_bytes, 256-byte aligned) into the arrays of `g` */
int    eco_graphs_bind(eco_graphs_t* g, void* workspace_dev, int32_t G, int32_t N);
/* copy G*N*N int8 couplings from host memory into the padded device layout (async on stream) and prepare */
int    eco_graphs_upload(eco_graphs_t* g, const int8_t* J_host, void* stream);
/* same, source already on the device, dense [G, N, N] */
int    eco_graphs_load_dev(eco_graphs_t* g, const int8_t* J_dev, void* stream);
/* replace the graphs in slots [first, first + count) (J_dev dense [count, N, N]) and refresh their constants: the
 * graph ring of the DQN trainer (a new random graph per episode, reference spinsystem.py:196) */
int    eco_graphs_update(eco_graphs_t* g, int32_t first, int32_t count, const int8_t* J_dev, void* stream);
/* Sparse ingest: the graphs of slots [first, first + count) from EDGE LISTS already on the device -- graph k owns entries
 * offsets_dev[k] .. offsets_dev[k+1]-1 of rows_dev / cols_dev (0-based vertices) / weights_dev -- without a dense N x N copy
 * crossing PCIe or existing on the host: the slots are zeroed, J[i][j] (and J[j][i] when `symmetric` != 0) are set to the
 * entry's weight, then the constants are refreshed.  This is how the GSet `.mc` instances and the scipy-CSR pickles of the
 * reference's loaders (experiments/utils.py:391-432: edge list -> dense float64 -> torch) reach the device: CSR is
 * rows = repeat(arange(N), diff(indptr)), cols = indices, symmetric = 0.  Duplicate entries: the last writer wins (the
 * reference's `matrix[i, j] = w` assignment); entries outside [0, N) make the call fail with ECO_ERR_INVALID (checked on
 * the device, reported after a stream synchronise).  n_entries = offsets[count], passed by the caller. */
int    eco_graphs_load_edges_dev(eco_graphs_t* g, int32_t first, int32_t count, const int64_t* offsets_dev,
                                 const int32_t* rows_dev, const int32_t* cols_dev, const int8_t* weights_dev,
                                 int64_t n_entries, int32_t symmetric, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Batched environment state (struct of arrays), B independent episodes.
 * Replaces SpinSystemBase's per-episode Python state (reference src/envs/spinsystem.py:183-259, 355-559):
 * self.state rows 0..6, score / normalized_score, best_* trackers, current_step, HistoryBuffer.
 * --------------------------------------------------------------------------------------------------------- */
typedef struct {          /* 96 bytes per episode                                                            */
    int32_t step;         /* current_step                                                                    */
    int32_t cut;          /* cut value of the current spins (integer for integer couplings)                  */
    int32_t best_cut;     /* best_solution                                                                   */
    int32_t dist;         /* Hamming distance to best_obs_spins (observable row 4)                           */
    int32_t n_improving;  /* #{i : s_i h_i > 0} (observable row 5 numerator; 0 <=> local optimum)            */
    int32_t flags;        /* bit0 done, bit1 greedy-stopped                                                  */
    int32_t n_visited;    /* entries in the visited-set table                                                */
    int32_t reserved;
    double  score, nscore, best_score, best_nscore;
    uint64_t key[2];      /* 128-bit Zobrist key of the set of vertices flipped w.r.t. the initial spins     */
    double  total_reward; /* running sum of rewards (solver.py:60-61 total_reward)                           */
    double  last_reward;
} eco_episode_t;

typedef struct {
    int32_t  B, N, NP, NW;          /* NW = NP/32 rounded up: words of the best-diff bitmask                 */
    int32_t  T, HCAP, use_basin, reserved;   /* reserved: ECO_ENV_* mode bits, set by the caller after eco_env_bind (0 = ECO-DQN) */
    double   basin_reward;          /* added when a NEW local optimum is reached (spinsystem.py:450-457)     */
    int8_t*        spins;           /* [B, NP]                                                               */
    int16_t*       hfield;          /* [B, NP]  local fields h = J s                                         */
    uint16_t*      last_flip;       /* [B, NP]  step at which vertex i was last flipped (0 = never)          */
    uint32_t*      diff_bits;       /* [B, NW]  bit i set <=> s_i != best_obs_spins_i                        */
    int32_t*       graph_idx;       /* [B]                                                                   */
    eco_episode_t* ep;              /* [B]                                                                   */
    uint64_t*      visited;         /* [B, HCAP, 2]  open-addressed set of 128-bit keys (utils.py:438-464)   */
    uint64_t*      zobrist;         /* [NP, 2]                                                               */
    float*         tsf_tab;         /* [T+1]  k-fold fp64 sum of 1/T, cast to fp32 (spinsystem.py:493)       */
    float*         imm_tab;         /* [T+1]  termination immanency per step (spinsystem.py:509-511)         */
    float*         xn;              /* [B, 3, NP] per-vertex observables: spin, s*h/mlr, time since flip     */
    float*         xg;              /* [B, 4]  global observables rows 3..6                                  */
    float*         frac_tab;        /* [N+1]  (float)((double)k / N): observable row 5 (spinsystem.py:513-514)  */
} eco_env_t;

size_t eco_env_workspace_bytes(int32_t B, int32_t N, int32_t T);
int    eco_env_bind(eco_env_t* env, void* workspace_dev, int32_t B, int32_t N, int32_t T,
                    double basin_reward /* < 0: none */);
/* upload Zobrist keys and the two fp32 tables (host -> device, async); tables have T+1 entries */
int    eco_env_set_tables(eco_env_t* env, const uint64_t* zobrist_host, const float* tsf_host,
                          const float* imm_host, void* stream);

/* reset(spins) for all B episodes: reference spinsystem.py:183-259 / 283-330.
 * graph_idx_dev [B] int32, init_spins_dev [B, N] int8 in {-1,+1} (dense, unpadded). */
int eco_env_reset(const eco_graphs_t* g, eco_env_t* env, const int32_t* graph_idx_dev,
                  const int8_t* init_spins_dev, void* stream);

/* step(action) for all B episodes: reference spinsystem.py:355-559.  Episodes whose done flag is set are
 * left untouched.  policy: ECO_POLICY_ACTIONS (actions_dev [B] int32 required) or ECO_POLICY_GREEDY.
 * reward_dev [B] double and done_dev [B] uint8 may be NULL.  hist_* may be NULL; when given they are
 * [B, T] arrays written at column (step-1): the action taken, the fp64 reward, the fp64 score. */
int eco_env_step(const eco_graphs_t* g, eco_env_t* env, int32_t policy, const int32_t* actions_dev,
                 double* reward_dev, uint8_t* done_dev, int32_t* hist_actions_dev, double* hist_rewards_dev,
                 double* hist_scores_dev, void* stream);

/* observation rows 0..6 as the reference's get_observation() returns them, cast to fp32 exactly as the
 * reference's drivers cast them (spinsystem.py:561-574; experiments/utils.py:174).  obs7_dev [B, 7, N]. */
int eco_env_observation(const eco_env_t* env, float* obs7_dev, void* stream);

/* argmax_i Q_i over the spins still at -1, lowest index on ties: the action selection of the reference's drivers for
 * irreversible spins (experiments/utils.py:67-74; the spins already flipped are filled with -1000).  q_dev [B, NP] fp32
 * (as written by eco_mpnn_forward), actions_dev [B] int32. */
int eco_env_masked_argmax(const eco_env_t* env, const float* q_dev, int32_t* actions_dev, void* stream);

/* best spins = current spins with the best-diff bits flipped.  best_spins_dev [B, N] int8. */
int eco_env_best_spins(const eco_env_t* env, int8_t* best_spins_dev, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * MPNN Q-network forward (+ fused argmax).  Replaces MPNN.forward, reference src/networks/mpnn.py:40-159,
 * and the argmax of experiments/utils.py:57-66 / src/agents/dqn/dqn.py:490-503.
 * Weights are fp32 device arrays in the reference's state_dict layout (SURVEY.md appendix A.3).
 * --------------------------------------------------------------------------------------------------------- */
typedef struct {
    const float* w_init;      /* node_init_embedding_layer.0.weight          (64, 7)   */
    const float* w_edge;      /* edge_embedding_layer.edge_embedding_NN.weight (63, 8) */
                              /* (S2V-DQN networks, n_obs_in = 1: (64, 1) and (63, 2) -- zero-pad the six missing
                               *  observable columns, the result is the same)                                   */
    const float* w_edge_feat; /* edge_embedding_layer.edge_feature_NN.weight (64, 64)  */
    const float* w_msg[3];    /* update_node_embedding_layer.l.message_layer.weight (64, 128) */
    const float* w_upd[3];    /* update_node_embedding_layer.l.update_layer.weight  (64, 128) */
    const float* w_pool;      /* readout_layer.layer_pooled.weight           (64, 64)  */
    const float* w_read;      /* readout_layer.layers_readout.0.weight       (1, 128)  */
    const float* b_read;      /* readout_layer.layers_readout.0.bias         (1,)      */
    const void*  packed;      /* eco_mpnn_pack() output for the tcgen05 path, or NULL  */
} eco_mpnn_t;

size_t eco_mpnn_scratch_bytes(int32_t B, int32_t N, int32_t impl);
size_t eco_mpnn_packed_bytes(void);
/* pre-split the weights into the bf16 hi/lo operand layout the tcgen05 kernel consumes (device -> device) */
int    eco_mpnn_pack(const eco_mpnn_t* w, void* packed_dev, void* stream);

/* ECO_MPNN_TCGEN05 / AUTO with couplings in {-1,0,1} run on the tensor cores: N <= 208 in one resident kernel (graphs
 * with NP <= 96 are processed 192/NP at a time as one block-diagonal graph), larger graphs as a pipeline of kernels
 * that exchange bf16 operand tiles through scratch_dev; other weights run on the CUDA-core kernel.
 * Q[b, i] for b < B from features xn [B,3,NP] / xg [B,4] and graph_idx [B] (use env->xn etc. for live
 * episodes, or replayed features for training).  norm_max: the batch-wide max degree the reference divides
 * by (mpnn.py:102); 0 means "max degree over the whole graph set", < 0 means "each episode's own graph" (what the
 * reference computes when it evaluates one environment at a time, e.g. DQN.act).
 * q_dev [B, NP] fp32 or NULL; actions_dev [B] int32 or NULL (argmax, lowest index on ties). */
int eco_mpnn_forward(const eco_graphs_t* g, const eco_mpnn_t* w, int32_t B, const int32_t* graph_idx_dev,
                     const float* xn_dev, const float* xg_dev, float norm_max, float* q_dev,
                     int32_t* actions_dev, void* scratch_dev, int32_t impl, void* stream);

/* The N x N product of a message-passing layer on the tensor cores (reference src/networks/mpnn.py:114-116:
 * torch.matmul(adj, node_features) / norm), any N <= ECO_MAX_SPINS, couplings in {-1,0,1}:
 *   out[b][i][f] = scale / max(1, deg_i) * sum_j J'[j][i] * x[b][j][f],   f < 64,   J' = J or |J| (use_abs)
 * x_dev, out_dev: [B, N, 64] fp32.  fp32-accurate (x is split into two bf16 terms, J is exact). */
int eco_graph_aggregate(const eco_graphs_t* g, int32_t B, const int32_t* graph_idx_dev, const float* x_dev,
                        int32_t use_abs, float scale, float* out_dev, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * DQN regression step: loss and its gradients for a replay minibatch.  Replaces (reference src/agents/dqn/dqn.py:436-447)
 *   q_value = self.network(states).gather(1, actions); loss = self.loss(q_value, td_target); loss.backward()
 * i.e. MPNN.forward (src/networks/mpnn.py:38-159) plus its autograd backward.  Couplings in {-1,0,1}.
 *   loss_dev [1] fp32 = mean_b l(Q[b, actions[b]] - targets[b]),  l = square (ECO_LOSS_MSE, F.mse_loss) or
 *   smooth-L1 with beta 1 (ECO_LOSS_HUBER, F.smooth_l1_loss)           (dqn.py:113-121)
 *   grad_dev [ECO_MPNN_N_PARAMS] fp32: d loss / d weights, the 12 tensors of eco_mpnn_t one after the other in
 *   state_dict order (w_init, w_edge, w_edge_feat, w_msg[0], w_upd[0], ..., w_pool, w_read, b_read).
 * features as for eco_mpnn_forward; actions_dev [B] int32, targets_dev [B] fp32.  Bit-reproducible (fixed-order sums).
 * --------------------------------------------------------------------------------------------------------- */
#define ECO_MPNN_N_PARAMS      58425
#define ECO_LOSS_MSE           0
#define ECO_LOSS_HUBER         1
size_t eco_mpnn_grad_scratch_bytes(int32_t B, int32_t N);
int    eco_mpnn_grad(const eco_graphs_t* g, const eco_mpnn_t* w, int32_t B, const int32_t* graph_idx_dev,
                     const float* xn_dev, const float* xg_dev, float norm_max, const int32_t* actions_dev,
                     const float* targets_dev, int32_t loss_kind, float* loss_dev, float* grad_dev,
                     void* scratch_dev, void* stream);
/* The same with the targets still being computed on ANOTHER stream: `targets_ready_event` (a cudaEvent_t recorded on that
 * stream after the last write of targets_dev, or NULL) is waited for on `stream` just before the readout -- the forward
 * pass with its saved activations (two thirds of the call) does not depend on the targets, so the Double-DQN target
 * (dqn.py:414-432: two forwards of the next states) overlaps it.  Capturable into a CUDA graph (becomes a graph edge). */
int    eco_mpnn_grad_ev(const eco_graphs_t* g, const eco_mpnn_t* w, int32_t B, const int32_t* graph_idx_dev,
                        const float* xn_dev, const float* xg_dev, float norm_max, const int32_t* actions_dev,
                        const float* targets_dev, int32_t loss_kind, float* loss_dev, float* grad_dev, void* scratch_dev,
                        void* targets_ready_event, void* stream);

/* The optimizer step that follows (reference src/agents/dqn/dqn.py:212 `optim.Adam(...)`, :449 `self.optimizer.step()`):
 * torch.optim.Adam semantics (weight_decay is added to the gradient, bias-corrected moments, no amsgrad) applied IN
 * PLACE to the 12 fp32 tensors `w` points at.  grad_dev as written by eco_mpnn_grad; exp_avg_dev / exp_avg_sq_dev
 * [ECO_MPNN_N_PARAMS] fp32 state (zero before the first step); step = 1, 2, ...  Re-run eco_mpnn_pack afterwards. */
int    eco_mpnn_adam(const eco_mpnn_t* w, const float* grad_dev, float* exp_avg_dev, float* exp_avg_sq_dev, int32_t step,
                     float lr, float beta1, float beta2, float eps, float weight_decay, void* stream);

/* The same step with its state on the device, for updates captured in a CUDA graph: *step_dev (int32, 0 before the first
 * step) is read as "steps done so far" and advanced by one; *lr_dev is the learning rate (the caller rewrites it when the
 * schedule of dqn.py:467-487 moves); the gradient is multiplied by grad_scale first (1 / world after a sum all-reduce). */
int    eco_mpnn_adam_dev(const eco_mpnn_t* w, const float* grad_dev, float* exp_avg_dev, float* exp_avg_sq_dev,
                         int32_t* step_dev, const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                         float grad_scale, void* stream);

/* Data-parallel form of the update (SURVEY.md section 8e; the reference is single-process: src/agents/dqn/dqn.py:403-451
 * runs on one device).  One process per GPU of one NVSwitch box; every rank calls eco_dp_adam once per update with ITS
 * gradient and gets the Adam step of the MEAN gradient applied to its parameters: the kernel publishes the gradient in a
 * buffer shared through CUDA IPC, waits for the peers' (system-scope flags over NVLink), sums all ranks' gradients straight
 * from peer memory in rank order (bit-identical on every rank) and updates -- all-reduce and optimizer in one launch.
 *   eco_dp_create    allocates this rank's exchange region;  eco_dp_handle  its 64-byte IPC handle (exchange them with any
 *   host-side all-gather);  eco_dp_open  maps the peers' regions ([world][64] handle bytes, own entry ignored).
 *   *err_dev (int32, device) becomes non-zero if a peer never arrives (the kernel traps instead of hanging).
 * Every rank must call eco_dp_adam the same number of times; step_dev / lr_dev as for eco_mpnn_adam_dev. */
#define ECO_DP_HANDLE_BYTES 64
typedef struct eco_dp eco_dp_t;
int  eco_dp_create(eco_dp_t** out, int32_t world, int32_t rank);
int  eco_dp_handle(const eco_dp_t* dp, void* handle64_host);
int  eco_dp_open(eco_dp_t* dp, const void* handles_host);
int  eco_dp_adam(eco_dp_t* dp, const eco_mpnn_t* w, const float* grad_dev, float* exp_avg_dev, float* exp_avg_sq_dev,
                 int32_t* step_dev, const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                 int32_t* err_dev, void* stream);
void eco_dp_destroy(eco_dp_t* dp);

/* ---------------------------------------------------------------------------------------------------------
 * Rollout: n_steps x [Q-eval + argmax -> env step] with no host round trip.  Replaces the hot loop of
 * __test_network_batched (reference experiments/utils.py:169-207) and, with ECO_POLICY_GREEDY, the Greedy
 * baseline (experiments/utils.py:218-227).  actions_scratch_dev [B] int32.  With ECO_ENV_IRREVERSIBLE the network
 * policy takes the argmax over the spins still at -1 (eco_env_masked_argmax) and episodes end when none is left.
 * For the plain ECO-DQN configuration on the resident tensor-core kernel (N <= 208, at least two episodes per SM) the whole
 * call is ONE kernel launch (forward + argmax + env step of every step; same results bit for bit); the environment
 * variable ECO_FUSED_STEP=0 selects two launches per step instead.
 * --------------------------------------------------------------------------------------------------------- */
int eco_rollout(const eco_graphs_t* g, eco_env_t* env, const eco_mpnn_t* w, int32_t n_steps, int32_t policy,
                float norm_max, int32_t* actions_scratch_dev, void* mpnn_scratch_dev, int32_t impl,
                int32_t* hist_actions_dev, double* hist_rewards_dev, double* hist_scores_dev, void* stream);

/* Collect per-episode results (async): best cut (int32), best spins [B,N] int8, step count. Any may be NULL. */
int eco_env_results(const eco_env_t* env, int32_t* best_cut_dev, int8_t* best_spins_dev,
                    int32_t* steps_dev, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Host-buffer entry point: the whole `test_network` inner job for one batch with HOST inputs and outputs
 * (what a caller of the reference's test_network holds): uploads graphs + init spins, resets, rolls out T
 * steps with the network policy, downloads best cuts / best spins.  Synchronises `stream` before returning.
 * A session owns the device workspaces so repeated calls do not allocate.
 * --------------------------------------------------------------------------------------------------------- */
typedef struct eco_session eco_session_t;
int  eco_session_create(eco_session_t** out, int32_t G, int32_t N, int32_t B, int32_t T, double basin_reward,
                        const float* const weights_host[12] /* state_dict order, appendix A.3 */, int32_t impl);
void eco_session_destroy(eco_session_t* s);
int  eco_session_rollout(eco_session_t* s, const int8_t* J_host /*[G,N,N]*/, const int32_t* graph_idx_host /*[B]*/,
                         const int8_t* init_spins_host /*[B,N]*/, int32_t policy, float norm_max,
                         int32_t* best_cut_host /*[B]*/, int8_t* best_spins_host /*[B,N] or NULL*/, void* stream);
/* counters for bench.py: kernels launched by this library since the last reset */
int64_t eco_launch_count(int reset);
/* Per-kernel device timing for bench.py's roofline: while enabled with on = k >= 1, every k-th MPNN forward kernel
 * (kind 0) and every k-th env-step kernel (kind 1) is bracketed by CUDA events on its launch stream (an event record
 * between two kernels costs about as much as a small kernel, so bench.py samples).  eco_profile_read synchronises the
 * device and returns the summed duration (ms) and the number of launches recorded since enabling.  Kind 2: the one-launch
 * rollouts of eco_rollout (MPNN forward + argmax + env step of every step inside one kernel): every such launch is
 * recorded and `launches` counts the rollout STEPS it covered, so total / launches is the time per [forward + env step]. */
#define ECO_PROF_MPNN 0
#define ECO_PROF_ENV_STEP 1
#define ECO_PROF_ROLLOUT 2
int eco_profile_enable(int on);
int eco_profile_read(int kind, double* total_ms, int64_t* launches);

/* ---------------------------------------------------------------------------------------------------------
 * Real-valued couplings (EdgeType.RANDOM: 2*rand-1 weights, reference src/envs/utils.py; any non-integer matrix of
 * SingleGraphGenerator / SetGraphGenerator / load_graph_set).  ECO-DQN rollout configuration only (CUT target, BLS
 * reward, reversible spins) plus the Greedy baseline.  Precision follows the reference:
 *   - the environment is fp64 (couplings, local fields, gains, score, normalised score, cut, rewards), as
 *     spinsystem.py computes with its fp64 `matrix`;
 *   - the MPNN reads fp32(J), because the reference's drivers cast the observation with .float()
 *     (experiments/utils.py:174): degree = #{j : fp32(J_ij) != 0}, edge stage and aggregation on fp32 couplings.
 * The tensor-core MPNN kernels stay {-1,0,1}-only: ECO_MPNN_TCGEN05 on a weighted set is ECO_ERR_UNSUPPORTED.
 * --------------------------------------------------------------------------------------------------------- */
#define ECO_WGRAPH_NO_DEGREE   2   /* gstat flag: every weighted degree is zero (the reference recurses forever)       */
#define ECO_WGRAPH_ASYMMETRIC  4   /* gstat flag: not symmetric, or a non-zero diagonal entry                          */
#define ECO_WGRAPH_NONFINITE   8   /* gstat flag: an entry is inf or nan                                               */

typedef struct {
    int32_t  G, N, NP, reserved;   /* reserved: 0 (OptimisationTarget.CUT only)                                        */
    double*  J;          /* [G, NP, NP]  fp64 couplings, zero padded                                               */
    float*   Jf;         /* [G, NP, NP]  fp32(J): what the MPNN reads                                              */
    double*  gscal;      /* [G, 4]       mlr (max non-zero weighted degree), qn, lb, sum_ij J_ij (score_solver.py:353-375) */
    float*   deg;        /* [G, NP]      max(1, #{j : fp32(J_ij) != 0})  (mpnn.py:34-38 on the fp32 observation)    */
    int32_t* gstat;      /* [G, 4]       max degree, nnz, 0, ECO_WGRAPH_* flags                                    */
    float*   dmax;       /* [1]          max degree over the whole set                                             */
} eco_wgraphs_t;

size_t eco_wgraphs_workspace_bytes(int32_t G, int32_t N);
int    eco_wgraphs_bind(eco_wgraphs_t* g, void* workspace_dev, int32_t G, int32_t N);
/* J_dev: dense [G, N, N] fp64 on the device.  Pads, writes the fp32 copy, the degrees, the flags and the scorer constants
 * in fp64 (replaces MaximumCutUnbiasedScorer.set_graph, score_solver.py:353-375, and mpnn.py:34-38). */
int    eco_wgraphs_load_dev(eco_wgraphs_t* g, const double* J_dev, void* stream);

/* Batched environment on a weighted set: the integer state `base` plus the fp64 arrays it cannot hold.  base.hfield and
 * the cut fields of base.ep are unused; every other array of `base` keeps its meaning, so eco_env_set_tables,
 * eco_env_observation, eco_env_best_spins and eco_env_masked_argmax take &base. */
typedef struct {
    eco_env_t base;
    double*   h;         /* [B, NP]  local fields h = J s in fp64                                                  */
    double*   cut;       /* [B, 2]   current cut, best cut (best_solution)                                         */
} eco_wenv_t;

size_t eco_wenv_workspace_bytes(int32_t B, int32_t N, int32_t T);
int    eco_wenv_bind(eco_wenv_t* env, void* workspace_dev, int32_t B, int32_t N, int32_t T, double basin_reward);
/* reset(spins): reference spinsystem.py:183-259 / 283-330, arguments as eco_env_reset */
int    eco_wenv_reset(const eco_wgraphs_t* g, eco_wenv_t* env, const int32_t* graph_idx_dev, const int8_t* init_spins_dev,
                      void* stream);
/* step: reference spinsystem.py:355-559 (ECO_POLICY_ACTIONS) or solver.py:105-131 (ECO_POLICY_GREEDY, key s_i h_i in
 * fp64, stop when the best gain is < 0); arguments and history arrays as eco_env_step */
int    eco_wenv_step(const eco_wgraphs_t* g, eco_wenv_t* env, int32_t policy, const int32_t* actions_dev, double* reward_dev,
                     uint8_t* done_dev, int32_t* hist_actions_dev, double* hist_rewards_dev, double* hist_scores_dev,
                     void* stream);
/* MPNN.forward (mpnn.py:40-159) on fp32(J) + argmax; arguments and norm_max modes as eco_mpnn_forward.  impl: AUTO or SIMT. */
int    eco_wmpnn_forward(const eco_wgraphs_t* g, const eco_mpnn_t* w, int32_t B, const int32_t* graph_idx_dev,
                         const float* xn_dev, const float* xg_dev, float norm_max, float* q_dev, int32_t* actions_dev,
                         void* scratch_dev, int32_t impl, void* stream);
/* rollout: experiments/utils.py:169-207 (ECO_POLICY_NETWORK) or :218-227 (ECO_POLICY_GREEDY); arguments as eco_rollout,
 * scratch sized by eco_mpnn_scratch_bytes(B, N, ECO_MPNN_SIMT) */
int    eco_wrollout(const eco_wgraphs_t* g, eco_wenv_t* env, const eco_mpnn_t* w, int32_t n_steps, int32_t policy,
                    float norm_max, int32_t* actions_scratch_dev, void* mpnn_scratch_dev, int32_t impl,
                    int32_t* hist_actions_dev, double* hist_rewards_dev, double* hist_scores_dev, void* stream);
/* best cut (fp64), best spins [B, N] int8, step count.  Any may be NULL. */
int    eco_wenv_results(const eco_wenv_t* env, double* best_cut_dev, int8_t* best_spins_dev, int32_t* steps_dev,
                        void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Sparse graph sets: G graphs of up to ECO_MAX_SPINS_SPARSE vertices stored as CSR, integer couplings in [-127, 127] -- the
 * GSet instances (G55: 5000 vertices, G70 / G72: 10 000, G81: 20 000) that the dense N x N layout cannot hold.  ECO-DQN
 * rollout configuration (CUT target, BLS and basin reward, reversible spins, Stopping.NORMAL) plus the Greedy baseline.
 * The environment is a plain eco_env_t (same layout and integer / fp64 rules as the int8 path), so eco_env_set_tables,
 * eco_env_observation, eco_env_best_spins and eco_env_results take it unchanged; for N <= ECO_MAX_SPINS every state array
 * equals the dense path's bit for bit.  The step costs O(degree) plus one O(N) feature row (time since flip); the MPNN
 * aggregates by gathering neighbour rows.  N is bounded by the uint16 last-flip steps with max_steps <= 65535 (the
 * reference's test scripts run 2N steps).  MIN_CUT and the S2V-DQN env modes are ECO_ERR_UNSUPPORTED.
 * --------------------------------------------------------------------------------------------------------- */
#define ECO_MAX_SPINS_SPARSE     32768
#define ECO_SGRAPH_FIELD_RANGE   8    /* gstat flag: a row's sum of |couplings| exceeds 32767 (the int16 local fields)       */
#define ECO_SGRAPH_NONCANONICAL  16   /* gstat flag: a row pointer, column or stored value breaks the CSR rules below        */

typedef struct {
    int32_t  G, N, NP, reserved;   /* reserved: ECO_GRAPHS_PM1 as for eco_graphs_t (informational); ECO_GRAPHS_MIN_CUT is not
                                      supported                                                                             */
    int64_t  nnz;        /* stored entries of all graphs                                                                */
    int64_t* row_ptr;    /* [G*N + 1]    global offsets: row i of graph g is entries row_ptr[g*N + i] .. row_ptr[g*N + i + 1] - 1 */
    int32_t* col;        /* [nnz]        column, strictly ascending within a row (every sum over a row has one fixed order)  */
    int8_t*  val;        /* [nnz]        coupling, non-zero; both directions of every edge are stored                       */
    double*  gscal;      /* [G, 4]       mlr, qn, lb, sum_ij J_ij (as eco_graphs_t)                                         */
    float*   deg;        /* [G, NP]      max(1, non-zeros of row i)                                                         */
    int32_t* gstat;      /* [G, 4]       max degree, nnz, max row sum of |J|, flags (eco_graphs_t meanings:
                                         bit0 weights outside {-1,0,1}, bit1 all weighted degrees zero, bit2 not symmetric /
                                         non-zero diagonal; plus ECO_SGRAPH_FIELD_RANGE, ECO_SGRAPH_NONCANONICAL)         */
    float*   dmax;       /* [1]          max degree over the whole set                                                      */
} eco_sgraphs_t;

size_t eco_sgraphs_workspace_bytes(int32_t G, int32_t N, int64_t nnz);
int    eco_sgraphs_bind(eco_sgraphs_t* g, void* workspace_dev, int32_t G, int32_t N, int64_t nnz);
/* canonical CSR already on the device (row_ptr_dev [G*N + 1] int64 with row_ptr_dev[0] = 0 and row_ptr_dev[G*N] = nnz,
 * col_dev [nnz] int32, val_dev [nnz] int8): copied into the workspace (async), then the constants and flags are computed */
int    eco_sgraphs_load_dev(eco_sgraphs_t* g, const int64_t* row_ptr_dev, const int32_t* col_dev, const int8_t* val_dev,
                            void* stream);

/* an eco_env_t for 1 <= N <= ECO_MAX_SPINS_SPARSE (eco_env_workspace_bytes / eco_env_bind with the sparse size limit) */
size_t eco_senv_workspace_bytes(int32_t B, int32_t N, int32_t T);
int    eco_senv_bind(eco_env_t* env, void* workspace_dev, int32_t B, int32_t N, int32_t T, double basin_reward);
/* reset / step: arguments, policies (ECO_POLICY_ACTIONS, ECO_POLICY_GREEDY) and history arrays as eco_env_reset / eco_env_step */
int    eco_senv_reset(const eco_sgraphs_t* g, eco_env_t* env, const int32_t* graph_idx_dev, const int8_t* init_spins_dev,
                      void* stream);
int    eco_senv_step(const eco_sgraphs_t* g, eco_env_t* env, int32_t policy, const int32_t* actions_dev, double* reward_dev,
                     uint8_t* done_dev, int32_t* hist_actions_dev, double* hist_rewards_dev, double* hist_scores_dev,
                     void* stream);
/* MPNN.forward (mpnn.py:40-159) + argmax on fp32 CUDA cores; arguments and norm_max modes as eco_mpnn_forward.
 * scratch_dev >= eco_smpnn_scratch_bytes(B, N), 16-byte aligned. */
size_t eco_smpnn_scratch_bytes(int32_t B, int32_t N);
int    eco_smpnn_forward(const eco_sgraphs_t* g, const eco_mpnn_t* w, int32_t B, const int32_t* graph_idx_dev,
                         const float* xn_dev, const float* xg_dev, float norm_max, float* q_dev, int32_t* actions_dev,
                         void* scratch_dev, void* stream);
/* rollout: ECO_POLICY_NETWORK (n_steps x [forward + argmax -> step]) or ECO_POLICY_GREEDY; arguments as eco_rollout,
 * mpnn_scratch_dev sized by eco_smpnn_scratch_bytes */
int    eco_srollout(const eco_sgraphs_t* g, eco_env_t* env, const eco_mpnn_t* w, int32_t n_steps, int32_t policy,
                    float norm_max, int32_t* actions_scratch_dev, void* mpnn_scratch_dev, int32_t* hist_actions_dev,
                    double* hist_rewards_dev, double* hist_scores_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ECODQN_B200_H */
