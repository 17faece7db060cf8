/*
 * corollout.h -- C ABI of libcorollout.so, the B200 (sm_100a) rollout engine behind
 * rl4co's env / decoder API.
 *
 * The reference (ai4co/rl4co) is 100% Python and has no FFI on this path; its only FFI
 * precedent is ctypes -> libhgscvrp.so (rl4co/envs/routing/cvrp/local_search.py:8-24).
 * Each entry point below replaces the reference function(s) cited next to it; the
 * Python-side ctypes binding a maintainer would add is shown in INTEGRATION.md and
 * implemented in rl4co_b200/native.py.
 *
 * Conventions (SURVEY.md section 8b)
 *   - every pointer is a DEVICE pointer into memory owned by the caller (PyTorch);
 *     the library never allocates, frees or retains device memory;
 *   - tensors are contiguous row-major with exactly the reference TensorDict dtypes:
 *     int64 actions / node ids, 1-byte bool masks, uint8 visited, float32 the rest;
 *   - all work is enqueued asynchronously on `stream` (a cudaStream_t passed as void*);
 *     no call synchronises the device;
 *   - return value: CO_OK (0) or a negative CO_ERR_*; co_last_error_string() describes
 *     the last failure on the calling thread.  No C++ exception crosses the boundary.
 *   - embed_dim E = 128, heads H = 8 (head dim 16) are compile-time constants of the
 *     AttentionModel this path serves (rl4co/models/zoo/am/policy.py:50-56).
 */
#ifndef COROLLOUT_H_
#define COROLLOUT_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CO_VERSION 100 /* 0.1.0 */

#define CO_OK 0
#define CO_ERR_BAD_ARG (-1)
#define CO_ERR_UNSUPPORTED (-2) /* shape outside what a kernel is instantiated for */
#define CO_ERR_CUDA (-3)        /* launch / runtime error; see co_last_error_string */

#define CO_EMBED_DIM 128
#define CO_NUM_HEADS 8

/* environment kinds (env.name in the reference: "tsp", "cvrp") */
#define CO_ENV_TSP 0
#define CO_ENV_CVRP 1
#define CO_ENV_SDVRP 2 /* split-delivery VRP: VRP context + dynamic embedding */
#define CO_ENV_OP 3    /* orienteering: budget context, length mask, prize reward (co_rollout; the step kernels are co_op_*) */
#define CO_ENV_PCTSP 4 /* prize-collecting TSP: remaining-prize context, depot rule on the collected prize (co_pctsp_*) */

/* action-selection modes (rl4co/utils/decoding.py:426-461) */
#define CO_SELECT_GREEDY 0       /* Greedy._step: argmax, first index on ties            */
#define CO_SELECT_SAMPLE_NOISE 1 /* Sampling._step with caller-supplied Exp(1) draws q:    */
                                 /*   argmax(exp(logp)/q) == torch.multinomial(p,1)        */
#define CO_SELECT_EVALUATE 2     /* Evaluate._step: action supplied, only logp computed    */
#define CO_SELECT_SAMPLE_PHILOX 3/* Sampling with in-kernel Philox4x32-10 Exp(1) draws     */

int co_version(void);
const char* co_last_error_string(void);
/* number of SMs / max dyn smem of the current device (cached); used to size grids */
int co_device_sm_count(void);

/* ------------------------------------------------------------------ environments */

/* TSPEnv._step  (rl4co/envs/routing/tsp/env.py:60-86)
 *   mask_out = mask_in with column action[b] cleared; done = no column left;
 *   first_node = action where i[b]==0 else kept; current_node = action; i += 1.
 * mask_in may alias mask_out (in-place step). */
int co_tsp_step(const int64_t* action, const uint8_t* mask_in, uint8_t* mask_out,
                int64_t* first_node, int64_t* current_node, int64_t* i, uint8_t* done,
                int B, int N, void* stream);

/* CVRPEnv.get_action_mask  (rl4co/envs/routing/cvrp/env.py:126-136)
 *   N counts the depot (node 0); demand is [B, N-1]; mask_out[b,n]=1 means feasible. */
int co_cvrp_action_mask(const float* demand, const float* used_capacity,
                        const float* vehicle_capacity, const uint8_t* visited,
                        const int64_t* current_node, uint8_t* mask_out, int B, int N,
                        void* stream);

/* CVRPEnv._step  (rl4co/envs/routing/cvrp/env.py:66-96), including the trailing
 * get_action_mask.  visited_in may alias visited_out, used_in may alias used_out. */
int co_cvrp_step(const int64_t* action, const float* demand, const float* vehicle_capacity,
                 const float* used_in, float* used_out, const uint8_t* visited_in,
                 uint8_t* visited_out, int64_t* current_node, uint8_t* done,
                 uint8_t* mask_out, int B, int N, void* stream);

/* TSPEnv._get_reward / CVRPEnv._get_reward
 * (tsp/env.py:150-156, cvrp/env.py:138-147 -> rl4co/utils/ops.py:54-90)
 *   reward[b] = - sum_t || x[a_{t+1}] - x[a_t] ||_2 over the cyclic tour; with_depot=1
 *   prepends node 0 (CVRP).  locs [B_locs,N,2]; actions [B,T]; trajectory j uses
 *   instance j % B_locs (multistart / augmentation share locs). */
/* SDVRPEnv (rl4co/envs/routing/sdvrp/env.py): `demand_with_depot` [B,N] f32 is the dynamic state (depot entry 0).
 * co_sdvrp_step = _step :55-82 (deliver min(demand, capacity - used), scatter_add, done) + get_action_mask :110-116;
 * outputs may alias inputs (in-place update). */
int co_sdvrp_action_mask(const float* demand_with_depot, const float* used_capacity,
                         const float* vehicle_capacity, const int64_t* current_node, uint8_t* mask_out,
                         int B, int N, void* stream);
int co_sdvrp_step(const int64_t* action, const float* demand_in, float* demand_out,
                  const float* vehicle_capacity, const float* used_in, float* used_out,
                  int64_t* current_node, uint8_t* done, uint8_t* mask_out, int B, int N, void* stream);

/* OPEnv (rl4co/envs/routing/op/env.py; sibling env, orienteering): locs [B,N,2] with the depot at 0, prize [B,N] (depot 0),
 * max_length [B,N] (per node: the budget minus the way back to the depot, env.py:121-123), visited [B,N] bool,
 * tour_length / current_total_prize [B] f32, current_node / i [B] i64 (updated in place by co_op_step).
 * co_op_step = _step :72-105 + get_action_mask :140-155 (done = depot re-entered after step 0);
 * co_op_reward = _get_reward :157-165 (sum of the collected prizes over actions [B,T]). */
int co_op_action_mask(const float* locs, const float* max_length, const uint8_t* visited, const float* tour_length,
                      const int64_t* current_node, uint8_t* mask_out, int B, int N, void* stream);
int co_op_step(const int64_t* action, const float* locs, const float* prize, const float* max_length,
               const uint8_t* visited_in, uint8_t* visited_out, float* tour_length, float* current_total_prize,
               int64_t* current_node, int64_t* i, uint8_t* done, uint8_t* mask_out, int B, int N, void* stream);
int co_op_reward(const float* prize, const int64_t* actions, float* reward, int B, int N, int T, void* stream);

/* PCTSPEnv (rl4co/envs/routing/pctsp/env.py; sibling env, prize-collecting TSP): real_prize / penalty [B,N] (depot 0),
 * visited [B,N] bool, cur_total_prize / cur_total_penalty [B] f32, current_node / i [B] i64 (in place).
 * co_pctsp_step = _step :62-93 + get_action_mask :143-151; the reward (:153-172) is co_op_reward over the penalties plus
 * co_tour_length. */
int co_pctsp_action_mask(const uint8_t* visited, const float* cur_total_prize, uint8_t* mask_out, int B, int N, void* stream);
int co_pctsp_step(const int64_t* action, const float* real_prize, const float* penalty, const uint8_t* visited_in,
                  uint8_t* visited_out, float* cur_total_prize, float* cur_total_penalty, int64_t* current_node, int64_t* i,
                  uint8_t* done, uint8_t* mask_out, int B, int N, void* stream);

int co_tour_length(const float* locs, const int64_t* actions, float* reward, int B,
                   int B_locs, int N, int T, int with_depot, void* stream);

/* TSPEnv.check_solution_validity / CVRPEnv.check_solution_validity
 * (tsp/env.py:158-164, cvrp/env.py:149-177).  *bad_count (device int32, caller-zeroed)
 * receives the number of invalid tours; demand==NULL selects the TSP rule. */
int co_check_tours(const int64_t* actions, const float* demand,
                   const float* vehicle_capacity, int32_t* bad_count, int B, int B_inst,
                   int N, int T, void* stream);

/* TSPEnv.local_search (rl4co/envs/routing/tsp/env.py:184-188 -> tsp/local_search.py:16-81): 2-opt on each tour,
 * best improvement per scan, bit for bit the reference's result.  locs [B,N,2] f32, tours_in / tours_out [B,N] int64
 * (may alias; the input is read whole before a row is written), moves_out [B] int32 or NULL: moves applied per row,
 * at most max_iterations (0 leaves every row unchanged).  A row holding a node index outside [0, N) is copied
 * unchanged and gets moves_out = -1.  No N x N matrix: shared memory per CTA is 16 * N bytes. */
#define CO_TWO_OPT_MAX_NODES 1024
int co_tsp_two_opt(const float* locs, const int64_t* tours_in, int64_t* tours_out, int32_t* moves_out,
                   int B, int N, int max_iterations, void* stream);

/* ------------------------------------------------------------------ decoder, one step */

/* Weights of the decoder path, device pointers, all float32, no biases
 * (rl4co/models/zoo/am/policy.py:65,70).  *_t tensors are TRANSPOSED copies
 * ([in, out] row-major) prepared once per weight update by the host side. */
typedef struct co_decoder_weights {
  const float* project_context_t; /* [ctx_dim, E]; ctx_dim = 2E (tsp) or E+1 (cvrp)   */
  const float* w_placeholder;     /* [2E] (tsp only, else NULL)                       */
  const float* project_out_t;     /* [E, E] transposed pointer.project_out.weight, or  */
                                  /* NULL when logit_key is pre-multiplied by it       */
  /* dynamic embedding (sdvrp: SDVRPDynamicEmbedding, nn/env_embeddings/dynamic.py:60-78; am/decoder.py:142-154):
   * glimpse_key / glimpse_val / logit_key of node n get + dynamic_feature[j, n] * dynamic_w[0:E | E:2E | 2E:3E].
   * Both NULL for static embeddings (tsp, cvrp). */
  const float* dynamic_w;         /* [3E] = projection.weight[:, 0]; the logit third folded with project_out   */
                                  /* (W_out^T w_l) when project_out_t == NULL                                   */
  const float* dynamic_feature;   /* [B_traj, N] per-step node feature (sdvrp: remaining demand, depot = 0)     */
} co_decoder_weights;

/* AttentionModelDecoder.forward (rl4co/models/zoo/am/decoder.py:156-193):
 * context embedding (nn/env_embeddings/context.py:116-134 | 61-74,147-149) + graph
 * context, PointerAttention (nn/attention.py:274-320) -> raw logits [B_traj, N]
 * (unmasked, unclipped, already in the reference's "(s b) l" order).
 * Trajectory j reads the cache of instance j % B_inst (multistart shares K/V/L).
 *   tsp : first_node, current_node [B_traj] int64, i [B_traj] int64 (i==0 -> placeholder)
 *   cvrp: current_node [B_traj] int64, used_capacity / vehicle_capacity [B_traj] f32
 * glimpse_key / glimpse_val / logit_key rows are `ld` floats apart (ld = E for the
 * reference's contiguous tensors, or the fused-cache row width for views into it; 0 = E).
 * w->project_out_t == NULL means logit_key already holds the folded rows
 * logit_key @ project_out.weight (block 2 of the rollout cache) and the projection is skipped. */
int co_pointer_logits(int env_kind, const co_decoder_weights* w, const float* node_emb,
                      const float* graph_ctx /* [B_inst,E] or NULL */,
                      const float* glimpse_key, const float* glimpse_val,
                      const float* logit_key, const uint8_t* action_mask,
                      const int64_t* first_node, const int64_t* current_node,
                      const int64_t* i, const float* used_capacity,
                      const float* vehicle_capacity, float* logits_out, int B_traj,
                      int B_inst, int N, int ld, void* stream);

/* DecodingStrategy.step (rl4co/utils/decoding.py:344-385): process_logits (:138-188:
 * tanh clip, mask -> -inf, temperature, log_softmax; top-k/top-p unsupported) then
 * Greedy / Sampling / Evaluate selection and logp gather.
 *   noise        : [B,N] Exp(1) draws for CO_SELECT_SAMPLE_NOISE, else NULL
 *   action_io    : [B] int64; read for CO_SELECT_EVALUATE, written otherwise
 *   logprobs_out : optional [B,N] full log-probabilities (store_all_logp), or NULL */
int co_select_action(const float* logits, const uint8_t* action_mask, const float* noise,
                     int64_t* action_io, float* logp_out, float* logprobs_out, int mode,
                     float tanh_clipping, float temperature, int mask_logits,
                     uint64_t seed, uint64_t offset, int B, int N, void* stream);

/* ------------------------------------------------------------------ whole-episode rollout */

/* Persistent fused rollout: replaces the whole `while not td["done"].all()` loop of
 * ConstructivePolicy.forward (rl4co/models/common/constructive/base.py:219-251):
 * decoder.forward + strategy.step + env.step per node selection, then
 * post_decoder_hook / get_reward / get_log_likelihood, in ONE kernel launch with no host
 * synchronisation.  One CTA owns one instance for the whole episode: its glimpse-key /
 * glimpse-value / folded logit-key rows live in registers, the per-node context table in
 * shared memory; the visited set is a bitmask in registers.
 *
 * The cache is the layout written by FusedAttentionModelDecoder._precompute_cache:
 *   cache[B_inst][N][co_cache_width(env_kind)] float32, column blocks of E floats:
 *     0: glimpse_key   1: glimpse_val   2: logit_key @ project_out (folded)
 *     3: node_emb @ Wctx[:, :E]^T  (tsp: "first node" table; cvrp: current-node table)
 *     4: node_emb @ Wctx[:, E:2E]^T (tsp only: current-node table)
 */
#define CO_ROLLOUT_FORCED_START 1 /* S>1: first action of start s is forced (multistart) */
#define CO_ROLLOUT_NO_PREFETCH 2  /* diagnostic: do not prefetch the next instance's cache rows into L2 */

typedef struct co_rollout_args {
  int32_t env_kind;     /* CO_ENV_*                                                    */
  int32_t select_mode;  /* CO_SELECT_*                                                 */
  int32_t B_inst;       /* instances (cache rows)                                      */
  int32_t num_starts;   /* S >= 1 trajectories per instance; S > 1 = multistart with   */
                        /* forced first action s % num_loc (+1 for cvrp), ops.py:128-149 */
  int32_t N;            /* nodes incl. depot                                           */
  int32_t T_max;        /* columns of actions_out / logp_out (tsp: N, cvrp: 2(N-1))     */
  int32_t num_loc;      /* generator.num_loc used by select_start_nodes                */
  int32_t flags;        /* CO_ROLLOUT_* bits                                           */
  float tanh_clipping;  /* 10.0 for AM                                                 */
  float temperature;    /* 1.0                                                         */
  const float* cache;        /* [B_inst, N, W]                                         */
  const float* graph_ctx;    /* [B_inst, E] or NULL (POMO: use_graph_context=False)    */
  const float* q_placeholder;/* [E] = Wctx @ W_placeholder (tsp step-0 context)        */
  const float* w_capacity;   /* [E] = Wctx[:, E] (cvrp remaining-capacity column)      */
  const float* locs;         /* [B_inst, N, 2]                                         */
  const float* demand;       /* [B_inst, N-1] (cvrp) or NULL                           */
  const float* vehicle_capacity; /* [B_inst] (cvrp) or NULL (=1.0)                     */
  const int64_t* forced_actions; /* [B_traj, T_max] for CO_SELECT_EVALUATE else NULL   */
  const float* noise;        /* [T_max, B_traj, N] Exp(1) for CO_SELECT_SAMPLE_NOISE   */
  uint64_t seed, offset;     /* Philox stream for CO_SELECT_SAMPLE_PHILOX              */
  int64_t* actions_out;      /* [B_traj, T_max]; B_traj = S * B_inst, row j = s*B + b  */
  float* logp_out;           /* [B_traj, T_max] per-step log-prob of the chosen action */
  float* reward_out;         /* [B_traj]  = -tour length                               */
  float* loglik_out;         /* [B_traj]  = sum_t logp                                 */
  int32_t* steps_out;        /* [B_traj]  decode steps until done (incl. forced start) */
  int32_t* max_steps_out;    /* [1] device int32, caller-zeroed: max over trajectories */
  float* used_capacity_out;  /* [B_traj] final used capacity (cvrp) or NULL            */
  /* round 2: narrow tsp cache (no first-node table) -- the first-node half of project_context
   * (context.py:129-133) becomes one 128x128 GEMV per episode inside the kernel            */
  const float* node_emb;     /* [B_inst, N, E] encoder output; tsp with cache_width 4E  */
  const float* w_first;      /* [E, E] = project_context.weight[:, :E] row-major; same   */
  int32_t cache_width;       /* floats per row of `cache`: 4E, or 5E = tsp layout with   */
                             /* the first-node table; 0 = co_cache_width(env_kind)       */
  int32_t reserved0;
  /* sdvrp: dynamic-embedding weights [wk | wv | W_out^T wl] = SDVRPDynamicEmbedding.projection.weight[:, 0] with
   * the logit third folded like block 2 of the cache (nn/env_embeddings/dynamic.py:60-78); NULL otherwise */
  const float* dyn_w;        /* [3E] */
  /* op: per-node length budget max_length [B_inst, N] (op/env.py:121-123); `demand` carries the customers' prizes
   * [B_inst, N-1], `vehicle_capacity` the budget at the depot max_length[:, 0], reward_out the collected prize;
   * pctsp: penalty per node [B_inst, N] (depot 0); `demand` = real prizes [B_inst, N-1], `vehicle_capacity` = prize_required */
  const float* node_limit;
} co_rollout_args;

int co_cache_width(int env_kind); /* floats per node row of the widest rollout cache layout (tsp 5E, cvrp 4E) */
/* largest N the persistent kernel is instantiated for (else CO_ERR_UNSUPPORTED) */
int co_rollout_max_nodes(void);
int co_rollout(const co_rollout_args* args, void* stream);

/* ------------------------------------------------------------------ dense projections
 *
 * fp32-accurate GEMM on tcgen05 tensor cores (kind::tf32, 3xTF32 hi/lo split, fp32 TMEM
 * accumulators):  C[M,Nout] = epilogue(A[M,K] @ W[Nout,K]^T),
 *   epilogue(v) = relu?((v + bias[n]) + residual[m,n]) * scale[n] + shift[n]   (each optional)
 * Replaces the nn.Linear calls of AttentionModelDecoder._precompute_cache
 * (rl4co/models/zoo/am/decoder.py:201-228) and of the AM encoder (nn/attention.py:110-134,
 * nn/mlp.py:45-60; skip connection nn/ops.py:9-15 and eval-mode BatchNorm nn/ops.py:30-46 fold
 * into residual / scale / shift).  W is passed pre-split (co_split_tf32): Whi = rna_tf32(W),
 * Wlo = W - Whi.  Requirements: K % 32 == 0, Nout % 4 == 0, row strides (lda, ldc, ldr, in
 * floats) % 4 == 0, 16-byte aligned pointers. */
int co_split_tf32(const float* w, float* hi, float* lo, long n, void* stream);
int co_gemm_tf32x3(const float* A, const float* Whi, const float* Wlo, float* C,
                   const float* bias, const float* residual, const float* scale,
                   const float* shift, int M, int Nout, int K, int lda, int ldc, int ldr,
                   int relu, void* stream);

/* Encoder feed-forward block in ONE kernel (the [M, 512] hidden activation never leaves the SM):
 *   out = ((x + relu(x W1^T + b1) W2^T + b2)) * scale + shift,  x [M,128], W1 [512,128], W2 [128,512]
 * = SkipConnection(MLP) + eval-mode BatchNorm of MultiHeadAttentionLayer (rl4co/models/nn/graph/attnnet.py:
 * 33-53, nn/mlp.py:45-60, nn/ops.py:9-15,30-46).  The weights are streamed by TMA bulk copies with cluster
 * multicast from a pre-tiled image: co_ffn_tile_weights builds it (once per weight version) from the co_split_tf32
 * parts of W1 and W2 into `wtiled` (co_ffn_tiled_weight_floats() floats, 128-byte aligned).
 * scale / shift NULL (both) for no affine; ldx / ldo row strides in floats (% 4 == 0); 16-byte aligned pointers. */
long co_ffn_tiled_weight_floats(void);
int co_ffn_tile_weights(const float* w1hi, const float* w1lo, const float* w2hi, const float* w2lo, float* wtiled,
                        void* stream);
int co_ffn_fused(const float* x, const float* wtiled, const float* b1, const float* b2, const float* scale,
                 const float* shift, float* out, int M, int ldx, int ldo, void* stream);

/* ------------------------------------------------------------------ data path (SURVEY.md 8f-3)
 * On-device instance generation (Philox4x32-10 keyed by seed / offset; same seed -> same data on every GPU) and
 * the dihedral-8 augmentation as streaming kernels.
 *   co_generate_uniform: out[i] = U[0,1) * (hi - lo) + lo           (envs/common/utils.py:61-62 "uniform")
 *   co_generate_demand : out[i] = (int(U * (max-min) + (min-1)) + 1) / capacity   (cvrp/generator.py:126-137)
 *   co_dihedral8       : out[a*B + b] = a-th image of locs[b], a = 0..7            (data/transforms.py:16-38) */
int co_generate_uniform(float* out, long n, uint64_t seed, uint64_t offset, float lo, float hi, void* stream);
int co_generate_demand(float* out, long n, uint64_t seed, uint64_t offset, int min_demand, int max_demand,
                       float capacity, void* stream);
int co_dihedral8(const float* locs, float* out, long B, int N, void* stream);

/* Encoder self-attention core: F.scaled_dot_product_attention of MultiHeadAttention
 * (rl4co/models/nn/attention.py:110-134) on the packed projection qkv [B*N, 3E] ("three h d"),
 * 8 heads x 16, no mask, fp32 -> out [B*N, E] ("h d"); N <= 128. */
int co_encoder_mha(const float* qkv, float* out, int B, int N, void* stream);

/* ------------------------------------------------------------------ training step: differentiable attention core
 * (SURVEY.md 8f-2).  o = softmax(q k^T / sqrt(16) [masked]) v per head, 8 heads x 16 channels, fp32; forward saves the
 * per-row log-sum-exp (log2 units of the scaled scores), backward recomputes the probabilities -- no [M, N] tensor in
 * memory.  Replaces F.scaled_dot_product_attention under autograd in the AM encoder
 * (rl4co/models/nn/attention.py:110-134) and in the glimpse of the teacher-forced log-likelihood pass
 * (nn/attention.py:300-314 with the T decode steps of an instance as T queries; utils/decoding.py:448-461).
 * All tensors are [B, rows, 128] with the head slice h at column 16 h, last dimension contiguous; row / batch strides
 * (in floats, multiples of 4) are free, so column views of the fused cache or of a packed qkv projection need no
 * copy.  mask: [B, M, 4] uint32, bit n % 32 of word n / 32 set = key n may be attended (NULL = no mask); a fully
 * masked row yields o = 0.  N <= 128 keys, M <= 256 queries per call. */
typedef struct co_attn_args {
  const float* q;        /* [B, M, E] */
  const float* k;        /* [B, N, E] */
  const float* v;        /* [B, N, E] */
  const uint32_t* mask;  /* [B, M, 4] or NULL */
  float* o;              /* [B, M, E]   (forward: out; backward: in) */
  float* lse;            /* [B, 8, M]   (forward: out; backward: in) */
  const float* dO;       /* [B, M, E], strides of o; backward only */
  float* dq;             /* [B, M, E] backward out */
  float* dk;             /* [B, N, E] backward out */
  float* dv;             /* [B, N, E] backward out */
  int32_t B, M, N, reserved0;
  int64_t q_bs, k_bs, v_bs, o_bs, dq_bs, dk_bs, dv_bs; /* batch strides (floats) */
  int32_t q_rs, k_rs, v_rs, o_rs, dq_rs, dk_rs, dv_rs; /* row strides (floats)   */
  float scale;                                         /* 1 / sqrt(head_dim) = 0.25 */
} co_attn_args;
int co_attn_fwd(const co_attn_args* args, void* stream);
int co_attn_bwd(const co_attn_args* args, void* stream);

/* Instance normalisation of the encoder (nn.InstanceNorm1d(E, affine=True) on x.permute(0,2,1),
 * rl4co/models/nn/ops.py:30-54; POMO's `normalization="instance"`): per (instance, channel) mean / biased variance over
 * the N nodes, y = (x - mean) / sqrt(var + eps) * gamma + beta.  x, out [B, N, 128] contiguous (out may alias x);
 * gamma / beta [128] or NULL. */
int co_instance_norm(const float* x, const float* gamma, const float* beta, float* out, long B, int N, float eps,
                     void* stream);

/* REINFORCE baseline statistics (rl4co/models/rl/reinforce/baselines.py:75-81):
 * out[0] += sum(reward), out[1] += count, in float64 so the cross-rank sum is
 * order-independent enough to reproduce the single-process mean. */
int co_reward_stats(const float* reward, double* out2, int B, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* COROLLOUT_H_ */
