/* libpqn_b200.so — C ABI of the B200-native PQN rollout-and-update hot path.
 *
 * The reference (mttga/purejaxql) has no FFI boundary of its own: its hot path
 * is traced Python/JAX.  The entry points below are what a binding for that
 * path would call; each cites the reference interface it replaces
 * (paths relative to the reference repo).  INTEGRATION.md shows the
 * reference-side ctypes stub.
 *
 * Conventions
 *  - plain C, no torch types; every pointer is a DEVICE pointer unless the
 *    name ends in _host; the caller owns every buffer; the library allocates
 *    nothing.
 *  - every call enqueues work on `stream` (a cudaStream_t passed as void*) and
 *    returns immediately: 0 = PQN_OK, negative = PQN_E_*; pqn_last_error()
 *    returns a thread-local message for the last failure.
 *  - `rng_mode`: 0 = jax "original" threefry counter layout (default of the
 *    reference's pinned jax<=0.4.38), 1 = jax_threefry_partitionable=True.
 *  - env state is an opaque word-major SoA block: uint32 state[words][N]
 *    (pqn_env_info gives `state_words`; layout documented in DESIGN.md and
 *    mirrored by purejaxql_b200/envs.py for import/export to gymnax fields).
 *  - batched over N = num_seeds * num_envs flat environments; seed s owns
 *    envs [s*num_envs, (s+1)*num_envs).
 */
#ifndef PQN_B200_H
#define PQN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PQN_OK 0
#define PQN_E_INVALID (-1)   /* bad argument (unknown env id, null pointer, bad size) */
#define PQN_E_CUDA (-2)      /* a CUDA runtime / launch error; see pqn_last_error() */
#define PQN_E_UNSUPPORTED (-3)

/* env ids (gymnax registry names in comments) */
#define PQN_ENV_BREAKOUT 0        /* "Breakout-MinAtar" */
#define PQN_ENV_ASTERIX 1         /* "Asterix-MinAtar" */
#define PQN_ENV_SPACE_INVADERS 2  /* "SpaceInvaders-MinAtar" */
#define PQN_ENV_FREEWAY 3         /* "Freeway-MinAtar" */
#define PQN_ENV_SEAQUEST 4        /* "Seaquest-MinAtar" */
#define PQN_ENV_CARTPOLE 16       /* "CartPole-v1" */
#define PQN_ENV_ACROBOT 17        /* "Acrobot-v1" */
#define PQN_ENV_MEMORY_CHAIN 32   /* "MemoryChain-bsuite" (num_bits = 1) */

typedef struct pqn_env_info_t {
  int32_t state_words;      /* uint32 words per env in the SoA state block (incl. 5 LogWrapper words) */
  int32_t obs_dim;          /* flattened observation length (400 for Breakout, 4 CartPole, 6 Acrobot, 3 MemoryChain) */
  int32_t obs_shape[3];     /* (H, W, C) for MinAtar, (D, 1, 1) for classic control */
  int32_t num_actions;      /* env.action_space(params).n  — pqn_minatar.py:151 */
  int32_t max_steps;        /* env_params.max_steps_in_episode default — pqn_minatar.py:105 */
  int32_t binary_obs;       /* 1: obs are {0,1}; the rollout buffer stores them bit-packed */
  int32_t packed_obs_words; /* uint32 words per packed obs row (64-byte multiple), 0 if !binary_obs */
} pqn_env_info_t;

const char* pqn_last_error(void);
int pqn_version(void);

/* ---- launch accounting (bench.py: gpu_launches, per-kernel roofline) -------
 * pqn_launch_count: kernels launched by this library since load.
 * pqn_profile_enable(1): bracket every kernel launch with CUDA events on the
 * launching stream; pqn_profile_read sums elapsed ms / launch counts per kernel
 * id (arrays of pqn_num_kernels() entries on the host) and optionally resets. */
long long pqn_launch_count(void);
int pqn_num_kernels(void);
const char* pqn_kernel_name(int id);
int pqn_profile_enable(int on);
int pqn_profile_read(double* ms_host, long long* count_host, int reset);

/* gymnax.make(name) metadata — pqn_minatar.py:103-105,151,157. */
int pqn_env_info(int env_id, pqn_env_info_t* out_host);

/* ---- jax.random plumbing on device ------------------------------------- */
/* out[n][num][2] = jax.random.split(keys[n], num)   (pqn_minatar.py:108,112,183,459) */
int pqn_rng_split(const uint32_t* keys, int64_t n, int32_t num, uint32_t* out, int rng_mode, void* stream);
/* Threefry-2x32-20 block function on n (key, counter) pairs: KAT hook for tests. */
int pqn_threefry2x32(const uint32_t* key_pairs, const uint32_t* ctr_pairs, uint32_t* out_pairs, int64_t n,
                     void* stream);
/* out[n][len] = jax.random.random_bits(keys[n], 32, (len,)) — sort keys of jax.random.permutation (:303) */
int pqn_rng_bits(const uint32_t* keys, int64_t n, int64_t len, uint32_t* out, int rng_mode, void* stream);
/* out[S][n] (int32) = jax.random.permutation(keys[s], n) as an index permutation, i.e. the shuffle that
 * `jax.random.permutation(rng, x)` applies to every leaf of the flattened rollout (pqn_minatar.py:299-315): jax's
 * rounds of a stable sort by fresh 32-bit keys, done as an exact bucket + rank sort (csrc/pqn_perm.cu).
 * out_chunk > 0 (must divide n) writes the minibatch layout out[n / out_chunk][S][out_chunk] instead of out[S][n]
 * (:316-321: minibatch i of seed s = positions [i * chunk, (i+1) * chunk)).  workspace: pqn_permutation_workspace_bytes. */
/* test hook: target bucket size 2^log2_elems of the bucket sort (default 6; > 8 forces the global-memory rank path);
 * returns the previous value.  Set it before pqn_permutation_workspace_bytes. */
int pqn_set_permutation_bucket_log2(int log2_elems);
int64_t pqn_permutation_workspace_bytes(int64_t n, int32_t S);
int pqn_permutation(const uint32_t* keys, int64_t n, int32_t S, int rng_mode, int32_t* out, int64_t out_chunk,
                    void* workspace, void* stream);

/* ---- the environment operator: vmapped LogWrapper(env).reset / .step ------
 * replaces vmap_reset / vmap_step, pqn_minatar.py:107-112 (gymnax protocol:
 * env.reset(key, params) -> (obs, state); env.step(key, state, action, params)
 * -> (obs, state, reward, done, info)).  keys: uint32[N][2] (one per env, i.e.
 * the caller already did jax.random.split(rng, n_envs)).  obs: float32[N][obs_dim].
 * info outputs may be NULL.  max_steps <= 0 selects the env default. */
int pqn_env_reset(int env_id, const uint32_t* keys, uint32_t* state, float* obs, int64_t N, int max_steps,
                  int rng_mode, void* stream);
/* gymnax EnvParams beyond the step limit.  max_steps <= 0 selects the env default (max_steps_in_episode).
 * memory_length: MemoryChain's memory_length (>= 1; 5 is gymnax's default, which pqn_env_reset uses); ignored by
 * envs without that parameter.  MemoryChain keeps it in its state, so pqn_env_step / pqn_rollout_act_step and their
 * auto-resets use the value the envs were reset with. */
typedef struct pqn_env_params_t {
  int32_t max_steps;
  int32_t memory_length;
} pqn_env_params_t;
/* pqn_env_reset with explicit env parameters (params_host: a host pointer, not NULL).  Returns PQN_E_INVALID for
 * memory_length < 1 on an env that has the parameter. */
int pqn_env_reset_params(int env_id, const uint32_t* keys, uint32_t* state, float* obs, int64_t N,
                         const pqn_env_params_t* params_host, int rng_mode, void* stream);
int pqn_env_step(int env_id, const uint32_t* keys, uint32_t* state, const int32_t* action, float* obs,
                 float* reward, uint8_t* done, float* info_discount, float* info_returned_episode_returns,
                 int32_t* info_returned_episode_lengths, int32_t* info_timestep, int64_t N, int max_steps,
                 int rng_mode, void* stream);
/* current observation of `state` as packed bits (binary_obs envs): uint32[N][packed_obs_words] */
int pqn_env_obs_packed(int env_id, const uint32_t* state, uint32_t* obs_packed, int64_t N, void* stream);
/* current observation of `state` as float32[N][obs_dim] (MemoryChain: the observation its last reset or step
 * returned, i.e. get_obs of the state before that step, as bsuite's step emits it) */
int pqn_env_obs(int env_id, const uint32_t* state, float* obs, int64_t N, void* stream);

/* ---- epsilon-greedy (eps_greedy_exploration, pqn_minatar.py:115-128,194-196) */
int pqn_eps_greedy(const uint32_t* keys /*[N][2]*/, const float* q /*[N][A]*/, const float* eps /*[1] device*/,
                   int32_t* action, int64_t N, int32_t A, int rng_mode, void* stream);

/* ---- fused rollout step (_step_env body, pqn_minatar.py:181-210) -----------
 * One launch = for every (seed s, env e): per-env keys from the step's
 * (rng_a, rng_s) pair, argmax + eps-greedy on q, LogWrapper(env).step with
 * auto-reset, and the stores of this step's transition row.
 *   step_keys: uint32[S][2][2]   (rng_a, rng_s) of this step for each seed
 *   q:         float32[S*E][A]   Q(last_obs) from the Q-network forward
 *   eps:       float32[1]        device scalar (eps_scheduler(n_updates), :195)
 *   obs_next:  row (s,e) of new_obs goes to row  s*obs_seed_stride + e  of
 *              obs_next: packed uint32[packed_obs_words] rows (binary envs) or
 *              float32[obs_dim] rows (classic control).  The rollout buffer is
 *              [S][T+1][E] rows, so the caller passes the step's base pointer
 *              and obs_seed_stride = (T+1)*E.
 *   action/reward/done/maxq: element (s,e) goes to  s*tr_seed_stride + e
 *              (buffers are [S][T][E]; tr_seed_stride = T*E); reward is scaled
 *              by rew_scale (:205); maxq = max_a q (next_q of the Q(lambda) scan)
 *   info_sums: float64[S][5] running sums over the update of
 *              (returned_episode_returns, returned_episode_lengths, timestep,
 *               returned_episode, discount) — :338 takes their means.  With
 *              info_done_only != 0 only steps with done contribute (the
 *              nanmean-where-returned_episode of get_test_metrics, :403-412).
 *   env_total / env_offset: the E envs of this call are envs [env_offset, env_offset + E) of a vmap over env_total
 *              envs (env-sharded data parallelism): per-env keys are split(key, env_total)[env_offset + e].
 *              env_total <= 0 means env_total = E, env_offset = 0. */
int pqn_rollout_act_step(int env_id, const uint32_t* step_keys, const float* q, const float* eps,
                         uint32_t* state, void* obs_next, int64_t obs_seed_stride, int32_t* action,
                         float* reward, uint8_t* done, float* maxq, int64_t tr_seed_stride, double* info_sums,
                         int info_done_only, int32_t S, int32_t E, int32_t env_total, int32_t env_offset, int max_steps,
                         float rew_scale, int rng_mode, void* stream);
/* keys_out[T][S][2][2], rng_inout[S][2]: the scan carry chain
 * rng, rng_a, rng_s = split(rng, 3) for T steps (pqn_minatar.py:183). */
int pqn_rollout_keys(uint32_t* rng_inout, uint32_t* keys_out, int32_t S, int32_t T, int rng_mode, void* stream);

/* ---- Q(lambda) targets (last_q bootstrap + reverse scan, pqn_minatar.py:227-260)
 *   q_last: float32[S*E][A] = Q(next_obs[T-1]);  reward/maxq/targets float32[S][T][E],
 *   done uint8[S][T][E]                                                        */
int pqn_qlambda(const float* reward, const uint8_t* done, const float* maxq, const float* q_last,
                float* targets, int32_t T, int32_t S, int32_t E, int32_t A, float gamma, float lambda,
                void* stream);

/* ---- Q-network (QNetwork/CNN pqn_minatar.py:24-69; MLP QNetwork pqn_gymnax.py:29-58)
 * All network entry points are batched over S independent seeds: parameter
 * blocks are float32[S][P] with the per-seed layout given by pqn_net_layout. */
#define PQN_NET_MINATAR_CNN 0
#define PQN_NET_MLP 1
#define PQN_NET_RNN 2   /* RNNQNetwork (GRU) of pqn_rnn_gymnax.py:57-105: MLP trunk + one-hot last action + scanned GRU + head */

typedef struct pqn_net_desc_t {
  int32_t kind;        /* PQN_NET_* */
  int32_t in_c;        /* CNN: input channels C (obs 10x10xC)   | MLP: input dim D */
  int32_t hidden;      /* CNN: 128 (fixed)                      | MLP: HIDDEN_SIZE */
  int32_t layers;      /* CNN: ignored                          | MLP: NUM_LAYERS (1 or 2) */
  int32_t num_actions; /* A */
  int32_t norm_type;   /* NORM_TYPE: 0 layer_norm (default), 1 batch_norm, 2 none   (pqn_minatar.py:31-36) */
  int32_t norm_input;  /* NORM_INPUT: 1 = the input BatchNorm normalises the observation (replaces x/255 in the CNN)
                          and is trained; 0 = it is the dummy of pqn_minatar.py:61-66 */
} pqn_net_desc_t;
#define PQN_NORM_LAYER 0
#define PQN_NORM_BATCH 1
#define PQN_NORM_NONE 2

/* offsets (in floats) of each tensor inside one seed's parameter block; flax
 * names: see SURVEY Appendix C.  Unused entries are -1. */
typedef struct pqn_net_layout_t {
  int64_t total;                 /* floats per seed */
  int64_t bn_scale, bn_bias;     /* BatchNorm_0 (dummy input norm)      [in] */
  int64_t conv_w, conv_b;        /* CNN_0/Conv_0 kernel [3,3,C,16] HWIO, bias [16] */
  int64_t ln0_scale, ln0_bias;   /* CNN: CNN_0/LayerNorm_0 [16] | MLP: LayerNorm_0 [H] */
  int64_t d0_w, d0_b;            /* CNN: CNN_0/Dense_0 [1024,128]/[128] | MLP: Dense_0 [D,H]/[H] */
  int64_t ln1_scale, ln1_bias;   /* CNN: CNN_0/LayerNorm_1 [128] | MLP: LayerNorm_1 [H] (layers==2) */
  int64_t d1_w, d1_b;            /* MLP only: Dense_1 [H,H]/[H] (layers==2) */
  int64_t head_w, head_b;        /* final Dense [H,A]/[A] */
  /* PQN_NET_RNN only (-1 otherwise): ScannedRNN_0/GRUCell_0/{ir,iz,in} kernel [H+A,H] + bias [H], {hr,hz} kernel [H,H],
   * hn kernel [H,H] + bias [H] */
  int64_t gru_ir_w, gru_ir_b, gru_iz_w, gru_iz_b, gru_in_w, gru_in_b, gru_hr_w, gru_hz_w, gru_hn_w, gru_hn_b;
} pqn_net_layout_t;

int pqn_net_layout(const pqn_net_desc_t* desc_host, pqn_net_layout_t* out_host);
/* floats per seed of the batch_stats block (flax "batch_stats" collection): [mean in][var in] of the input BatchNorm,
 * then, for norm_type == batch_norm, (mean[n], var[n]) of every hidden BatchNorm in network order (CNN: 16, 128;
 * MLP: hidden x layers).  With norm_type none the ln*_scale / ln*_bias layout entries are -1 (no such parameters). */
int64_t pqn_net_stats_floats(const pqn_net_desc_t* desc_host);
/* bytes of scratch the forward/backward need for `rows` samples per seed */
int64_t pqn_net_workspace_bytes(const pqn_net_desc_t* desc_host, int32_t S, int64_t rows);

/* network.init (pqn_minatar.py:156-170) on the device: flax-default initialisers (he_normal / lecun_normal
 * truncated normals, zero biases, unit norm scales) drawn counter-based from keys[S][2]. */
int pqn_net_init(const pqn_net_desc_t* desc_host, const uint32_t* keys, float* params, int32_t S, void* stream);

/* q[S][rows][A] = network.apply(params, obs, train=False) — pqn_minatar.py:184-191,227-234.
 *  obs: packed uint32[S][rows_total][packed_words] (CNN) or float32[S][rows_total][D] (MLP);
 *  gather (may be NULL): int32[S][rows] row indices into the seed's obs rows
 *  (minibatch gather of preprocess_transition, :299-307); obs_rows_per_seed is
 *  the stride of the obs buffer in rows.  batch_stats: float32[S][pqn_net_stats_floats] running statistics, read by
 *  the batch_norm / NORM_INPUT variants (train=False => use_running_average); may be NULL for the default network. */
int pqn_qnet_forward(const pqn_net_desc_t* desc_host, const float* params, const float* batch_stats, const void* obs,
                     const int32_t* gather, int64_t obs_rows_per_seed, float* q, int32_t S, int64_t rows,
                     void* workspace, void* stream);

/* One _learn_phase gradient (pqn_minatar.py:266-291): loss = 0.5*mean((Q(obs)[a]-target)^2),
 * action/target: [S][tr_rows_per_seed] indexed through `gather` like obs;
 * grads[S][P] (overwritten), loss_sum[S] += loss, qsa_sum[S] += mean(q_sa),
 * bn_sums: float32[S][2*in] += per-feature (sum x, sum x^2) of the raw obs minibatch
 * (input BatchNorm statistics, :65,293-296; consumed by pqn_bn_stats_update); may be NULL.
 * batch_stats (may be NULL for the default network): the running statistics of the HIDDEN BatchNorm layers are
 * updated in place (train=True, mutable batch_stats, :277-281); the input BatchNorm's go through bn_sums. */
int pqn_qnet_loss_grad(const pqn_net_desc_t* desc_host, const float* params, float* batch_stats, const void* obs,
                       const int32_t* gather, int64_t obs_rows_per_seed, const int32_t* action,
                       const float* target, int64_t tr_rows_per_seed, float* grads, float* loss_sum,
                       float* qsa_sum, float* bn_sums, int32_t S, int64_t rows, void* workspace, void* stream);

/* ---- recurrent Q-network (PQN_NET_RNN; purejaxql/pqn_rnn_gymnax.py) -------------------------------------------
 * One time step of network.apply(params, hs, obs[None], done[None], last_action[None], train=False) for S x E envs
 * (rollout :201-213, evaluation :447-459, memory warm-up :517-529):
 *   hs float32[S][E][H] carry, updated in place; obs float32 rows (row (s,e) at s*obs_rows_per_seed + e);
 *   last_done uint8[S][E] resets the carry to zero BEFORE the cell (:41-45); last_action int32[S][E] is appended
 *   one-hot to the GRU input (:84-85); q float32[S*E][A]. */
int pqn_rnn_step(const pqn_net_desc_t* desc_host, const float* params, float* hs, const float* obs,
                 int64_t obs_rows_per_seed, const uint8_t* last_done, const int32_t* last_action, float* q, int32_t S,
                 int32_t E, void* workspace, void* stream);
/* _loss_fn + value_and_grad of one minibatch window (:330-366): forward of the whole [T][B] window from the stored
 * carry hs0[S][B][H] (train=True), in-loss Q(lambda) targets from the stop-gradient q values (:295-323, bootstrap
 * max_a q[T-1]), loss = 0.5 mean over t < T-1, BPTT through the scanned GRU and the trunk.  All [S][T][B] tensors are
 * time-major per seed.  grads[S][P] is overwritten; loss_sum[S] += loss, qsa_sum[S] += mean chosen q. */
int pqn_rnn_loss_grad(const pqn_net_desc_t* desc_host, const float* params, const float* hs0, const float* obs,
                      const uint8_t* last_done, const int32_t* last_action, const int32_t* action, const float* reward,
                      const uint8_t* done, float* grads, float* loss_sum, float* qsa_sum, int32_t S, int32_t T, int32_t B,
                      float gamma, float lambda, void* workspace, void* stream);

/* optax.chain(clip_by_global_norm(max_norm), radam(lr_t)) + apply_updates
 * (pqn_minatar.py:159-162,292).  sched: float32[num_steps][4] per optimizer step
 * (lr, 1-b1^t, 1-b2^t, rect (0 => un-rectified step)); step_counter: int32[1]
 * device counter (grad_steps), incremented by the call. */
int pqn_radam_clip_step(float* params, const float* grads, float* mu, float* nu, const float* sched,
                        int32_t* step_counter, float* gnorm_scratch /*[S][64]*/, int32_t S, int64_t P,
                        float max_norm, float b1, float b2, float eps, void* stream);

/* dummy input BatchNorm running statistics (flax nn.BatchNorm momentum 0.99;
 * pqn_minatar.py:65,293-296): batch_stats float32[S][2][F] (mean, var),
 * bn_sums float32[S][2][F] (sum x, sum x^2 over `count` elements per feature);
 * bn_sums is zeroed for the next minibatch.  stats_seed_stride: floats between the seeds' batch_stats blocks
 * (pqn_net_stats_floats; 0 => 2*F). */
int pqn_bn_stats_update(float* batch_stats, float* bn_sums, int32_t S, int32_t F, int64_t stats_seed_stride,
                        float count, float momentum, void* stream);

/* Implementation selectors of the CNN (process-wide; the defaults are the fast paths, the others are kept as A/B
 * references for the parity tests):
 *  tensor-core path of the dense layer (forward, wgrad, dgrad): 2 (default) = tcgen05 kind::f16 on fp16-split (hi, lo')
 *  operand planes; 1 = tcgen05 3xTF32 with the lo operand derived in the kernel; 0 = fp32 FFMA kernels. */
int pqn_set_tensor_core_path(int on);
/*  3x3 conv forward: 1 (default) = fp16 mma.sync (exponent-coded im2col bits, fp16-split weights); 3 = the tf32
 *  mma.sync kernel of round 1; 2 = tcgen05 (correct, slower: per-pixel epilogue); 0 = fp32 CUDA cores.  The conv
 *  weight gradient runs on tf32 mma.sync for 1-3. */
int pqn_set_conv_mma_path(int on);

/* ---- tcgen05 (5th-gen tensor core) path of the dense contractions ----------
 * lo[i] = x[i] - trunc_tf32(x[i]): the error-compensation operand of 3xTF32. */
int pqn_tc_split_lo(const float* x, float* lo, int64_t n, void* stream);
/* Test hook: D[s] = A[s].B[s] through the TMA -> tcgen05.mma(kind::tf32) -> TMEM pipeline.
 *  a_mn=0: A is [S][M][K]; a_mn=1: A is [S][K][M].  b_mn=0: B is [S][N][K]; b_mn=1: B is [S][K][N].
 *  split3: 3xTF32 with the *_lo operands from pqn_tc_split_lo; else one TF32 pass.  N % 128 == 0. */
int pqn_tc_gemm_test(const float* a, const float* a_lo, const float* b, const float* b_lo, float* d, int32_t S,
                     int32_t M, int32_t N, int32_t K, int a_mn, int b_mn, int split3, void* stream);

/* fp16-split planes for the default tensor-core path: hi = fp16(x*scale), lo = fp16((x*scale - hi) * 2^11), so that
 * x*scale = hi + lo * 2^-11 to 22 significant bits (saturating at +-65000).  hi/lo: __half[n]. */
int pqn_tc_split16(const float* x, void* hi, void* lo, int64_t n, float scale, void* stream);
/* Test hook: D[s] = (A[s].B[s]) * out_scale through TMA -> tcgen05.mma(kind::f16) -> TMEM with the operands given as
 * (hi, lo) fp16 planes (3 products per k-step: hi.hi into the main accumulator, lo.hi + hi.lo into the 2^-11 one). */
int pqn_tc_gemm16_test(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo, float* d, int32_t S,
                       int32_t M, int32_t N, int32_t K, int a_mn, int b_mn, float out_scale, void* stream);

/* Debug hook: one 128x128x32 tile; dumps the TMA-written smem tiles and the TMEM accumulator. */
int pqn_tc_debug(const float* a, const float* b, float* dump_a, float* dump_b, float* out_d, uint32_t* info,
                 int a_mn, int b_mn, int nk, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PQN_B200_H */
