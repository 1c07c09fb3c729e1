/*
 * gsmarl_b200.h — C ABI of the B200-native batched GS-MARL environment hot path.
 *
 * STATUS OF THE REFERENCE (read this first).  The interface this library is a
 * drop-in for is the vectorised-env boundary of finleygou/GS-MARL:
 *   gsmarl/envs/mpe_env/env_wrappers.py          (GSMARL.egg-info/SOURCES.txt:11)
 *   gsmarl/envs/mpe_env/multiagent/environment.py (SOURCES.txt:15; classes named in readme.md:27-41)
 *   gsmarl/envs/mpe_env/multiagent/core.py        (SOURCES.txt:14)
 *   gsmarl/envs/mpe_env/multiagent/scenarios/<name>.py (SOURCES.txt:21-25)
 * Those files are WITHHELD in the mounted reference (readme.md:1, "hidden during
 * review"); only the manifest lines above prove they are supposed to exist.  The
 * reference has no FFI of its own (pure Python, setup.py:12-25 builds no extension),
 * so there is no reference C signature to copy.  Every entry point below therefore
 * cites the manifest line / readme line of the Python method it stands in for, and
 * every numeric constant of the model is an EXPLICIT field of gsm_config with no
 * default inside the library (SURVEY.md Appendix B) — nothing from upstream MPE can
 * leak in silently.  The model's arithmetic is the declared one in /SPEC.md;
 * parity with the real GS-MARL env is UNPINNED until its sources are mounted.
 *
 * Conventions: extern "C", plain pointers and sizes, int status return (0 = OK,
 * negative = gsm_status), caller-owned buffers, stream-ordered (no host sync) for
 * every call that takes a stream.  `real` below means float when cfg.dtype ==
 * GSM_F32 (production) and double when GSM_F64 (verification mode, compiled
 * without FMA contraction).
 */
#ifndef GSMARL_B200_H
#define GSMARL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSM_ABI_VERSION 7

#define GSM_OBS_DIM 6        /* vx, vy, px, py, target_dx, target_dy          (SPEC.md §6) */
#define GSM_NBR_FEAT_DIM 6   /* dx, dy, dvx, dvy, dist, (real)entity_type     (SPEC.md §6) */
#define GSM_MAX_DISCRETE 16
#define GSM_MAX_LSA_N 32     /* one warp lane per assignment column */
#define GSM_POLICY_HIDDEN 64       /* hidden width of the declared graph actor (SPEC.md §10) */
#define GSM_POLICY_MAX_ACTIONS 9   /* rows of head_w; compiled instances: n_actions 5 and 9  */
#define GSM_POLICY_VALUE_HEADS 2   /* critics on the same embedding: reward value, cost value */

typedef enum gsm_status {
  GSM_OK = 0,
  GSM_ERR_INVALID_ARG = -1,
  GSM_ERR_CUDA = -2,
  GSM_ERR_ABI = -3,
  GSM_ERR_UNSUPPORTED = -4,
  GSM_ERR_NO_DEVICE = -5
} gsm_status;

typedef enum gsm_dtype { GSM_F32 = 0, GSM_F64 = 1 } gsm_dtype;

/* Scenario families named by the reference: cooperative navigation (readme.md:44,71),
 * polygon = scenarios/simple_formation.py (SOURCES.txt:24, readme.md:89),
 * line = scenarios/simple_line.py (SOURCES.txt:25, readme.md:90). */
typedef enum gsm_scenario {
  GSM_SCN_NAVIGATION = 0,
  GSM_SCN_POLYGON = 1,
  GSM_SCN_LINE = 2
} gsm_scenario;

typedef enum gsm_action_mode {
  GSM_ACT_DISCRETE = 0,   /* int32 index into cfg.discrete_u                       */
  GSM_ACT_CONTINUOUS = 1  /* real[2] control                                        */
} gsm_action_mode;

typedef enum gsm_entity_type {
  GSM_ENT_AGENT = 0,
  GSM_ENT_GOAL = 1,
  GSM_ENT_OBSTACLE = 2,
  GSM_ENT_MARKER = 3      /* polygon centre / line end-points                       */
} gsm_entity_type;

/*
 * World + scenario description.  Stands in for scenario.make_world(args)
 * (scenarios/<name>.py, SOURCES.txt:21-25) and the World constants of core.py
 * (SOURCES.txt:14).  Entities are indexed agents first (0..n_agents-1) then
 * landmarks (n_agents..n_agents+n_landmarks-1).  All pointer fields are HOST arrays
 * copied at gsm_create; none may be NULL unless stated.
 */
typedef struct gsm_config {
  uint32_t struct_size;        /* = sizeof(gsm_config); checked                     */
  uint32_t abi_version;        /* = GSM_ABI_VERSION; checked                        */
  int32_t dtype;               /* gsm_dtype                                         */
  int32_t scenario;            /* gsm_scenario                                      */
  int32_t action_mode;         /* gsm_action_mode                                   */
  int32_t n_agents;            /* N >= 1                                            */
  int32_t n_landmarks;         /* L >= 0                                            */
  int32_t max_nbrs;            /* K: padded neighbour rows per agent, 1..N+L-1      */
  int32_t episode_length;      /* done when t >= episode_length (readme.md:101)     */
  int32_t n_discrete_actions;  /* 1..GSM_MAX_DISCRETE (ignored for CONTINUOUS)      */
  int32_t share_reward;        /* 0: per-agent reward, 1: mean over agents          */
  int32_t cost_obstacles;      /* 1: obstacle overlaps also count into the cost     */
  int32_t own_goal_always;     /* navigation: own goal is a neighbour at any range  */
  int32_t reserved0;
  double dt;
  double damping;
  double contact_force;
  double contact_margin;
  double sensing_radius;       /* neighbour iff dist < sensing_radius (strict)      */
  double w_dist;               /* reward = -w_dist*d + (d < goal_tol ? w_goal : 0)  */
  double w_goal;
  double goal_tol;
  double polygon_radius;       /* POLYGON only (readme.md:89: 0.5 in the paper)     */
  double spawn_extent[4];      /* per gsm_entity_type: reset draws U(-e, e)^2       */
  const double* discrete_u;    /* [n_discrete_actions][2] control per action index  */
  const double* size;          /* [N+L] entity radii                                */
  const uint8_t* collide;      /* [N+L] 1: takes part in contact force              */
  const int32_t* type;         /* [N+L] gsm_entity_type; agents first               */
  const double* mass;          /* [N]                                               */
  const double* accel;         /* [N] force = accel * u                             */
  const double* max_speed;     /* [N] <= 0: no clamp                                */
  const double* slot_table;    /* POLYGON: [N][2] unit offsets; LINE: [N][2] with   */
                               /* [k][0] = fraction along A->B; NAVIGATION: NULL    */
} gsm_config;

/*
 * Per-step buffers.  Stands in for the tuple the reference's step returns —
 * `obs, graph/adjacency, rewards, costs, dones, infos` (BASELINE.json north_star;
 * environment.py, SOURCES.txt:15).  All pointers are caller-owned.  For gsm_step /
 * gsm_reset / gsm_observe they are DEVICE pointers (so a runner can aim them at
 * slot t of its rollout buffer, SURVEY.md §8 f2); for the *_host variants they are
 * HOST pointers.  Any output pointer may be NULL to skip that output.
 */
typedef struct gsm_step_io {
  const void* actions;  /* DISCRETE: int32 [n_envs][N]; CONTINUOUS: real [n_envs][N][2] */
  void* obs;            /* real  [n_envs][N][GSM_OBS_DIM]                               */
  int32_t* nbr_idx;     /* int32 [n_envs][N][K]   entity index, ascending, -1 padded    */
  void* nbr_feat;       /* real  [n_envs][N][K][GSM_NBR_FEAT_DIM], zero padded          */
  int32_t* nbr_cnt;     /* int32 [n_envs][N]      rows written (<= K)                   */
  uint32_t* adj;        /* u32   [n_envs][N][adj_words] neighbour bitmask over entities */
  void* reward;         /* real  [n_envs][N]                                            */
  void* cost;           /* real  [n_envs][N]      integer-valued collision count        */
  uint8_t* done;        /* u8    [n_envs][N]                                            */
  int32_t* assign;      /* int32 [n_envs][N]      POLYGON/LINE: slot of agent i         */
} gsm_step_io;

typedef struct gsm_io_sizes {   /* bytes of each gsm_step_io buffer for this handle */
  size_t actions, obs, nbr_idx, nbr_feat, nbr_cnt, adj, reward, cost, done, assign;
  size_t agent_state;   /* real [n_envs][N][4]  (px,py,vx,vy)  */
  size_t landmark_pos;  /* real [n_envs][L][2]                 */
  size_t step_count;    /* int32 [n_envs]                      */
  int32_t adj_words;    /* ceil((N+L)/32)                      */
  int32_t real_bytes;   /* 4 or 8                              */
} gsm_io_sizes;

typedef struct gsm_env gsm_env;   /* opaque */

int gsm_abi_version(void);
const char* gsm_status_string(int status);
/* Last error text for a handle (or for gsm_create when h == NULL). */
const char* gsm_last_error(const gsm_env* h);

/* make_env / MultiAgentGraphConstrainEnv.__init__ (make_env.py SOURCES.txt:12;
 * environment.py SOURCES.txt:15).  env_offset is the global index of this shard's
 * first env: reset draws depend on (seed, env_offset + i, episode) only, so any
 * sharding of the same global env range gives identical states. */
int gsm_create(const gsm_config* cfg, int64_t n_envs, int64_t env_offset, int device,
               gsm_env** out);
int gsm_destroy(gsm_env* h);
int gsm_get_io_sizes(const gsm_env* h, gsm_io_sizes* out);

/* MultiAgentGraphConstrainEnv.reset (environment.py SOURCES.txt:15; scenario
 * reset_world, scenarios/<name>.py).  mask: NULL = every env; else device u8, env i is
 * reset iff mask[i*mask_stride] != 0 (mask_stride = N lets a `done` buffer be
 * passed directly).  Writes obs / nbr_* / adj (and assign) of the reset envs only. */
int gsm_reset(gsm_env* h, uint64_t seed, const uint8_t* mask, int64_t mask_stride,
              const gsm_step_io* io, void* stream);

/* MultiAgentGraphConstrainEnv.step -> World.step + per-agent obs/graph/reward/cost/
 * done (environment.py SOURCES.txt:15; core.py SOURCES.txt:14). */
int gsm_step(gsm_env* h, const gsm_step_io* io, void* stream);

/* T consecutive steps, one launch sequence replayed from a CUDA graph: step s reads
 * actions + s*action_stride bytes and writes every non-NULL output at
 * + s*<that buffer's gsm_io_sizes entry> (i.e. io points at slot 0 of [T][...]
 * rollout-buffer tensors; SURVEY.md §8 f2). */
int gsm_rollout(gsm_env* h, int32_t n_steps, const gsm_step_io* io, void* stream);

/* Auto-reset inside gsm_rollout (the vec-env wrapper's "reset when done", env_wrappers.py
 * SOURCES.txt:11): when enabled, an env whose step counter reaches episode_length at step s
 * keeps its terminal outputs in slot s and is re-drawn (same Philox stream as gsm_reset with
 * the handle's current seed) before step s+1.  gsm_step is not affected. */
int gsm_set_auto_reset(gsm_env* h, int enabled);

/* Slot stride of gsm_rollout, in envs: the io pointers aim at this handle's first env inside
 * [T][slot_envs][...] tensors that are wider than the handle (slot_envs >= n_envs; 0 restores
 * the handle's own n_envs).  Lets several handles that each own a contiguous env range of one
 * GPU — sub-shards on their own CUDA streams, so the tail of one fused rollout overlaps the body
 * of another's — fill ONE rollout buffer (the buffer insert of utils/graph_separated_buffer.py,
 * SOURCES.txt:33, stays a no-op).  gsm_step / gsm_reset are not affected: their tensors are one
 * slot, and a contiguous env slice of it is already a valid io. */
int gsm_set_slot_envs(gsm_env* h, int64_t slot_envs);

/* _get_obs + graph build for the current state, no physics (environment.py). */
int gsm_observe(gsm_env* h, const gsm_step_io* io, void* stream);

/* State injection / extraction (device pointers; NULL = skip that part).  Used by
 * the parity tests to start from oracle-generated states, and for checkpointing. */
int gsm_set_state(gsm_env* h, const void* agent_state, const void* landmark_pos,
                  const int32_t* step_count, void* stream);
int gsm_get_state(gsm_env* h, void* agent_state, void* landmark_pos, int32_t* step_count,
                  void* stream);

/* Episode counters (device int32 [n_envs]; NULL = skip): the reset draws are keyed by (seed, global
 * env index, episode), so a checkpoint that restores agent_state / landmark_pos / step_count must
 * restore these too for the NEXT re-draws to repeat. */
int gsm_set_episode(gsm_env* h, const int32_t* episode, void* stream);
int gsm_get_episode(gsm_env* h, int32_t* episode, void* stream);

/* Host-buffer variants: every pointer in io / arguments is HOST memory.  The call
 * stages through pinned memory, copies H2D, runs the device path on the handle's own
 * stream, copies D2H and synchronises — this is the numpy-facing drop-in path the
 * reference's env_wrappers.py (SOURCES.txt:11) exposes to the runner. */
/* Library-owned PINNED host buffers laid out as one arena (out receives the ten
 * sub-buffer pointers).  Passing exactly these to the *_host calls makes a step one
 * H2D copy (actions) + one kernel + one D2H copy (all outputs). */
int gsm_host_io(gsm_env* h, gsm_step_io* out);
/* What the *_host calls deliver into the gsm_host_io buffers, and how.
 * out_mask: bit k = deliver output k, k in the order of gsm_step_io (1 obs, 2 nbr_idx, 3 nbr_feat,
 *   4 nbr_cnt, 5 adj, 6 reward, 7 cost, 8 done, 9 assign); a runner that reads the graph through
 *   adj + nbr_feat can drop nbr_idx (redundant), navigation can drop assign (the identity).  Outputs
 *   that are switched off keep whatever the host buffer held.  Default: all.
 * sparse != 0 (default): the pinned arena is mapped and a kernel writes the outputs into it over
 *   PCIe, sending only the nbr_cnt[i] valid rows of nbr_feat per agent (71 % of a dense step's
 *   bytes are nbr_feat, about half of its rows are padding) — the padding rows of the host buffer
 *   already hold zeros and rows that stop being valid are cleared — and of nbr_idx only the 16-byte
 *   pieces that differ from what the host already holds (neighbour sets change slowly), so the host
 *   arrays stay bit-identical to the device tensors.  sparse == 0: one dense D2H copy per call.
 *   In sparse mode the library relies on the host arena holding what it last delivered: treat the output
 *   buffers as READ-ONLY (copy before modifying in place); calling gsm_set_host_outputs again with the same
 *   arguments forces a dense re-synchronisation if they were overwritten.
 * A change takes effect with a dense re-synchronisation on the next *_host call. */
int gsm_set_host_outputs(gsm_env* h, uint32_t out_mask, int32_t sparse);
int gsm_reset_host(gsm_env* h, uint64_t seed, const uint8_t* mask, int64_t mask_stride,
                   const gsm_step_io* io);
int gsm_step_host(gsm_env* h, const gsm_step_io* io);
int gsm_observe_host(gsm_env* h, const gsm_step_io* io);
int gsm_set_state_host(gsm_env* h, const void* agent_state, const void* landmark_pos,
                       const int32_t* step_count);
int gsm_get_state_host(gsm_env* h, void* agent_state, void* landmark_pos,
                       int32_t* step_count);

/* Number of this library's kernels launched on behalf of the handle so far
 * (graph replays count the kernels inside the graph). */
int64_t gsm_kernel_launches(const gsm_env* h);

/* Stand-alone batched linear sum assignment (scipy.optimize.linear_sum_assignment,
 * scipy==1.7.3 in requirements.txt:101; rectangular_lsap shortest-augmenting-path,
 * square case).  cost: device real [n_problems][n][n] row-major; col4row: device
 * int32 [n_problems][n].  dtype: gsm_dtype.  1 <= n <= GSM_MAX_LSA_N. */
int gsm_lsa(const void* cost, int32_t* col4row, int64_t n_problems, int32_t n,
            int32_t dtype, int device, void* stream);

/* ---- SURVEY.md §8 "next" rows f3 + f1: actor forward over the padded graph, collect loop ------
 * Reference side (withheld): the GNN actor of gsmarl/algorithms (torch-geometric,
 * requirements.txt:119) evaluated once per env step by runner/mpe_runner.py's collect
 * (SOURCES.txt:28), whose results go into utils/graph_separated_buffer.py (SOURCES.txt:33).
 * The architecture is the DECLARED one of SPEC.md §10 (parameters shared by all agents):
 *   e = relu(ego_w obs + ego_b); m_r = relu(nbr_w feat_r + nbr_b) for the nbr_cnt valid rows;
 *   a = softmax_r(att_w . m_r + att_b); z = head_w [e ; sum_r a_r m_r] + head_b;
 *   action = argmax_k(z_k - log(-log(u_k))), u from Philox4x32-10 with key = seed and counter
 *   (row_offset + row, step, 0x80000000 | k/4) — or argmax_k z_k when greedy != 0.
 * Weight matrices are row-major [out][in] like torch.nn.Linear.weight; HOST memory (they travel
 * in the kernel's parameter space).  fp32 only. */
typedef struct gsm_policy_weights {
  uint32_t struct_size;          /* = sizeof(gsm_policy_weights); checked */
  int32_t n_actions;             /* 5 or 9 */
  float ego_w[GSM_POLICY_HIDDEN][GSM_OBS_DIM];
  float ego_b[GSM_POLICY_HIDDEN];
  float nbr_w[GSM_POLICY_HIDDEN][GSM_NBR_FEAT_DIM];
  float nbr_b[GSM_POLICY_HIDDEN];
  float att_w[GSM_POLICY_HIDDEN];
  float att_b;
  float head_w[GSM_POLICY_MAX_ACTIONS][2 * GSM_POLICY_HIDDEN];   /* rows >= n_actions ignored */
  float head_b[GSM_POLICY_MAX_ACTIONS];
  float value_w[GSM_POLICY_VALUE_HEADS][2 * GSM_POLICY_HIDDEN];  /* v = value_w [e ; sum_r a_r m_r] + value_b */
  float value_b[GSM_POLICY_VALUE_HEADS];                         /* [0] reward critic, [1] cost critic   */
} gsm_policy_weights;

typedef struct gsm_policy_io {   /* DEVICE pointers; a "row" is one agent of one env */
  const float* obs;        /* [n_rows][GSM_OBS_DIM]                     */
  const float* nbr_feat;   /* [n_rows][max_nbrs][GSM_NBR_FEAT_DIM]      */
  const int32_t* nbr_cnt;  /* [n_rows]  valid rows (clamped to [0, max_nbrs]) */
  int32_t* actions;        /* [n_rows]  out                             */
  float* logp;             /* [n_rows]  out, log pi(action); NULL = skip */
  float* logits;           /* [n_rows][n_actions] out; NULL = skip       */
  float* values;           /* [n_rows][GSM_POLICY_VALUE_HEADS] out; NULL = skip (actor-only kernel) */
  int64_t n_rows;
  uint64_t row_offset;     /* global index of row 0 (env_offset * N): sharding-invariant draws */
  uint64_t seed, step;
  int32_t max_nbrs;
  int32_t greedy;
} gsm_policy_io;

int gsm_policy_act(const gsm_policy_weights* w, const gsm_policy_io* io, int device, void* stream);
const char* gsm_policy_last_error(void);

/* ---- learner pass (SPEC.md §12): evaluate_actions of the same actor, forward and backward ------
 * Stands in for the lineage's evaluate_actions / get_values (SOURCES.txt:8, withheld).  The weights
 * are a DEVICE float vector in torch.nn.utils.parameters_to_vector(GraphAttentionActor) order:
 *   ego_w[64][6], ego_b[64], nbr_w[64][6], nbr_b[64], att_w[64], att_b, head_w[A][128], head_b[A],
 *   value_w[2][128], value_b[2]   -> GSM_POLICY_N_PARAMS(A) floats (1864 for A = 5, 2380 for A = 9).
 * No host copy and no host sync: a minibatch step can be captured in a CUDA graph.  Row i of the
 * call reads source row src = rows ? rows[i] : i of obs / nbr_feat / nbr_cnt / actions and writes
 * element i of every output.  Only the nbr_cnt[src] valid neighbour rows are read.  fp32 only. */
#define GSM_POLICY_N_PARAMS(n_actions) (961 + 129 * (n_actions) + 2 * (2 * GSM_POLICY_HIDDEN + 1))

typedef struct gsm_policy_eval_io {   /* DEVICE pointers */
  uint32_t struct_size;      /* = sizeof(gsm_policy_eval_io); checked                          */
  int32_t n_actions;         /* 5 or 9                                                         */
  const float* params;       /* [GSM_POLICY_N_PARAMS(n_actions)]                               */
  const float* obs;          /* [src_rows][GSM_OBS_DIM]                                        */
  const float* nbr_feat;     /* [src_rows][max_nbrs][GSM_NBR_FEAT_DIM]                         */
  const int32_t* nbr_cnt;    /* [src_rows]  valid rows (clamped to [0, max_nbrs])              */
  const int32_t* actions;    /* [src_rows]  an action outside [0, n_actions) gives NaN logp / grad */
  const int64_t* rows;       /* [n_rows] source row of row i (caller keeps it in range); NULL = i */
  float* logp;               /* [n_rows] out, z_a - logsumexp(z); NULL = skip                  */
  float* entropy;            /* [n_rows] out, logsumexp(z) - sum_k p_k z_k; NULL = skip        */
  float* values;             /* [n_rows][GSM_POLICY_VALUE_HEADS] out; NULL = skip              */
  int64_t n_rows;
  int32_t max_nbrs;
  int32_t reserved;          /* 0 */
} gsm_policy_eval_io;

/* logp / values bit-identical to what gsm_policy_act / gsm_collect wrote for the same rows and actions. */
int gsm_policy_evaluate(const gsm_policy_eval_io* io, int device, void* stream);

/* Workspace bytes gsm_policy_backward needs for n_rows rows (a function of n_rows and n_actions
 * only); GSM_ERR_INVALID_ARG for n_rows < 0, GSM_ERR_UNSUPPORTED for n_actions not 5 or 9. */
int64_t gsm_policy_backward_workspace(int64_t n_rows, int32_t n_actions);

/* grad [GSM_POLICY_N_PARAMS] (overwritten) = d/dparams of
 *   sum_i d_logp[i] logp[i] + d_entropy[i] entropy[i] + d_values[i] . values[i]
 * over the rows of io (its output pointers are not used).  d_logp, d_entropy [n_rows] and d_values
 * [n_rows][2] may each be NULL (= zero).  Deterministic: per-block partial sums into `workspace`
 * (a partition of the rows that depends on n_rows only), combined in a fixed order; no atomics.
 * n_rows == 0 leaves grad untouched. */
int gsm_policy_backward(const gsm_policy_eval_io* io, const float* d_logp, const float* d_entropy,
                        const float* d_values, float* grad, void* workspace, size_t workspace_bytes,
                        int device, void* stream);

/* ---- Gaussian actor for GSM_ACT_CONTINUOUS worlds (SPEC.md §10b / §12b) ----------------------
 * The same embedding h = [e ; sum_r a_r m_r] as above, with a diagonal Gaussian head:
 *   mean = mean_w h + mean_b [2];  sigma = exp(log_std), log_std [2] a free parameter (not a function
 *   of the state);  action = mean + sigma * eps, eps by Box-Muller from words 0 and 1 of
 *   Philox4x32-10(key = seed, counter = (row lo, row hi, step, 0x80000000)) — or action = mean when
 *   greedy != 0.  Actions are not clipped or squashed.
 *   logp = sum_d (-1/2 delta_d^2 - log_std_d) - log(2 pi), delta_d = (a_d - mean_d) exp(-log_std_d)
 *   (NaN for a non-finite action);  entropy = sum_d (log_std_d + 1/2 (1 + log 2 pi)).
 * The learner's parameter vector is parameters_to_vector(GaussianGraphActor) order:
 *   ego_w[64][6], ego_b[64], nbr_w[64][6], nbr_b[64], att_w[64], att_b, mean_w[2][128], mean_b[2],
 *   log_std[2], value_w[2][128], value_b[2]   -> GSM_POLICY_GAUSS_N_PARAMS floats. */
#define GSM_POLICY_GAUSS_DIM 2
#define GSM_POLICY_GAUSS_N_PARAMS 1479

typedef struct gsm_policy_gauss_weights {   /* HOST memory, row-major [out][in] */
  uint32_t struct_size;          /* = sizeof(gsm_policy_gauss_weights); checked */
  float ego_w[GSM_POLICY_HIDDEN][GSM_OBS_DIM];
  float ego_b[GSM_POLICY_HIDDEN];
  float nbr_w[GSM_POLICY_HIDDEN][GSM_NBR_FEAT_DIM];
  float nbr_b[GSM_POLICY_HIDDEN];
  float att_w[GSM_POLICY_HIDDEN];
  float att_b;
  float mean_w[GSM_POLICY_GAUSS_DIM][2 * GSM_POLICY_HIDDEN];
  float mean_b[GSM_POLICY_GAUSS_DIM];
  float log_std[GSM_POLICY_GAUSS_DIM];
  float value_w[GSM_POLICY_VALUE_HEADS][2 * GSM_POLICY_HIDDEN];
  float value_b[GSM_POLICY_VALUE_HEADS];
} gsm_policy_gauss_weights;

typedef struct gsm_policy_gauss_io {   /* gsm_policy_io with float actions and the mean; DEVICE pointers */
  const float* obs;        /* [n_rows][GSM_OBS_DIM]                     */
  const float* nbr_feat;   /* [n_rows][max_nbrs][GSM_NBR_FEAT_DIM]      */
  const int32_t* nbr_cnt;  /* [n_rows]  valid rows (clamped to [0, max_nbrs]) */
  float* actions;          /* [n_rows][GSM_POLICY_GAUSS_DIM] out        */
  float* logp;             /* [n_rows]  out, log pi(action); NULL = skip */
  float* mean;             /* [n_rows][GSM_POLICY_GAUSS_DIM] out; NULL = skip */
  float* values;           /* [n_rows][GSM_POLICY_VALUE_HEADS] out; NULL = skip (actor-only kernel) */
  int64_t n_rows;
  uint64_t row_offset;     /* global index of row 0 (env_offset * N): sharding-invariant draws */
  uint64_t seed, step;
  int32_t max_nbrs;
  int32_t greedy;
} gsm_policy_gauss_io;

int gsm_policy_act_gauss(const gsm_policy_gauss_weights* w, const gsm_policy_gauss_io* io, int device,
                         void* stream);

typedef struct gsm_policy_gauss_eval_io {   /* gsm_policy_eval_io with float actions; DEVICE pointers */
  uint32_t struct_size;      /* = sizeof(gsm_policy_gauss_eval_io); checked                    */
  int32_t action_dim;        /* GSM_POLICY_GAUSS_DIM                                           */
  const float* params;       /* [GSM_POLICY_GAUSS_N_PARAMS]                                    */
  const float* obs;          /* [src_rows][GSM_OBS_DIM]                                        */
  const float* nbr_feat;     /* [src_rows][max_nbrs][GSM_NBR_FEAT_DIM]                         */
  const int32_t* nbr_cnt;    /* [src_rows]  valid rows (clamped to [0, max_nbrs])              */
  const float* actions;      /* [src_rows][GSM_POLICY_GAUSS_DIM]                               */
  const int64_t* rows;       /* [n_rows] source row of row i (caller keeps it in range); NULL = i */
  float* logp;               /* [n_rows] out; NULL = skip                                      */
  float* entropy;            /* [n_rows] out; NULL = skip                                      */
  float* values;             /* [n_rows][GSM_POLICY_VALUE_HEADS] out; NULL = skip              */
  int64_t n_rows;
  int32_t max_nbrs;
  int32_t reserved;          /* 0 */
} gsm_policy_gauss_eval_io;

/* As gsm_policy_evaluate / gsm_policy_backward_workspace / gsm_policy_backward, for the Gaussian
 * head: logp / values bit-identical to what gsm_policy_act_gauss / gsm_collect_gauss wrote; grad
 * [GSM_POLICY_GAUSS_N_PARAMS]; the same determinism rule.  A non-finite action gives NaN logp, and a
 * NaN gradient only where its d_logp != 0. */
int gsm_policy_evaluate_gauss(const gsm_policy_gauss_eval_io* io, int device, void* stream);
int64_t gsm_policy_backward_workspace_gauss(int64_t n_rows);
int gsm_policy_backward_gauss(const gsm_policy_gauss_eval_io* io, const float* d_logp, const float* d_entropy,
                              const float* d_values, float* grad, void* workspace, size_t workspace_bytes,
                              int device, void* stream);

/* ---- PPO-Lagrangian update (SPEC.md §14): the loss fused into the learner backward, one Adam step ----
 * Declared stand-in for the lineage's MAPPO-Lagrangian learner (withheld).  One minibatch of n rows; row
 * i reads source row src = rows ? rows[i] : i of the buffer's obs / nbr_feat / nbr_cnt / actions (the
 * eval io, whose output pointers are ignored) and of old_logp / old_values / returns / advantages:
 *   Ahat_h = (A_h - mu_h) / (sigma_h + 1e-5);  Abar = Ahat_0 - lambda Ahat_1;  rho = exp(logp - old_logp)
 *   L_pi = -(1/n) sum min(rho Abar, clip(rho, 1 - clip, 1 + clip) Abar)
 *   vc_h = old_v_h + clip(v_h - old_v_h, -value_clip, value_clip)
 *   L_V  = (1/n) sum_h sum max(1/2 (v_h - R_h)^2, 1/2 (vc_h - R_h)^2)
 *   L    = L_pi + value_coef L_V - entropy_coef (1/n) sum entropy
 * logp, entropy and values are gsm_policy_evaluate's (bit-identical).  grad = dL/dparams through the seeds
 *   d_logp = -rho Abar / n where rho Abar <= clip(rho) Abar, else 0;  d_entropy = -entropy_coef / n;
 *   d_v_h = value_coef (v_h - R_h) / n where (v_h - R_h)^2 >= (vc_h - R_h)^2, else value_coef (vc_h - R_h) / n
 *   where |v_h - old_v_h| <= value_clip, else 0  (torch autograd of L except at exact ties);
 * stats [GSM_PPO_STAT_FIELDS] = means over the n rows of: L_pi, L_V reward head, L_V cost head, entropy,
 * rho, clipped (|rho - 1| > clip), approx KL (old_logp - logp), then L.  Deterministic (a fixed partition
 * of the rows, fixed-order sums, no atomics); three launches with gsm_adam_step, no host sync. */
#define GSM_PPO_STAT_FIELDS 8

typedef struct gsm_ppo_loss_io {   /* DEVICE pointers */
  uint32_t struct_size;          /* = sizeof(gsm_ppo_loss_io); checked                                */
  int32_t reserved;              /* 0 */
  const float* old_logp;         /* [src_rows]     the buffer's logp                                  */
  const float* old_values;       /* [src_rows][2]  the buffer's values[:-1]                           */
  const float* returns;          /* [src_rows][2]  gsm_gae returns                                    */
  const float* advantages;       /* [src_rows][2]  gsm_gae advantages                                 */
  const float* adv_moments;      /* [4] (mu_0, sigma_0, mu_1, sigma_1) over the whole rollout         */
  const float* lagrange;         /* [1] lambda >= 0                                                   */
  float* stats;                  /* [GSM_PPO_STAT_FIELDS] out                                         */
  float clip;                    /* > 0 */
  float value_clip;              /* > 0 */
  float value_coef;              /* >= 0 */
  float entropy_coef;            /* >= 0 */
} gsm_ppo_loss_io;

/* Workspace bytes gsm_ppo_backward(_gauss) needs (a function of n_rows and n_actions only);
 * GSM_ERR_INVALID_ARG for n_rows < 0, GSM_ERR_UNSUPPORTED for n_actions not 5 or 9. */
int64_t gsm_ppo_backward_workspace(int64_t n_rows, int32_t n_actions);
int64_t gsm_ppo_backward_workspace_gauss(int64_t n_rows);

/* GSM_ERR_ABI for a bad struct_size; GSM_ERR_INVALID_ARG for a missing pointer, a short workspace,
 * clip <= 0, value_clip <= 0 or a negative coefficient.  n_rows == 0 leaves grad and stats untouched. */
int gsm_ppo_backward(const gsm_policy_eval_io* io, const gsm_ppo_loss_io* loss, float* grad, void* workspace,
                     size_t workspace_bytes, int device, void* stream);
int gsm_ppo_backward_gauss(const gsm_policy_gauss_eval_io* io, const gsm_ppo_loss_io* loss, float* grad,
                           void* workspace, size_t workspace_bytes, int device, void* stream);

/* torch.nn.utils.clip_grad_norm_(max_grad_norm) then torch.optim.Adam (no weight decay, no amsgrad), one
 * launch over n floats:  norm = ||grad||_2 (fixed-order sum);  g = grad min(1, max_grad_norm / (norm + 1e-6));
 * t = *step + 1;  m = beta1 m + (1 - beta1) g;  v = beta2 v + (1 - beta2) g^2;
 * params -= (lr / (1 - beta1^t)) m / (sqrt(v) / sqrt(1 - beta2^t) + eps)  (bias corrections in fp64);
 * *step = t;  *grad_norm = norm.  A non-finite norm skips the step: params, m, v and *step are left
 * unchanged (torch would write NaN); *grad_norm is still written.  grad is not modified.  DEVICE pointers.
 * GSM_ERR_INVALID_ARG for a missing pointer, n < 1, beta1 or beta2 outside [0, 1), lr < 0, eps < 0 or
 * max_grad_norm <= 0. */
int gsm_adam_step(float* params, const float* grad, float* m, float* v, int32_t* step, int64_t n, float lr,
                  float beta1, float beta2, float eps, float max_grad_norm, float* grad_norm, int device,
                  void* stream);

/* n_steps of {actor forward + sampling, env step} enqueued on `stream` with no host sync (2
 * kernels per step; capturable into a CUDA graph).  io->obs / nbr_* / adj / assign point at slot 0
 * of [n_steps+1][...] tensors whose slot 0 already holds the current observation (gsm_reset,
 * gsm_observe or the previous collect's last slot); io->actions / reward / cost / done point at
 * slot 0 of [n_steps][...] tensors; logp: float [n_steps][n_envs][N] or NULL; values: float
 * [n_steps][n_envs][N][GSM_POLICY_VALUE_HEADS] or NULL (the critics' predictions for the observation
 * the action was taken in — the buffer's value_preds / cost_preds).  Step t: the actor
 * reads observation slot t and writes actions (and logp) slot t with Philox step first_step + t;
 * gsm_step writes reward / cost / done slot t and the next observation into slot t + 1 — the
 * buffer "insert" is where the kernels write.  Slot strides follow gsm_get_io_sizes /
 * gsm_set_slot_envs.  With gsm_set_auto_reset enabled, envs that finish at step t keep their terminal
 * reward / cost / done in slot t and are re-drawn, their first observation replacing slot t + 1.
 * Needs a GSM_F32, GSM_ACT_DISCRETE handle with n_discrete_actions ==
 * w->n_actions. */
int gsm_collect(gsm_env* h, const gsm_policy_weights* w, int32_t n_steps, const gsm_step_io* io,
                float* logp, float* values, uint64_t seed, uint64_t first_step, int32_t greedy,
                void* stream);

/* gsm_collect with the Gaussian actor: io->actions is float [n_steps][n_envs][N][2].  Needs a
 * GSM_F32, GSM_ACT_CONTINUOUS handle; everything else as gsm_collect. */
int gsm_collect_gauss(gsm_env* h, const gsm_policy_gauss_weights* w, int32_t n_steps, const gsm_step_io* io,
                      float* logp, float* values, uint64_t seed, uint64_t first_step, int32_t greedy,
                      void* stream);

/* buffer.compute_returns + compute_cost_returns (utils/graph_separated_buffer.py, SOURCES.txt:33;
 * withheld: the on-policy lineage's GAE recursion, declared in SPEC.md §11) for both critics in one
 * launch.  DEVICE pointers over the rollout buffer's slots, slot stride = slot_rows rows:
 * reward, cost: float [T][slot_rows]; done: u8 [T][slot_rows]; values: float [T+1][slot_rows][2]
 * (slot T = bootstrap prediction for the last observation); returns, advantages (may be NULL):
 * float [T][slot_rows][2].  For t = T-1..0, head h (0: reward, 1: cost):
 *   mask = done[t] ? 0 : 1;  delta = r_h[t] + gamma * V_h[t+1] * mask - V_h[t];
 *   gae = delta + gamma * lam * mask * gae;  advantages[t] = gae;  returns[t] = gae + V_h[t]. */
int gsm_gae(const float* reward, const float* cost, const float* values, const uint8_t* done,
            int32_t n_steps, int64_t n_rows, int64_t slot_rows, float gamma, float lam,
            float* returns, float* advantages, int device, void* stream);

/* ---- episode statistics (SPEC.md §13): the runner's per-episode logging over the buffer slots --------
 * Episode return, cost and length per agent row and per team, across calls: rollouts shorter or longer
 * than an episode and staggered episode ends are handled by a per-row fp64 carry.  Slot t with done = 1
 * is the last step of an episode (the gsm_gae rule).  Per row, for t = 0 .. T-1:
 *   R += (double)reward[t];  C += (double)cost[t];  n += 1;  if done[t]: agent episode (R, C, n), carry = 0.
 * An env's team episode ends where its agent 0's done is set: team return = (sum_j R_j) / N, team cost =
 * sum_j C_j (j ascending, fp64), team length = n of agent 0.  Safe: cost == 0; over the limit: cost >
 * agent_cost_limit (agent episodes) or > team_cost_limit (team episodes).
 * totals [GSM_EPISODE_STAT_FIELDS] (overwritten every call; additive across calls and ranks):
 *   agent episodes  0 count, 1 sum return, 2 sum return^2, 3 sum cost, 4 sum cost^2, 5 sum length,
 *                   6 safe count, 7 over-limit count;  team episodes  8 .. 15, the same fields.
 * Deterministic: per-block partials in `workspace` (a partition of the rows that depends on n_rows and
 * agents_per_env only), combined in a fixed order; no atomics.  Two launches, no host sync. */
#define GSM_EPISODE_STAT_FIELDS 16

typedef struct gsm_episode_io {   /* DEVICE pointers; row = one agent of one env, rows [g*N, (g+1)*N) = env g */
  uint32_t struct_size;          /* = sizeof(gsm_episode_io); checked                                 */
  int32_t dtype;                 /* gsm_dtype of reward / cost                                        */
  const void* reward;            /* real [n_steps][slot_rows]                                         */
  const void* cost;              /* real [n_steps][slot_rows]                                         */
  const uint8_t* done;           /* u8   [n_steps][slot_rows]                                         */
  double* carry_return;          /* [n_rows] in/out: the partial episode of each row                  */
  double* carry_cost;            /* [n_rows] in/out                                                   */
  int32_t* carry_length;         /* [n_rows] in/out                                                   */
  double* totals;                /* [GSM_EPISODE_STAT_FIELDS] out                                     */
  int32_t* episodes;             /* [n_rows / N] out: team episodes each env completed in this call   */
  double* last_return;           /* [n_rows] the last agent episode completed in this call; rows that */
  double* last_cost;             /* [n_rows]   completed none are left untouched; NULL = skip         */
  int32_t* last_length;          /* [n_rows]                                                          */
  double* team_last_return;      /* [n_rows / N] the same rule per env; NULL = skip                   */
  double* team_last_cost;        /* [n_rows / N]                                                      */
  int64_t n_rows;                /* a multiple of agents_per_env; 0 = no-op                           */
  int64_t slot_rows;             /* slot stride in rows, >= n_rows                                    */
  int32_t n_steps;               /* T >= 1                                                            */
  int32_t agents_per_env;        /* N, 1 .. 1024                                                      */
  double agent_cost_limit;
  double team_cost_limit;
} gsm_episode_io;

/* Workspace bytes gsm_episode_stats needs (a function of n_rows and agents_per_env only);
 * GSM_ERR_INVALID_ARG for n_rows < 0, agents_per_env outside [1, 1024] or n_rows % agents_per_env != 0. */
int64_t gsm_episode_stats_workspace(int64_t n_rows, int32_t agents_per_env);

/* GSM_ERR_ABI for a bad struct_size; GSM_ERR_INVALID_ARG for a missing reward / cost / done / carry /
 * totals / episodes pointer, n_steps < 1, a bad agents_per_env or n_rows (as above), slot_rows < n_rows,
 * an unknown dtype or a workspace smaller than gsm_episode_stats_workspace. */
int gsm_episode_stats(const gsm_episode_io* io, void* workspace, size_t workspace_bytes, int device,
                      void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GSMARL_B200_H */
