/*
 * muzero_b200 — C ABI of the B200-native MuZero search-and-inference engine.
 *
 * Drop-in boundary for the self-play hot path of michaelnny/muzero.  The
 * reference has no FFI; its boundary is three Python call signatures
 *   muzero/mcts.py:302-312      uct_search(...)
 *   muzero/network.py:62-84     MuZeroNet.initial_inference(x)
 *   muzero/network.py:86-111    MuZeroNet.recurrent_inference(hidden, action)
 * which muzero_b200/{mcts,network}.py keep; those modules call ONLY the entry
 * points below (ctypes, raw device pointers + the current CUDA stream).  Each
 * entry point cites the reference lines it replaces.
 *
 * Conventions
 *   - every function returns 0 on success, a negative MZ_E* code otherwise and
 *     never throws; mz_last_error() gives the thread-local message;
 *   - every pointer marked "dev" is device memory owned by the caller; the
 *     library allocates no device memory: pools and nets live inside an arena
 *     the caller allocates (size from mz_*_arena_bytes) and keeps alive;
 *   - kernels are enqueued on `stream` (a cudaStream_t) and nothing
 *     synchronises except where stated, so a whole simulation loop can be
 *     captured into a CUDA graph;
 *   - a handle is not thread-safe.
 */
#ifndef MUZERO_B200_H
#define MUZERO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MZ_OK            0
#define MZ_EINVAL       -1   /* bad argument                                  */
#define MZ_ECUDA        -2   /* CUDA runtime error (message has the detail)   */
#define MZ_ENOMEM       -3   /* arena too small                               */
#define MZ_ESTATE       -4   /* call out of order (e.g. expand before select) */

typedef struct mz_pool mz_pool;   /* node pool + per-tree search state for B trees */
typedef struct mz_net  mz_net;    /* repacked network weights + launch plan        */
typedef void* mz_stream;          /* cudaStream_t                                  */

const char* mz_last_error(void);
int mz_version(void);
/* Programmatic dependent launch between the short kernels of the per-simulation chain (tree kernel <-> tcgen05 MLP
 * kernel): a kernel's prologue overlaps its predecessor's tail.  Scheduling only, no effect on results.  Default on;
 * enable = 0 (or MZ_NO_PDL=1 in the environment) launches every kernel the ordinary way. */
int mz_set_pdl(int enable);
/* sm count and compute capability of `device`; fails on anything but sm_100. */
int mz_device_check(int device, int* sm_count, int* cc);

/* ------------------------------------------------------------------------
 * Search pool  (replaces Node / MinMaxStats objects, mcts.py:33-217)
 * ---------------------------------------------------------------------- */
typedef struct mz_pool_config {
  int32_t num_trees;          /* B                                                    */
  int32_t num_actions;        /* A                                                    */
  int32_t num_simulations;    /* S; a tree has exactly S+1 expanded nodes; S <= 65534 */
  int32_t hidden_bytes;       /* bytes of one node's hidden-state slot (multiple of 16) */
  int32_t is_board_game;      /* config.is_board_game   (mcts.py:147-155,169-171)     */
  int32_t has_known_bounds;   /* config.known_bounds is not None (mcts.py:36-38)      */
  double  bound_min, bound_max;
  double  discount;           /* config.discount                                      */
} mz_pool_config;

/* buffers inside the arena that tests / the host wrapper may look at */
enum mz_view {
  MZ_VIEW_EDGES = 0,     /* [B, S+1, A] 8-byte HOT records {u32 child << 16 | N (child 0xFFFF = none), f32 child_Q}: statistics of child (node, a) in the PARENT's row -- all the pUCT descent reads; child_Q = Node.child_Q of the edge (float32, min-max normalised; 0 for unvisited edges), refreshed by expand_backup */
  MZ_VIEW_PRIOR,         /* f64 [B, A]   the one prior every node of a tree uses (mcts.py:386)             */
  MZ_VIEW_ROOT_W,        /* f64 [B]                                                                          */
  MZ_VIEW_ROOT_N,        /* i32 [B]                                                                          */
  MZ_VIEW_MINMAX,        /* f64 [B, 2]   (min, max)                                                          */
  MZ_VIEW_COUNT,         /* i32 [B]      expanded nodes so far                                               */
  MZ_VIEW_LEAF_PARENT,   /* i32 [B]      node the last select stopped at                                     */
  MZ_VIEW_LEAF_ACTION,   /* i32 [B]                                                                          */
  MZ_VIEW_LEAF_DEPTH,    /* i32 [B]      depth of the leaf about to be created (>= 1)                        */
  MZ_VIEW_SRC_SLOT,      /* i32 [B]      tree*(S+1)+leaf_parent : hidden slot to read                        */
  MZ_VIEW_DST_SLOT,      /* i32 [B]      tree*(S+1)+count       : hidden slot to write                       */
  MZ_VIEW_PATH,          /* u32 [B, S+1] edge index (node*A+action) per level of the last select             */
  MZ_VIEW_NODE_PARENT,   /* i32 [B, S+1] parent node of each expanded node (-1 for the root)                 */
  MZ_VIEW_NODE_MOVE,     /* i32 [B, S+1] action that led to each expanded node                               */
  MZ_VIEW_NODE_VALUE,    /* f32 [B, S+1] value the network gave each node when it was expanded (debug/replay) */
  MZ_VIEW_RNG_KEY,       /* u32 [B, 624] MT19937 state (numpy legacy stream)                                 */
  MZ_VIEW_RNG_POS,       /* i32 [B]                                                                          */
  MZ_VIEW_HIDDEN,        /* u8  [B, S+1, hidden_bytes]                                                       */
  MZ_VIEW_REWARD,        /* f32 [B]      scratch the network writes, expand_backup reads                     */
  MZ_VIEW_VALUE,         /* f32 [B]                                                                          */
  MZ_VIEW_ERROR,         /* i32 [1]      sticky device-side error bits (MZ_DEVERR_*)                         */
  MZ_VIEW_STATS,         /* u64 [8]      {sum of select depths, select calls*B, tie-break draws, mt twists, then (MZ_TREE_TIMING only) min / max block start and max block end of the fused tree kernel, ns} */
  MZ_VIEW_EDGE_W,        /* f64 [B, S+1, A] Node.W of every edge     (COLD: read and written by the backup only; defined where N > 0) */
  MZ_VIEW_EDGE_REWARD,   /* f32 [B, S+1, A] Node.reward of every edge (COLD; written once, when the edge's child is expanded)       */
  MZ_VIEW__COUNT
};
#define MZ_DEVERR_POOL_FULL   1   /* more than S expansions                       */
#define MZ_DEVERR_NAN_POLICY  2   /* visit policy has NaN (all visits masked)     */

int mz_pool_arena_bytes(const mz_pool_config* cfg, size_t* bytes);
/* pb_c_table_host: float64[S+2], (log((n+base+1)/base)+init)*sqrt(n) computed by the
 * caller with CPython math exactly as mcts.py:193-195 does; copied synchronously. */
int mz_pool_create(const mz_pool_config* cfg, const double* pb_c_table_host,
                   void* arena_dev, size_t arena_bytes, mz_pool** out);
int mz_pool_destroy(mz_pool* pool);
/* Scheduling knob for pipelined sub-batches (no effect on results): num_ctas > 0 makes mz_expand_backup_select run as
 * that many persistent 1024-thread CTAs that pull trees off a counter and request more shared memory than is left
 * beside a persistent conv CTA, so the tree kernel of one sub-batch occupies `num_ctas` SMs of its own while the other
 * sub-batch's tower (capped to the remaining SMs with mz_net_set_cta_limit) runs undisturbed.  0 = warp-per-tree grid
 * over all SMs. */
int mz_pool_set_tree_ctas(mz_pool* pool, int num_ctas);
int mz_pool_view(mz_pool* pool, int which, void** dev_ptr, size_t* bytes);

/* np.random.seed(seed[t]) for every tree (init_genrand), on device. */
int mz_rng_seed(mz_pool* pool, const uint32_t* seeds_dev, mz_stream stream);

/* Dirichlet(alpha) noise from each tree's MT19937 stream with numpy's legacy
 * gamma sampler (mcts.py:244-245).  Same algorithm and draws as numpy; log/pow
 * are CUDA's, so samples agree with numpy to a few ulp, not bit-for-bit —
 * parity tests inject numpy's own noise through mz_search_reset instead. */
int mz_dirichlet(mz_pool* pool, double alpha, double* noise_out_dev /* [B,A] */, mz_stream stream);

/* Root preparation: Dirichlet mix, illegal-action masking + renormalisation,
 * root expansion, MinMaxStats reset.  Replaces mcts.py:353-367 (+244-246, 283-299).
 *   pi_probs    f32 [B,A]  softmax output of initial_inference
 *   noise       f64 [B,A]  or NULL (deterministic / alpha == 0: prior stays float32)
 *   eps         config.root_exploration_eps
 *   mask        u8  [B,A]  or NULL (actions_mask is None)
 *   players     i32 [B,2]  (current_player, opponent_player) or NULL (= (1,1))
 *   root_reward f32 [B]    or NULL (= 0, network.py:77)                         */
int mz_search_reset(mz_pool* pool, const float* pi_probs, const double* noise, double eps,
                    const uint8_t* mask, const int32_t* players, const float* root_reward,
                    mz_stream stream);

/* One warp per tree: pUCT descent with min-max normalised Q, float32 scores,
 * MT19937 tie-breaks, until an unexpanded child.  Replaces the select loop
 * mcts.py:372-379 and Node.best_child/child_Q/child_U (mcts.py:104-127,159-200).
 * Results land in the LEAF_* / SRC_SLOT / DST_SLOT / PATH views. */
int mz_select(mz_pool* pool, mz_stream stream);

/* Expand the selected leaf with (reward, value) of recurrent_inference and back
 * the value up to the root.  Replaces Node.expand (mcts.py:75-102, called at
 * mcts.py:386) and Node.backup (mcts.py:129-157).  reward/value: f32 [B] dev,
 * or NULL to use the pool's REWARD / VALUE scratch. */
int mz_expand_backup(mz_pool* pool, const float* reward, const float* value, mz_stream stream);

/* mz_expand_backup of this simulation followed by mz_select of the next one, in one launch (same results as
 * the two calls; saves a launch per simulation). */
int mz_expand_backup_select(mz_pool* pool, const float* reward, const float* value, mz_stream stream);

/* Visit counts -> masked policy -> action.  Replaces mcts.py:392-407 and
 * generate_play_policy (mcts.py:250-280).
 *   mask         u8  [B,A] or NULL
 *   temperature  f64 [B]
 *   deterministic  argmax(visits) instead of sampling
 *   action i32 [B], pi f64 [B,A], root_value f64 [B], visits i32 [B,A] (nullable) */
int mz_root_policy(mz_pool* pool, const uint8_t* mask, const double* temperature, int deterministic,
                   int32_t* action, double* pi, double* root_value, int32_t* visits, mz_stream stream);

/* ------------------------------------------------------------------------
 * Networks  (replace MuZeroNet.initial_inference / recurrent_inference,
 *            network.py:62-111, with util.py:31-36 and util.py:70-93 fused in)
 * ---------------------------------------------------------------------- */
enum mz_net_kind { MZ_NET_MLP = 0, MZ_NET_BOARD = 1, MZ_NET_ATARI = 2 };

typedef struct mz_net_config {
  int32_t kind;              /* mz_net_kind                                              */
  int32_t in_channels, in_h, in_w;   /* observation shape (MLP: flattened = c*h*w)       */
  int32_t num_actions;
  int32_t num_planes;        /* MLP width / conv channels                                */
  int32_t num_res_blocks;    /* conv nets                                                */
  int32_t hidden_dim;        /* MLP hidden-state size                                    */
  int32_t value_support, reward_support;   /* 1 = scalar head (network.py:126-134)       */
} mz_net_config;

/* bytes of one hidden-state slot in the layout the net's kernels use */
int mz_net_hidden_bytes(const mz_net_config* cfg, int32_t* bytes);
int mz_net_arena_bytes(const mz_net_config* cfg, int32_t max_batch, size_t* bytes);
/* weights: array of `num_weights` device pointers to float32 tensors in the
 * reference's state_dict order and PyTorch layouts (see muzero_b200/network.py);
 * they are repacked (transposed / BatchNorm folded / converted) into the arena
 * synchronously, so the caller may free them afterwards. */
int mz_net_create(const mz_net_config* cfg, const float* const* weights, int32_t num_weights,
                  int32_t max_batch, void* arena_dev, size_t arena_bytes, mz_net** out);
int mz_net_destroy(mz_net* net);

/* initial_inference for `batch` observations (network.py:62-84).
 *   obs        f32 [batch, c*h*w]
 *   hidden_out slot array; row i goes to slot dst_index[i] (or i when NULL)
 *   pi_probs   f32 [batch, A] softmax;  value f32 [batch] (support -> scalar applied) */
int mz_net_initial(mz_net* net, int32_t batch, const float* obs, void* hidden_out,
                   const int32_t* dst_index, float* pi_probs, float* value, mz_stream stream);

/* initial_inference for MuZeroAtariNet observations in their COMPACT form.  The reference's Atari observation
 * (gym_env.py:306-313, StackFrameAndAction.observation) is k uint8 frames cast to float32 followed by k constant
 * action planes (action + 1) / num_actions; uploading that float32 tensor is 4x the bytes of what it encodes.
 *   frames        u8  [batch, k, h, w]     (k = in_channels / 2)
 *   plane_values  f32 [batch, k]           the value of each constant plane
 * Results are identical to mz_net_initial on the expanded float32 observation. */
int mz_net_initial_frames(mz_net* net, int32_t batch, const uint8_t* frames, const float* plane_values,
                          void* hidden_out, const int32_t* dst_index, float* pi_probs, float* value,
                          mz_stream stream);

/* initial_inference of the B observations of a search WITH the root preparation fused into the policy epilogue
 * (mcts.py:355-367 in one go): the warp that computes tree t's softmax also draws its Dirichlet noise
 * (noise_mode 2: from the tree's MT19937 stream, exactly mz_dirichlet; 1: reads `noise`; 0: none), mixes, masks,
 * renormalises, expands the root and resets MinMaxStats -- bit-identical to mz_net_initial [+ mz_dirichlet] +
 * mz_search_reset, two launches fewer.  Pass `obs` (f32) or (`frames`, `plane_values`) as in mz_net_initial_frames, the
 * other NULL.  batch must equal the pool's num_trees; row i is tree i.  In mode 2 the drawn sample is also written to
 * `noise` (f64 [B, A]). */
int mz_net_initial_search(mz_net* net, mz_pool* pool, int32_t batch, const float* obs, const uint8_t* frames,
                          const float* plane_values, void* hidden_out, const int32_t* dst_index, float* pi_probs,
                          float* value, int32_t noise_mode, double* noise, double alpha, double eps,
                          const uint8_t* mask, const int32_t* players, mz_stream stream);

/* recurrent_inference (network.py:86-111): row i reads slot src_index[i] of
 * hidden_in, applies action[i], writes slot dst_index[i] of hidden_out.
 * pi_probs may be NULL: the search never uses it (mcts.py:386 passes the root
 * prior to every expansion), so the policy head is skipped. */
int mz_net_recurrent(mz_net* net, int32_t batch, const void* hidden_in, const int32_t* src_index,
                     const int32_t* action, void* hidden_out, const int32_t* dst_index,
                     float* reward, float* value, float* pi_probs, mz_stream stream);

/* All num_simulations simulations of the pool's trees -- select -> recurrent_inference -> expand + backup, the loop of
 * mcts.py:372-390 -- after the roots were prepared (mz_net_initial_search or mz_search_reset); leaves the pool as the
 * last mz_expand_backup would.  Either the per-simulation launch chain (mz_select, then S x (mz_net_recurrent,
 * mz_expand_backup[_select])), enqueued here so that a search is three C calls, or ONE launch of a persistent kernel
 * whose CTAs own their trees for the whole search:
 *   - MuZeroMLPNet, 5..32 actions, at most 32 trees per SM of the device: a CTA of 32 warps owns 32 trees; warp w runs
 *     tree w's backup and descent, then the CTA runs the tcgen05 chain on the 32 gathered rows (default where it
 *     applies);
 *   - MuZeroMLPNet, up to 12 actions, any batch: a CTA owns 128 trees, one thread per tree (only on request: measured
 *     slower than the chain).
 * Results are bit-identical in all three forms (tests/test_network_gpu.py::
 * test_one_launch_search_kernel_equals_the_launch_chain). */
int mz_search_run(mz_net* net, mz_pool* pool, mz_stream stream);

/* Which form mz_search_run uses (scheduling knob, no effect on results): -1 (default) one launch where that is the
 * faster form, 0 always the launch chain, 1 one launch wherever a kernel exists.  MZ_FUSED_SEARCH=0/1 in the
 * environment overrides it process-wide. */
int mz_net_set_fused_search(mz_net* net, int32_t enable);

/* Cap the grid of the net's persistent kernels (0 = one CTA per SM).  Two engines that are driven from two
 * streams (sub-batches of one search) can each be given half of the SMs so that their towers run side by side:
 * small batches are bound by the layer-to-layer tile dependencies, not by SM count. */
int mz_net_set_cta_limit(mz_net* net, int32_t max_ctas);

/* Per-kernel device timing of a net's launches (measurement aid for bench.py's roofline):
 * between begin and end every kernel the net launches EAGERLY is bracketed by CUDA events on
 * its stream; end synchronises and returns milliseconds and counts per kernel class
 * {0: conv3x3 (tcgen05; counted in conv LAYERS, one launch runs many), 1: heads, 2: observation packing,
 *  3: fused MLP, 4: conv3x3 again, counted in kernel LAUNCHES (same milliseconds as class 0)}. */
int mz_net_profile_begin(mz_net* net);
int mz_net_profile_end(mz_net* net, double* ms_by_class /* [5] */, int64_t* launches_by_class /* [5] */);

/* ------------------------------------------------------------------------
 * Callers of the search path, device-resident (SURVEY.md 8f: f-1, f-3)
 * ---------------------------------------------------------------------- */
/* Batched board-game environments: replace BoardGameEnv.reset / step / observation
 * (games/env.py:100-154, 242-271) with the last-move win check of games/gomoku.py:72-116 and
 * games/tictactoe.py:33-77.  num_actions = board_size^2 + 1 (the last action resigns).
 * Players: 1 = black (moves first), 2 = white.  Observations are written as float32
 * [G, 2*stack_history+1, N, N] from the side to move: [X_t, Y_t, X_t-1, Y_t-1, ..., colour]. */
typedef struct mz_env mz_env;
int mz_env_arena_bytes(int32_t games, int32_t board_size, int32_t stack_history, size_t* bytes);
int mz_env_create(int32_t games, int32_t board_size, int32_t stack_history, int32_t num_to_win, void* arena_dev,
                  size_t arena_bytes, mz_env** out);
int mz_env_destroy(mz_env* env);
/* views: 0 board i8[G,N*N], 1 history i8[G,2,stack,N*N], 2 mask u8[G,A], 3 player i32[G], 4 steps i32[G],
 *        5 winner i32[G], 6 done u8[G], 7 error i32[1] (bit 0: an illegal action was submitted)            */
int mz_env_view(mz_env* env, int32_t which, void** ptr, size_t* bytes);
/* reset the games with which[g] != 0 (all when NULL); obs may be NULL */
int mz_env_reset(mz_env* env, const uint8_t* which /* [G] */, float* obs, mz_stream stream);
/* one move per unfinished game: reward f64[G] and done u8[G] of THIS move, mover i32[G] = who played it,
 * obs = the next observation; finished games are left untouched (reward 0, done 1) */
int mz_env_step(mz_env* env, const int32_t* action /* [G] */, double* reward, uint8_t* done, int32_t* mover,
                float* obs, mz_stream stream);

/* Trajectories [G, max_len] (lengths i32[G]) -> training targets.  float64 in the reference's operation order:
 * targets and priorities are bit-identical to compute_n_step_target (pipeline.py:632-671; pow_table[i] =
 * discount**i evaluated by the caller with CPython floats, i = 0..td_steps), compute_mc_return_target
 * (pipeline.py:674-706) and priorities = |root_value - target| (pipeline.py:128,152).                       */
int mz_targets_nstep(int32_t games, int32_t max_len, const int32_t* lengths, const double* rewards,
                     const double* root_values, int32_t td_steps, const double* pow_table_dev, double* targets,
                     double* priorities /* nullable */, mz_stream stream);
int mz_targets_mc(int32_t games, int32_t max_len, const int32_t* lengths, const double* rewards,
                  const int32_t* player_ids, const double* root_values /* nullable with priorities */,
                  double* targets, double* priorities /* nullable */, mz_stream stream);
/* make_unroll_sequence (pipeline.py:709-767): per (game, step) the next unroll_steps actions / rewards / targets /
 * search policies with absorbing padding (action 0, reward 0, value 0, uniform policy).  Outputs are laid out
 * [G, max_len, unroll_steps(, A)]; valid u8[G, max_len] marks real steps.  Actions stay int32 (the reference's
 * int8 cast wraps for more than 127 actions, pipeline.py:753).                                               */
int mz_unroll_sequences(int32_t games, int32_t max_len, int32_t unroll_steps, int32_t num_actions,
                        const int32_t* lengths, const int32_t* actions, const double* rewards, const double* targets,
                        const float* pi /* [G,max_len,A] */, int32_t* out_action, float* out_reward, float* out_value,
                        float* out_pi, uint8_t* valid /* nullable */, mz_stream stream);

/* ---- device-resident replay (SURVEY.md 8 f-4; reference: muzero/replay.py:38-142) ---------------------------------
 * The caller (muzero_b200/replay.py) owns every buffer; rng_key u32[624] / rng_pos i32[1] are numpy legacy MT19937
 * states on the device (same format as MZ_VIEW_RNG_KEY / MZ_VIEW_RNG_POS).                                        */
/* PrioritizedReplay.sample with priority_exponent == 0 (replay.py:89-91): out_index[k] = trunc(size * u_k) for
 * consecutive doubles of the replay's OWN stream, out_weight[k] = 1.                                               */
int mz_replay_sample_uniform(int64_t size, int32_t batch, uint32_t* rng_key, int32_t* rng_pos, int64_t* out_index,
                             float* out_weight, mz_stream stream);
/* PrioritizedReplay.sample with priority_exponent != 0 (replay.py:93-100): float32 priorities ** exponent / their
 * float32 pairwise sum, np.random.choice(p=...) on the stream passed in (the reference draws from the GLOBAL numpy
 * stream here), importance weights ((1/size) / p[idx]) ** importance_exponent / max.  scratch_probs: f32[size + 1026],
 * scratch_cdf: f64[size + size / 2048 + 1].  Bit-exact for exponents 1, 2 and 0.5 (numpy's exact paths), powf
 * otherwise.  The float32 pairwise total is evaluated in parallel along numpy's own (fixed) recursion tree; the
 * float64 running sum by a parallel scan whenever no addition can round (every probability >= 2^-29), else in order. */
int mz_replay_sample_prioritized(int64_t size, int32_t batch, const float* priorities, float priority_exponent,
                                 float importance_exponent, uint32_t* rng_key, int32_t* rng_pos, float* scratch_probs,
                                 double* scratch_cdf, int64_t* out_index, float* out_weight, mz_stream stream);
/* PrioritizedReplay.add for n items at once (replay.py:70-79): storage[(start + i) % capacity] = rows[i]            */
int mz_replay_scatter(const void* rows, void* storage, int64_t n, int64_t row_bytes, int64_t start, int64_t capacity,
                      mz_stream stream);
/* PrioritizedReplay.get + the np.stack of sample (replay.py:81-83,102-104): rows[i] = storage[index[i]]            */
int mz_replay_gather(const void* storage, const int64_t* index, void* rows, int64_t n, int64_t row_bytes,
                     mz_stream stream);
/* PrioritizedReplay.update_priorities (replay.py:107-114): in order, later duplicates win                          */
int mz_replay_update_priorities(float* priorities, const int64_t* index, const float* values, int32_t n,
                                mz_stream stream);

/* ---- training step of the ResNet towers (SURVEY.md 8 f-2) -------------------------------------------------------
 * Replaces, for MuZeroBoardGameNet with num_planes == 128, what autograd + cuDNN execute for the towers inside
 * calc_loss (pipeline.py:541-612): network.represent / dynamics / prediction (network.py:353-395, 398-448, 451-500)
 * up to the tower outputs, forward and backward, in train mode (batch statistics, running-statistics update).
 * Heads, hidden-state normalisation, losses and the gradient-scale hooks stay with the caller (PyTorch autograd).
 * All tensors are float32 NCHW device buffers owned by the caller; the handle keeps fp16 / bf16 operand copies and the
 * saved activations in the caller's arena.  Towers: 0 representation, 1 dynamics, 2 prediction; `call` is the unroll
 * index (dynamics / prediction are evaluated unroll_steps times per step, each call keeps its own activations).      */
typedef struct mz_train mz_train;
typedef struct mz_train_config {
  int32_t in_channels;      /* observation planes (representation's first conv)                   */
  int32_t board_h, board_w;
  int32_t num_actions;      /* <= 128                                                              */
  int32_t num_planes;       /* 128                                                                 */
  int32_t num_res_blocks;
  int32_t batch;
  int32_t unroll_steps;
} mz_train_config;
int mz_train_arena_bytes(const mz_train_config* cfg, size_t* bytes);
int mz_train_create(const mz_train_config* cfg, void* arena_dev, size_t arena_bytes, mz_train** out);
int mz_train_destroy(mz_train* t);
/* 8 device pointers per 3x3 convolution, convolutions in module order (representation conv_block, its res_blocks'
 * conv_block1 / conv_block2 ..., dynamics conv_block, its res_blocks, prediction res_blocks):
 * conv weight f32 [128][ci][3][3], its gradient, BatchNorm weight, its gradient, BatchNorm bias, its gradient,
 * running_mean, running_var.  Gradients are ACCUMULATED (+=) like autograd's: BatchNorm parameters by the tower
 * backward calls, conv weights by mz_train_end_step.                                                              */
int mz_train_bind(mz_train* t, void* const* ptrs, int32_t n, mz_stream stream);
/* once per step before the first tower: re-pack the (updated) weights into operand layouts, clear the statistics   */
int mz_train_begin_step(mz_train* t, mz_stream stream);
/* x: observation [B,in_channels,H,W] (tower 0) or hidden state [B,128,H,W]; action i64 [B] (tower 1 only);
 * out: the tower's output [B,128,H,W] (after the last ReLU, before normalize_hidden_state / the heads)              */
int mz_train_tower_forward(mz_train* t, int32_t tower, int32_t call, const float* x, const int64_t* action, float* out,
                           mz_stream stream);
/* grad_out: dL/d out [B,128,H,W]; grad_in: dL/d x [B,128,H,W] (towers 1, 2; NULL for tower 0)                      */
int mz_train_tower_backward(mz_train* t, int32_t tower, int32_t call, const float* grad_out, float* grad_in,
                            mz_stream stream);
/* The K prediction-tower calls of an unroll (network.py:398-470 called from pipeline.py:580) do not depend on one
 * another, only on the dynamics chain: ncalls of them (calls call .. call + ncalls - 1) run as ONE launch chain over
 * the stacked inputs x [ncalls * B,128,H,W] (call-major).  Every call keeps its own train-mode BatchNorm batch
 * statistics, running statistics and parameter gradients receive the calls' contributions in call order: the same
 * arithmetic as ncalls separate calls.  *max_calls: how many calls may be stacked for this handle (1: none).
 * out_norm (optional): the output's per-position min-max normalisation over the channels (util.py:31-36) -- what the
 * representation and dynamics functions hand on (network.py:353-395, 440-470) -- written by the same pass; out may then
 * be NULL.  grad_norm (optional): dL/d out_norm, folded into the gradient with respect to the tower's output together
 * with grad_out (either may be NULL).                                                                               */
int mz_train_stacked_calls(mz_train* t, int32_t* max_calls);
int mz_train_tower_forward_calls(mz_train* t, int32_t tower, int32_t call, int32_t ncalls, const float* x, const int64_t* action,
                                 float* out, float* out_norm, mz_stream stream);
int mz_train_tower_backward_calls(mz_train* t, int32_t tower, int32_t call, int32_t ncalls, const float* grad_out,
                                  const float* grad_norm, float* grad_in, mz_stream stream);
/* the weight-gradient kernels of the tower backward calls run on a stream of the handle's own, beside the caller's:
 * make `stream` wait for them (capture-safe; mz_train_end_step does it itself)                                     */
int mz_train_join(mz_train* t, mz_stream stream);
/* after the last tower backward of a step: reduce the split-K partials into the conv weight gradients              */
int mz_train_end_step(mz_train* t, mz_stream stream);
/* parity tests: which = 0 tower input planes, 1 raw conv output of `layer`, 2 its activated output, 3 its
 * batch statistics f32 [128][2] (mean, 1/sqrt(var + eps)).  Planes are 16-bit [groups][plane_rows][8],
 * row P of the padded (H+1)x(W+1) grid at plane row front_rows + P.  A prediction call that ran stacked in this
 * step's forward returns the stacked buffers (plane_rows of unroll_steps calls, front_rows past the earlier calls
 * of its stack): the same values a separate forward of that call stores.                                           */
int mz_train_debug_view(mz_train* t, int32_t tower, int32_t call, int32_t layer, int32_t which, void** ptr, size_t* bytes,
                        int32_t* plane_rows, int32_t* front_rows);

/* ---- the learner's optimizer step (pipeline.py:246-252 optimizer.step(); torch.optim.Adam of */
/* gomoku/run_training.py:110) as ONE launch over all parameter tensors.  tensors: device array, one record per parameter
 * (parameter, gradient, exp_avg, exp_avg_sq: float32, the same dense layout, n elements) -- the optimizer's own state
 * tensors, updated in place; chunk_tensor / chunk_start: for every chunk of mz_adam_chunk_elements() elements the
 * index of its tensor and its first element; step: device scalar holding the ALREADY incremented step count (torch's
 * capturable per-parameter `step`); lr: device scalar.  L2 weight decay is added to the gradient, like torch.optim.Adam. */
typedef struct mz_adam_tensor {
  float* p;
  const float* g;
  float* m;
  float* v;
  int64_t n;
} mz_adam_tensor;
int mz_adam_chunk_elements(void);
int mz_adam_step(const mz_adam_tensor* tensors_dev, const int32_t* chunk_tensor_dev, const int64_t* chunk_start_dev, int32_t n_chunks,
                 const float* step_dev, const float* lr_dev, double beta1, double beta2, double eps, double weight_decay,
                 mz_stream stream);

/* ---- the heads' 1x1 convolutions (network.py:398-470, Conv2d(planes, 1 | 2, kernel_size=1, bias=False)) over stacked tower
 * outputs: x f32 [n][c][hw], w f32 [m][c] (m <= 4, c <= 256), y f32 [n][m][hw].  Backward: dx f32 [n][c][hw] (written),
 * dw f32 [m][c] (written: per-block partial sums in `scratch`, mz_head_conv_scratch_bytes, are added in a fixed order). */
int mz_head_conv_forward(const float* x, const float* w, float* y, int64_t n, int32_t c, int32_t hw, int32_t m, mz_stream stream);
size_t mz_head_conv_scratch_bytes(int64_t n, int32_t c, int32_t m);
int mz_head_conv_backward(const float* x, const float* w, const float* dy, float* dx, float* dw, void* scratch, int64_t n, int32_t c,
                          int32_t hw, int32_t m, mz_stream stream);

/* ---- the rest of a head (BatchNorm2d(mid) in train mode + ReLU + Flatten + Linear(mid * hw, o); network.py:398-470) over the
 * stacked 1x1-convolution outputs y f32 [calls * b][mid][hw] of `calls` forward calls, every call with its own batch statistics
 * (mid <= 4, mid * hw <= 1024, o <= 128).  forward: saved f32 [calls][mid][3] (mean, 1/sqrt(var + eps), var), z f32
 * [calls * b][mid * hw] (the activated features, kept for the backward pass), out f32 [calls * b][o]; running_mean / running_var
 * take the calls' updates in call order.  backward: dout f32 [calls * b][o] -> dy (like y), dgamma / dbeta [mid] (WRITTEN, not
 * accumulated) and dzr (like z) = dL/dz after the ReLU mask; the Linear layer's own gradients are the plain products
 * dout^T z and sum(dout) (left to the caller's GEMM); sums f32 [calls][mid][2] is scratch.                                 */
int mz_head_tail_forward(const float* y, const float* gamma, const float* beta, const float* w, const float* bias, float* running_mean,
                         float* running_var, float* saved, float* z, float* out, int32_t calls, int32_t b, int32_t mid, int32_t hw, int32_t o,
                         float eps, float momentum, mz_stream stream);
int mz_head_tail_backward(const float* dout, const float* y, const float* gamma, const float* w, const float* saved, const float* z, float* dzr,
                          float* sums, float* dy, float* dgamma, float* dbeta, int32_t calls, int32_t b, int32_t mid, int32_t hw, int32_t o,
                          mz_stream stream);

/* number of kernels the library has launched since load (bench's gpu_launches) */
uint64_t mz_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* MUZERO_B200_H */
