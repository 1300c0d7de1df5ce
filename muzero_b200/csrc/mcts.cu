// Batched MCTS over a GPU-resident struct-of-arrays node pool: one warp per tree.
//
// Bit-exactness contract (SURVEY.md §2.1, Appendix A): every float64 operation
// of the reference's CPython arithmetic is issued as a separate IEEE
// round-to-nearest instruction (__dadd_rn/__dmul_rn/__ddiv_rn — never
// contracted into FMA), float32 score arithmetic uses __fmul_rn/__fadd_rn, the
// pb_c term comes from a host table computed with CPython math, tie-breaks
// consume numpy's legacy MT19937 stream with numpy's masked rejection.
#include "common.cuh"
#include "rng.cuh"
#include "pool.cuh"
#include "tree_thread.cuh"
#include "tree_warp.cuh"
#include <vector>

namespace mz {

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
constexpr int kTreesPerBlock = 4;  // 128 threads

// ---------------------------------------------------------------------------
// mz_rng_seed: init_genrand(seed) per tree
// ---------------------------------------------------------------------------
__global__ void rng_seed_kernel(PoolDev p, const uint32_t* __restrict__ seeds) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= p.B) return;
  uint32_t* key = p.rng_key + (size_t)t * 624;
  uint32_t s = seeds[t];
  for (int i = 0; i < 624; ++i) {
    key[i] = s;
    s = 1812433253u * (s ^ (s >> 30)) + (uint32_t)i + 1u;
  }
  p.rng_pos[t] = 624;
}

// ---------------------------------------------------------------------------
// mz_search_reset
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kTreesPerBlock * 32)
reset_kernel(PoolDev p, const float* __restrict__ pi, const double* __restrict__ noise, double eps,
             float one_minus_eps_f32, const uint8_t* __restrict__ mask, const int32_t* __restrict__ players,
             const float* __restrict__ root_reward) {
  const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (t >= p.B) return;
  const size_t o = (size_t)t * p.A;
  root_setup_tree(p, t, lane, pi + o, noise ? noise + o : nullptr, eps, one_minus_eps_f32, mask ? mask + o : nullptr,
                  players ? players + 2 * t : nullptr, root_reward ? root_reward + t : nullptr);
}

// ---------------------------------------------------------------------------
// mz_select
// ---------------------------------------------------------------------------
extern __shared__ __align__(16) unsigned char smem_raw[];

template <int NCH>
__global__ void __launch_bounds__(kTreesPerBlock * 32)
select_kernel(PoolDev p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t = blockIdx.x * kTreesPerBlock + warp;
  double* sT = reinterpret_cast<double*>(smem_raw);                       // [S+2] pb_c table
  // RN(1/n): read through L1 (__ldg), not staged -- 3.2 KB of shared memory per CTA would no longer fit beside the
  // persistent conv kernel of the other sub-batch (228 KB - 223.75 KB - two 1 KB reservations)
  const double* sR = p.T + (p.S + 2);
  float* sc = reinterpret_cast<float*>(sT + (p.S + 2)) + (size_t)warp * ((p.A + 3) & ~3);
  __shared__ unsigned long long s_stats[4];
  pdl_trigger();
  if (threadIdx.x < 4) s_stats[threadIdx.x] = 0;
  for (int i = threadIdx.x; i < p.S + 2; i += blockDim.x) sT[i] = p.T[i];
  __syncthreads();
  pdl_wait();
  if (t < p.B) select_tree<NCH>(p, t, lane, sT, sR, sc, s_stats);
  flush_stats(p, s_stats);
}

// ---------------------------------------------------------------------------
// mz_expand_backup
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kTreesPerBlock * 32)
expand_backup_kernel(PoolDev p, const float* __restrict__ reward_in, const float* __restrict__ value_in) {
  pdl_trigger();
  pdl_wait();
  const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (t >= p.B) return;
  expand_backup_tree(p, t, lane, reward_in[t], value_in[t]);
}

// expand+backup of simulation s and select of simulation s+1 in ONE launch: both are warp-per-tree and touch only
// their own tree, so the second half simply runs on the statistics the first half just wrote (ordered by
// __syncwarp).  Saves a launch and a cold pass over the path per simulation -- what the MLP configurations, whose
// whole simulation lasts ~50 us, are bound by.
template <int NCH>
__global__ void __launch_bounds__(kTreesPerBlock * 32)
backup_select_kernel(PoolDev p, const float* __restrict__ reward_in, const float* __restrict__ value_in) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t = blockIdx.x * kTreesPerBlock + warp;
  double* sT = reinterpret_cast<double*>(smem_raw);
  const double* sR = p.T + (p.S + 2);
  float* sc = reinterpret_cast<float*>(sT + (p.S + 2)) + (size_t)warp * ((p.A + 3) & ~3);
  __shared__ unsigned long long s_stats[4];
  pdl_trigger();
  if (threadIdx.x < 4) s_stats[threadIdx.x] = 0;
  for (int i = threadIdx.x; i < p.S + 2; i += blockDim.x) sT[i] = p.T[i];
  __syncthreads();
  pdl_wait();
  if (t < p.B) {
    if (p.timing && threadIdx.x == 0) {
      const unsigned long long t0 = globaltimer_ns();
      atomicMin(p.stats + 4, t0);
      atomicMax(p.stats + 5, t0);
    }
    expand_backup_tree(p, t, lane, reward_in[t], value_in[t]);
    __syncwarp();
    select_tree<NCH>(p, t, lane, sT, sR, sc, s_stats);
    if (p.timing && lane == 0) atomicMax(p.stats + 6, globaltimer_ns());
  }
  flush_stats(p, s_stats);
}

// ---------------------------------------------------------------------------
// Tiny action spaces (A <= kThreadA: CartPole 2, LunarLander 4): ONE THREAD per tree.  A warp per tree keeps 2 of 32
// lanes busy there and needs as many warps as trees (16 384 for config 1: two waves of latency-bound warps); a thread
// per tree needs 512.  Same arithmetic, instruction for instruction (puct via the child_Q cache, div_by_count,
// child_q, the backup recurrence), same MT19937 stream (sequential twist), same memory -- only the work split differs,
// and the lock-step / golden tests with A = 2 and A = 4 run through these kernels.
// ---------------------------------------------------------------------------
constexpr int kThreadA = 4;
constexpr int kThreadBlock = 64;

// mode: 1 select, 2 expand+backup, 3 expand+backup then select
__global__ void __launch_bounds__(kThreadBlock)
tree_thread_kernel(PoolDev p, const float* __restrict__ reward_in, const float* __restrict__ value_in, int mode) {
  double* sT = reinterpret_cast<double*>(smem_raw);          // pb_c table, then RN(1/n): [2 * (S + 2)]
  const double* sR = sT + (p.S + 2);
  pdl_trigger();
  for (int i = threadIdx.x; i < 2 * (p.S + 2); i += blockDim.x) sT[i] = p.T[i];
  __syncthreads();
  pdl_wait();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned member = __ballot_sync(kFull, t < p.B);
  if (t >= p.B) return;
  if (mode & 2) expand_backup_tree_thread(p, t, reward_in[t], value_in[t]);
  if (mode & 1) {
    TreeThreadStats st;
    select_tree_thread<kThreadA>(p, t, sT, sR, st);
    // statistics: one atomic per warp and counter (`member` = the lanes of this warp that own a tree)
    __syncwarp(member);
    const unsigned d = __reduce_add_sync(member, st.depth);
    const unsigned dr = __reduce_add_sync(member, st.draws);
    const unsigned tw = __reduce_add_sync(member, st.twists);
    if ((threadIdx.x & 31) == 0) {
      atomicAdd(p.stats + 0, (unsigned long long)d);
      atomicAdd(p.stats + 1, (unsigned long long)__popc(member));
      if (dr) atomicAdd(p.stats + 2, (unsigned long long)dr);
      if (tw) atomicAdd(p.stats + 3, (unsigned long long)tw);
    }
  }
}

// The same, CONFINED to a few SMs: `gridDim.x` CTAs of 32 warps pull trees off a counter.  For PipelinedSearchPlan,
// where the tree kernels of one sub-batch are meant to run in the shadow of the other sub-batch's conv tower.
// Spread over all SMs (one small CTA beside every persistent conv CTA) they do start there, but a latency-bound warp
// beside the tower's warps runs 2-10x slower per instruction (FP64 9.5x) AND slows the tower's MMA issue by ~25 %
// (tools/coresident_probe.py) -- worse than not overlapping at all.  So the tower is launched on
// num_sms - gridDim.x SMs and this kernel asks for more shared memory than is left beside a conv CTA: its CTAs can
// only land on the SMs the tower leaves free, and at most gridDim.x SMs are ever withheld from the (cooperative)
// tower launch of the other sub-batch.
constexpr int kConfinedThreads = 1024;
constexpr int kConfinedSmem = 40 * 1024;
template <int NCH>
__global__ void __launch_bounds__(kConfinedThreads)
backup_select_confined_kernel(PoolDev p, const float* __restrict__ reward_in, const float* __restrict__ value_in) {
  const int lane = threadIdx.x & 31;
  double* sT = reinterpret_cast<double*>(smem_raw);
  const double* sR = p.T + (p.S + 2);
  __shared__ unsigned long long s_stats[4];
  pdl_trigger();
  if (threadIdx.x < 4) s_stats[threadIdx.x] = 0;
  for (int i = threadIdx.x; i < p.S + 2; i += blockDim.x) sT[i] = p.T[i];
  __syncthreads();
  pdl_wait();
  while (true) {
    unsigned t = 0;
    if (lane == 0) t = atomicAdd(p.work, 1u);
    t = __shfl_sync(kFull, t, 0);
    if (t >= (unsigned)p.B) break;
    expand_backup_tree(p, (int)t, lane, reward_in[t], value_in[t]);
    __syncwarp();
    select_tree<NCH>(p, (int)t, lane, sT, sR, nullptr, s_stats);
  }
  flush_stats(p, s_stats);
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(p.work + 1, 1u) == gridDim.x - 1) {   // last CTA out: every CTA has left its loop
      p.work[0] = 0;
      p.work[1] = 0;
      __threadfence();
    }
  }
}

// ---------------------------------------------------------------------------
// mz_root_policy
// ---------------------------------------------------------------------------
// v ** e for integral e in [1,5], correctly rounded (what a faithful pow returns)
__device__ double pow_int_exact(uint32_t v, int e) {
  unsigned __int128 pw = 1;
  for (int i = 0; i < e; ++i) pw *= (unsigned __int128)v;
  const unsigned long long hi64 = (unsigned long long)(pw >> 64), lo64 = (unsigned long long)pw;
  if (hi64 == 0 && lo64 < (1ULL << 53)) return (double)lo64;
  const int msb = hi64 ? 127 - __clzll((long long)hi64) : 63 - __clzll((long long)lo64);
  const int shift = msb - 52;
  unsigned long long mant = (unsigned long long)(pw >> shift);
  const unsigned __int128 rem = pw & ((((unsigned __int128)1) << shift) - 1);
  const unsigned __int128 half = ((unsigned __int128)1) << (shift - 1);
  if (rem > half || (rem == half && (mant & 1ULL))) ++mant;
  return ldexp((double)mant, shift);
}

__global__ void __launch_bounds__(kTreesPerBlock * 32)
root_policy_kernel(PoolDev p, const uint8_t* __restrict__ mask, const double* __restrict__ temperature,
                   int deterministic, int32_t* __restrict__ action, double* __restrict__ pi_out,
                   double* __restrict__ root_value, int32_t* __restrict__ visits_out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t = blockIdx.x * kTreesPerBlock + warp;
  if (t >= p.B) return;
  const int A = p.A;
  double* x = reinterpret_cast<double*>(smem_raw) + (size_t)warp * A;
  const HotEdge* row = p.hot + (size_t)t * p.max_nodes * A;
  const double T = temperature[t];

  int best_v = -1, best_a = 0;
  long long isum = 0;
  double e = 1.0;
  bool e_int = true;
  if (T > 0.0) {
    e = __ddiv_rn(1.0, T);
    e = (e < 5.0) ? e : 5.0;     // min(5.0, 1/T)
    e = (1.0 > e) ? 1.0 : e;     // max(1.0, .)
    e_int = (e == floor(e));
  }
  for (int a0 = 0; a0 < A; a0 += 32) {
    const int a = a0 + lane;
    int v = -1;
    if (a < A) {
      v = (int)(row[a].x & 0xffffu);
      if (mask != nullptr && mask[(size_t)t * A + a] == 0) v = 0;
      if (visits_out) visits_out[(size_t)t * A + a] = v;
      x[a] = (T > 0.0) ? (e_int ? pow_int_exact((uint32_t)v, (int)e) : pow((double)v, e)) : (double)v;
      isum += v;
    }
    // first maximum of the visit counts (np.argmax)
    int bv = v, ba = a;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const int ov = __shfl_xor_sync(kFull, bv, o), oa = __shfl_xor_sync(kFull, ba, o);
      if (ov > bv || (ov == bv && oa < ba)) { bv = ov; ba = oa; }
    }
    if (bv > best_v) { best_v = bv; best_a = ba; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) isum += __shfl_xor_sync(kFull, isum, o);
  __syncwarp();
  const double s = (T > 0.0) ? pairwise_sum<double>(x, A) : (double)isum;
  __syncwarp();
  bool has_nan = false;
  for (int a = lane; a < A; a += 32) {
    const double pr = __ddiv_rn(x[a], s);
    x[a] = pr;
    pi_out[(size_t)t * A + a] = pr;
    has_nan |= (pr != pr);
  }
  has_nan = __any_sync(kFull, has_nan);
  __syncwarp();
  int act = best_a;
  if (!deterministic) {
    if (has_nan) {
      if (lane == 0) atomicOr(p.error, MZ_DEVERR_NAN_POLICY);
      act = -1;
    } else {
      // np.random.choice(A, p=pi): cdf = cumsum(p); cdf /= cdf[-1]; searchsorted(cdf, u, 'right')
      WarpRng rng;
      rng.load(p.rng_key + (size_t)t * 624, p.rng_pos + t, lane);
      const double u = rng.next_double();
      rng.store(p.rng_pos + t);
      double acc = 0.0;
      for (int a = 0; a < A; ++a) acc = __dadd_rn(acc, x[a]);
      const double last = acc;
      acc = 0.0;
      int idx = 0;
      for (int a = 0; a < A; ++a) {
        acc = __dadd_rn(acc, x[a]);
        if (__ddiv_rn(acc, last) <= u) idx = a + 1; else break;
      }
      act = idx;
    }
  }
  if (lane == 0) {
    action[t] = act;
    const int rn = p.rootN[t];
    root_value[t] = rn > 0 ? __ddiv_rn(p.rootW[t], (double)rn) : 0.0;
  }
}

// ---------------------------------------------------------------------------
// mz_dirichlet: numpy legacy_standard_gamma / dirichlet on the tree's stream
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kTreesPerBlock * 32)
dirichlet_kernel(PoolDev p, double alpha, double* __restrict__ out) {
  const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (t >= p.B) return;
  dirichlet_tree(p, t, lane, alpha, out + (size_t)t * p.A);
}

}  // namespace mz

// ===========================================================================
// host side of the C ABI
// ===========================================================================
using namespace mz;

namespace {

struct Carve {
  size_t off = 0;
  size_t take(size_t bytes) {
    const size_t o = off;
    off = align_up(off + bytes, 256);
    return o;
  }
};

void layout(const mz_pool_config& c, size_t* offs, size_t* sizes, size_t* extra_offs, size_t* total) {
  const size_t B = c.num_trees, A = c.num_actions, n = (size_t)c.num_simulations + 1;
  Carve cv;
  auto put = [&](int which, size_t bytes) { offs[which] = cv.take(bytes); sizes[which] = bytes; };
  put(MZ_VIEW_EDGES, B * n * A * sizeof(HotEdge));
  put(MZ_VIEW_PRIOR, B * A * 8);
  put(MZ_VIEW_ROOT_W, B * 8);
  put(MZ_VIEW_ROOT_N, B * 4);
  put(MZ_VIEW_MINMAX, B * 16);
  put(MZ_VIEW_COUNT, B * 4);
  put(MZ_VIEW_LEAF_PARENT, B * 4);
  put(MZ_VIEW_LEAF_ACTION, B * 4);
  put(MZ_VIEW_LEAF_DEPTH, B * 4);
  put(MZ_VIEW_SRC_SLOT, B * 4);
  put(MZ_VIEW_DST_SLOT, B * 4);
  put(MZ_VIEW_PATH, B * n * 4);
  put(MZ_VIEW_NODE_PARENT, B * n * 4);
  put(MZ_VIEW_NODE_MOVE, B * n * 4);
  put(MZ_VIEW_NODE_VALUE, B * n * 4);
  put(MZ_VIEW_RNG_KEY, B * 624 * 4);
  put(MZ_VIEW_RNG_POS, B * 4);
  put(MZ_VIEW_HIDDEN, B * n * (size_t)c.hidden_bytes);
  put(MZ_VIEW_REWARD, B * 4);
  put(MZ_VIEW_VALUE, B * 4);
  put(MZ_VIEW_ERROR, 4);
  put(MZ_VIEW_STATS, 8 * 8);
  put(MZ_VIEW_EDGE_W, B * n * A * 8);
  put(MZ_VIEW_EDGE_REWARD, B * n * A * 4);
  extra_offs[0] = cv.take((size_t)(c.num_simulations + 2) * 16); // pb_c table, then RN(1/n)
  extra_offs[1] = cv.take(B);                                     // same_player
  extra_offs[2] = cv.take(B * 8);                                 // root_reward
  extra_offs[3] = cv.take(B);                                     // f32_prior
  extra_offs[4] = cv.take(16);                                    // work counters of the confined tree kernel
  *total = cv.off;
}

int check_cfg(const mz_pool_config* c) {
  MZ_CHECK_ARG(c != nullptr, "config is NULL");
  MZ_CHECK_ARG(c->num_trees > 0, "num_trees must be positive, got %d", c->num_trees);
  MZ_CHECK_ARG(c->num_actions > 0 && c->num_actions <= 65535, "num_actions out of range: %d", c->num_actions);
  MZ_CHECK_ARG(c->num_simulations > 0 && c->num_simulations <= 65534,
               "num_simulations must be in [1, 65534], got %d", c->num_simulations);
  MZ_CHECK_ARG(c->hidden_bytes >= 0 && c->hidden_bytes % 16 == 0, "hidden_bytes must be a multiple of 16, got %d",
               c->hidden_bytes);
  MZ_CHECK_ARG((size_t)c->num_trees * (c->num_simulations + 1) < (size_t)1 << 31, "too many node slots");
  MZ_CHECK_ARG((size_t)(c->num_simulations + 1) * c->num_actions < (size_t)1 << 32, "tree too large for u32 edge ids");
  MZ_CHECK_ARG(c->num_simulations <= 4000, "num_simulations > 4000 not supported (pb_c table lives in shared memory)");
  if (c->is_board_game)  // mcts.py:349-350
    MZ_CHECK_ARG(c->discount == 1.0, "board games require discount == 1.0 (mcts.py:349), got %g", c->discount);
  return MZ_OK;
}

}  // namespace
namespace mz {
PoolDev pool_dev(const mz_pool* h) {
  PoolDev d;
  d.B = h->B; d.A = h->A; d.S = h->S; d.max_nodes = h->max_nodes;
  d.board = h->cfg.is_board_game;
  d.discount = h->cfg.discount;
  d.dp = h->cfg.discount * (h->cfg.is_board_game ? -1.0 : 1.0);   // mcts.py:169-174: discount * p
  d.hot = (HotEdge*)h->view_ptr[MZ_VIEW_EDGES];
  d.ew = (double*)h->view_ptr[MZ_VIEW_EDGE_W];
  d.er = (float*)h->view_ptr[MZ_VIEW_EDGE_REWARD];
  d.prior = (double*)h->view_ptr[MZ_VIEW_PRIOR];
  d.rootW = (double*)h->view_ptr[MZ_VIEW_ROOT_W];
  d.rootN = (int*)h->view_ptr[MZ_VIEW_ROOT_N];
  d.minmax = (double*)h->view_ptr[MZ_VIEW_MINMAX];
  d.count = (int*)h->view_ptr[MZ_VIEW_COUNT];
  d.leaf_parent = (int*)h->view_ptr[MZ_VIEW_LEAF_PARENT];
  d.leaf_action = (int*)h->view_ptr[MZ_VIEW_LEAF_ACTION];
  d.leaf_depth = (int*)h->view_ptr[MZ_VIEW_LEAF_DEPTH];
  d.src_slot = (int*)h->view_ptr[MZ_VIEW_SRC_SLOT];
  d.dst_slot = (int*)h->view_ptr[MZ_VIEW_DST_SLOT];
  d.path = (uint32_t*)h->view_ptr[MZ_VIEW_PATH];
  d.node_parent = (int*)h->view_ptr[MZ_VIEW_NODE_PARENT];
  d.node_move = (int*)h->view_ptr[MZ_VIEW_NODE_MOVE];
  d.node_value = (float*)h->view_ptr[MZ_VIEW_NODE_VALUE];
  d.rng_key = (uint32_t*)h->view_ptr[MZ_VIEW_RNG_KEY];
  d.rng_pos = (int*)h->view_ptr[MZ_VIEW_RNG_POS];
  d.reward = (float*)h->view_ptr[MZ_VIEW_REWARD];
  d.value = (float*)h->view_ptr[MZ_VIEW_VALUE];
  d.error = (int*)h->view_ptr[MZ_VIEW_ERROR];
  d.stats = (unsigned long long*)h->view_ptr[MZ_VIEW_STATS];
  d.T = h->pb_c_table;
  d.same_player = h->same_player;
  d.root_reward = h->root_reward;
  d.f32_prior = h->f32_prior;
  d.work = h->work;
  d.bound_min = h->cfg.bound_min; d.bound_max = h->cfg.bound_max;
  d.has_bounds = h->cfg.has_known_bounds;
  static const int timing = getenv("MZ_TREE_TIMING") != nullptr;
  d.timing = timing;
  return d;
}
}  // namespace mz
namespace {
inline PoolDev dev_of(const mz_pool* h) { return pool_dev(h); }

// early start of the tree kernels only for batches whose kernels leave SMs free (see launch_pdl in mlp.cu)
inline bool pdl_ok(const mz_pool* pool) { return pool->B <= 8192; }
inline int tree_blocks(int B) { return (B + kTreesPerBlock - 1) / kTreesPerBlock; }
// thread-per-tree kernels: tiny action spaces and enough trees to fill warps (MZ_TREE_THREAD=0/1 overrides)
inline bool use_thread_kernels(const mz_pool* pool) {
  static const int force = getenv("MZ_TREE_THREAD") ? atoi(getenv("MZ_TREE_THREAD")) : -1;
  if (pool->A > kThreadA) return false;
  if (force >= 0) return force != 0;
  return pool->B >= 512;
}

}  // namespace

extern "C" int mz_pool_arena_bytes(const mz_pool_config* cfg, size_t* bytes) {
  int rc = check_cfg(cfg);
  if (rc) return rc;
  MZ_CHECK_ARG(bytes != nullptr, "bytes is NULL");
  size_t offs[MZ_VIEW__COUNT], sizes[MZ_VIEW__COUNT], extra[5];
  layout(*cfg, offs, sizes, extra, bytes);
  return MZ_OK;
}

extern "C" int mz_pool_create(const mz_pool_config* cfg, const double* pb_c_table_host, void* arena_dev,
                              size_t arena_bytes, mz_pool** out) {
  int rc = check_cfg(cfg);
  if (rc) return rc;
  MZ_CHECK_ARG(pb_c_table_host && arena_dev && out, "NULL argument");
  MZ_CHECK_ARG(((uintptr_t)arena_dev & 255) == 0, "arena must be 256-byte aligned");
  size_t offs[MZ_VIEW__COUNT], sizes[MZ_VIEW__COUNT], extra[5], total;
  layout(*cfg, offs, sizes, extra, &total);
  {
    // The per-simulation tree kernels must be able to share an SM with the persistent conv kernel of ANOTHER
    // sub-batch (PipelinedSearchPlan), which runs with the maximum shared-memory carve-out; a kernel that
    // prefers a different L1/shared split cannot be co-resident with it.
    const int mx = (int)cudaSharedmemCarveoutMaxShared;
    cudaFuncSetAttribute(select_kernel<0>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(select_kernel<1>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(select_kernel<2>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(select_kernel<3>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(select_kernel<4>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(expand_backup_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(backup_select_kernel<0>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(backup_select_kernel<1>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(backup_select_kernel<2>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(backup_select_kernel<3>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(backup_select_kernel<4>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(backup_select_confined_kernel<1>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(backup_select_confined_kernel<2>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(backup_select_confined_kernel<3>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaFuncSetAttribute(backup_select_confined_kernel<4>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
    cudaGetLastError();
  }
  if (arena_bytes < total) {
    set_error("arena too small: %zu < %zu", arena_bytes, total);
    return MZ_ENOMEM;
  }
  mz_pool* h = new mz_pool();
  h->cfg = *cfg;
  h->B = cfg->num_trees; h->A = cfg->num_actions; h->S = cfg->num_simulations; h->max_nodes = h->S + 1;
  h->arena = arena_dev; h->arena_bytes = arena_bytes;
  char* base = (char*)arena_dev;
  for (int i = 0; i < MZ_VIEW__COUNT; ++i) { h->view_ptr[i] = base + offs[i]; h->view_bytes[i] = sizes[i]; }
  h->pb_c_table = (double*)(base + extra[0]);
  h->same_player = (uint8_t*)(base + extra[1]);
  h->root_reward = (double*)(base + extra[2]);
  h->f32_prior = (uint8_t*)(base + extra[3]);
  h->work = (unsigned*)(base + extra[4]);
  h->tree_ctas = 0;
  h->selected = 0;
  cudaError_t e = cudaMemcpy(h->pb_c_table, pb_c_table_host, (size_t)(h->S + 2) * 8, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    // correctly rounded reciprocals of the visit counts (host IEEE division) for div_by_count
    std::vector<double> rcp((size_t)h->S + 2);
    for (int i = 0; i < h->S + 2; ++i) rcp[i] = 1.0 / (double)(i > 0 ? i : 1);
    e = cudaMemcpy(h->pb_c_table + (h->S + 2), rcp.data(), rcp.size() * 8, cudaMemcpyHostToDevice);
  }
  if (e == cudaSuccess) e = cudaMemset(h->work, 0, 16);
  if (e == cudaSuccess) e = cudaMemset(h->view_ptr[MZ_VIEW_EDGE_W], 0, sizes[MZ_VIEW_EDGE_W]);
  if (e == cudaSuccess) e = cudaMemset(h->view_ptr[MZ_VIEW_EDGE_REWARD], 0, sizes[MZ_VIEW_EDGE_REWARD]);
  if (e == cudaSuccess) e = cudaMemset(h->view_ptr[MZ_VIEW_ERROR], 0, 4);
  if (e == cudaSuccess) e = cudaMemset(h->view_ptr[MZ_VIEW_STATS], 0, 64);
  if (e == cudaSuccess) e = cudaMemset(h->view_ptr[MZ_VIEW_LEAF_DEPTH], 0, sizes[MZ_VIEW_LEAF_DEPTH]);
  if (e == cudaSuccess) e = cudaMemset(h->view_ptr[MZ_VIEW_RNG_KEY], 0, sizes[MZ_VIEW_RNG_KEY]);
  if (e == cudaSuccess) e = cudaMemset(h->view_ptr[MZ_VIEW_RNG_POS], 0, sizes[MZ_VIEW_RNG_POS]);
  if (e != cudaSuccess) {
    set_error("pool initialisation failed: %s", cudaGetErrorString(e));
    delete h;
    return MZ_ECUDA;
  }
  *out = h;
  return MZ_OK;
}

extern "C" int mz_pool_set_tree_ctas(mz_pool* pool, int num_ctas) {
  MZ_CHECK_ARG(pool, "NULL argument");
  MZ_CHECK_ARG(num_ctas >= 0 && num_ctas <= 64, "num_ctas out of range: %d", num_ctas);
  MZ_CHECK_ARG((size_t)(pool->S + 2) * 8 <= (size_t)kConfinedSmem, "pb_c table does not fit the confined kernel");
  pool->tree_ctas = num_ctas;
  return MZ_OK;
}

extern "C" int mz_pool_destroy(mz_pool* pool) {
  delete pool;
  return MZ_OK;
}

extern "C" int mz_pool_view(mz_pool* pool, int which, void** dev_ptr, size_t* bytes) {
  MZ_CHECK_ARG(pool && dev_ptr && bytes, "NULL argument");
  MZ_CHECK_ARG(which >= 0 && which < MZ_VIEW__COUNT, "unknown view %d", which);
  *dev_ptr = pool->view_ptr[which];
  *bytes = pool->view_bytes[which];
  return MZ_OK;
}

extern "C" int mz_rng_seed(mz_pool* pool, const uint32_t* seeds_dev, mz_stream stream) {
  MZ_CHECK_ARG(pool && seeds_dev, "NULL argument");
  rng_seed_kernel<<<(pool->B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(dev_of(pool), seeds_dev);
  MZ_LAUNCH_CHECK("rng_seed_kernel");
  return MZ_OK;
}

extern "C" int mz_dirichlet(mz_pool* pool, double alpha, double* noise_out_dev, mz_stream stream) {
  MZ_CHECK_ARG(pool && noise_out_dev, "NULL argument");
  // mcts.py:241-242 restricts alpha to [0, 1]; numpy rejects alpha <= 0
  MZ_CHECK_ARG(alpha > 0.0 && alpha <= 1.0, "Expect `alpha` to be a float in the range (0.0, 1.0], got %g", alpha);
  dirichlet_kernel<<<tree_blocks(pool->B), kTreesPerBlock * 32, 0, (cudaStream_t)stream>>>(dev_of(pool), alpha,
                                                                                          noise_out_dev);
  MZ_LAUNCH_CHECK("dirichlet_kernel");
  return MZ_OK;
}

extern "C" int mz_search_reset(mz_pool* pool, const float* pi_probs, const double* noise, double eps,
                               const uint8_t* mask, const int32_t* players, const float* root_reward,
                               mz_stream stream) {
  MZ_CHECK_ARG(pool && pi_probs, "NULL argument");
  // mcts.py:239-240
  MZ_CHECK_ARG(eps >= 0.0 && eps <= 1.0, "Expect `eps` to be a float in the range [0.0, 1.0], got %g", eps);
  const float ome = (float)(1.0 - eps);
  reset_kernel<<<tree_blocks(pool->B), kTreesPerBlock * 32, 0, (cudaStream_t)stream>>>(
      dev_of(pool), pi_probs, noise, eps, ome, mask, players, root_reward);
  MZ_LAUNCH_CHECK("reset_kernel");
  pool->selected = 0;
  return MZ_OK;
}

extern "C" int mz_select(mz_pool* pool, mz_stream stream) {
  MZ_CHECK_ARG(pool, "NULL argument");
  const int A = pool->A;
  const size_t smem = (size_t)(pool->S + 2) * 8 + (A > 128 ? (size_t)kTreesPerBlock * ((A + 3) & ~3) * sizeof(float) : 0);
  const dim3 grid(tree_blocks(pool->B)), block(kTreesPerBlock * 32);
  cudaStream_t st = (cudaStream_t)stream;
  const PoolDev d = dev_of(pool);
  if (use_thread_kernels(pool)) {
    launch_pdl(pdl_ok(pool), tree_thread_kernel, dim3((pool->B + kThreadBlock - 1) / kThreadBlock), dim3(kThreadBlock), (size_t)(pool->S + 2) * 16, st, d, nullptr, nullptr, 1);
    MZ_LAUNCH_CHECK("tree_thread_kernel");
    pool->selected = 1;
    return MZ_OK;
  }
  if (A <= 32) launch_pdl(pdl_ok(pool), select_kernel<1>, grid, block, smem, st, d);
  else if (A <= 64) launch_pdl(pdl_ok(pool), select_kernel<2>, grid, block, smem, st, d);
  else if (A <= 96) launch_pdl(pdl_ok(pool), select_kernel<3>, grid, block, smem, st, d);
  else if (A <= 128) launch_pdl(pdl_ok(pool), select_kernel<4>, grid, block, smem, st, d);
  else launch_pdl(pdl_ok(pool), select_kernel<0>, grid, block, smem, st, d);
  MZ_LAUNCH_CHECK("select_kernel");
  pool->selected = 1;
  return MZ_OK;
}

extern "C" int mz_expand_backup_select(mz_pool* pool, const float* reward, const float* value, mz_stream stream) {
  MZ_CHECK_ARG(pool, "NULL argument");
  if (!pool->selected) {
    set_error("mz_expand_backup_select called without a preceding mz_select");
    return MZ_ESTATE;
  }
  const int A = pool->A;
  const size_t smem = (size_t)(pool->S + 2) * 8 + (A > 128 ? (size_t)kTreesPerBlock * ((A + 3) & ~3) * sizeof(float) : 0);
  const dim3 grid(tree_blocks(pool->B)), block(kTreesPerBlock * 32);
  cudaStream_t st = (cudaStream_t)stream;
  const PoolDev d = dev_of(pool);
  const float* r = reward ? reward : d.reward;
  const float* v = value ? value : d.value;
  if (use_thread_kernels(pool)) {
    launch_pdl(pdl_ok(pool), tree_thread_kernel, dim3((pool->B + kThreadBlock - 1) / kThreadBlock), dim3(kThreadBlock), (size_t)(pool->S + 2) * 16, st, d, r, v, 3);
    MZ_LAUNCH_CHECK("tree_thread_kernel");
    pool->selected = 1;
    return MZ_OK;
  }
  if (pool->tree_ctas > 0 && A <= 128) {
    const dim3 cgrid(pool->tree_ctas), cblock(kConfinedThreads);
    if (A <= 32) launch_pdl_pairs(pdl_ok(pool), backup_select_confined_kernel<1>, cgrid, cblock, (size_t)kConfinedSmem, st, d, r, v);
    else if (A <= 64) launch_pdl_pairs(pdl_ok(pool), backup_select_confined_kernel<2>, cgrid, cblock, (size_t)kConfinedSmem, st, d, r, v);
    else if (A <= 96) launch_pdl_pairs(pdl_ok(pool), backup_select_confined_kernel<3>, cgrid, cblock, (size_t)kConfinedSmem, st, d, r, v);
    else launch_pdl_pairs(pdl_ok(pool), backup_select_confined_kernel<4>, cgrid, cblock, (size_t)kConfinedSmem, st, d, r, v);
    MZ_LAUNCH_CHECK("backup_select_confined_kernel");
    pool->selected = 1;
    return MZ_OK;
  }
  if (A <= 32) launch_pdl(pdl_ok(pool), backup_select_kernel<1>, grid, block, smem, st, d, r, v);
  else if (A <= 64) launch_pdl(pdl_ok(pool), backup_select_kernel<2>, grid, block, smem, st, d, r, v);
  else if (A <= 96) launch_pdl(pdl_ok(pool), backup_select_kernel<3>, grid, block, smem, st, d, r, v);
  else if (A <= 128) launch_pdl(pdl_ok(pool), backup_select_kernel<4>, grid, block, smem, st, d, r, v);
  else launch_pdl(pdl_ok(pool), backup_select_kernel<0>, grid, block, smem, st, d, r, v);
  MZ_LAUNCH_CHECK("backup_select_kernel");
  pool->selected = 1;
  return MZ_OK;
}

extern "C" int mz_expand_backup(mz_pool* pool, const float* reward, const float* value, mz_stream stream) {
  MZ_CHECK_ARG(pool, "NULL argument");
  if (!pool->selected) {
    set_error("mz_expand_backup called without a preceding mz_select");
    return MZ_ESTATE;
  }
  const PoolDev d = dev_of(pool);
  if (use_thread_kernels(pool)) {
    launch_pdl(pdl_ok(pool), tree_thread_kernel, dim3((pool->B + kThreadBlock - 1) / kThreadBlock), dim3(kThreadBlock), (size_t)(pool->S + 2) * 16, (cudaStream_t)stream, d, reward ? reward : d.reward, value ? value : d.value, 2);
    MZ_LAUNCH_CHECK("tree_thread_kernel");
    pool->selected = 0;
    return MZ_OK;
  }
  launch_pdl(pdl_ok(pool), expand_backup_kernel, dim3(tree_blocks(pool->B)), dim3(kTreesPerBlock * 32), (size_t)0, (cudaStream_t)stream,
             d, reward ? reward : d.reward, value ? value : d.value);
  MZ_LAUNCH_CHECK("expand_backup_kernel");
  pool->selected = 0;
  return MZ_OK;
}

extern "C" int mz_root_policy(mz_pool* pool, const uint8_t* mask, const double* temperature, int deterministic,
                              int32_t* action, double* pi, double* root_value, int32_t* visits, mz_stream stream) {
  MZ_CHECK_ARG(pool && temperature && action && pi && root_value, "NULL argument");
  const size_t smem = (size_t)kTreesPerBlock * pool->A * sizeof(double);
  root_policy_kernel<<<tree_blocks(pool->B), kTreesPerBlock * 32, smem, (cudaStream_t)stream>>>(
      dev_of(pool), mask, temperature, deterministic, action, pi, root_value, visits);
  MZ_LAUNCH_CHECK("root_policy_kernel");
  return MZ_OK;
}
