// Shared declarations of the muzero_b200 library (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>

#include "../../include/muzero_b200.h"

namespace mz {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);
void set_pdl(int on);

#define MZ_CHECK_ARG(cond, ...)            \
  do {                                     \
    if (!(cond)) {                         \
      mz::set_error(__VA_ARGS__);          \
      return MZ_EINVAL;                    \
    }                                      \
  } while (0)

#define MZ_CUDA(call)                                                                  \
  do {                                                                                 \
    cudaError_t e__ = (call);                                                          \
    if (e__ != cudaSuccess) {                                                          \
      mz::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, \
                    __LINE__);                                                         \
      return MZ_ECUDA;                                                                 \
    }                                                                                  \
  } while (0)

#define MZ_LAUNCH_CHECK(name)                                                         \
  do {                                                                                \
    cudaError_t e__ = cudaGetLastError();                                             \
    if (e__ != cudaSuccess) {                                                         \
      mz::set_error("launch of %s failed: %s", name, cudaGetErrorString(e__));        \
      return MZ_ECUDA;                                                                \
    }                                                                                 \
    mz::count_launch();                                                               \
  } while (0)

constexpr int kWarp = 32;
constexpr uint16_t kNoChild = 0xFFFF;

// One (node, action) edge of a tree = the statistics of the child that action leads to, stored in the PARENT's row
// and split by who reads it:
//   HOT  (mz_view EDGES, 8 bytes):  .x = child << 16 | N   (u16 node index of the expanded child or kNoChild, u16 Node.N)
//                                   .y = Node.child_Q of the edge as the next descent needs it (float32 bits, min-max
//                                        normalised; 0 for an unvisited edge), refreshed by the backup
//        -- everything the pUCT descent reads: one coalesced 8-byte-per-lane load gives a warp a node's whole child set;
//   COLD (EDGE_W f64, EDGE_REWARD f32): Node.W and Node.reward, touched by the backup only, for the edges of one path.
// Unvisited child = N 0, child kNoChild (the reference creates such children eagerly, mcts.py:98-100; N=0, W=0,
// reward=0 makes lazy creation observationally identical).  The cold words of an edge are DEFINED only once N > 0
// (the expansion writes them): nothing reads them before, so expanding a node zeroes its hot row only.
typedef uint2 HotEdge;
__host__ __device__ inline uint32_t hot_word(uint32_t N, uint32_t child) { return (N & 0xffffu) | (child << 16); }

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Programmatic dependent launch (PDL).  The per-simulation chain of the MLP configurations alternates two short,
// latency-bound kernels (tree kernel, tcgen05 MLP kernel); with a full kernel boundary between them the second pays the
// launch latency and its prologue (table staging, TMEM allocation, barrier set-up) after the first has drained.
// Launched with the programmatic-serialisation attribute a kernel may start while its predecessor still runs; it does
// everything that does not depend on the predecessor, then pdl_wait() blocks until the predecessor grid has completed
// and its writes are visible.  pdl_trigger() lets the successor start that early.  Both are no-ops in a kernel that was
// launched the ordinary way.  MZ_NO_PDL=1 launches everything the ordinary way.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(bool allow, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args... args) {
  cudaLaunchConfig_t lc = {};
  lc.gridDim = grid; lc.blockDim = block; lc.dynamicSmemBytes = smem; lc.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = (allow && pdl_enabled()) ? 1 : 0;
  lc.attrs = at; lc.numAttrs = 1;
  return cudaLaunchKernelEx(&lc, kernel, static_cast<KArgs>(args)...);
}
// the same with the grid launched as 2-CTA clusters when it has an even number of CTAs: a 2-CTA cluster is placed on
// the two SMs of one TPC, so such a grid holds whole SM pairs and leaves every other pair to an SM-pair launch (the
// conv towers) running beside it
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl_pairs(bool allow, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                    cudaStream_t st, Args... args) {
  cudaLaunchConfig_t lc = {};
  lc.gridDim = grid; lc.blockDim = block; lc.dynamicSmemBytes = smem; lc.stream = st;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = (allow && pdl_enabled()) ? 1 : 0;
  at[1].id = cudaLaunchAttributeClusterDimension;
  at[1].val.clusterDim.x = 2; at[1].val.clusterDim.y = 1; at[1].val.clusterDim.z = 1;
  lc.attrs = at; lc.numAttrs = grid.x % 2 == 0 ? 2 : 1;
  return cudaLaunchKernelEx(&lc, kernel, static_cast<KArgs>(args)...);
}

}  // namespace mz

// Search pool: every pointer aims into the caller's arena.
struct mz_pool {
  mz_pool_config cfg;
  int B, A, S, max_nodes;
  void* arena;
  size_t arena_bytes;
  void* view_ptr[MZ_VIEW__COUNT];
  size_t view_bytes[MZ_VIEW__COUNT];
  double* pb_c_table;  // dev f64 [S+2]
  uint8_t* same_player;  // dev u8 [B]: current_player == opponent_player
  double* root_reward;   // dev f64 [B]
  uint8_t* f32_prior;    // dev u8 [B]: prior is float32 (no-noise path)
  unsigned* work;        // dev u32 [2]: work counters of the confined tree kernel
  int tree_ctas;         // > 0: the fused tree kernel runs as that many persistent CTAs (mz_pool_set_tree_ctas)
  int selected;          // host-side call-order check
};
