// Internal interface every network family implements behind the mz_net handle.
#pragma once
#include "common.cuh"
#include "pool.cuh"
#include <vector>

namespace mz {

// Optional per-kernel timing (mz_net_profile_begin/end): CUDA events recorded on the launching
// stream around every kernel the net launches, summed per kernel class.  Eager launches only.
enum ProfClass { kProfConv = 0, kProfHead = 1, kProfPack = 2, kProfMlp = 3, kProfConvLaunches = 4, kProfClasses = 5 };

struct NetImpl {
  bool profiling = false;
  int cta_limit = 0;                    // persistent kernels use at most this many CTAs (0: one per SM)
  int fused_search = -1;                // mz_search_run: -1 one launch per search where it is the faster form, 0 never
                                        // (launch chain), 1 wherever a one-launch kernel exists (mz_net_set_fused_search)
  const RootSetup* pending_root = nullptr;   // set around initial() by mz_net_initial_search: the policy epilogue
                                             // also prepares the search roots (Dirichlet, mask, renormalise, reset)
  std::vector<cudaEvent_t> prof_ev;     // pairs (begin, end)
  std::vector<int> prof_cls, prof_weight;   // weight: how many layers one launch covers
  void prof_mark(int cls, cudaStream_t st, int weight = 1) {
    if (!profiling) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, st);
    prof_ev.push_back(e);
    if (cls >= 0) { prof_cls.push_back(cls); prof_weight.push_back(weight); }
  }
  virtual ~NetImpl() {
    for (cudaEvent_t e : prof_ev) cudaEventDestroy(e);
  }
  virtual int initial(int batch, const float* obs, void* hidden_out, const int32_t* dst_index, float* pi_probs,
                      float* value, cudaStream_t st) = 0;
  virtual int initial_frames(int, const uint8_t*, const float*, void*, const int32_t*, float*, float*, cudaStream_t) {
    set_error("mz_net_initial_frames: this network family takes float32 observations");
    return MZ_EINVAL;
  }
  // all simulations of a search in ONE launch (persistent kernel that owns the trees); > 0: this net / pool is not
  // covered, the caller enqueues the per-simulation launch chain instead
  virtual int search(mz_pool*, cudaStream_t) { return 1; }
  virtual int recurrent(int batch, const void* hidden_in, const int32_t* src_index, const int32_t* action,
                        void* hidden_out, const int32_t* dst_index, float* reward, float* value, float* pi_probs,
                        cudaStream_t st) = 0;
  // test aid (mz_net_debug_*): every family implements it
  virtual int debug_capture_bytes(int, size_t*) = 0;
  virtual int debug_capture(void*, size_t) = 0;
  virtual int debug_tensor(int, mz_debug_tensor*, int32_t*) = 0;
  virtual int debug_launch(int, mz_debug_launch*, int32_t*) = 0;
};

int mlp_hidden_bytes(const mz_net_config& c, int32_t* bytes);
int mlp_arena_bytes(const mz_net_config& c, size_t* bytes);
int mlp_create(const mz_net_config& c, const float* const* w, int nw, void* arena, size_t arena_bytes, NetImpl** out);

int conv_hidden_bytes(const mz_net_config& c, int32_t* bytes);
int conv_arena_bytes(const mz_net_config& c, int max_batch, size_t* bytes);
int conv_create(const mz_net_config& c, const float* const* w, int nw, int max_batch, void* arena,
                size_t arena_bytes, NetImpl** out);

}  // namespace mz

struct mz_net {
  mz_net_config cfg;
  int max_batch;
  mz::NetImpl* impl;
};
