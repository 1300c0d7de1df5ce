// C ABI of the network handles: dispatch on the network family.
#include "net.cuh"

using namespace mz;

extern "C" int mz_net_hidden_bytes(const mz_net_config* cfg, int32_t* bytes) {
  MZ_CHECK_ARG(cfg && bytes, "NULL argument");
  switch (cfg->kind) {
    case MZ_NET_MLP: return mlp_hidden_bytes(*cfg, bytes);
    case MZ_NET_BOARD:
    case MZ_NET_ATARI: return conv_hidden_bytes(*cfg, bytes);
  }
  set_error("unknown network kind %d", cfg->kind);
  return MZ_EINVAL;
}

extern "C" int mz_net_arena_bytes(const mz_net_config* cfg, int32_t max_batch, size_t* bytes) {
  MZ_CHECK_ARG(cfg && bytes, "NULL argument");
  MZ_CHECK_ARG(max_batch > 0, "max_batch must be positive");
  switch (cfg->kind) {
    case MZ_NET_MLP: return mlp_arena_bytes(*cfg, bytes);
    case MZ_NET_BOARD:
    case MZ_NET_ATARI: return conv_arena_bytes(*cfg, max_batch, bytes);
  }
  set_error("unknown network kind %d", cfg->kind);
  return MZ_EINVAL;
}

extern "C" int mz_net_create(const mz_net_config* cfg, const float* const* weights, int32_t num_weights,
                             int32_t max_batch, void* arena_dev, size_t arena_bytes, mz_net** out) {
  MZ_CHECK_ARG(cfg && weights && arena_dev && out, "NULL argument");
  MZ_CHECK_ARG(max_batch > 0, "max_batch must be positive");
  MZ_CHECK_ARG(((uintptr_t)arena_dev & 255) == 0, "arena must be 256-byte aligned");
  for (int i = 0; i < num_weights; ++i) MZ_CHECK_ARG(weights[i] != nullptr, "weights[%d] is NULL", i);
  NetImpl* impl = nullptr;
  int rc;
  switch (cfg->kind) {
    case MZ_NET_MLP: rc = mlp_create(*cfg, weights, num_weights, arena_dev, arena_bytes, &impl); break;
    case MZ_NET_BOARD:
    case MZ_NET_ATARI: rc = conv_create(*cfg, weights, num_weights, max_batch, arena_dev, arena_bytes, &impl); break;
    default: set_error("unknown network kind %d", cfg->kind); return MZ_EINVAL;
  }
  if (rc) return rc;
  mz_net* h = new mz_net();
  h->cfg = *cfg;
  h->max_batch = max_batch;
  h->impl = impl;
  *out = h;
  return MZ_OK;
}

extern "C" int mz_net_destroy(mz_net* net) {
  if (net) { delete net->impl; delete net; }
  return MZ_OK;
}

extern "C" int mz_net_initial(mz_net* net, int32_t batch, const float* obs, void* hidden_out,
                              const int32_t* dst_index, float* pi_probs, float* value, mz_stream stream) {
  MZ_CHECK_ARG(net && obs && hidden_out && value, "NULL argument");
  MZ_CHECK_ARG(batch > 0 && batch <= net->max_batch, "batch %d outside (0, %d]", batch, net->max_batch);
  return net->impl->initial(batch, obs, hidden_out, dst_index, pi_probs, value, (cudaStream_t)stream);
}

extern "C" int mz_net_initial_frames(mz_net* net, int32_t batch, const uint8_t* frames, const float* plane_values,
                                     void* hidden_out, const int32_t* dst_index, float* pi_probs, float* value,
                                     mz_stream stream) {
  MZ_CHECK_ARG(net && frames && plane_values && hidden_out && value, "NULL argument");
  MZ_CHECK_ARG(batch > 0 && batch <= net->max_batch, "batch %d outside (0, %d]", batch, net->max_batch);
  return net->impl->initial_frames(batch, frames, plane_values, hidden_out, dst_index, pi_probs, value,
                                   (cudaStream_t)stream);
}

extern "C" int mz_net_initial_search(mz_net* net, mz_pool* pool, int32_t batch, const float* obs, const uint8_t* frames,
                                     const float* plane_values, void* hidden_out, const int32_t* dst_index,
                                     float* pi_probs, float* value, int32_t noise_mode, double* noise, double alpha,
                                     double eps, const uint8_t* mask, const int32_t* players, mz_stream stream) {
  MZ_CHECK_ARG(net && pool && hidden_out && pi_probs && value, "NULL argument");
  MZ_CHECK_ARG((obs != nullptr) != (frames != nullptr), "pass either obs or (frames, plane_values)");
  MZ_CHECK_ARG(frames == nullptr || plane_values != nullptr, "frames without plane_values");
  MZ_CHECK_ARG(batch == pool->B && batch <= net->max_batch, "batch %d must equal the pool's %d trees (net max %d)", batch,
               pool->B, net->max_batch);
  MZ_CHECK_ARG(net->cfg.num_actions == pool->A, "network has %d actions, pool %d", net->cfg.num_actions, pool->A);
  MZ_CHECK_ARG(noise_mode >= 0 && noise_mode <= 2, "noise_mode must be 0 (none), 1 (given) or 2 (device draw)");
  MZ_CHECK_ARG(noise_mode == 0 || noise != nullptr, "noise buffer is NULL");
  if (noise_mode) {
    // mcts.py:239-242
    MZ_CHECK_ARG(eps >= 0.0 && eps <= 1.0, "Expect `eps` to be a float in the range [0.0, 1.0], got %g", eps);
    if (noise_mode == 2)
      MZ_CHECK_ARG(alpha > 0.0 && alpha <= 1.0, "Expect `alpha` to be a float in the range (0.0, 1.0], got %g", alpha);
  }
  RootSetup rs;
  rs.pool = pool_dev(pool);
  rs.enabled = 1;
  rs.noise_mode = noise_mode; rs.noise = noise; rs.alpha = alpha; rs.eps = noise_mode ? eps : 0.0;
  rs.one_minus_eps_f32 = (float)(1.0 - rs.eps);
  rs.mask = mask; rs.players = players;
  net->impl->pending_root = &rs;
  const int rc = frames ? net->impl->initial_frames(batch, frames, plane_values, hidden_out, dst_index, pi_probs, value,
                                                    (cudaStream_t)stream)
                        : net->impl->initial(batch, obs, hidden_out, dst_index, pi_probs, value, (cudaStream_t)stream);
  net->impl->pending_root = nullptr;
  if (rc == MZ_OK) pool->selected = 0;
  return rc;
}

extern "C" int mz_net_recurrent(mz_net* net, int32_t batch, const void* hidden_in, const int32_t* src_index,
                                const int32_t* action, void* hidden_out, const int32_t* dst_index, float* reward,
                                float* value, float* pi_probs, mz_stream stream) {
  MZ_CHECK_ARG(net && hidden_in && action && hidden_out && reward && value, "NULL argument");
  MZ_CHECK_ARG(batch > 0 && batch <= net->max_batch, "batch %d outside (0, %d]", batch, net->max_batch);
  return net->impl->recurrent(batch, hidden_in, src_index, action, hidden_out, dst_index, reward, value, pi_probs,
                              (cudaStream_t)stream);
}

extern "C" int mz_search_run(mz_net* net, mz_pool* pool, mz_stream stream) {
  MZ_CHECK_ARG(net && pool, "NULL argument");
  MZ_CHECK_ARG(pool->cfg.hidden_bytes > 0, "the pool has no hidden-state slots (it was made for an external network)");
  MZ_CHECK_ARG(pool->B <= net->max_batch, "pool has %d trees, the net was created for batches of at most %d", pool->B,
               net->max_batch);
  MZ_CHECK_ARG(net->cfg.num_actions == pool->A, "network has %d actions, pool %d", net->cfg.num_actions, pool->A);
  int rc = net->impl->search(pool, (cudaStream_t)stream);
  if (rc <= 0) {
    if (rc == MZ_OK) pool->selected = 0;
    return rc;
  }
  // launch chain: select, then S x (recurrent inference, expand + backup [+ select of the next simulation])
  void* hidden = pool->view_ptr[MZ_VIEW_HIDDEN];
  const int32_t* src = (const int32_t*)pool->view_ptr[MZ_VIEW_SRC_SLOT];
  const int32_t* dst = (const int32_t*)pool->view_ptr[MZ_VIEW_DST_SLOT];
  const int32_t* act = (const int32_t*)pool->view_ptr[MZ_VIEW_LEAF_ACTION];
  float* rew = (float*)pool->view_ptr[MZ_VIEW_REWARD];
  float* val = (float*)pool->view_ptr[MZ_VIEW_VALUE];
  if ((rc = mz_select(pool, stream))) return rc;
  for (int sim = 0; sim < pool->S; ++sim) {
    // pi_probs = NULL: the search never reads the recurrent policy (mcts.py:386)
    if ((rc = mz_net_recurrent(net, pool->B, hidden, src, act, hidden, dst, rew, val, nullptr, stream))) return rc;
    rc = sim + 1 < pool->S ? mz_expand_backup_select(pool, nullptr, nullptr, stream)
                           : mz_expand_backup(pool, nullptr, nullptr, stream);
    if (rc) return rc;
  }
  return MZ_OK;
}

extern "C" int mz_net_set_fused_search(mz_net* net, int32_t enable) {
  MZ_CHECK_ARG(net, "NULL argument");
  net->impl->fused_search = enable < 0 ? -1 : (enable != 0 ? 1 : 0);
  return MZ_OK;
}

extern "C" int mz_net_set_cta_limit(mz_net* net, int32_t max_ctas) {
  MZ_CHECK_ARG(net && max_ctas >= 0, "bad argument");
  net->impl->cta_limit = max_ctas;
  return MZ_OK;
}

extern "C" int mz_net_debug_capture_bytes(mz_net* net, int32_t batch, size_t* bytes) {
  MZ_CHECK_ARG(net && bytes, "NULL argument");
  MZ_CHECK_ARG(batch > 0 && batch <= net->max_batch, "batch %d outside (0, %d]", batch, net->max_batch);
  return net->impl->debug_capture_bytes(batch, bytes);
}

extern "C" int mz_net_debug_capture(mz_net* net, void* buf, size_t bytes) {
  MZ_CHECK_ARG(net, "NULL argument");
  MZ_CHECK_ARG(((uintptr_t)buf & 255) == 0, "capture buffer must be 256-byte aligned");
  return net->impl->debug_capture(buf, bytes);
}

extern "C" int mz_net_debug_tensor(mz_net* net, int32_t index, mz_debug_tensor* out, int32_t* count) {
  MZ_CHECK_ARG(net && count && (index < 0 || out), "NULL argument");
  return net->impl->debug_tensor(index, out, count);
}

extern "C" int mz_net_debug_launch(mz_net* net, int32_t index, mz_debug_launch* out, int32_t* count) {
  MZ_CHECK_ARG(net && count && (index < 0 || out), "NULL argument");
  return net->impl->debug_launch(index, out, count);
}

extern "C" int mz_net_profile_begin(mz_net* net) {
  MZ_CHECK_ARG(net, "NULL argument");
  NetImpl* n = net->impl;
  for (cudaEvent_t e : n->prof_ev) cudaEventDestroy(e);
  n->prof_ev.clear();
  n->prof_cls.clear();
  n->prof_weight.clear();
  n->profiling = true;
  return MZ_OK;
}

extern "C" int mz_net_profile_end(mz_net* net, double* ms_by_class, int64_t* launches_by_class) {
  MZ_CHECK_ARG(net && ms_by_class && launches_by_class, "NULL argument");
  NetImpl* n = net->impl;
  n->profiling = false;
  MZ_CUDA(cudaDeviceSynchronize());
  for (int c = 0; c < kProfClasses; ++c) { ms_by_class[c] = 0.0; launches_by_class[c] = 0; }
  for (size_t i = 0; i < n->prof_cls.size(); ++i) {
    float ms = 0.0f;
    MZ_CUDA(cudaEventElapsedTime(&ms, n->prof_ev[2 * i], n->prof_ev[2 * i + 1]));
    ms_by_class[n->prof_cls[i]] += ms;
    launches_by_class[n->prof_cls[i]] += n->prof_weight[i];
    if (n->prof_cls[i] == kProfConv) { ms_by_class[kProfConvLaunches] += ms; launches_by_class[kProfConvLaunches] += 1; }
  }
  for (cudaEvent_t e : n->prof_ev) cudaEventDestroy(e);
  n->prof_ev.clear();
  n->prof_cls.clear();
  n->prof_weight.clear();
  return MZ_OK;
}
