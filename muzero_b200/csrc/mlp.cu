// Fused fp32 inference kernels for the MuZeroMLPNet family (network.py:140-267).
//
// One CTA runs the whole initial_inference / recurrent_inference chain for a
// tile of 32 rows (trees): hidden-state gather by slot index, one-hot action as
// a weight-row gather, both Linear-ReLU-Linear stacks, min-max normalisation
// (util.py:31-36), softmax and the support->scalar transform (util.py:70-93)
// never leave shared memory.  These nets are 0.18-0.40 MFLOP per row: the path
// is launch/latency bound, so the design goal is ONE launch per network call.
#include "common.cuh"
#include "net.cuh"
#include "umma.cuh"
#include <algorithm>
#include <type_traits>
#include "tree_thread.cuh"
#include "tree_warp.cuh"
#include <cuda_fp16.h>
#include <cstdlib>

namespace mz {
using namespace umma;

constexpr int kRows = 32;
constexpr int kThreads = 256;
constexpr int kInitThreads = 512;

struct MlpDev {
  int in_dim, A, P, HD, Sv, Sr;
  int in_pad;   // in_dim rounded up to 4
  // transposed [in, out] weights
  const float *rep1_wt, *rep1_b, *rep2_wt, *rep2_b;
  const float *dyn1_wt, *dyn1_b, *dyn2_wt, *dyn2_b;
  const float *rew1_wt, *rew1_b, *rew2_wt, *rew2_w, *rew2_b;   // *_w: original [out, in] layout for tiny heads
  const float *pol1_wt, *pol1_b, *pol2_wt, *pol2_w, *pol2_b;
  const float *val1_wt, *val1_b, *val2_wt, *val2_w, *val2_b;
};

// out[r][j] = act(bias[j] + sum_k in[r][k] * Wt[k][j] (+ Wt[extra_row[r]][j]))
// thread -> (column j, row group g); RPT rows per thread held in registers.
template <int RPT>
__device__ void dense_cols(const float* __restrict__ Wt, const float* __restrict__ bias, const float* in, int ldin,
                           int K, int OUT, bool relu, float* out, int ldout, const int* extra_row) {
  constexpr int G = kRows / RPT;
  const int items = OUT * G;
  for (int idx = threadIdx.x; idx < items; idx += blockDim.x) {
    const int j = idx % OUT, g = idx / OUT;
    const float* x0 = in + (size_t)g * RPT * ldin;
    float acc[RPT];
    const float b = bias[j];
#pragma unroll
    for (int r = 0; r < RPT; ++r) acc[r] = b;
    int k = 0;
    const int K4 = K & ~3;
#pragma unroll 2
    for (; k < K4; k += 4) {
      const float w0 = __ldg(Wt + (size_t)(k + 0) * OUT + j);
      const float w1 = __ldg(Wt + (size_t)(k + 1) * OUT + j);
      const float w2 = __ldg(Wt + (size_t)(k + 2) * OUT + j);
      const float w3 = __ldg(Wt + (size_t)(k + 3) * OUT + j);
#pragma unroll
      for (int r = 0; r < RPT; ++r) {
        const float4 xv = *reinterpret_cast<const float4*>(x0 + (size_t)r * ldin + k);
        acc[r] = fmaf(xv.x, w0, acc[r]);
        acc[r] = fmaf(xv.y, w1, acc[r]);
        acc[r] = fmaf(xv.z, w2, acc[r]);
        acc[r] = fmaf(xv.w, w3, acc[r]);
      }
    }
    for (; k < K; ++k) {
      const float w = __ldg(Wt + (size_t)k * OUT + j);
#pragma unroll
      for (int r = 0; r < RPT; ++r) acc[r] = fmaf(x0[(size_t)r * ldin + k], w, acc[r]);
    }
#pragma unroll
    for (int r = 0; r < RPT; ++r) {
      float v = acc[r];
      if (extra_row) v += __ldg(Wt + (size_t)extra_row[g * RPT + r] * OUT + j);
      if (relu) v = fmaxf(v, 0.0f);
      out[(size_t)(g * RPT + r) * ldout + j] = v;
    }
  }
}

// tiny heads (OUT < 16): a warp per (row, output), lanes split K; W in [OUT, K] layout
__device__ void dense_tiny(const float* __restrict__ W, const float* __restrict__ bias, const float* in, int ldin,
                           int K, int OUT, float* out, int ldout) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int item = warp; item < kRows * OUT; item += blockDim.x / 32) {
    const int r = item / OUT, j = item % OUT;
    float acc = 0.0f;
    for (int k = lane; k < K; k += 32) acc = fmaf(in[(size_t)r * ldin + k], __ldg(W + (size_t)j * K + k), acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) out[(size_t)r * ldout + j] = acc + bias[j];
  }
}

__device__ void dense(const float* Wt, const float* W, const float* bias, const float* in, int ldin, int K, int OUT,
                      bool relu, float* out, int ldout, const int* extra_row = nullptr) {
  // rows per thread: as many as still give every thread of the CTA an item (256 threads: 32 for OUT >= 256, 16 for
  // >= 128, ...; 512 threads: one step fewer).  The summation order of an output element does not depend on it.
  int rpt = 32;
  while (rpt > 2 && OUT * (kRows / rpt) < (int)blockDim.x) rpt >>= 1;
  if (OUT < 16 && W != nullptr && !relu && extra_row == nullptr) dense_tiny(W, bias, in, ldin, K, OUT, out, ldout);
  else if (rpt == 32) dense_cols<32>(Wt, bias, in, ldin, K, OUT, relu, out, ldout, extra_row);
  else if (rpt == 16) dense_cols<16>(Wt, bias, in, ldin, K, OUT, relu, out, ldout, extra_row);
  else if (rpt == 8) dense_cols<8>(Wt, bias, in, ldin, K, OUT, relu, out, ldout, extra_row);
  else if (rpt == 4) dense_cols<4>(Wt, bias, in, ldin, K, OUT, relu, out, ldout, extra_row);
  else dense_cols<2>(Wt, bias, in, ldin, K, OUT, relu, out, ldout, extra_row);
  __syncthreads();
}

// util.py:25-28 signed_parabolic, float32, same operation order as the torch expression
__device__ __forceinline__ float signed_parabolic(float x) {
  const float eps = 1e-3f;
  float z = __fadd_rn(1.0f, __fmul_rn(4.0f * eps, __fadd_rn(eps + 1.0f, fabsf(x))));
  z = __fsqrt_rn(z);
  z = __fdiv_rn(__fdiv_rn(z, 2.0f), eps);
  z = __fsub_rn(z, 500.0f);                           // 1 / 2 / eps
  const float r = __fsub_rn(__fmul_rn(z, z), 1.0f);
  return x > 0.0f ? r : (x < 0.0f ? -r : 0.0f * r);
}

// util.py:70-93: softmax over the support, expectation, inverse value transform.  One warp per row.
__device__ void support_to_scalar(const float* logits, int ld, int S, float* out_global, int row0, int batch) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = warp; r < kRows; r += blockDim.x / 32) {
    if (row0 + r >= batch) continue;
    const float* l = logits + (size_t)r * ld;
    if (S == 1) {                                     // scalar head, network.py:126-134
      if (lane == 0) out_global[row0 + r] = l[0];
      continue;
    }
    float m = -INFINITY;
    for (int i = lane; i < S; i += 32) m = fmaxf(m, l[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    const int maxv = (S - 1) / 2;
    const float step = S > 1 ? (float)(2 * maxv) / (float)(S - 1) : 0.0f;
    float den = 0.0f, num = 0.0f;
    for (int i = lane; i < S; i += 32) {
      const float e = expf(l[i] - m);
      den += e;
      num += e * ((float)(-maxv) + step * (float)i);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      den += __shfl_xor_sync(0xffffffffu, den, o);
      num += __shfl_xor_sync(0xffffffffu, num, o);
    }
    if (lane == 0) out_global[row0 + r] = signed_parabolic(num / den);
  }
  __syncthreads();
}

__device__ void softmax_rows(const float* logits, int ld, int A, float* out_global, int row0, int batch) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = warp; r < kRows; r += blockDim.x / 32) {
    if (row0 + r >= batch) continue;
    const float* l = logits + (size_t)r * ld;
    float m = -INFINITY;
    for (int i = lane; i < A; i += 32) m = fmaxf(m, l[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float den = 0.0f;
    for (int i = lane; i < A; i += 32) den += expf(l[i] - m);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) den += __shfl_xor_sync(0xffffffffu, den, o);
    for (int i = lane; i < A; i += 32) out_global[(size_t)(row0 + r) * A + i] = expf(l[i] - m) / den;
  }
  __syncthreads();
}

// util.py:31-36 over the feature dimension; writes the normalised state to smem and to its slot
__device__ void normalise_and_store(const float* hraw, float* hn, int HD, float* hidden_out,
                                    const int32_t* dst_index, int row0, int batch) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = warp; r < kRows; r += blockDim.x / 32) {
    const float* h = hraw + (size_t)r * HD;
    float mn = INFINITY, mx = -INFINITY;
    for (int i = lane; i < HD; i += 32) { mn = fminf(mn, h[i]); mx = fmaxf(mx, h[i]); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    const float den = __fadd_rn(__fsub_rn(mx, mn), 1e-8f);
    const bool live = row0 + r < batch;
    float* dst = nullptr;
    if (live) dst = hidden_out + (size_t)(dst_index ? dst_index[row0 + r] : row0 + r) * HD;
    for (int i = lane; i < HD; i += 32) {
      const float v = __fdiv_rn(__fsub_rn(h[i], mn), den);
      hn[(size_t)r * HD + i] = v;
      if (live) dst[i] = v;
    }
  }
  __syncthreads();
}

struct Smem {
  float *x, *h1, *hraw, *hn, *lg;
  int *arow;
  int ldx, ldh, ldl;
};
// row strides are multiples of 4 floats: dense_cols reads its input rows as float4
__device__ Smem carve(const MlpDev& n, float* base) {
  Smem s;
  s.ldx = max(n.in_pad, n.HD);
  s.ldh = (n.P + 3) & ~3;
  s.ldl = (max(max(n.A, n.Sv), n.Sr) + 3) & ~3;
  s.x = base;
  s.h1 = s.x + kRows * s.ldx;
  s.hraw = s.h1 + kRows * s.ldh;
  s.hn = s.hraw + kRows * n.HD;
  s.lg = s.hn + kRows * n.HD;
  s.arow = reinterpret_cast<int*>(s.lg + kRows * s.ldl);
  return s;
}
size_t smem_bytes(const MlpDev& n) {
  const int ldx = n.in_pad > n.HD ? n.in_pad : n.HD;
  int m = n.A > n.Sv ? n.A : n.Sv;
  m = m > n.Sr ? m : n.Sr;
  const int ldl = (m + 3) & ~3;
  const int ldh = (n.P + 3) & ~3;
  return sizeof(float) * ((size_t)kRows * ldx + (size_t)kRows * ldh + 2 * (size_t)kRows * n.HD + (size_t)kRows * ldl) +
         sizeof(int) * kRows;
}

extern __shared__ __align__(16) float mlp_smem[];

// Test aid (mz_net_debug_capture): where the SIMT kernels copy every dense output and the normalised state, each to a
// [batch][columns] fp32 region of its own (nullptr: not captured).  Every captured shared-memory tensor is next written
// at least one dense() -- and so one barrier -- later, so the copy needs no barrier of its own.
enum SimtCapSlot { kCapNet0L0 = 0, kCapNet0L1, kCapNorm, kCapRewL0, kCapRewL1, kCapPolL0, kCapPolL1, kCapValL0, kCapValL1,
                   kCapSlots };
struct MlpSimtCap {
  float* t[kCapSlots];
};
__device__ void cap_rows(float* dst, const float* src, int ld, int cols, int row0, int batch) {
  if (dst == nullptr) return;
  for (int i = threadIdx.x; i < kRows * cols; i += blockDim.x) {
    const int r = i / cols, j = i % cols;
    if (row0 + r < batch) dst[(size_t)(row0 + r) * cols + j] = src[(size_t)r * ld + j];
  }
}

// prediction heads on the normalised state in s.hn (network.py:223-233)
__device__ void prediction_heads(const MlpDev& n, const Smem& s, float* pi_probs, float* value, int row0, int batch,
                                 const MlpSimtCap& cap) {
  if (pi_probs != nullptr) {
    dense(n.pol1_wt, nullptr, n.pol1_b, s.hn, n.HD, n.HD, n.P, true, s.h1, s.ldh);
    cap_rows(cap.t[kCapPolL0], s.h1, s.ldh, n.P, row0, batch);
    dense(n.pol2_wt, n.pol2_w, n.pol2_b, s.h1, s.ldh, n.P, n.A, false, s.lg, s.ldl);
    cap_rows(cap.t[kCapPolL1], s.lg, s.ldl, n.A, row0, batch);
    softmax_rows(s.lg, s.ldl, n.A, pi_probs, row0, batch);
  }
  dense(n.val1_wt, nullptr, n.val1_b, s.hn, n.HD, n.HD, n.P, true, s.h1, s.ldh);
  cap_rows(cap.t[kCapValL0], s.h1, s.ldh, n.P, row0, batch);
  dense(n.val2_wt, n.val2_w, n.val2_b, s.h1, s.ldh, n.P, n.Sv, false, s.lg, s.ldl);
  cap_rows(cap.t[kCapValL1], s.lg, s.ldl, n.Sv, row0, batch);
  support_to_scalar(s.lg, s.ldl, n.Sv, value, row0, batch);
}

// kInitThreads = 512: sixteen warps, so that the root preparation fused behind the softmax (root_setup_fused: a
// sequential Dirichlet sampler per tree) has two rows per warp instead of four
__global__ void __launch_bounds__(kInitThreads)
mlp_initial_kernel(MlpDev n, int batch, const float* __restrict__ obs, float* __restrict__ hidden_out,
                   const int32_t* __restrict__ dst_index, float* __restrict__ pi_probs, float* __restrict__ value,
                   const __grid_constant__ RootSetup rs, const __grid_constant__ MlpSimtCap cap) {
  const Smem s = carve(n, mlp_smem);
  const int row0 = blockIdx.x * kRows;
  for (int i = threadIdx.x; i < kRows * s.ldx; i += blockDim.x) {
    const int r = i / s.ldx, k = i % s.ldx;
    s.x[i] = (row0 + r < batch && k < n.in_dim) ? obs[(size_t)(row0 + r) * n.in_dim + k] : 0.0f;
  }
  __syncthreads();
  dense(n.rep1_wt, nullptr, n.rep1_b, s.x, s.ldx, n.in_dim, n.P, true, s.h1, s.ldh);
  cap_rows(cap.t[kCapNet0L0], s.h1, s.ldh, n.P, row0, batch);
  dense(n.rep2_wt, nullptr, n.rep2_b, s.h1, s.ldh, n.P, n.HD, false, s.hraw, n.HD);
  cap_rows(cap.t[kCapNet0L1], s.hraw, n.HD, n.HD, row0, batch);
  normalise_and_store(s.hraw, s.hn, n.HD, hidden_out, dst_index, row0, batch);
  cap_rows(cap.t[kCapNorm], s.hn, n.HD, n.HD, row0, batch);
  prediction_heads(n, s, pi_probs, value, row0, batch, cap);
  if (rs.enabled) {
    // fused root preparation (mz_net_initial_search): the warp that wrote row r's softmax (softmax_rows: warp r % 8,
    // lane i -> actions i, i + 32, ...) draws the tree's Dirichlet noise, mixes, masks, renormalises and resets the tree
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int r = warp; r < kRows; r += blockDim.x / 32)
      if (row0 + r < batch) root_setup_fused(rs, row0 + r, lane, pi_probs + (size_t)(row0 + r) * n.A);
  }
}

__global__ void __launch_bounds__(kThreads)
mlp_recurrent_kernel(MlpDev n, int batch, const float* __restrict__ hidden_in, const int32_t* __restrict__ src_index,
                     const int32_t* __restrict__ action, float* __restrict__ hidden_out,
                     const int32_t* __restrict__ dst_index, float* __restrict__ reward, float* __restrict__ value,
                     float* __restrict__ pi_probs, const __grid_constant__ MlpSimtCap cap) {
  const Smem s = carve(n, mlp_smem);
  const int row0 = blockIdx.x * kRows;
  // leaf gather: parent hidden state by slot index + the action as a weight-row index
  for (int i = threadIdx.x; i < kRows * (n.HD / 4); i += blockDim.x) {
    const int r = i / (n.HD / 4), k4 = i % (n.HD / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row0 + r < batch) {
      const size_t slot = src_index ? src_index[row0 + r] : row0 + r;
      v = *reinterpret_cast<const float4*>(hidden_in + slot * n.HD + 4 * k4);
    }
    *reinterpret_cast<float4*>(s.x + (size_t)r * s.ldx + 4 * k4) = v;
  }
  if (threadIdx.x < kRows) {
    const int r = threadIdx.x;
    int a = (row0 + r < batch) ? action[row0 + r] : 0;
    a = min(max(a, 0), n.A - 1);
    s.arow[r] = n.HD + a;      // one-hot(action) concatenated after the state (network.py:191-193)
  }
  __syncthreads();
  dense(n.dyn1_wt, nullptr, n.dyn1_b, s.x, s.ldx, n.HD, n.P, true, s.h1, s.ldh, s.arow);
  cap_rows(cap.t[kCapNet0L0], s.h1, s.ldh, n.P, row0, batch);
  dense(n.dyn2_wt, nullptr, n.dyn2_b, s.h1, s.ldh, n.P, n.HD, false, s.hraw, n.HD);
  cap_rows(cap.t[kCapNet0L1], s.hraw, n.HD, n.HD, row0, batch);
  // reward head reads the UN-normalised state (network.py:195-196)
  dense(n.rew1_wt, nullptr, n.rew1_b, s.hraw, n.HD, n.HD, n.P, true, s.h1, s.ldh);
  cap_rows(cap.t[kCapRewL0], s.h1, s.ldh, n.P, row0, batch);
  dense(n.rew2_wt, n.rew2_w, n.rew2_b, s.h1, s.ldh, n.P, n.Sr, false, s.lg, s.ldl);
  cap_rows(cap.t[kCapRewL1], s.lg, s.ldl, n.Sr, row0, batch);
  support_to_scalar(s.lg, s.ldl, n.Sr, reward, row0, batch);
  normalise_and_store(s.hraw, s.hn, n.HD, hidden_out, dst_index, row0, batch);
  cap_rows(cap.t[kCapNorm], s.hn, n.HD, n.HD, row0, batch);
  prediction_heads(n, s, pi_probs, value, row0, batch, cap);
}

__global__ void transpose_kernel(const float* __restrict__ w, float* __restrict__ wt, int out, int in) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < out * in) {
    const int o = i / in, k = i % in;
    wt[(size_t)k * out + o] = w[i];
  }
}


// ---------------------------------------------------------------------------
// tcgen05 path of recurrent_inference (the per-simulation call of the search)
// ---------------------------------------------------------------------------
// One CTA owns tiles of 128 rows (trees) and runs the whole chain for a tile on the tensor
// cores with every activation staying on chip:
//   transition: [h(64) | onehot(a)] -> P -> 64     reward: h_raw -> P -> Sr     value: h' -> P -> Sv   [policy]
// Each two-layer net is processed in chunks of 256 hidden units:
//   D1[128 x 256] = A_in[128 x 64] . W1c^T      (4 MMAs  M128 N256 K16, fp32 in TMEM columns 0..255)
//   epilogue 1: + bias (+ the action's weight column, a [A][P] fp32 table) , ReLU, fp16 -> A_mid (smem, K-major)
//   D2[128 x N2] (+)= A_mid[128 x 256] . W2c^T  (16 MMAs M128 N{32,64,..} K16, TMEM columns 256..)
// followed by the net's own epilogue 2 (min-max normalisation of util.py:31-36, support -> scalar of
// util.py:70-93, softmax).  Operands are fp16 (the hidden state is normalised to [0,1]), accumulation fp32.
// Weights are pre-packed per (net, chunk, layer) block in exactly the shared-memory core-matrix layout and
// streamed by a producer warp with 1-D bulk copies (TMA) through a 3-slot mbarrier ring, so the next block
// loads while the current one is multiplied.  Widths 256 and 512 only: MlpTcParams holds kTcMaxBlocks = 16 blocks, two
// per chunk of each of the three nets a search runs (the policy's adds two more per chunk); mlp_create sends every
// other width to the SIMT kernels.

constexpr int kTcRows = 128;          // rows per tile == compute threads
constexpr int kTcCompute = 256;       // 8 compute warps: warps 0-3 own the tile's rows (thread = row), warps 4-7 share
                                      // their TMEM lane quadrants and take half of the first-layer epilogue's columns
constexpr int kTcThreads = 288;       // + 1 producer warp
constexpr int kTcChunk = 256;         // hidden units per chunk
constexpr int kTcSlots = 3;           // weight ring
constexpr int kTcSlotBytes = 32768;
constexpr int kTcMaxBlocks = 16;

struct MlpTcParams {
  const unsigned char* wpack;
  uint32_t blk_off[kTcMaxBlocks], blk_bytes[kTcMaxBlocks];
  int nblk, nnets, chunks;
  int nsplit;                         // 2: two CTAs per tile -- both run the transition net, one adds the reward net, the other
                                      // the value (and policy) net; 1: one CTA runs all nets of its tiles
  int P, A, Apad, Sr, Sv;
  int tab_in_smem;                    // the [A][P] action table fits beside the tiles in shared memory
  const float* tabA;                  // [A][P]: first-layer weight column of each action (network.py:191-193)
  const float* b1[4];
  const float* b2[4];
  int batch;
  const float* hidden_in; const int32_t* src_index; const int32_t* action;
  float* hidden_out; const int32_t* dst_index; float* reward; float* value; float* pi;
  long long* dbg;                     // MZ_MLP_DEBUG: clock64 stamps of CTA 0 / thread 0 (measurement aid)
};
// Test aid (mz_net_debug_capture, read by the kCap instantiation only), per net and CTA part: the fp16 hidden layer as
// epilogue 1 stores it ([batch][P]) and the fp32 second-layer output + bias before its transform ([batch][64 | 32 | 32 |
// A]).  The last kernel parameter, so that the parameters before it keep their offsets in every instantiation.
struct MlpTcCap {
  __half* mid[4][2];
  float* out[4][2];
};

__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  __half2 t = __floats2half2_rn(fminf(fmaxf(a, -65504.0f), 65504.0f), fminf(fmaxf(b, -65504.0f), 65504.0f));
  return *reinterpret_cast<uint32_t*>(&t);
}

// softmax expectation over a support of S <= 32 logits held by one thread, then the inverse value transform
__device__ __forceinline__ float support_scalar_regs(const float (&l)[32], int S) {
  if (S == 1) return l[0];
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < 32; ++i) if (i < S) m = fmaxf(m, l[i]);
  const int maxv = (S - 1) / 2;
  const float step = (float)(2 * maxv) / (float)(S - 1);
  float den = 0.0f, num = 0.0f;
#pragma unroll
  for (int i = 0; i < 32; ++i)
    if (i < S) {
      const float e = expf(l[i] - m);
      den += e;
      num += e * ((float)(-maxv) + step * (float)i);
    }
  return signed_parabolic(num / den);
}

// leaf gather: parent hidden state of row `row` of tile `tile` by slot index -> fp16 operand tile in shared memory
__device__ __forceinline__ void gather_tile(const MlpTcParams& p, int tile, int row, uint32_t sIn_a) {
  const int grow = tile * kTcRows + row;
  const bool live = grow < p.batch;
  const size_t slot = live ? (p.src_index ? (size_t)p.src_index[grow] : (size_t)grow) : 0;
  const float4* src = reinterpret_cast<const float4*>(p.hidden_in + slot * 64);
#pragma unroll
  for (int g = 0; g < 8; ++g) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    if (live) { a = src[2 * g]; b = src[2 * g + 1]; }
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sIn_a + (uint32_t)(g * 128 + row) * 16),
                 "r"(pack_h2(a.x, a.y)), "r"(pack_h2(a.z, a.w)), "r"(pack_h2(b.x, b.y)), "r"(pack_h2(b.z, b.w)) : "memory");
  }
}

// the same for one row whose slot is already known (persistent search kernel: the thread just selected the leaf)
__device__ __forceinline__ void gather_row(const float* hidden_in, size_t slot, bool live, int row, uint32_t sIn_a) {
  const float4* src = reinterpret_cast<const float4*>(hidden_in + slot * 64);
#pragma unroll
  for (int g = 0; g < 8; ++g) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
    if (live) { a = src[2 * g]; b = src[2 * g + 1]; }
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sIn_a + (uint32_t)(g * 128 + row) * 16),
                 "r"(pack_h2(a.x, a.y)), "r"(pack_h2(a.z, a.w)), "r"(pack_h2(b.x, b.y)), "r"(pack_h2(b.z, b.w)) : "memory");
  }
}

// What the persistent per-search form of the kernel needs besides the network: the pool whose trees it searches.
struct SearchArgs {
  PoolDev pool;
  int sims;                           // simulations to run (the pool's num_simulations)
};

// kSearch = false: recurrent_inference of `batch` rows (one launch per simulation of the launch-chain search, or a
// stand-alone network call).
// kSearch = true: ONE launch per SEARCH.  A CTA owns the trees of its 128-row tiles for all simulations: the thread that
// owns row i of the tile also owns tree i and runs its pUCT descent and its backup (tree_thread.cuh: thread-per-tree
// forms of the tree kernels, TA = compile-time bound on the number of actions) around the tensor-core chain
//   [backup of simulation s-1] -> select -> gather the leaf's parent state -> transition -> reward -> value -> ...
// so a simulation costs no launch, no prologue (TMEM allocation, bias / action-table staging, barrier set-up happen
// once per search) and the leaf action, reward and value never leave the thread's registers.  Trees of different
// CTAs never interact, so there is no inter-CTA synchronisation at all.
// kCap: the test instantiation that also copies every intermediate to the capture regions of MlpTcParams.
template <bool kSearch, int TA, bool kCap = false>
__global__ void __launch_bounds__(kTcThreads, 1) mlp_tc_kernel(const __grid_constant__ MlpTcParams p,
                                                               const __grid_constant__ SearchArgs sa,
                                                               const __grid_constant__ MlpTcCap cap) {
  extern __shared__ __align__(1024) unsigned char tsm[];
  unsigned char* sIn = tsm;                       // [8][128][16]  h_in   (fp16, K-major core matrices)
  unsigned char* sRaw = sIn + 16384;              // h_raw
  unsigned char* sNorm = sRaw + 16384;            // h' (normalised)
  unsigned char* sMid = sNorm + 16384;            // [32][128][16] hidden chunk
  unsigned char* sW = sMid + 65536;               // [kTcSlots][32 KB]
  uint64_t* w_full = reinterpret_cast<uint64_t*>(sW + kTcSlots * kTcSlotBytes);
  uint64_t* w_empty = w_full + kTcSlots;
  uint64_t* bar_mma = w_empty + kTcSlots;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bar_mma + 1);
  float* sB1 = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_holder + 4) + 15) & ~(uintptr_t)15);   // [4][P] first-layer biases
  float* sTab = sB1 + 4 * p.P;                                      // [A][P] action columns (when they fit)
  // search form: pb_c table (float64 [S + 2]) and the action each row's thread selected (read by the helper warps)
  double* sT = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(sTab + (p.tab_in_smem ? p.A * (p.P + 4) : 0)) + 15) & ~(uintptr_t)15);
  int* sAct = reinterpret_cast<int*>(sT + (kSearch ? 2 * (sa.sims + 2) : 0));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  int dbg_n = 0;
  auto stamp = [&]() { if (p.dbg && blockIdx.x == 0 && tid == 0 && dbg_n < 60) p.dbg[dbg_n++] = clock64(); };
  stamp();
  // the first tile's leaf gather (two dependent global round trips) overlaps the staging below and the TMEM allocation
  const int nsplit = kSearch ? 1 : p.nsplit, part = (int)blockIdx.x % nsplit;
  const int nsims = kSearch ? sa.sims : 1;
  // the nets this CTA runs, in order: everything, or transition + its share of the heads
  uint32_t net_list = 0;              // 4 bits per entry (an indexed array would live in local memory)
  int nn = 0;
  for (int n = 0; n < p.nnets; ++n)
    if (nsplit == 1 || n == 0 || (n == 1) == (part == 0)) net_list |= (uint32_t)n << (4 * nn++);
  auto net_at = [&](int ni) { return (int)((net_list >> (4 * ni)) & 15u); };
  const int bpn = 2 * p.chunks;       // weight blocks per net
  const int first_tile = (int)blockIdx.x / nsplit, tile_step = (int)gridDim.x / nsplit;
  pdl_trigger();          // the next kernel of the chain may start its own prologue now
  if (kSearch)
    for (int i = tid; i < 2 * (sa.sims + 2); i += kTcThreads) sT[i] = sa.pool.T[i];     // pb_c table, then RN(1/n)
  // first-layer biases and the action table are read by every row of every tile: stage them once per CTA
  // (from global they cost an exposed L2 round trip per 32-column chunk of every epilogue)
  for (int i = tid; i < p.nnets * p.P; i += kTcThreads) sB1[i] = p.b1[i / p.P][i % p.P];
  // rows of the table are padded by 4 floats: rows of a warp pick different actions, and with a stride of P floats
  // (a multiple of 32 banks) every action's column c sits in the same bank -- a 10-way conflict per float4
  const int tabP = p.P + 4;
  if (p.tab_in_smem)
    for (int i = tid; i < p.A * p.P; i += kTcThreads) sTab[(i / p.P) * tabP + i % p.P] = p.tabA[i];

  if (tid == 0) {
    for (int s = 0; s < kTcSlots; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 1); }
    mbar_init(bar_mma, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(tmem_holder, 512);
  // everything above is independent of the previous kernel of the stream (programmatic dependent launch: it overlaps
  // that kernel's tail); the leaf gather below reads what the tree kernel selected
  pdl_wait();
  // the first tile's leaf gather (two dependent global round trips) is issued before the prologue barrier
  if (!kSearch && tid < 128 && first_tile * kTcRows < p.batch) gather_tile(p, first_tile, tid, smem_u32(sIn));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_holder;
  const int ntiles = (p.batch + kTcRows - 1) / kTcRows;
  stamp();

  if (warp == kTcCompute / 32) {
    // ------------------------------------------------ weight producer
    if (lane == 0) {
      uint32_t it = 0;
      for (int tile = first_tile; tile < ntiles; tile += tile_step)
       for (int sim = 0; sim < nsims; ++sim)
        for (int ni = 0; ni < nn; ++ni)
          for (int b = net_at(ni) * bpn; b < (net_at(ni) + 1) * bpn; ++b, ++it) {
            const uint32_t s = it % kTcSlots, ph = (it / kTcSlots) & 1;
            mbar_wait(&w_empty[s], ph ^ 1);
            mbar_arrive_expect_tx(&w_full[s], p.blk_bytes[b]);
            bulk_g2s(sW + (size_t)s * kTcSlotBytes, p.wpack + p.blk_off[b], p.blk_bytes[b], &w_full[s]);
          }
    }
  } else {
    // ------------------------------------------------ compute: thread (warps 0-3) = row of the tile; warps 4-7 help
    // with epilogue 1, the longest serial piece of a tile (256 columns per row): a warp can only read the TMEM lanes
    // of its quadrant (warp % 4), so warp w + 4 takes columns 128..255 of the rows warp w owns
    const int row = tid & 127;
    const bool owner = tid < 128;
    const int qbeg = owner ? 0 : 4;
    const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);    // this warp's TMEM lanes
    const uint32_t sIn_a = smem_u32(sIn), sRaw_a = smem_u32(sRaw), sNorm_a = smem_u32(sNorm), sMid_a = smem_u32(sMid);
    uint32_t wit = 0, mma_ph = 0;
    auto bar128 = []() { asm volatile("bar.sync 1, 256;" ::: "memory"); };   // all compute warps
    // tid 0 issues `n` K-steps of D(+)= A.B^T on the weight block at the head of the ring, then every thread
    // waits for them (one mbarrier, alternating phase)
    // One warp issues the MMAs, and what it executes between two of them is latency the tensor pipe sits out: the K steps
    // are unrolled four to an election (compile-time count), the descriptors' high words built once per group and their
    // low words stepped by additions, the ring slot and its phase kept incrementally (csrc/train.cu, tools/issue_bench2.cu).
    uint32_t slot = 0, slot_ph = 0;
    auto mma_group = [&](uint32_t a_addr, auto ksteps_c, uint32_t dcol, uint32_t N, bool accumulate) {
      constexpr int ksteps = decltype(ksteps_c)::value;
      static_assert(ksteps % 4 == 0, "K steps are issued four to an election");
      if (warp == 0) {
        mbar_wait(&w_full[slot], slot_ph);
        tc_fence_after();
        const uint32_t idesc = instr_desc_f16(128, N);
        const uint64_t at = smem_desc(a_addr, 2048, 128), bt = smem_desc(smem_u32(sW) + slot * kTcSlotBytes, N * 16, 128);
        const uint32_t a_lo = (uint32_t)at, a_hi = (uint32_t)(at >> 32), b_lo = (uint32_t)bt, b_hi = (uint32_t)(bt >> 32);
        const uint32_t bs = 2u * N;                  // 32 N bytes per K step, in 16-byte units (A: 4096 bytes = 256 units)
        auto d64 = [](uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; };
#pragma unroll
        for (int ks = 0; ks < ksteps; ks += 4)
          mma4_f16_elect(tmem + dcol, d64(a_lo + ks * 256u, a_hi), d64(a_lo + (ks + 1) * 256u, a_hi), d64(a_lo + (ks + 2) * 256u, a_hi),
                         d64(a_lo + (ks + 3) * 256u, a_hi), d64(b_lo + ks * bs, b_hi), d64(b_lo + (ks + 1) * bs, b_hi),
                         d64(b_lo + (ks + 2) * bs, b_hi), d64(b_lo + (ks + 3) * bs, b_hi), idesc, (accumulate || ks > 0) ? 1u : 0u);
        commit_elect(&w_empty[slot]);
        commit_elect(bar_mma);
      }
      if (++slot == kTcSlots) { slot = 0; slot_ph ^= 1u; }
      ++wit;
      mbar_wait(bar_mma, mma_ph);
      mma_ph ^= 1;
      tc_fence_after();
    };

    TreeThreadStats tstats;
    const double* sR = sT + (kSearch ? sa.sims + 2 : 0);                   // RN(1/n)
    for (int tile = first_tile; tile < ntiles; tile += tile_step) {
      const int grow = tile * kTcRows + row;
      const bool live = grow < p.batch;
      float rew_reg = 0.0f, val_reg = 0.0f;       // reward / value of this row's last inference (search form)
      const int node0 = (kSearch && owner && live) ? sa.pool.count[grow] : 0;     // nodes of the tree so far (1 after a reset)
     for (int sim = 0; sim < nsims; ++sim) {
      int act;
      size_t dst_slot = 0;
      if (kSearch) stamp();
      if constexpr (kSearch) {
        // tree phase: this thread's tree -- backup of the previous simulation, then the descent of this one
        act = 0;
        if (owner) {
          size_t src_slot = 0;
          if (live) {
            if (sim > 0) expand_backup_tree_thread(sa.pool, grow, rew_reg, val_reg);
            stamp();
            const int2 leaf = select_tree_thread<TA>(sa.pool, grow, sT, sR, tstats);
            stamp();
            act = leaf.y;
            src_slot = (size_t)grow * sa.pool.max_nodes + leaf.x;
            dst_slot = (size_t)grow * sa.pool.max_nodes + min(node0 + sim, sa.pool.max_nodes - 1);
          }
          gather_row(p.hidden_in, src_slot, live, row, sIn_a);
          sAct[row] = act;
        }
      } else {
        // leaf gather (the CTA's first tile was gathered before the prologue barrier)
        if (owner && tile != first_tile) gather_tile(p, tile, row, sIn_a);
        act = live ? p.action[grow] : 0;
      }
      fence_proxy_async();
      tc_fence_before();
      bar128();
      if (kSearch && !owner) act = sAct[row];
      act = min(max(act, 0), p.A - 1);
      stamp();

      for (int ni = 0; ni < nn; ++ni) {
        const int net = net_at(ni);
        const uint32_t a_in = net == 0 ? sIn_a : (net == 1 ? sRaw_a : sNorm_a);
        const uint32_t N2 = net == 0 ? 64u : (net == 3 ? (uint32_t)p.Apad : 32u);
        const float* b1 = sB1 + net * p.P;
        const float* tab = net == 0 ? (p.tab_in_smem ? sTab + (size_t)act * tabP : p.tabA + (size_t)act * p.P) : nullptr;
        for (int c = 0; c < p.chunks; ++c) {
          mma_group(a_in, std::integral_constant<int, 4>{}, 0u, 256u, false);                        // D1 = A_in . W1c^T
          stamp();
          // epilogue 1: bias (+ action column) + ReLU -> fp16 hidden chunk in shared memory
#pragma unroll 1
          for (int q = qbeg; q < qbeg + 4; ++q) {
            uint32_t r[32];
            tmem_ld32(trow + (uint32_t)(q * 32), r);
            tmem_ld_wait();
            const int col0 = c * kTcChunk + q * 32;
            float v[32];
#pragma unroll
            for (int e = 0; e < 32; e += 4) {
              const float4 b4 = *reinterpret_cast<const float4*>(b1 + col0 + e);
              v[e] = __uint_as_float(r[e]) + b4.x; v[e + 1] = __uint_as_float(r[e + 1]) + b4.y;
              v[e + 2] = __uint_as_float(r[e + 2]) + b4.z; v[e + 3] = __uint_as_float(r[e + 3]) + b4.w;
            }
            if (tab) {
#pragma unroll
              for (int e = 0; e < 32; e += 4) {
                const float4 t4 = *reinterpret_cast<const float4*>(tab + col0 + e);
                v[e] += t4.x; v[e + 1] += t4.y; v[e + 2] += t4.z; v[e + 3] += t4.w;
              }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float* w = v + 8 * u;
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sMid_a + (uint32_t)((q * 4 + u) * 128 + row) * 16),
                           "r"(pack_h2(fmaxf(w[0], 0.f), fmaxf(w[1], 0.f))), "r"(pack_h2(fmaxf(w[2], 0.f), fmaxf(w[3], 0.f))),
                           "r"(pack_h2(fmaxf(w[4], 0.f), fmaxf(w[5], 0.f))), "r"(pack_h2(fmaxf(w[6], 0.f), fmaxf(w[7], 0.f))) : "memory");
            }
            if constexpr (kCap) {
              if (live) {
                uint4* dst = reinterpret_cast<uint4*>(cap.mid[net][part] + (size_t)grow * p.P + col0);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  const float* w = v + 8 * u;
                  dst[u] = make_uint4(pack_h2(fmaxf(w[0], 0.f), fmaxf(w[1], 0.f)), pack_h2(fmaxf(w[2], 0.f), fmaxf(w[3], 0.f)),
                                      pack_h2(fmaxf(w[4], 0.f), fmaxf(w[5], 0.f)), pack_h2(fmaxf(w[6], 0.f), fmaxf(w[7], 0.f)));
                }
              }
            }
          }
          fence_proxy_async();
          tc_fence_before();
          bar128();
          stamp();
          mma_group(sMid_a, std::integral_constant<int, 16>{}, 256u, N2, c > 0);                     // D2 (+)= A_mid . W2c^T
          stamp();
        }
        // epilogue 2
        const float* b2 = p.b2[net];
        if (!owner) {
          // helpers have no part in the second-layer epilogues
        } else if (net == 0) {
          // transition output: h_raw (for the reward net) and its min-max normalisation (util.py:31-36)
          float h[64];
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            uint32_t r[32];
            tmem_ld32(trow + 256u + (uint32_t)(q * 32), r);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 32; ++e) h[q * 32 + e] = __uint_as_float(r[e]) + __ldg(b2 + q * 32 + e);
          }
          if constexpr (kCap) {
            if (live) {
              float4* dst = reinterpret_cast<float4*>(cap.out[0][part] + (size_t)grow * 64);
#pragma unroll
              for (int g = 0; g < 16; ++g) dst[g] = make_float4(h[4 * g], h[4 * g + 1], h[4 * g + 2], h[4 * g + 3]);
            }
          }
          stamp();
          float mn = INFINITY, mx = -INFINITY;
#pragma unroll
          for (int e = 0; e < 64; ++e) { mn = fminf(mn, h[e]); mx = fmaxf(mx, h[e]); }
          // (h - min) * (1 / den): 64 IEEE divisions per row serialise behind their slow-path checks (measured 10 k
          // cycles of a 42 k-cycle tile with only the four row-owner warps active); the product differs from the
          // quotient by at most 1 ulp of fp32, three orders of magnitude below the fp16 operand rounding
          const float inv = __fdiv_rn(1.0f, __fadd_rn(__fsub_rn(mx, mn), 1e-8f));
#pragma unroll
          for (int g = 0; g < 8; ++g)
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sRaw_a + (uint32_t)(g * 128 + row) * 16),
                         "r"(pack_h2(h[8 * g], h[8 * g + 1])), "r"(pack_h2(h[8 * g + 2], h[8 * g + 3])),
                         "r"(pack_h2(h[8 * g + 4], h[8 * g + 5])), "r"(pack_h2(h[8 * g + 6], h[8 * g + 7])) : "memory");
#pragma unroll
          for (int e = 0; e < 64; ++e) h[e] = __fmul_rn(__fsub_rn(h[e], mn), inv);
#pragma unroll
          for (int g = 0; g < 8; ++g)
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sNorm_a + (uint32_t)(g * 128 + row) * 16),
                         "r"(pack_h2(h[8 * g], h[8 * g + 1])), "r"(pack_h2(h[8 * g + 2], h[8 * g + 3])),
                         "r"(pack_h2(h[8 * g + 4], h[8 * g + 5])), "r"(pack_h2(h[8 * g + 6], h[8 * g + 7])) : "memory");
          stamp();
          if (live && part == 0) {
            const size_t slot = kSearch ? dst_slot : (p.dst_index ? (size_t)p.dst_index[grow] : (size_t)grow);
            float4* dst = reinterpret_cast<float4*>(p.hidden_out + slot * 64);
#pragma unroll
            for (int g = 0; g < 16; ++g) dst[g] = make_float4(h[4 * g], h[4 * g + 1], h[4 * g + 2], h[4 * g + 3]);
          }
          stamp();
        } else if (net == 1 || net == 2) {
          uint32_t r[32];
          tmem_ld32(trow + 256u, r);
          tmem_ld_wait();
          const int S = net == 1 ? p.Sr : p.Sv;
          float l[32];
#pragma unroll
          for (int e = 0; e < 32; ++e) l[e] = __uint_as_float(r[e]) + (e < S ? __ldg(b2 + e) : 0.0f);
          if constexpr (kCap) {
            if (live) {
#pragma unroll
              for (int e = 0; e < 32; ++e)
                if (e < S) cap.out[net][part][(size_t)grow * 32 + e] = l[e];
            }
          }
          const float out = support_scalar_regs(l, S);
          if (kSearch) { if (net == 1) rew_reg = out; else val_reg = out; }
          else if (live) (net == 1 ? p.reward : p.value)[grow] = out;
        } else {
          // policy: softmax over A logits spread over Apad TMEM columns (three passes over TMEM)
          float m = -INFINITY, den = 0.0f;
          for (int pass = 0; pass < 3; ++pass)
            for (int q = 0; q * 32 < p.Apad; ++q) {
              uint32_t r[32];
              tmem_ld32(trow + 256u + (uint32_t)(q * 32), r);
              tmem_ld_wait();
#pragma unroll
              for (int e = 0; e < 32; ++e) {
                const int a = q * 32 + e;
                if (a < p.A) {
                  const float lg = __uint_as_float(r[e]) + __ldg(b2 + a);
                  if constexpr (kCap) {
                    if (pass == 0 && live) cap.out[3][part][(size_t)grow * p.A + a] = lg;
                  }
                  if (pass == 0) m = fmaxf(m, lg);
                  else if (pass == 1) den += expf(lg - m);
                  else if (live) p.pi[(size_t)grow * p.A + a] = expf(lg - m) / den;
                }
              }
            }
        }
        fence_proxy_async();
        tc_fence_before();
        bar128();
        stamp();
      }
     }   // simulations
      if (kSearch && owner && live) expand_backup_tree_thread(sa.pool, grow, rew_reg, val_reg);    // the last simulation
    }
    if constexpr (kSearch) {
      // statistics of this CTA's descents: one atomic per warp and counter
      if (owner) {
        unsigned n_live = 0;
        for (int tile = first_tile; tile < ntiles; tile += tile_step) n_live += (tile * kTcRows + row < p.batch) ? 1u : 0u;
        const unsigned d = __reduce_add_sync(0xffffffffu, tstats.depth), dr = __reduce_add_sync(0xffffffffu, tstats.draws);
        const unsigned tw = __reduce_add_sync(0xffffffffu, tstats.twists), nl = __reduce_add_sync(0xffffffffu, n_live);
        if (lane == 0) {
          atomicAdd(sa.pool.stats + 0, (unsigned long long)d);
          atomicAdd(sa.pool.stats + 1, (unsigned long long)nl * (unsigned long long)sa.sims);
          if (dr) atomicAdd(sa.pool.stats + 2, (unsigned long long)dr);
          if (tw) atomicAdd(sa.pool.stats + 3, (unsigned long long)tw);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  stamp();
  if (warp == 0) tmem_dealloc(tmem, 512);
}


// ---------------------------------------------------------------------------
// One launch per search, warp per tree (mz_search_run for MuZeroMLPNet with 5..32 actions when the batch fits one wave
// of 32-tree CTAs): a CTA of 32 warps owns 32 trees for ALL simulations.
//   tree phase : warp w runs tree w's backup (of the previous simulation) and pUCT descent -- the warp-per-tree code of
//                the tree kernels (tree_warp.cuh), 32 trees side by side on the SM -- and gathers the leaf's parent
//                state into row w of the operand tile;
//   net phase  : the tcgen05 chain of mlp_tc_kernel (transition -> reward -> value, hidden layer in chunks of 256) on a
//                128-row tile whose first 32 rows are the trees.  Those rows are TMEM lanes 0..31, which only warps with
//                warp % 4 == 0 can read: the 8 such warps split the 256 columns of the first-layer epilogue (32 each);
//                thread 0 issues the MMAs and, knowing when a weight slot is free (it waits for its own MMAs), also
//                issues the TMA loads of the weight ring -- no producer warp.
// Reward and value go back to the tree warps through shared memory.  Nothing is launched, allocated or staged per
// simulation and the trees never leave their SM; trees of different CTAs never interact (no inter-CTA synchronisation).
// ---------------------------------------------------------------------------
constexpr int kS32Trees = 32;
constexpr int kS32Threads = 1024;

__global__ void __launch_bounds__(kS32Threads, 1) mlp_search32_kernel(const __grid_constant__ MlpTcParams p,
                                                                      const __grid_constant__ SearchArgs sa) {
  extern __shared__ __align__(1024) unsigned char tsm[];
  unsigned char* sIn = tsm;                       // [8][128][16]  h_in   (fp16, K-major core matrices; rows 0..31 live)
  unsigned char* sRaw = sIn + 16384;              // h_raw
  unsigned char* sNorm = sRaw + 16384;            // h' (normalised)
  unsigned char* sMid = sNorm + 16384;            // [32][128][16] hidden chunk
  unsigned char* sW = sMid + 65536;               // [kTcSlots][32 KB]
  uint64_t* w_full = reinterpret_cast<uint64_t*>(sW + kTcSlots * kTcSlotBytes);
  uint64_t* bar_mma = w_full + kTcSlots;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bar_mma + 1);
  float* sB1 = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_holder + 4) + 15) & ~(uintptr_t)15);   // [3][P]
  float* sTab = sB1 + 4 * p.P;                    // [A][P + 4] action columns (when they fit)
  const int tabP = p.P + 4;
  double* sT = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(sTab + (p.tab_in_smem ? p.A * tabP : 0)) + 15) & ~(uintptr_t)15);
  const double* sR = sa.pool.T + (sa.sims + 2);   // RN(1/n): select_tree reads it with ld.global.nc (__ldg), so NOT the shared copy
  float* sRew = reinterpret_cast<float*>(sT + 2 * (sa.sims + 2));   // [32] reward of each tree's last inference
  float* sVal = sRew + kS32Trees;
  int* sAct = reinterpret_cast<int*>(sVal + kS32Trees);             // [32] action each tree selected
  unsigned long long* sDst = reinterpret_cast<unsigned long long*>(sAct + kS32Trees);   // [32] hidden slot of the new node
  float2* sMM = reinterpret_cast<float2*>(sDst + kS32Trees);        // [2][32] partial (min, max) of the transition output
  unsigned long long* s_stats = reinterpret_cast<unsigned long long*>(sMM + 2 * kS32Trees);   // [4]

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const PoolDev& pool = sa.pool;
  const int S = sa.sims;
  int dbg_n = 0;
  auto stamp = [&]() { if (p.dbg && blockIdx.x == 0 && tid == 0 && dbg_n < 62) p.dbg[dbg_n++] = clock64(); };
  stamp();
  // ---- prologue (once per search)
  for (int i = tid; i < 2 * (S + 2); i += kS32Threads) sT[i] = pool.T[i];
  for (int i = tid; i < 3 * p.P; i += kS32Threads) sB1[i] = p.b1[i / p.P][i % p.P];
  if (p.tab_in_smem)
    for (int i = tid; i < p.A * p.P; i += kS32Threads) sTab[(i / p.P) * tabP + i % p.P] = p.tabA[i];
  for (int i = tid; i < (3 * 16384 + 65536) / 16; i += kS32Threads)       // operand tiles: rows 32..127 stay zero
    reinterpret_cast<int4*>(tsm)[i] = make_int4(0, 0, 0, 0);
  if (tid < 4) s_stats[tid] = 0;
  if (tid == 0) {
    for (int s = 0; s < kTcSlots; ++s) mbar_init(&w_full[s], 1);
    mbar_init(bar_mma, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(tmem_holder, 512);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_holder;
  const uint32_t sIn_a = smem_u32(sIn), sRaw_a = smem_u32(sRaw), sNorm_a = smem_u32(sNorm), sMid_a = smem_u32(sMid);
  const int bps = p.nblk;                           // weight blocks per simulation (3 nets x chunks x 2 layers)
  const int ntiles = (p.batch + kS32Trees - 1) / kS32Trees;
  int my_tiles = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) ++my_tiles;
  const long long total_blocks = (long long)my_tiles * S * bps;
  long long gb = 0;                                 // weight blocks consumed so far (thread 0's view == everyone's)
  uint32_t mma_ph = 0;
  // thread 0: fill slot (g % kTcSlots) with block g of the CTA's block stream
  auto issue_block = [&](long long g) {
    const int b = (int)(g % bps), s = (int)(g % kTcSlots);
    mbar_arrive_expect_tx(&w_full[s], p.blk_bytes[b]);
    bulk_g2s(sW + (size_t)s * kTcSlotBytes, p.wpack + p.blk_off[b], p.blk_bytes[b], &w_full[s]);
  };
  if (tid == 0)
    for (long long g = 0; g < kTcSlots && g < total_blocks; ++g) issue_block(g);
  // D (+)= A . B^T on the weight block at the head of the stream; the epilogue warps wait for the MMAs, thread 0 then
  // refills the slot they just released
  const bool epi = (warp & 3) == 0;                 // warps whose TMEM lane quadrant holds the 32 live rows
  const int ej = warp >> 2;                         // 0..7: this epilogue warp's 32-column share of 256 columns
  auto mma_group = [&](uint32_t a_addr, int ksteps, uint32_t dcol, uint32_t N, bool accumulate) {
    if (warp == 0) {
      // the WHOLE warp walks the issue loop and one lane is elected inside each tcgen05 asm statement: an `if (tid == 0)`
      // around the MMAs makes ptxas wrap every UTCHMMA in a convergence loop (~100 cycles per MMA, measured 1.6 k cycles
      // for the 16 MMAs of a second layer that the tensor pipe finishes in 0.5 k)
      const int s = (int)(gb % kTcSlots);
      mbar_wait(&w_full[s], (uint32_t)((gb / kTcSlots) & 1));
      tc_fence_after();
      const uint32_t idesc = instr_desc_f16(128, N);
      const uint32_t b_addr = smem_u32(sW) + (uint32_t)s * kTcSlotBytes;
      for (int ks = 0; ks < ksteps; ++ks) {
        const uint64_t ad = smem_desc(a_addr + (uint32_t)ks * 4096u, 2048, 128);
        const uint64_t bd = smem_desc(b_addr + (uint32_t)ks * 32u * N, N * 16, 128);
        mma_f16_elect(tmem + dcol, ad, bd, idesc, (accumulate || ks > 0) ? 1u : 0u);
      }
      commit_elect(bar_mma);
    }
    if (epi) {
      mbar_wait(bar_mma, mma_ph);
      tc_fence_after();
      if (tid == 0 && gb + kTcSlots < total_blocks) issue_block(gb + kTcSlots);
    }
    mma_ph ^= 1;
    ++gb;
  };

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int t = tile * kS32Trees + warp;          // this warp's tree
    const bool live = t < p.batch;
    const int node0 = live ? pool.count[t] : 0;     // nodes of the tree so far (1 after a reset)
    for (int sim = 0; sim < S; ++sim) {
      stamp();
      // ---------------- tree phase: one warp per tree
      size_t src_slot = 0;
      if (live) {
        if (sim > 0) { expand_backup_tree(pool, t, lane, sRew[warp], sVal[warp]); __syncwarp(); }
        stamp();
        const int2 leaf = select_tree<1>(pool, t, lane, sT, sR, nullptr, s_stats);
        stamp();
        src_slot = (size_t)t * pool.max_nodes + leaf.x;
        if (lane == 0) {
          sAct[warp] = leaf.y;
          sDst[warp] = (unsigned long long)t * pool.max_nodes + min(node0 + sim, pool.max_nodes - 1);
        }
      } else if (lane == 0) {
        sAct[warp] = 0;
      }
      // leaf gather: 64 floats of the parent's state -> row `warp` of the fp16 operand tile (lane l: floats 4l..4l+3)
      if (lane < 16) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (live) v = reinterpret_cast<const float4*>(p.hidden_in + src_slot * 64)[lane];
        asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(sIn_a + (uint32_t)((lane >> 1) * 128 + warp) * 16 + (lane & 1) * 8),
                     "r"(pack_h2(v.x, v.y)), "r"(pack_h2(v.z, v.w)) : "memory");
      }
      fence_proxy_async();
      tc_fence_before();
      __syncthreads();
      tc_fence_after();
      stamp();
      // ---------------- net phase
      const int row = lane;                         // epilogue threads: lane == row of the tile == tree of the tile
      const uint32_t trow = tmem;                   // TMEM lanes 0..31
      int act = sAct[row];
      act = min(max(act, 0), p.A - 1);
      for (int net = 0; net < 3; ++net) {
        const uint32_t a_in = net == 0 ? sIn_a : (net == 1 ? sRaw_a : sNorm_a);
        const uint32_t N2 = net == 0 ? 64u : 32u;
        const float* b1 = sB1 + net * p.P;
        const float* tab = net == 0 ? (p.tab_in_smem ? sTab + (size_t)act * tabP : p.tabA + (size_t)act * p.P) : nullptr;
        for (int c = 0; c < p.chunks; ++c) {
          mma_group(a_in, 4, 0u, 256u, false);                        // D1 = A_in . W1c^T
          stamp();
          if (epi) {
            // epilogue 1: bias (+ action column) + ReLU -> fp16 hidden chunk; this warp's 32 of the 256 columns
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              uint32_t r[16];
              tmem_ld16(trow + (uint32_t)(ej * 32 + half * 16), r);
              tmem_ld_wait();
              const int col0 = c * kTcChunk + ej * 32 + half * 16;
              float v[16];
#pragma unroll
              for (int e = 0; e < 16; e += 4) {
                const float4 b4 = *reinterpret_cast<const float4*>(b1 + col0 + e);
                v[e] = __uint_as_float(r[e]) + b4.x; v[e + 1] = __uint_as_float(r[e + 1]) + b4.y;
                v[e + 2] = __uint_as_float(r[e + 2]) + b4.z; v[e + 3] = __uint_as_float(r[e + 3]) + b4.w;
              }
              if (tab) {
#pragma unroll
                for (int e = 0; e < 16; e += 4) {
                  const float4 t4 = *reinterpret_cast<const float4*>(tab + col0 + e);
                  v[e] += t4.x; v[e + 1] += t4.y; v[e + 2] += t4.z; v[e + 3] += t4.w;
                }
              }
#pragma unroll
              for (int u = 0; u < 2; ++u) {
                const float* w = v + 8 * u;
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sMid_a + (uint32_t)((ej * 4 + half * 2 + u) * 128 + row) * 16),
                             "r"(pack_h2(fmaxf(w[0], 0.f), fmaxf(w[1], 0.f))), "r"(pack_h2(fmaxf(w[2], 0.f), fmaxf(w[3], 0.f))),
                             "r"(pack_h2(fmaxf(w[4], 0.f), fmaxf(w[5], 0.f))), "r"(pack_h2(fmaxf(w[6], 0.f), fmaxf(w[7], 0.f))) : "memory");
              }
            }
          }
          fence_proxy_async();
          tc_fence_before();
          __syncthreads();
          tc_fence_after();
          stamp();
          mma_group(sMid_a, 16, 256u, N2, c > 0);                     // D2 (+)= A_mid . W2c^T
          stamp();
        }
        // epilogue 2
        const float* b2 = p.b2[net];
        if (net == 0) {
          // transition output: warps 0 and 4 take 32 of its 64 columns each; h_raw (for the reward net) and its
          // min-max normalisation (util.py:31-36) over all 64, combined through shared memory
          if (epi && ej < 2) {
            float h[32];
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              uint32_t r[16];
              tmem_ld16(trow + 256u + (uint32_t)(ej * 32 + half * 16), r);
              tmem_ld_wait();
#pragma unroll
              for (int e = 0; e < 16; ++e) h[half * 16 + e] = __uint_as_float(r[e]) + __ldg(b2 + ej * 32 + half * 16 + e);
            }
            float mn = INFINITY, mx = -INFINITY;
#pragma unroll
            for (int e = 0; e < 32; ++e) { mn = fminf(mn, h[e]); mx = fmaxf(mx, h[e]); }
            sMM[ej * kS32Trees + row] = make_float2(mn, mx);
#pragma unroll
            for (int g = 0; g < 4; ++g)
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sRaw_a + (uint32_t)((ej * 4 + g) * 128 + row) * 16),
                           "r"(pack_h2(h[8 * g], h[8 * g + 1])), "r"(pack_h2(h[8 * g + 2], h[8 * g + 3])),
                           "r"(pack_h2(h[8 * g + 4], h[8 * g + 5])), "r"(pack_h2(h[8 * g + 6], h[8 * g + 7])) : "memory");
            asm volatile("bar.sync 1, 64;" ::: "memory");              // warps 0 and 4
            const float2 o = sMM[(ej ^ 1) * kS32Trees + row];
            mn = fminf(mn, o.x); mx = fmaxf(mx, o.y);
            // (h - min) * (1 / den), as mlp_tc_kernel does (bit-identical hidden states)
            const float inv = __fdiv_rn(1.0f, __fadd_rn(__fsub_rn(mx, mn), 1e-8f));
#pragma unroll
            for (int e = 0; e < 32; ++e) h[e] = __fmul_rn(__fsub_rn(h[e], mn), inv);
#pragma unroll
            for (int g = 0; g < 4; ++g)
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sNorm_a + (uint32_t)((ej * 4 + g) * 128 + row) * 16),
                           "r"(pack_h2(h[8 * g], h[8 * g + 1])), "r"(pack_h2(h[8 * g + 2], h[8 * g + 3])),
                           "r"(pack_h2(h[8 * g + 4], h[8 * g + 5])), "r"(pack_h2(h[8 * g + 6], h[8 * g + 7])) : "memory");
            if (tile * kS32Trees + row < p.batch) {
              float4* dst = reinterpret_cast<float4*>(p.hidden_out + sDst[row] * 64 + ej * 32);
#pragma unroll
              for (int g = 0; g < 8; ++g) dst[g] = make_float4(h[4 * g], h[4 * g + 1], h[4 * g + 2], h[4 * g + 3]);
            }
          }
        } else if (warp == 0) {
          float l[32];
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            uint32_t r[16];
            tmem_ld16(trow + 256u + (uint32_t)(half * 16), r);
            tmem_ld_wait();
            const int Sn = net == 1 ? p.Sr : p.Sv;
#pragma unroll
            for (int e = 0; e < 16; ++e) l[half * 16 + e] = __uint_as_float(r[e]) + (half * 16 + e < Sn ? __ldg(b2 + half * 16 + e) : 0.0f);
          }
          const float out = support_scalar_regs(l, net == 1 ? p.Sr : p.Sv);
          (net == 1 ? sRew : sVal)[row] = out;
        }
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
      }
    }   // simulations
    if (live) expand_backup_tree(pool, t, lane, sRew[warp], sVal[warp]);     // the last simulation
    __syncthreads();
  }
  flush_stats(pool, s_stats);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

// W [out x in_total] fp32 (row-major, PyTorch Linear.weight) -> fp16 block [K/8][N][8]:
// rows n0 .. n0+N-1 (zero beyond `out`), input columns k0 .. k0+K-1
__global__ void pack_linear_kernel(const float* __restrict__ w, __half* __restrict__ dst, int out, int in_total, int n0,
                                   int N, int k0, int K) {
  const int total = K * N;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int e = i % 8, n = (i / 8) % N, g = i / (8 * N);
    const int k = k0 + g * 8 + e, row = n0 + n;
    const float v = (row < out) ? w[(size_t)row * in_total + k] : 0.0f;
    dst[i] = __float2half_rn(fminf(fmaxf(v, -65504.0f), 65504.0f));
  }
}
// tab[a][p] = W1[p][HD + a]
__global__ void action_column_kernel(const float* __restrict__ w, float* __restrict__ tab, int P, int HD, int A) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < A * P) {
    const int a = i / P, pp = i % P;
    tab[i] = w[(size_t)pp * (HD + A) + HD + a];
  }
}


// ---------------------------------------------------------------------------
struct MlpNet : NetImpl {
  MlpDev d;
  size_t smem;
  bool tc = false;                  // tcgen05 recurrent path available for these dimensions
  MlpTcParams tcp;
  int tc_blocks_no_policy = 0, tc_blocks_policy = 0, num_sms = 148;
  size_t tc_smem = 0;

  // ---- test aid (mz_net_debug_capture): every intermediate of a call in a region of its own ----
  // Nets of a record: 0 representation, 1 transition, 2 reward, 3 value, 4 policy.  Layers: 0 the hidden layer (bias,
  // action column, ReLU), 1 the second Linear + bias before its transform, 2 the normalised state (SIMT kernels).
  char* cap_buf = nullptr;
  size_t cap_size = 0, cap_used = 0;
  bool cap_full = false;
  std::vector<mz_debug_tensor> cap_tensors;
  std::vector<mz_debug_launch> cap_launches;
  bool capturing() const { return cap_buf != nullptr; }
  void cap_begin() { cap_used = 0; cap_full = false; cap_tensors.clear(); cap_launches.clear(); }
  // a region [batch][stride] for one tensor and its record (nullptr and cap_full: the buffer is too small)
  void* cap_take(int net, int layer, int batch, int cols, int stride, int ebytes, int part, int src) {
    const size_t bytes = align_up((size_t)batch * stride * ebytes, 256);
    if (cap_full || cap_used + bytes > cap_size) { cap_full = true; return nullptr; }
    void* r = cap_buf + cap_used;
    cap_used += bytes;
    mz_debug_tensor t = {};
    t.ptr = r; t.kind = MZ_DEBUG_MLP; t.stage = net; t.index = layer; t.plane_rows = batch; t.groups = cols;
    t.h = stride; t.w = ebytes; t.batch = part; t.src = src; t.residual = -1;
    cap_tensors.push_back(t);
    return r;
  }
  int cap_last() const { return (int)cap_tensors.size() - 1; }
  int cap_fail() {
    set_error("mz_net_debug_capture: buffer of %zu bytes too small", cap_size);
    return MZ_ENOMEM;
  }
  void cap_launch(int recurrent, int tile_rows, int nsplit, int grid, int tiles, int chunks, int nets, bool policy,
                  int tab_in_smem, int batch) {
    mz_debug_launch L = {};
    L.num_layers = nets; L.tile_rows = tile_rows; L.pair = nsplit; L.grid = grid; L.num_tiles = tiles;
    L.multi_pass = chunks; L.n = policy ? 1 : 0; L.resident = tab_in_smem; L.sub = recurrent;
    L.h = d.P; L.w = d.A; L.batch = batch;
    cap_launches.push_back(L);
  }
  // the regions of a SIMT call (slots of MlpSimtCap), recorded in execution order
  MlpSimtCap cap_simt(bool recurrent, int batch, bool policy) {
    MlpSimtCap c = {};
    const int net0 = recurrent ? 1 : 0;
    c.t[kCapNet0L0] = (float*)cap_take(net0, 0, batch, d.P, d.P, 4, 0, -1);
    const int l0 = cap_last();
    c.t[kCapNet0L1] = (float*)cap_take(net0, 1, batch, d.HD, d.HD, 4, 0, l0);
    const int raw = cap_last();
    if (recurrent) {
      c.t[kCapRewL0] = (float*)cap_take(2, 0, batch, d.P, d.P, 4, 0, raw);
      c.t[kCapRewL1] = (float*)cap_take(2, 1, batch, d.Sr, d.Sr, 4, 0, cap_last());
    }
    c.t[kCapNorm] = (float*)cap_take(net0, 2, batch, d.HD, d.HD, 4, 0, raw);
    const int norm = cap_last();
    if (policy) {
      c.t[kCapPolL0] = (float*)cap_take(4, 0, batch, d.P, d.P, 4, 0, norm);
      c.t[kCapPolL1] = (float*)cap_take(4, 1, batch, d.A, d.A, 4, 0, cap_last());
    }
    c.t[kCapValL0] = (float*)cap_take(3, 0, batch, d.P, d.P, 4, 0, norm);
    c.t[kCapValL1] = (float*)cap_take(3, 1, batch, d.Sv, d.Sv, 4, 0, cap_last());
    return c;
  }
  // the regions of a tcgen05 call: per CTA part, the nets it runs (value and policy read the normalisation of their
  // part's transition output)
  void cap_tc(const MlpTcParams& q, MlpTcCap& c) {
    const int S2[4] = {64, 32, 32, q.A};
    const int cols2[4] = {64, q.Sr, q.Sv, q.A};
    for (int part = 0; part < q.nsplit; ++part) {
      int raw = -1;
      for (int n = 0; n < q.nnets; ++n) {
        if (!(q.nsplit == 1 || n == 0 || (n == 1) == (part == 0))) continue;
        c.mid[n][part] = (__half*)cap_take(n + 1, 0, q.batch, q.P, q.P, 2, part, n == 0 ? -1 : raw);
        c.out[n][part] = (float*)cap_take(n + 1, 1, q.batch, cols2[n], S2[n], 4, part, cap_last());
        if (n == 0) raw = cap_last();
      }
    }
  }
  int debug_capture_bytes(int batch, size_t* bytes) override {
    // more than any one call takes: the SIMT kernels' nine fp32 regions, or the tcgen05 kernel's eight fp16 hidden
    // layers and eight fp32 outputs (two CTA parts)
    const int m = std::max(std::max(std::max(d.P, d.HD), std::max(d.A, 64)), std::max(d.Sv, d.Sr));
    const size_t simt = (size_t)kCapSlots * align_up((size_t)batch * m * 4, 256);
    const size_t tc_b = 8 * align_up((size_t)batch * d.P * 2, 256) + 8 * align_up((size_t)batch * std::max(d.A, 64) * 4, 256);
    *bytes = std::max(simt, tc_b);
    return MZ_OK;
  }
  int debug_capture(void* buf, size_t bytes) override {
    cap_buf = (char*)buf; cap_size = buf ? bytes : 0;
    cap_begin();
    return MZ_OK;
  }
  int debug_tensor(int index, mz_debug_tensor* out, int32_t* count) override {
    *count = (int32_t)cap_tensors.size();
    if (index < 0) return MZ_OK;
    MZ_CHECK_ARG(index < *count, "tensor %d of %d", index, *count);
    *out = cap_tensors[index];
    return MZ_OK;
  }
  int debug_launch(int index, mz_debug_launch* out, int32_t* count) override {
    *count = (int32_t)cap_launches.size();
    if (index < 0) return MZ_OK;
    MZ_CHECK_ARG(index < *count, "launch %d of %d", index, *count);
    *out = cap_launches[index];
    return MZ_OK;
  }

  int search(mz_pool* pool, cudaStream_t st) override;
  int initial(int batch, const float* obs, void* hidden_out, const int32_t* dst_index, float* pi_probs,
              float* value, cudaStream_t st) override {
    MlpSimtCap cap = {};
    const int grid = (batch + kRows - 1) / kRows;
    if (capturing()) {
      cap_begin();
      cap = cap_simt(false, batch, pi_probs != nullptr);
      if (cap_full) return cap_fail();
      cap_launch(0, kRows, 1, grid, grid, 0, pi_probs ? 3 : 2, pi_probs != nullptr, 0, batch);
    }
    prof_mark(kProfMlp, st);
    RootSetup rs;
    if (pending_root) rs = *pending_root; else rs.enabled = 0;
    mlp_initial_kernel<<<grid, kInitThreads, smem, st>>>(d, batch, obs, (float*)hidden_out, dst_index, pi_probs, value,
                                                         rs, cap);
    prof_mark(-1, st);
    MZ_LAUNCH_CHECK("mlp_initial_kernel");
    return MZ_OK;
  }
  int recurrent(int batch, const void* hidden_in, const int32_t* src_index, const int32_t* action, void* hidden_out,
                const int32_t* dst_index, float* reward, float* value, float* pi_probs, cudaStream_t st) override {
    if (capturing()) cap_begin();
    if (tc && (pi_probs == nullptr || tc_blocks_policy > 0)) {
      MlpTcParams q = tcp;
      q.batch = batch; q.hidden_in = (const float*)hidden_in; q.src_index = src_index; q.action = action;
      q.hidden_out = (float*)hidden_out; q.dst_index = dst_index; q.reward = reward; q.value = value; q.pi = pi_probs;
      q.nnets = pi_probs ? 4 : 3;
      q.nblk = pi_probs ? tc_blocks_policy : tc_blocks_no_policy;
      const int ntiles = (batch + kTcRows - 1) / kTcRows;
      // few tiles: two CTAs per tile share the heads (the four nets of a tile otherwise run back to back on one SM)
      static const bool no_split = getenv("MZ_MLP_NO_SPLIT") != nullptr;
      q.nsplit = (!no_split && 2 * ntiles <= num_sms) ? 2 : 1;
      static const bool debug = getenv("MZ_MLP_DEBUG") != nullptr;
      q.dbg = nullptr;
      if (debug) { cudaMalloc(&q.dbg, 64 * sizeof(long long)); cudaMemset(q.dbg, 0, 64 * sizeof(long long)); }
      prof_mark(kProfMlp, st);
      SearchArgs none;
      none.sims = 0;
      // programmatic dependent launch only while the grid leaves SMs free: CTAs of a dependent kernel that start early
      // sit on their SMs spinning until the predecessor drains, and with one 208 KB CTA per SM on most of the GPU
      // (CartPole, 128 tiles) they held up the kernels they were waiting for (172 -> 120 M simulations/s)
      const int grid = q.nsplit == 2 ? 2 * ntiles : (ntiles < num_sms ? ntiles : num_sms);
      MlpTcCap cap = {};
      if (capturing()) {
        cap_tc(q, cap);
        if (cap_full) return cap_fail();
        cap_launch(1, kTcRows, q.nsplit, grid, ntiles, q.chunks, q.nnets, pi_probs != nullptr, q.tab_in_smem, batch);
      }
      launch_pdl(2 * grid <= num_sms, capturing() ? mlp_tc_kernel<false, 4, true> : mlp_tc_kernel<false, 4>, dim3(grid),
                 dim3(kTcThreads), tc_smem, st, q, none, cap);
      prof_mark(-1, st);
      MZ_LAUNCH_CHECK("mlp_recurrent_tc_kernel");
      if (debug) {   // measurement aid: cycle stamps of CTA 0 (start, prologue, gather, then per net: MMA1, epi1, MMA2, epi2; end)
        cudaDeviceSynchronize();
        long long h[64];
        cudaMemcpy(h, q.dbg, sizeof(h), cudaMemcpyDeviceToHost);
        cudaFree(q.dbg);
        fprintf(stderr, "[mlp dbg] cycles since start:");
        for (int i = 1; i < 64 && h[i]; ++i) fprintf(stderr, " %lld", h[i] - h[0]);
        fprintf(stderr, "\n");
      }
      return MZ_OK;
    }
    MlpSimtCap cap = {};
    const int grid = (batch + kRows - 1) / kRows;
    if (capturing()) {
      cap = cap_simt(true, batch, pi_probs != nullptr);
      if (cap_full) return cap_fail();
      cap_launch(1, kRows, 1, grid, grid, 0, pi_probs ? 4 : 3, pi_probs != nullptr, 0, batch);
    }
    prof_mark(kProfMlp, st);
    mlp_recurrent_kernel<<<grid, kThreads, smem, st>>>(d, batch, (const float*)hidden_in, src_index, action,
                                                       (float*)hidden_out, dst_index, reward, value, pi_probs, cap);
    prof_mark(-1, st);
    MZ_LAUNCH_CHECK("mlp_recurrent_kernel");
    return MZ_OK;
  }
};

int MlpNet::search(mz_pool* pool, cudaStream_t st) {
  // mode: -1 auto (one launch where it measured faster: the warp-per-tree kernel), 0 launch chain, 1 one launch wherever a
  // kernel exists.  MZ_FUSED_SEARCH=0/1 in the environment overrides the handle's setting process-wide.
  static const int env_mode = getenv("MZ_FUSED_SEARCH") ? atoi(getenv("MZ_FUSED_SEARCH")) : -2;
  const int mode = env_mode >= 0 ? (env_mode != 0) : fused_search;
  if (mode == 0 || !tc || pool->A != d.A || pool->cfg.hidden_bytes != d.HD * 4) return 1;
  MlpTcParams q = tcp;
  q.batch = pool->B;
  q.hidden_in = (const float*)pool->view_ptr[MZ_VIEW_HIDDEN];
  q.hidden_out = (float*)pool->view_ptr[MZ_VIEW_HIDDEN];
  q.src_index = nullptr; q.dst_index = nullptr; q.action = nullptr; q.reward = nullptr; q.value = nullptr; q.pi = nullptr;
  q.nnets = 3;                       // the search never reads the recurrent policy (mcts.py:386)
  q.nblk = tc_blocks_no_policy;
  q.nsplit = 1;
  q.dbg = nullptr;
  SearchArgs sa;
  sa.pool = pool_dev(pool);
  sa.sims = pool->S;
  // (a) warp per tree, 32 trees per CTA: needs an action row that fills a useful part of a warp and a batch that fits
  // one wave of CTAs (every CTA runs its trees' whole search)
  const int ntiles32 = (pool->B + kS32Trees - 1) / kS32Trees;
  if (pool->A > 4 && pool->A <= 32 && ntiles32 <= num_sms) {
    const size_t smem32 = tc_smem + (size_t)(pool->S + 2) * 16 + 2048;
    if (smem32 <= 227 * 1024) {
      static const bool debug32 = getenv("MZ_MLP_DEBUG") != nullptr;
      if (debug32) { cudaMalloc(&q.dbg, 64 * sizeof(long long)); cudaMemset(q.dbg, 0, 64 * sizeof(long long)); }
      prof_mark(kProfMlp, st);
      mlp_search32_kernel<<<ntiles32, kS32Threads, smem32, st>>>(q, sa);
      prof_mark(-1, st);
      MZ_LAUNCH_CHECK("mlp_search32_kernel");
      if (debug32) {   // cycle stamps of CTA 0 / thread 0 (tree 0): start, then per simulation: start, backup done, select done, gather + barrier, per net: MMA1, epilogue 1 + barrier, MMA2
        cudaDeviceSynchronize();
        long long h[64];
        cudaMemcpy(h, q.dbg, sizeof(h), cudaMemcpyDeviceToHost);
        cudaFree(q.dbg);
        fprintf(stderr, "[mlp search32 dbg] cycles since start:");
        for (int i = 1; i < 64 && h[i]; ++i) fprintf(stderr, " %lld", h[i] - h[0]);
        fprintf(stderr, "\n");
      }
      return MZ_OK;
    }
  }
  // (b) thread per tree, 128 trees per CTA: measured slower than the launch chain at every size (DESIGN.md section 4),
  // so only on request
  if (mode != 1 || pool->A > 12) return 1;
  static const bool debug = getenv("MZ_MLP_DEBUG") != nullptr;
  if (debug) { cudaMalloc(&q.dbg, 64 * sizeof(long long)); cudaMemset(q.dbg, 0, 64 * sizeof(long long)); }
  const size_t smem_need = tc_smem + (size_t)(pool->S + 2) * 16 + kTcRows * sizeof(int) + 64;
  if (smem_need > 227 * 1024) return 1;
  const int ntiles = (pool->B + kTcRows - 1) / kTcRows;
  const int grid = ntiles < num_sms ? ntiles : num_sms;
  prof_mark(kProfMlp, st);
  const MlpTcCap no_cap = {};
  if (pool->A <= 4) mlp_tc_kernel<true, 4><<<grid, kTcThreads, smem_need, st>>>(q, sa, no_cap);
  else mlp_tc_kernel<true, 12><<<grid, kTcThreads, smem_need, st>>>(q, sa, no_cap);
  prof_mark(-1, st);
  MZ_LAUNCH_CHECK("mlp_tc_kernel<search>");
  if (debug) {   // cycle stamps of CTA 0 / thread 0: start, prologue, then per simulation: sim start, tree phase + gather done, ...
    cudaDeviceSynchronize();
    long long h[64];
    cudaMemcpy(h, q.dbg, sizeof(h), cudaMemcpyDeviceToHost);
    cudaFree(q.dbg);
    fprintf(stderr, "[mlp search dbg] cycles since start:");
    for (int i = 1; i < 64 && h[i]; ++i) fprintf(stderr, " %lld", h[i] - h[0]);
    fprintf(stderr, "\n");
  }
  return MZ_OK;
}

static int mlp_dims(const mz_net_config& c, int* in_dim) {
  MZ_CHECK_ARG(c.hidden_dim > 0 && c.hidden_dim % 4 == 0, "hidden_dim must be a positive multiple of 4, got %d",
               c.hidden_dim);
  MZ_CHECK_ARG(c.num_planes > 0 && c.num_actions > 0 && c.value_support > 0 && c.reward_support > 0,
               "bad MLP dimensions");
  *in_dim = c.in_channels * c.in_h * c.in_w;
  MZ_CHECK_ARG(*in_dim > 0, "bad observation shape");
  return MZ_OK;
}

int mlp_hidden_bytes(const mz_net_config& c, int32_t* bytes) {
  int in_dim;
  int rc = mlp_dims(c, &in_dim);
  if (rc) return rc;
  *bytes = c.hidden_dim * 4;
  return MZ_OK;
}

// shapes of the 20 state_dict tensors, in order (network.py:143-147,170-180,210-220)
static void mlp_shapes(const mz_net_config& c, int in_dim, int (*sh)[2]) {
  const int P = c.num_planes, H = c.hidden_dim, A = c.num_actions;
  const int s[20][2] = {{P, in_dim}, {P, 1}, {H, P}, {H, 1},
                        {P, H + A}, {P, 1}, {H, P}, {H, 1},
                        {P, H}, {P, 1}, {c.reward_support, P}, {c.reward_support, 1},
                        {P, H}, {P, 1}, {A, P}, {A, 1},
                        {P, H}, {P, 1}, {c.value_support, P}, {c.value_support, 1}};
  memcpy(sh, s, sizeof(s));
}

int mlp_arena_bytes(const mz_net_config& c, size_t* bytes) {
  int in_dim;
  int rc = mlp_dims(c, &in_dim);
  if (rc) return rc;
  int sh[20][2];
  mlp_shapes(c, in_dim, sh);
  size_t tot = 0;
  for (int i = 0; i < 20; ++i) tot += 2 * align_up((size_t)sh[i][0] * sh[i][1] * 4, 256);   // [out,in] + transposed
  // tcgen05 recurrent path: packed fp16 weight blocks (4 nets x chunks x 2 layers, <= 32 KB each) + action table
  tot += (size_t)4 * ((c.num_planes + kTcChunk - 1) / kTcChunk) * 2 * kTcSlotBytes +
         align_up((size_t)c.num_actions * c.num_planes * 4, 256) + 1024;
  *bytes = tot;
  return MZ_OK;
}

int mlp_create(const mz_net_config& c, const float* const* w, int nw, void* arena, size_t arena_bytes, NetImpl** out) {
  int in_dim;
  int rc = mlp_dims(c, &in_dim);
  if (rc) return rc;
  MZ_CHECK_ARG(nw == 20, "MuZeroMLPNet has 20 state_dict tensors, got %d", nw);
  size_t need;
  mlp_arena_bytes(c, &need);
  if (arena_bytes < need) { set_error("net arena too small: %zu < %zu", arena_bytes, need); return MZ_ENOMEM; }
  int sh[20][2];
  mlp_shapes(c, in_dim, sh);
  char* p = (char*)arena;
  const float* orig[20];
  const float* tr[20];
  for (int i = 0; i < 20; ++i) {
    const size_t n = (size_t)sh[i][0] * sh[i][1];
    float* o = (float*)p; p += align_up(n * 4, 256);
    float* t = (float*)p; p += align_up(n * 4, 256);
    MZ_CUDA(cudaMemcpy(o, w[i], n * 4, cudaMemcpyDeviceToDevice));
    if (sh[i][1] > 1) {
      transpose_kernel<<<(int)((n + 255) / 256), 256>>>(o, t, sh[i][0], sh[i][1]);
      MZ_LAUNCH_CHECK("transpose_kernel");
    }
    orig[i] = o; tr[i] = t;
  }
  MZ_CUDA(cudaDeviceSynchronize());
  MlpNet* net = new MlpNet();
  MlpDev& d = net->d;
  d.in_dim = in_dim; d.A = c.num_actions; d.P = c.num_planes; d.HD = c.hidden_dim;
  d.Sv = c.value_support; d.Sr = c.reward_support; d.in_pad = (in_dim + 3) & ~3;
  d.rep1_wt = tr[0];  d.rep1_b = orig[1];  d.rep2_wt = tr[2];  d.rep2_b = orig[3];
  d.dyn1_wt = tr[4];  d.dyn1_b = orig[5];  d.dyn2_wt = tr[6];  d.dyn2_b = orig[7];
  d.rew1_wt = tr[8];  d.rew1_b = orig[9];  d.rew2_wt = tr[10]; d.rew2_w = orig[10]; d.rew2_b = orig[11];
  d.pol1_wt = tr[12]; d.pol1_b = orig[13]; d.pol2_wt = tr[14]; d.pol2_w = orig[14]; d.pol2_b = orig[15];
  d.val1_wt = tr[16]; d.val1_b = orig[17]; d.val2_wt = tr[18]; d.val2_w = orig[18]; d.val2_b = orig[19];
  // ---- tcgen05 recurrent path (hidden 64, hidden layers in chunks of 256, supports and actions that fit one block)
  {
    const int P = d.P, A = d.A;
    const int apad = (A + 15) / 16 * 16;
    const char* simt = getenv("MZ_MLP_SIMT");
    // the transition, reward and value nets' 2 blocks per chunk must fit the kTcMaxBlocks entries of MlpTcParams (so
    // P <= 512), and the kernel's shared memory a block; wider nets run on the SIMT kernel
    const size_t tc_smem_base = 3 * 16384 + 65536 + (size_t)kTcSlots * kTcSlotBytes + 256 + (size_t)4 * P * 4;
    net->tc = d.HD == 64 && P % kTcChunk == 0 && 3 * (P / kTcChunk) * 2 <= kTcMaxBlocks && tc_smem_base <= 227 * 1024 &&
              d.Sr <= 32 && d.Sv <= 32 && !(simt && simt[0] == '1');
    if (net->tc) {
      const int chunks = P / kTcChunk;
      const bool pol = apad <= 64 && 4 * chunks * 2 <= kTcMaxBlocks;
      p = (char*)align_up((size_t)p, 1024);
      unsigned char* wp = (unsigned char*)p;
      MlpTcParams& q = net->tcp;
      memset(&q, 0, sizeof(q));
      q.wpack = wp; q.chunks = chunks; q.P = P; q.A = A; q.Apad = apad; q.Sr = d.Sr; q.Sv = d.Sv;
      const int w1_idx[4] = {4, 8, 16, 12}, in_tot[4] = {d.HD + A, d.HD, d.HD, d.HD};
      const int n2[4] = {64, 32, 32, apad}, out2[4] = {d.HD, d.Sr, d.Sv, A};
      size_t off = 0;
      int nb = 0;
      for (int net_i = 0; net_i < (pol ? 4 : 3); ++net_i) {
        q.b1[net_i] = orig[w1_idx[net_i] + 1];
        q.b2[net_i] = orig[w1_idx[net_i] + 3];
        for (int ch = 0; ch < chunks; ++ch) {
          if (nb + 2 > kTcMaxBlocks) {
            set_error("internal: MLP weight block %d of at most %d", nb + 1, kTcMaxBlocks);
            delete net;
            return MZ_EINVAL;
          }
          // layer 1 block: rows ch*256.., K = 64
          pack_linear_kernel<<<64, 256>>>(orig[w1_idx[net_i]], (__half*)(wp + off), P, in_tot[net_i], ch * kTcChunk,
                                          kTcChunk, 0, 64);
          MZ_LAUNCH_CHECK("pack_linear_kernel");
          q.blk_off[nb] = (uint32_t)off; q.blk_bytes[nb] = 64 * kTcChunk * 2; off += kTcSlotBytes; ++nb;
          // layer 2 block: N2 rows (zero-padded), input columns ch*256..
          pack_linear_kernel<<<64, 256>>>(orig[w1_idx[net_i] + 2], (__half*)(wp + off), out2[net_i], P, 0, n2[net_i],
                                          ch * kTcChunk, kTcChunk);
          MZ_LAUNCH_CHECK("pack_linear_kernel");
          q.blk_off[nb] = (uint32_t)off; q.blk_bytes[nb] = (uint32_t)(kTcChunk * n2[net_i] * 2); off += kTcSlotBytes; ++nb;
        }
        if (net_i == 2) net->tc_blocks_no_policy = nb;
      }
      net->tc_blocks_policy = pol ? nb : 0;
      p += off;
      float* tab = (float*)p; p += align_up((size_t)A * P * 4, 256);
      action_column_kernel<<<(A * P + 255) / 256, 256>>>(orig[4], tab, P, d.HD, A);
      MZ_LAUNCH_CHECK("action_column_kernel");
      q.tabA = tab;
      MZ_CUDA(cudaDeviceSynchronize());
      if ((size_t)(p - (char*)arena) > arena_bytes) { set_error("internal: MLP arena overrun"); delete net; return MZ_ENOMEM; }
      net->tc_smem = tc_smem_base;
      q.tab_in_smem = net->tc_smem + (size_t)A * (P + 4) * 4 <= 227 * 1024 ? 1 : 0;
      if (q.tab_in_smem) net->tc_smem += (size_t)A * (P + 4) * 4;
      int dev = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&net->num_sms, cudaDevAttrMultiProcessorCount, dev);
      const int smem_cap = 227 * 1024;
      MZ_CUDA(cudaFuncSetAttribute(mlp_tc_kernel<false, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_cap));
      MZ_CUDA(cudaFuncSetAttribute(mlp_tc_kernel<false, 4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_cap));
      MZ_CUDA(cudaFuncSetAttribute(mlp_tc_kernel<true, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_cap));
      MZ_CUDA(cudaFuncSetAttribute(mlp_tc_kernel<true, 12>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_cap));
      MZ_CUDA(cudaFuncSetAttribute(mlp_search32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_cap));
    }
  }
  net->smem = smem_bytes(d);
  if (net->smem > 227 * 1024) {
    set_error("MLP too wide for the fused kernel: needs %zu bytes of shared memory", net->smem);
    delete net;
    return MZ_EINVAL;
  }
  MZ_CUDA(cudaFuncSetAttribute(mlp_initial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)net->smem));
  MZ_CUDA(cudaFuncSetAttribute(mlp_recurrent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)net->smem));
  *out = net;
  return MZ_OK;
}

}  // namespace mz
