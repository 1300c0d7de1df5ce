// Training forward / backward of the ResNet towers of MuZeroBoardGameNet (network.py:273-300,353-395,398-470) for the
// K-step unroll of pipeline.py:541-612, on the Blackwell tensor cores.  SURVEY.md 8 f-2.
//
// What runs here: every 3x3 convolution of the representation / dynamics / prediction towers -- forward, data
// gradient and weight gradient as tcgen05 implicit GEMMs -- the train-mode BatchNorm + ReLU + residual around them,
// forward and backward, and the min-max normalisation of the hidden state (util.py:31-36) at the tower boundary, forward
// and backward.  The heads (1x1 convolution, BatchNorm, ReLU, Linear) and the optimizer step are in optim.cu; the losses
// and the two gradient-scale hooks stay PyTorch autograd (muzero_b200/train_engine.py, training.py).
//
// Layout: padded channel-group planes: a board is (H+1)*(W+1) positions, position q = y*(W+1) + x, column W and row H
// are a ZERO halo shared with the next row / board, an activation tensor is C/8 planes of [rows][8 channels] 16-bit.
// With zeros at the halo every 3x3 tap is an unmasked constant row offset in all three GEMMs:
//   forward   Y[P][co]    = sum_tap sum_ci  A[P + off(tap)][ci]  * W[co][ci][tap]          M = rows, N = co, K = 9*ci
//   dgrad     dA[P][ci]   = sum_tap sum_co dY[P + off(tap)][co]  * W[co][ci][8 - tap]      the same kernel, other weights
//   wgrad     dW[tap][co][ci] = sum_P     dY[P][co] * A[P + off(tap)][ci]                  M = co, N = ci, K = rows
// For forward / dgrad the planes are the no-swizzle K-major operand layout (as in conv.cu).  For wgrad K runs along
// the ROWS, and the very same planes are the no-swizzle MN-major operand layout (8 channels contiguous, consecutive
// K = consecutive 16-byte rows), so both operands are again plain 1-D bulk copies and a tap is a shifted start address.
// Every plane has `front` zero rows before row 0 and a zero tail, so that no tile needs a special case.
//
// Precision: activations and weights fp16 (like the inference engine; with bf16 the towers are 7e-3 instead of 8e-4 from
// fp32 at the same step time, DESIGN.md 4), gradients bf16 (fp32 range, no loss scaling), fp32 accumulation in TMEM,
// fp32 BatchNorm statistics and parameter gradients.
// kind::f16 MMAs take fp16 x fp16 or bf16 x bf16 but not a mix (an fp16 x bf16 descriptor raises an illegal-instruction
// fault), so every activation a weight gradient needs is ALSO kept as a bf16 copy, written by the kernel that produces
// it: the forward chain keeps fp16's three extra mantissa bits, dW = dY^T A runs bf16 x bf16.
#include "common.cuh"
#include "umma.cuh"
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <cstdlib>
#include <type_traits>
#include <vector>

namespace mz {
using namespace umma;

namespace {

constexpr int kC = 128;            // tower width this engine is built for
constexpr int kFront = 64;         // zero rows before row 0 of every plane (>= W + 2)
constexpr int kTail = 448;         // zero rows after the last 128-row tile (wgrad splits overshoot by < 16 * splits + halo)
constexpr int kSplits = 4;         // row splits of a weight-gradient launch
constexpr int kWgStage = 128;      // rows per wgrad pipeline stage
constexpr int kWgStages = 3;
constexpr int kConvStagesMax = 8;
constexpr float kBnEps = 1e-5f, kBnMomentum = 0.1f;
constexpr int kTimelineMax = 8192;
constexpr int kDyRing = 6;         // dY buffers in flight between the dgrad / BatchNorm chain and the weight-gradient streams
constexpr int kSideStreams = 3;    // weight-gradient launches alternate between these: consecutive ones may overlap

// ---- 16-bit element helpers: T = __half (forward tensors) or __nv_bfloat16 (gradients, wgrad operand copies) -------
template <typename T>
__device__ __forceinline__ float2 unpack2(uint32_t v) {
  if constexpr (std::is_same_v<T, __nv_bfloat16>) return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v));
  else return __half22float2(*reinterpret_cast<const __half2*>(&v));
}
template <typename T>
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  uint32_t d;
  if constexpr (std::is_same_v<T, __nv_bfloat16>) {
    __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
    d = *reinterpret_cast<uint32_t*>(&t);
  } else {
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
  }
  return d;
}
template <typename T>
__device__ __forceinline__ void unpack8(const int4& r, float (&v)[8]) {
  const uint32_t w[4] = {(uint32_t)r.x, (uint32_t)r.y, (uint32_t)r.z, (uint32_t)r.w};
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const float2 f = unpack2<T>(w[u]);
    v[2 * u] = f.x; v[2 * u + 1] = f.y;
  }
}
template <typename T>
__device__ __forceinline__ int4 pack8(const float* v) {
  return make_int4((int)pack2<T>(v[0], v[1]), (int)pack2<T>(v[2], v[3]), (int)pack2<T>(v[4], v[5]), (int)pack2<T>(v[6], v[7]));
}

// kind::f16 instruction descriptor with explicit operand formats (0 = fp16, 1 = bf16) and majors (1 = MN-major)
__host__ __device__ constexpr uint32_t idesc_of(uint32_t M, uint32_t N, uint32_t afmt, uint32_t bfmt, uint32_t mn_major) {
  return (1u << 4) | (afmt << 7) | (bfmt << 10) | (mn_major << 15) | (mn_major << 16) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// Batch statistics are accumulated with INTEGER atomics on fixed-point values: integer addition is associative, so the
// totals are the same bits whatever order the CTAs arrive in (float atomics are not), and a consumer needs one load per
// channel instead of a pass over per-CTA partials.  Activation sums use 2^-24 units (|sum| < 5e11), their squares 2^-16
// (sum < 1.4e14: even a tensor saturated at fp16's 65504 fits for 32 000 rows per call), gradient sums 2^-40 units
// (|sum| < 8e6): all far below float32's own rounding of the values that went in.
constexpr double kFixAct = 16777216.0, kFixActSq = 65536.0, kFixGrad = 1099511627776.0;
__device__ __forceinline__ void fix_add(long long* dst, float v, double scale) {
  atomicAdd(reinterpret_cast<unsigned long long*>(dst), (unsigned long long)__double2ll_rn((double)v * scale));
}
__device__ __forceinline__ float fix_get(const long long* src, double scale) {
  return (float)((double)__ldcg(src) / scale);
}

struct Geom {
  int B, H, W, Wp, PB, Ptot, R128, PR;     // PR: rows of one plane incl. front and tail
};

// MZ_TRAIN_TIMELINE=1 (measurement only): every chain kernel stamps %globaltimer into its own record
// [first CTA entered | first CTA past griddepcontrol.wait | last CTA done | first CTA done]
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void tl_stamp(unsigned long long* tl, int k) {
  if (tl && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.x == 0) tl[k] = gtimer();
}
__device__ __forceinline__ void tl_stamp_lane0(unsigned long long* tl, int k) {      // any warp of CTA 0
  if (tl && blockIdx.x == 0 && blockIdx.y == 0 && (threadIdx.x & 31) == 0) tl[k] = gtimer();
}
// kind: 1 forward conv, 2 dgrad, 3 bn_fwd, 4 bn_bwd_apply, 5 wgrad
__device__ __forceinline__ void tl_end(unsigned long long* tl, int kind) {
  if (tl && threadIdx.x == 0) {
    const unsigned long long t = gtimer();
    atomicMax(tl + 2, t);
    if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) { tl[3] = t; tl[8] = (unsigned long long)kind; }
  }
}

__device__ __forceinline__ bool is_halo(int P, int PB, int Wp, int W, int H) {
  const int q = P % PB, y = q / Wp, x = q - y * Wp;
  return x == W || y == H;
}

// column sums of a 32 x 32 register tile held as v[32] per lane (lane = row): returns the sum of column `lane`
__device__ __forceinline__ float warp_colsum32(float (&v)[32], int lane) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const bool up = (lane & s) != 0;
#pragma unroll
    for (int i = 0; i < s; ++i) {
      const float keep = up ? v[i + s] : v[i];
      const float send = up ? v[i] : v[i + s];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
    }
  }
  return v[0];
}

// ---------------------------------------------------------------------------------------------------------------
// forward conv / dgrad: one 128-row tile per CTA, N = 128 output channels, K = 9 taps x cg_in*8 channels
// ---------------------------------------------------------------------------------------------------------------
struct TConvParams {
  const uint16_t* in;       // planes [cg_in][PR][8]
  const uint16_t* w;        // packed [9][chunks][stage_g][128][8]
  uint16_t* out;            // planes [16][PR][8], zeros at halo rows
  const uint16_t* add;      // optional bf16 planes added to the result (dgrad: the skip connection's gradient)
  long long* stats;         // optional [128][2] += fixed-point (sum, sum of squares) over the real rows (forward: BatchNorm)
  // dgrad into a layer that ends in BatchNorm + ReLU: the result G = dL/dA of that layer is turned into
  // dZ = G * (A > 0) right here (that is all its consumers read) and the layer's BatchNorm-backward sums
  // (sum dZ, sum dZ * xhat) are taken from the fp32 values -- no separate reduction pass over the tensor
  const uint8_t* mask_bits; // the layer's ReLU mask [16][R128]: bit e of byte (g, row) = (A[row][8 g + e] > 0), or nullptr
  const uint16_t* mask_y;   // its raw conv output Y (fp16)
  const float* mask_saved;  // its [128][2] (mean, invstd)
  long long* mask_sums;     // its [128][2] += fixed-point (sum dZ, sum dZ * xhat)
  int cg_in, stage_g, chunks;   // a weight stage = stage_g channel groups of one tap; chunks stages per tap
  int Ptot, PB, Wp, W, H, PR, R128;
  int TP, TPs;              // rows of a tile incl. halo / rows of a shared-memory plane (odd)
  int sub_rows, stat_sub;   // several forward calls stacked along the rows: rows per call (a multiple of 128) and the distance
                            // (floats) between consecutive calls' statistics records -- a tile belongs to call row0 / sub_rows
  int stages, nbuf;
  uint32_t idesc;
  int dgrad;                // dgrad: bf16 operands and output; forward: fp16
  unsigned long long* tl;   // measurement only: timeline record or nullptr
};

constexpr int kTConvThreads = 320;   // w0 producer, w1 MMA issuer, w2-9 epilogue (lane quadrant warp % 4, column half (warp - 2) / 4)
constexpr int kWgThreads = 192;      // w0 producer, w1 MMA issuer, w2-5 epilogue

// kChunks: 1 / 2 = 128 / 256 input channels in 128-channel weight stages (compile-time issue loop); 0 = any other shape
template <int kChunks>
__global__ void __launch_bounds__(kTConvThreads) tconv_kernel(const __grid_constant__ TConvParams p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int halo = p.Wp + 1;
  const uint32_t stage_bytes = (uint32_t)p.stage_g * kC * 16;
  const uint32_t a_bytes = ((uint32_t)p.cg_in * p.TPs * 16 + 127) & ~127u;
  // A CTA walks the tiles blockIdx.x, blockIdx.x + gridDim.x, ...  With nbuf == 2 (launches with more tiles than SMs: the
  // stacked prediction calls) tile buffer and accumulator are double-buffered: tile i + 1 is fetched and its MMAs run
  // while the epilogue warps are still on tile i, and the weight ring streams on across tiles.
  const int nbuf = p.nbuf, ntiles = p.R128 / 128, G = (int)gridDim.x;

  unsigned char* sA = smem;                                       // [nbuf][cg_in][TPs][16]
  unsigned char* sW = smem + (size_t)nbuf * a_bytes;
  tl_stamp(p.tl, 0);
  uint64_t* bars = reinterpret_cast<uint64_t*>(sW + (size_t)p.stages * stage_bytes);
  uint64_t* w_full = bars;                           // [stages]
  uint64_t* w_empty = bars + kConvStagesMax;         // [stages]
  uint64_t* a_full = bars + 2 * kConvStagesMax;      // [2] tile fetched
  uint64_t* a_empty = a_full + 2;                    // [2] the MMAs that read the tile are done
  uint64_t* mma_done = a_empty + 2;                  // [2] accumulator complete
  uint64_t* acc_empty = mma_done + 2;                // [2] the epilogue has read the accumulator
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(acc_empty + 2);
  float* s_stat = reinterpret_cast<float*>(tmem_holder + 2);   // [2][4 quadrants][2][128] column sums
  float* s_saved = s_stat + 2 * 8 * kC;                          // [2][128][2] (mean, invstd) of the masked layer

  if (tid == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 1); }
    for (int k = 0; k < 2; ++k) { mbar_init(&a_full[k], 1); mbar_init(&a_empty[k], 1); mbar_init(&mma_done[k], 1); mbar_init(&acc_empty[k], 256); }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_holder, 256);
  pdl_trigger();            // the next kernel of the chain may set itself up beside this one
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_holder;
  const int total = 9 * p.chunks;

  if (warp == 0) {
    // The weights do not depend on the previous kernel of the chain (they were packed at the start of the step): fill the
    // ring first, then wait for the predecessor, then fetch the tiles it wrote.  The whole warp walks this code: lane 0
    // waits and posts byte counts, and a tile's cg_in plane copies are issued by as many LANES with one instruction
    // (sixteen copies issued one after the other by a single lane were 0.6 of the 1.2 us between griddepcontrol.wait and
    // the first MMA).
    const unsigned char* wsrc = reinterpret_cast<const unsigned char*>(p.w);
    auto fetch_tile = [&](int i, int t) {
      const int buf = nbuf == 2 ? (i & 1) : 0;
      if (lane == 0) {
        if (i >= nbuf) mbar_wait(&a_empty[buf], (uint32_t)((i / nbuf) - 1) & 1u);
        mbar_arrive_expect_tx(&a_full[buf], (uint32_t)p.cg_in * p.TP * 16u);
      }
      __syncwarp();
      unsigned char* dstA = sA + (size_t)buf * a_bytes;
      for (int g = lane; g < p.cg_in; g += 32)
        bulk_g2s(dstA + (size_t)g * p.TPs * 16, p.in + ((size_t)g * p.PR + kFront + t * 128 - halo) * 8, (uint32_t)p.TP * 16u, &a_full[buf]);
    };
    int s = 0;
    uint32_t ph = 0;
    bool wrapped = false;                     // the ring has been filled once: from then on a slot must be released first
    auto next_stage = [&](int it) {
      if (lane == 0) {
        if (wrapped) mbar_wait(&w_empty[s], ph);
        mbar_arrive_expect_tx(&w_full[s], stage_bytes);
        bulk_g2s(sW + (size_t)s * stage_bytes, wsrc + (size_t)it * stage_bytes, stage_bytes, &w_full[s]);
      }
      if (++s == p.stages) { s = 0; if (wrapped) ph ^= 1u; wrapped = true; }
    };
    int it = 0;
    for (; it < p.stages; ++it) next_stage(it);          // stages <= total: the first tile's leading stages
    pdl_wait();
    tl_stamp(p.tl, 1);
    if ((int)blockIdx.x < ntiles) fetch_tile(0, (int)blockIdx.x);
    // The next tile is requested once `stages` stages of this tile have been issued: by then the MMA warp is inside
    // this tile, so the buffer the next tile goes to (read by the tile before this one) is free without waiting, and
    // the fetch has the rest of this tile's MMAs to arrive.
    const int fetch_at = p.stages < total - 1 ? p.stages : total - 1;
    int i = 0;
    for (int t = (int)blockIdx.x; t < ntiles; t += G, ++i) {
      for (; it < total; ++it) {
        next_stage(it);
        if (nbuf == 2 && it == fetch_at && t + G < ntiles) fetch_tile(i + 1, t + G);
      }
      it = 0;
      if (nbuf == 1 && t + G < ntiles) fetch_tile(i + 1, t + G);
    }
  } else if (warp == 1) {
    // The issue loop is ONE warp running dependent scalar code, and it has to hand the tensor pipe an MMA every 64
    // cycles.  What that takes (tools/issue_bench2.cu, tools/ring_bench.cu): compile-time loop structure (a runtime trip
    // count, stage count by division or a descriptor rebuilt per MMA each cost more than the MMA: 145 cycles per MMA
    // measured), stage index / phase kept incrementally, descriptor high words hoisted and low words stepped by additions
    // (16-byte units), and operands that are PROVABLY warp-uniform (redux.sync) so that they live in uniform registers
    // instead of going through R2UR before every UTCHMMA.  Then one warp sustains 64.0 cycles per MMA including the
    // full / empty hand-over of the weight ring.
    auto U = [](uint32_t x) { return __reduce_max_sync(0xffffffffu, x); };
    const uint64_t a_t = smem_desc(smem_u32(sA) + (uint32_t)halo * 16u, (uint32_t)p.TPs * 16u, 128);
    const uint64_t b_t = smem_desc(smem_u32(sW), kC * 16, 128);
    const uint32_t a_hi = U((uint32_t)(a_t >> 32)), b_hi = U((uint32_t)(b_t >> 32));
    const uint32_t a_base0 = U((uint32_t)a_t), b_base = U((uint32_t)b_t), a_buf_units = U(a_bytes >> 4);
    const uint32_t a_step = U((uint32_t)(2 * p.TPs)), stage_units = U(stage_bytes >> 4);
    constexpr uint32_t b_step = 2u * kC;
    const uint32_t a_chunk = U((uint32_t)(p.stage_g * p.TPs));
    const uint32_t tm0 = U(tmem), idesc = U(p.idesc), nstages = U((uint32_t)p.stages), wp = U((uint32_t)p.Wp);
    auto d64 = [](uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; };
    uint32_t ph = 0, b_lo = b_base, s = 0;
    int i = 0;
    for (int t = (int)blockIdx.x; t < ntiles; t += G, ++i) {
      const int buf = nbuf == 2 ? (i & 1) : 0;
      const uint32_t use = (uint32_t)(i / nbuf);
      mbar_wait(&a_full[buf], use & 1u);
      if (i >= nbuf) mbar_wait(&acc_empty[buf], (use - 1u) & 1u);
      tc_fence_after();
      if (i == 0) tl_stamp_lane0(p.tl, 4);
      const uint32_t tm = tm0 + (uint32_t)buf * 128u, a_base = a_base0 + (uint32_t)buf * a_buf_units;
      if constexpr (kChunks > 0) {
        // 128-channel stages: eight K steps under two elections; kChunks stages per tap
        uint32_t a_tap = a_base - wp - 1u;      // tap (0, 0)
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
#pragma unroll
          for (int ch = 0; ch < kChunks; ++ch) {
            const uint32_t a_lo = a_tap + (uint32_t)ch * a_chunk;
            mbar_wait(&w_full[s], ph);
            tc_fence_after();
            mma4_f16_elect(tm, d64(a_lo, a_hi), d64(a_lo + a_step, a_hi), d64(a_lo + 2 * a_step, a_hi), d64(a_lo + 3 * a_step, a_hi),
                           d64(b_lo, b_hi), d64(b_lo + b_step, b_hi), d64(b_lo + 2 * b_step, b_hi), d64(b_lo + 3 * b_step, b_hi), idesc,
                           (tap | ch) ? 1u : 0u);
            mma4_f16_elect(tm, d64(a_lo + 4 * a_step, a_hi), d64(a_lo + 5 * a_step, a_hi), d64(a_lo + 6 * a_step, a_hi),
                           d64(a_lo + 7 * a_step, a_hi), d64(b_lo + 4 * b_step, b_hi), d64(b_lo + 5 * b_step, b_hi),
                           d64(b_lo + 6 * b_step, b_hi), d64(b_lo + 7 * b_step, b_hi), idesc, 1u);
            commit_elect(&w_empty[s]);
            b_lo += stage_units;
            if (++s == nstages) { s = 0; ph ^= 1u; b_lo = b_base; }
          }
          a_tap += (tap % 3 == 2) ? wp - 2u : 1u;
        }
      } else {
        // any other stage shape (the representation tower's first convolution)
        const int ksteps = p.stage_g / 2;
        uint32_t acc = 0;
        uint32_t a_tap = a_base - wp - 1u;
        for (int tap = 0; tap < 9; ++tap) {
          uint32_t a_lo = a_tap;
          for (int ch = 0; ch < p.chunks; ++ch) {
            mbar_wait(&w_full[s], ph);
            tc_fence_after();
            for (int ks = 0; ks < ksteps; ++ks) {
              mma_f16_elect(tm, d64(a_lo + (uint32_t)ks * a_step, a_hi), d64(b_lo + (uint32_t)ks * b_step, b_hi), idesc, acc);
              acc = 1;
            }
            commit_elect(&w_empty[s]);
            a_lo += a_chunk;
            b_lo += stage_units;
            if (++s == nstages) { s = 0; ph ^= 1u; b_lo = b_base; }
          }
          a_tap += (tap % 3 == 2) ? wp - 2u : 1u;
        }
      }
      if (i == 0) tl_stamp_lane0(p.tl, 5);
      commit_elect(&a_empty[buf]);
      commit_elect(&mma_done[buf]);
    }
  } else {
    // ---- epilogue: TMEM lane = tile row; a warp reads lane quadrant warp % 4, columns [64 half, 64 half + 64)
    const int quad = warp & 3, half = (warp - 2) >> 2;
    const int et = tid - 64;                  // 0..255
    const bool mask = p.mask_y != nullptr;
    // everything this role reads from global memory was written by earlier kernels of the chain: order it behind them
    pdl_wait();
    int i = 0;
    for (int t = (int)blockIdx.x; t < ntiles; t += G, ++i) {
      const int buf = nbuf == 2 ? (i & 1) : 0, sb = i & 1;      // shared-memory scratch alternates in either mode
      const uint32_t use = (uint32_t)(i / nbuf);
      const int row0 = t * 128;
      const int P = row0 + quad * 32 + lane;
      const bool inr = P < p.Ptot;
      const bool valid = inr && !is_halo(P, p.PB, p.Wp, p.W, p.H);
      const size_t rowoff = (size_t)kFront + (size_t)P;
      float* st_buf = s_stat + sb * 8 * kC;
      float* sv_buf = s_saved + sb * 2 * kC;
      const size_t sub_off = (size_t)(row0 / p.sub_rows) * (size_t)p.stat_sub;      // this tile's call: its statistics record
      if (mask) {
        sv_buf[et] = p.mask_saved[sub_off + et];
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
      // Everything the epilogue needs besides the accumulator -- the skip gradient, the masked layer's Y and ReLU bits for
      // this thread's row and 64 columns -- is requested NOW, while the MMAs run: no global round trip sits between the
      // last MMA and the stores.  Loads are UNCONDITIONAL per lane (every row of a plane up to its zero tail is readable;
      // halo rows are discarded by `valid` below): a predicate would turn each load into load + select.
      const bool do_add = p.add != nullptr;
      int4 py[8], pd[8];
      uint2 bits = make_uint2(0xffffffffu, 0xffffffffu);
      if (mask) {
        uint32_t bq[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) bq[u] = __ldcg(p.mask_bits + (size_t)(half * 8 + u) * p.R128 + P);
        bits.x = bq[0] | (bq[1] << 8) | (bq[2] << 16) | (bq[3] << 24);
        bits.y = bq[4] | (bq[5] << 8) | (bq[6] << 16) | (bq[7] << 24);
#pragma unroll
        for (int u = 0; u < 8; ++u) py[u] = __ldcg(reinterpret_cast<const int4*>(p.mask_y) + (size_t)(half * 8 + u) * p.PR + rowoff);
      }
      if (do_add) {
#pragma unroll
        for (int u = 0; u < 8; ++u) pd[u] = __ldcg(reinterpret_cast<const int4*>(p.add) + (size_t)(half * 8 + u) * p.PR + rowoff);
      }
      mbar_wait(&mma_done[buf], use & 1u);
      tc_fence_after();
      if (warp == 2 && i == 0) tl_stamp_lane0(p.tl, 6);
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t r[32];
        tmem_ld32(tmem + (uint32_t)buf * 128u + ((uint32_t)(quad * 32) << 16) + (uint32_t)(half * 64 + c * 32), r);
        tmem_ld_wait();
        if (c == 1) {                          // the accumulator is in registers: the MMAs of the tile after next may have it
          tc_fence_before();
          mbar_arrive(&acc_empty[buf]);
        }
        float v[32];
#pragma unroll
        for (int e = 0; e < 32; ++e) v[e] = valid ? __uint_as_float(r[e]) : 0.0f;
        if (do_add) {
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            float f[8];
            unpack8<__nv_bfloat16>(pd[c * 4 + u], f);
#pragma unroll
            for (int e = 0; e < 8; ++e) v[8 * u + e] = valid ? v[8 * u + e] + f[e] : 0.0f;
          }
        }
        float zx[32];
        if (mask) {
          // v := dZ = G * (A > 0);  zx := dZ * xhat
          const uint32_t word = c == 0 ? bits.x : bits.y;
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            float y8[8];
            unpack8<__half>(py[c * 4 + u], y8);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int col = half * 64 + c * 32 + 8 * u + e;
              const float dz = ((word >> (8 * u + e)) & 1u) ? v[8 * u + e] : 0.0f;
              v[8 * u + e] = dz;
              zx[8 * u + e] = dz * (y8[e] - sv_buf[2 * col]) * sv_buf[2 * col + 1];
            }
          }
        }
        if (inr) {
          int4 o[4];                           // packed before the stores: one store sequence for either type, fewer spills
#pragma unroll
          for (int u = 0; u < 4; ++u) o[u] = p.dgrad ? pack8<__nv_bfloat16>(v + 8 * u) : pack8<__half>(v + 8 * u);
#pragma unroll
          for (int u = 0; u < 4; ++u) reinterpret_cast<int4*>(p.out)[(size_t)(half * 8 + c * 4 + u) * p.PR + rowoff] = o[u];
        }
        const int col0 = half * 64 + c * 32;
        if (mask) {
          const float s1 = warp_colsum32(v, lane);
          const float s2 = warp_colsum32(zx, lane);
          st_buf[quad * 2 * kC + col0 + lane] = s1;
          st_buf[quad * 2 * kC + kC + col0 + lane] = s2;
        } else if (p.stats) {
          float sq[32];
#pragma unroll
          for (int e = 0; e < 32; ++e) sq[e] = v[e] * v[e];
          const float s1 = warp_colsum32(v, lane);
          const float s2 = warp_colsum32(sq, lane);
          st_buf[quad * 2 * kC + col0 + lane] = s1;
          st_buf[quad * 2 * kC + kC + col0 + lane] = s2;
        }
      }
      if (warp == 2 && i == 0) tl_stamp_lane0(p.tl, 7);
      long long* sums = mask ? p.mask_sums : p.stats;
      if (sums) {
        sums += sub_off / 2;
        asm volatile("bar.sync 1, 256;" ::: "memory");
        const int which = et >> 7, col = et & (kC - 1);
        float a = 0.0f;
#pragma unroll
        for (int q = 0; q < 4; ++q) a += st_buf[q * 2 * kC + which * kC + col];
        fix_add(sums + 2 * col + which, a, mask ? kFixGrad : (which ? kFixActSq : kFixAct));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 256);
  tl_end(p.tl, p.stats ? 1 : 2);
}

// ---------------------------------------------------------------------------------------------------------------
// wgrad: CTA (split s, tap row ky, ci block) accumulates dW[ky*3 + kx][co][ci] for kx = 0..2 over its rows
// ---------------------------------------------------------------------------------------------------------------
struct TWgradParams {
  const uint16_t* dy;       // bf16 planes [16][PR][8]
  const uint16_t* x;        // bf16 planes of the conv's input; ci block b starts at plane b * 16
  float* partial;           // [ci_blocks][slices][9][N/4][128 co][4]: a warp's lanes (co) store contiguous 16-byte pieces
  int n_groups;             // N / 8 of one ci block
  int Rs;                   // rows per split, multiple of 16
  int Wp, PR;
  int slices, slice0;       // slices of the tensor (calls x kSplits) / first slice of this call: every launch owns its slices,
                            // nothing is read back (a read-modify-write of 9.4 MB per launch cost more than the MMAs)
  uint32_t idesc;
  unsigned long long* tl;   // measurement only
};

__global__ void __launch_bounds__(kWgThreads) twgrad_kernel(const __grid_constant__ TWgradParams p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int split = blockIdx.x, ky = blockIdx.y, blk = blockIdx.z;
  const int ng = p.n_groups, N = ng * 8;
  tl_stamp(p.tl, 0);
  tl_stamp(p.tl, 1);
  const uint32_t dy_bytes = 16u * kWgStage * 16u, x_bytes = (uint32_t)ng * (kWgStage + 2) * 16u;
  const uint32_t st_bytes = dy_bytes + ((x_bytes + 127u) & ~127u);
  unsigned char* sS = smem;                                        // [kWgStages][dY | X]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kWgStages * (size_t)st_bytes);
  uint64_t* full = bars;                  // [kWgStages]
  uint64_t* empty = bars + kWgStages;     // [kWgStages]
  uint64_t* done = bars + 2 * kWgStages;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 2 * kWgStages + 1);

  if (tid == 0) {
    for (int s = 0; s < kWgStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(done, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_holder, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_holder;
  const int nst = (p.Rs + kWgStage - 1) / kWgStage;
  const int r_base = split * p.Rs;

  if (warp == 0) {
    // The whole warp produces: lane 0 waits for the slot and posts the byte count, then every lane issues ONE of the
    // stage's up to 32 plane copies (lanes 0-15: dY planes, 16-31: X planes) -- one instruction for all of them instead of
    // 32 issued one after the other by a single lane, which took longer than the stage's 24 MMAs.
    const uint16_t* xb = p.x + (size_t)blk * 16 * p.PR * 8;
    for (int st = 0; st < nst; ++st) {
      const int s = st % kWgStages;
      const uint32_t ph = (uint32_t)(st / kWgStages) & 1u;
      const int rows = (p.Rs - st * kWgStage) < kWgStage ? (p.Rs - st * kWgStage) : kWgStage;
      const int r0 = r_base + st * kWgStage;
      if (lane == 0) {
        mbar_wait(&empty[s], ph ^ 1u);
        mbar_arrive_expect_tx(&full[s], 16u * rows * 16u + (uint32_t)ng * (rows + 2) * 16u);
      }
      __syncwarp();
      unsigned char* d0 = sS + (size_t)s * st_bytes;
      if (lane < 16) {
        bulk_g2s(d0 + (size_t)lane * kWgStage * 16, p.dy + ((size_t)lane * p.PR + kFront + r0) * 8, (uint32_t)rows * 16u, &full[s]);
      } else if (lane - 16 < ng) {
        const int g = lane - 16;
        const int xr0 = r0 + (ky - 1) * p.Wp - 1;
        bulk_g2s(d0 + dy_bytes + (size_t)g * (kWgStage + 2) * 16, xb + ((size_t)g * p.PR + kFront + xr0) * 8,
                 (uint32_t)(rows + 2) * 16u, &full[s]);
      }
    }
  } else if (warp == 1) {
    // MN-major, no swizzle: consecutive K (rows) are consecutive 16-byte units, 8 rows = one 128-byte core matrix;
    // LBO = distance between core matrices along K (128 B), SBO = distance between 8-channel groups (one plane).
    // Same issue-loop discipline as tconv_kernel: hoisted descriptor words, warp-uniform operands, a compile-time body
    // for full 128-row stages.
    auto U = [](uint32_t x) { return __reduce_max_sync(0xffffffffu, x); };
    auto d64 = [](uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; };
    const uint64_t a_t = smem_desc(smem_u32(sS), 128, kWgStage * 16), b_t = smem_desc(smem_u32(sS) + dy_bytes, 128, (kWgStage + 2) * 16);
    const uint32_t a_hi = U((uint32_t)(a_t >> 32)), b_hi = U((uint32_t)(b_t >> 32));
    const uint32_t a_first = U((uint32_t)a_t), b_first = U((uint32_t)b_t), st16 = U(st_bytes >> 4);
    const uint32_t tm = U(tmem), idesc = U(p.idesc), n_cols = U((uint32_t)N);
    uint32_t s = 0, ph = 0, a_st = a_first, b_st = b_first;
    for (int st = 0; st < nst; ++st) {
      const int rows = (p.Rs - st * kWgStage) < kWgStage ? (p.Rs - st * kWgStage) : kWgStage;
      mbar_wait(&full[s], ph);
      tc_fence_after();
      if (st == 0) tl_stamp_lane0(p.tl, 4);
      const uint32_t acc0 = st > 0 ? 1u : 0u;
      if (rows == kWgStage) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {      // eight K steps (16 rows = 16 units each) under two elections per tap
          const uint32_t d = tm + (uint32_t)kx * n_cols, b0 = b_st + (uint32_t)kx;
          mma4_f16_elect(d, d64(a_st, a_hi), d64(a_st + 16, a_hi), d64(a_st + 32, a_hi), d64(a_st + 48, a_hi),
                         d64(b0, b_hi), d64(b0 + 16, b_hi), d64(b0 + 32, b_hi), d64(b0 + 48, b_hi), idesc, acc0);
          mma4_f16_elect(d, d64(a_st + 64, a_hi), d64(a_st + 80, a_hi), d64(a_st + 96, a_hi), d64(a_st + 112, a_hi),
                         d64(b0 + 64, b_hi), d64(b0 + 80, b_hi), d64(b0 + 96, b_hi), d64(b0 + 112, b_hi), idesc, 1u);
        }
      } else {
        for (int kx = 0; kx < 3; ++kx) {
          const uint32_t d = tm + (uint32_t)kx * n_cols;
          for (int ks = 0; ks < rows / 16; ++ks)
            mma_f16_elect(d, d64(a_st + (uint32_t)ks * 16u, a_hi), d64(b_st + (uint32_t)(ks * 16 + kx), b_hi), idesc,
                          (st > 0 || ks > 0) ? 1u : 0u);
        }
      }
      commit_elect(&empty[s]);
      a_st += st16; b_st += st16;
      if (++s == (uint32_t)kWgStages) { s = 0; ph ^= 1u; a_st = a_first; b_st = b_first; }
    }
    tl_stamp_lane0(p.tl, 5);
    commit_elect(done);
  } else {
    const int quad = warp & 3;
    const int co = quad * 32 + lane;
    // steps j = (tap kx, 16-column chunk c); the partials of step j + 1 are requested while step j is added and stored
    const int nc = N / 16, steps = 3 * nc;
    float4* base = reinterpret_cast<float4*>(p.partial) + ((size_t)blk * p.slices + p.slice0 + split) * 9 * (size_t)(N / 4) * kC + co;
    mbar_wait(done, 0);
    tc_fence_after();
    if (warp == 2) tl_stamp_lane0(p.tl, 6);
    for (int j = 0; j < steps; ++j) {
      const int kx = j / nc, c = j - kx * nc;
      float4* dst = base + ((size_t)(ky * 3 + kx) * (N / 4) + c * 4) * kC;
      uint32_t r[16];
      tmem_ld16(tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(kx * N + c * 16), r);
      tmem_ld_wait();
#pragma unroll
      for (int u = 0; u < 4; ++u)
        dst[(size_t)u * kC] = make_float4(__uint_as_float(r[4 * u]), __uint_as_float(r[4 * u + 1]), __uint_as_float(r[4 * u + 2]),
                                          __uint_as_float(r[4 * u + 3]));
    }
    if (warp == 2) tl_stamp_lane0(p.tl, 7);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem, 512);
  tl_end(p.tl, 5);
}

// ---------------------------------------------------------------------------------------------------------------
// elementwise / reduction kernels on the planes.  Thread = (plane g = blockIdx.y, row P): 8 channels, one 16-byte access
// ---------------------------------------------------------------------------------------------------------------
constexpr int kEwThreads = 256;
constexpr int kEwRows = 1;           // rows per thread

struct BnFwdParams {
  const uint16_t* y;        // raw conv output (fp16)
  const uint16_t* res;      // residual (fp16) or nullptr
  uint16_t* a;              // relu(bn(y) + res)
  uint16_t* a_b;            // optional bf16 copy (wgrad operand)
  uint8_t* bits;            // ReLU mask [16][R128]: bit e of byte (g, row) = (a[row][8 g + e] > 0): what the backward pass reads instead of a
  const long long* sums;    // [128][2] fixed-point totals from the conv epilogue
  float* saved;             // [128][2] (mean, invstd) for the backward pass
  const float *gamma, *beta;
  float *running_mean, *running_var;
  int Ptot, PB, Wp, W, H, PR, R128;
  int sub_rows, stat_sub, n_sub;   // stacked calls (blockIdx.z): rows per call, distance between their statistics records (floats)
  float inv_n, unbias;      // 1 / (B*H*W), n / (n - 1)
  unsigned long long* tl;
};

__global__ void __launch_bounds__(kEwThreads) bn_fwd_kernel(const BnFwdParams p) {
  __shared__ float s_scale[8], s_shift[8];
  const int g = blockIdx.y, sub = blockIdx.z;
  tl_stamp(p.tl, 0);
  pdl_trigger();
  pdl_wait();
  tl_stamp(p.tl, 1);
  // the thread's rows are requested FIRST (unconditional: rows past the call's end are the next call's or the plane's zero
  // tail): their round trip and the one that fetches the statistics overlap instead of following each other
  const size_t plane = (size_t)g * p.PR + kFront + (size_t)sub * p.sub_rows;
  int4 yr[kEwRows], rr[kEwRows];
#pragma unroll
  for (int k = 0; k < kEwRows; ++k) {
    const int L = (blockIdx.x * kEwRows + k) * kEwThreads + threadIdx.x;
    yr[k] = __ldcg(reinterpret_cast<const int4*>(p.y) + plane + L);
    if (p.res) rr[k] = __ldcg(reinterpret_cast<const int4*>(p.res) + plane + L);
  }
  if (threadIdx.x < 8) {
    const int c = g * 8 + threadIdx.x;
    const long long* sums = p.sums + (size_t)sub * (p.stat_sub / 2);
    const float mean = fix_get(sums + 2 * c, kFixAct) * p.inv_n;
    float var = fix_get(sums + 2 * c + 1, kFixActSq) * p.inv_n - mean * mean;
    var = var > 0.0f ? var : 0.0f;
    const float is = rsqrtf(var + kBnEps);
    const float sc = p.gamma[c] * is;
    s_scale[threadIdx.x] = sc;
    s_shift[threadIdx.x] = p.beta[c] - mean * sc;
    if (blockIdx.x == 0) {
      float* saved = p.saved + (size_t)sub * p.stat_sub;
      saved[2 * c] = mean; saved[2 * c + 1] = is;
      if (sub == 0) {
        // the running statistics take the stacked calls' updates one after the other, in call order
        float rm = p.running_mean[c], rv = p.running_var[c];
        for (int z = 0; z < p.n_sub; ++z) {
          const long long* sz = p.sums + (size_t)z * (p.stat_sub / 2);
          const float mz_ = fix_get(sz + 2 * c, kFixAct) * p.inv_n;
          float vz = fix_get(sz + 2 * c + 1, kFixActSq) * p.inv_n - mz_ * mz_;
          vz = vz > 0.0f ? vz : 0.0f;
          rm = (1.0f - kBnMomentum) * rm + kBnMomentum * mz_;
          rv = (1.0f - kBnMomentum) * rv + kBnMomentum * vz * p.unbias;
        }
        p.running_mean[c] = rm; p.running_var[c] = rv;
      }
    }
  }
  __syncthreads();
  float sc[8], sh[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { sc[e] = s_scale[e]; sh[e] = s_shift[e]; }
#pragma unroll
  for (int k = 0; k < kEwRows; ++k) {
    const int L = (blockIdx.x * kEwRows + k) * kEwThreads + threadIdx.x;
    if (L >= p.sub_rows) break;
    const int P = sub * p.sub_rows + L;
    int4 o = make_int4(0, 0, 0, 0), ob = o;
    uint32_t m = 0;
    if (P < p.Ptot && !is_halo(P, p.PB, p.Wp, p.W, p.H)) {
      float v[8];
      unpack8<__half>(yr[k], v);
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = v[e] * sc[e] + sh[e];
      if (p.res) {
        float r[8];
        unpack8<__half>(rr[k], r);
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] += r[e];
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = fmaxf(v[e], 0.0f);
      o = pack8<__half>(v);
      if (p.a_b) ob = pack8<__nv_bfloat16>(v);
      // the mask is taken from the STORED value (what bn_bwd_reduce_kernel's `a > 0` sees)
      float w[8];
      unpack8<__half>(o, w);
#pragma unroll
      for (int e = 0; e < 8; ++e) m |= (w[e] > 0.0f ? 1u : 0u) << e;
    }
    reinterpret_cast<int4*>(p.a)[plane + L] = o;
    if (p.a_b) reinterpret_cast<int4*>(p.a_b)[plane + L] = ob;
    p.bits[(size_t)g * p.R128 + P] = (uint8_t)m;
  }
  tl_end(p.tl, 3);
}

struct BnBwdParams {
  const uint16_t* g;        // gradient w.r.t. the activated output (bf16); with a == nullptr it is already dZ
  const uint16_t* a;        // the activated output (fp16): ReLU mask, or nullptr
  const uint16_t* y;        // raw conv output (fp16)
  const float* saved;       // [128][2] mean, invstd
  long long* sums;          // [128][2] fixed-point (sum dZ, sum dZ * xhat): from the reduce kernel / the dgrad epilogue
  const float* gamma;
  float *dgamma, *dbeta;    // += (apply kernel, blockIdx.x == 0)
  uint16_t* dy;             // gradient w.r.t. the raw conv output (bf16), zeros at halo rows
  uint16_t* dz;             // optional: the masked gradient itself (the residual branch's share), bf16
  int Ptot, PB, Wp, W, H, PR;
  int sub_rows, stat_sub, n_sub;   // stacked calls (blockIdx.z), as in BnFwdParams
  float inv_n;
  int rows_per_cta;         // reduce kernel
  unsigned long long* tl;
};

__global__ void __launch_bounds__(kEwThreads) bn_bwd_reduce_kernel(const BnBwdParams p) {
  const int g = blockIdx.y, sub = blockIdx.z;
  const float* saved = p.saved + (size_t)sub * p.stat_sub;
  float mean[8], is[8], s1[8], s2[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    mean[e] = saved[2 * (g * 8 + e)]; is[e] = saved[2 * (g * 8 + e) + 1];
    s1[e] = 0.0f; s2[e] = 0.0f;
  }
  const size_t plane = (size_t)g * p.PR + kFront + (size_t)sub * p.sub_rows;
  const int r_begin = blockIdx.x * p.rows_per_cta;
  const int r_end = (r_begin + p.rows_per_cta) < p.sub_rows ? (r_begin + p.rows_per_cta) : p.sub_rows;
  for (int L = r_begin + threadIdx.x; L < r_end; L += kEwThreads) {
    // halo rows: G is zero there, so they add nothing
    float gv[8], av[8], yv[8];
    unpack8<__nv_bfloat16>(__ldcg(reinterpret_cast<const int4*>(p.g) + plane + L), gv);
    unpack8<__half>(__ldcg(reinterpret_cast<const int4*>(p.a) + plane + L), av);
    unpack8<__half>(__ldcg(reinterpret_cast<const int4*>(p.y) + plane + L), yv);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float dz = av[e] > 0.0f ? gv[e] : 0.0f;
      s1[e] += dz;
      s2[e] += dz * (yv[e] - mean[e]) * is[e];
    }
  }
  __shared__ float red[kEwThreads / 32][16];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s1[e] += __shfl_xor_sync(0xffffffffu, s1[e], o);
      s2[e] += __shfl_xor_sync(0xffffffffu, s2[e], o);
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int e = 0; e < 8; ++e) { red[warp][e] = s1[e]; red[warp][8 + e] = s2[e]; }
  }
  __syncthreads();
  if (threadIdx.x < 16) {
    float t = 0.0f;
    for (int w = 0; w < kEwThreads / 32; ++w) t += red[w][threadIdx.x];
    const int e = threadIdx.x & 7, which = threadIdx.x >> 3;
    fix_add(p.sums + (size_t)sub * (p.stat_sub / 2) + 2 * (g * 8 + e) + which, t, kFixGrad);
  }
}

__global__ void __launch_bounds__(kEwThreads) bn_bwd_apply_kernel(const BnBwdParams p) {
  __shared__ float s_k[8][4];      // mean, invstd, gamma*invstd, and the two batch means
  __shared__ float s_m[8][2];
  const int g = blockIdx.y, sub = blockIdx.z;
  tl_stamp(p.tl, 0);
  pdl_trigger();
  pdl_wait();
  tl_stamp(p.tl, 1);
  const size_t plane = (size_t)g * p.PR + kFront + (size_t)sub * p.sub_rows;
  int4 gr[kEwRows], ar[kEwRows], yr[kEwRows];
#pragma unroll
  for (int k = 0; k < kEwRows; ++k) {
    const int L = (blockIdx.x * kEwRows + k) * kEwThreads + threadIdx.x;
    gr[k] = __ldcg(reinterpret_cast<const int4*>(p.g) + plane + L);
    yr[k] = __ldcg(reinterpret_cast<const int4*>(p.y) + plane + L);
    if (p.a) ar[k] = __ldcg(reinterpret_cast<const int4*>(p.a) + plane + L);
  }
  if (threadIdx.x < 8) {
    const int c = g * 8 + threadIdx.x;
    const long long* sums = p.sums + (size_t)sub * (p.stat_sub / 2);
    const float* saved = p.saved + (size_t)sub * p.stat_sub;
    const float S1 = fix_get(sums + 2 * c, kFixGrad), S2 = fix_get(sums + 2 * c + 1, kFixGrad);
    s_k[threadIdx.x][0] = saved[2 * c];
    s_k[threadIdx.x][1] = saved[2 * c + 1];
    s_k[threadIdx.x][2] = p.gamma[c] * saved[2 * c + 1];
    s_m[threadIdx.x][0] = S1 * p.inv_n;
    s_m[threadIdx.x][1] = S2 * p.inv_n;
    if (blockIdx.x == 0 && sub == 0) {      // the parameter gradients take the stacked calls' sums last call first: the
      float dg = p.dgamma[c], db = p.dbeta[c];   // order in which separate calls' backward passes would run
      for (int z = p.n_sub - 1; z >= 0; --z) {
        const long long* sz = p.sums + (size_t)z * (p.stat_sub / 2);
        dg += fix_get(sz + 2 * c + 1, kFixGrad);
        db += fix_get(sz + 2 * c, kFixGrad);
      }
      p.dgamma[c] = dg; p.dbeta[c] = db;
    }
  }
  __syncthreads();
  float mean[8], is[8], gi[8], m1[8], m2[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { mean[e] = s_k[e][0]; is[e] = s_k[e][1]; gi[e] = s_k[e][2]; m1[e] = s_m[e][0]; m2[e] = s_m[e][1]; }
#pragma unroll
  for (int k = 0; k < kEwRows; ++k) {
    const int L = (blockIdx.x * kEwRows + k) * kEwThreads + threadIdx.x;
    if (L >= p.sub_rows) break;
    const int P = sub * p.sub_rows + L;
    int4 o = make_int4(0, 0, 0, 0), oz = make_int4(0, 0, 0, 0);
    if (P < p.Ptot && !is_halo(P, p.PB, p.Wp, p.W, p.H)) {
      float gv[8], av[8], yv[8], dzv[8], dyv[8];
      unpack8<__nv_bfloat16>(gr[k], gv);
      if (p.a) unpack8<__half>(ar[k], av);
      unpack8<__half>(yr[k], yv);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        dzv[e] = (!p.a || av[e] > 0.0f) ? gv[e] : 0.0f;
        const float xh = (yv[e] - mean[e]) * is[e];
        dyv[e] = gi[e] * (dzv[e] - m1[e] - xh * m2[e]);
      }
      o = pack8<__nv_bfloat16>(dyv);
      oz = pack8<__nv_bfloat16>(dzv);
    }
    reinterpret_cast<int4*>(p.dy)[plane + L] = o;
    if (p.dz) reinterpret_cast<int4*>(p.dz)[plane + L] = oz;
  }
  tl_end(p.tl, 4);
}

// float32 [B][C][H][W] -> fp16 planes and their bf16 copy (zeros at halo positions and channels >= C); cg planes are written
__global__ void nchw_to_planes_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst, uint16_t* __restrict__ dst_b, int C,
                                      int cg, int Ptot, int PB, int Wp, int W, int H, int PR) {
  const int g = blockIdx.y;
  const int P = blockIdx.x * blockDim.x + threadIdx.x;
  if (P >= Ptot) return;
  const int b = P / PB, q = P - b * PB, y = q / Wp, x = q - y * Wp;
  float v[8];
  const int yc = y < H ? y : H - 1, xc = x < W ? x : W - 1;          // unconditional loads, the select afterwards
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = g * 8 + e;
    v[e] = __ldg(src + (((size_t)b * C + (c < C ? c : C - 1)) * H + yc) * W + xc);
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) v[e] = (g * 8 + e < C && y < H && x < W) ? v[e] : 0.0f;
  reinterpret_cast<int4*>(dst)[(size_t)g * PR + kFront + P] = pack8<__half>(v);
  reinterpret_cast<int4*>(dst_b)[(size_t)g * PR + kFront + P] = pack8<__nv_bfloat16>(v);
}

// bf16 gradient planes -> float32 [B][C][H][W]
__global__ void planes_to_nchw_kernel(const uint16_t* __restrict__ src, float* __restrict__ dst, int C, int Ptot, int PB, int Wp,
                                      int W, int H, int PR) {
  const int g = blockIdx.y;
  const int P = blockIdx.x * blockDim.x + threadIdx.x;
  if (P >= Ptot) return;
  const int b = P / PB, q = P - b * PB, y = q / Wp, x = q - y * Wp;
  if (y >= H || x >= W) return;
  float v[8];
  unpack8<__nv_bfloat16>(__ldcg(reinterpret_cast<const int4*>(src) + (size_t)g * PR + kFront + P), v);
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = g * 8 + e;
    if (c < C) dst[(((size_t)b * C + c) * H + y) * W + x] = v[e];
  }
}


// A tower's output for autograd: raw [B][128][H][W] float32 and / or its per-position min-max normalisation over the 128
// channels (util.py:31-36: (h - lo) / (hi - lo + 1e-8), the float32 operations of the reference on the same values).
// Block = 32 rows x 16 channel groups: warp g loads the 32 rows' 16-byte records of plane g (coalesced), the channel
// minimum / maximum of a row is combined over the 16 warps through shared memory, every thread stores its 8 channels.
constexpr int kTowerIoThreads = 512;

__global__ void __launch_bounds__(kTowerIoThreads) tower_out_kernel(const uint16_t* __restrict__ src, float* __restrict__ raw,
                                                                    float* __restrict__ norm, int Ptot, int PB, int Wp, int W, int H,
                                                                    int PR) {
  __shared__ float s_lo[16][33], s_hi[16][33];
  const int g = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int P = blockIdx.x * 32 + lane;
  const int b = P / PB, q = P - b * PB, y = q / Wp, x = q - y * Wp;
  const bool real = P < Ptot && y < H && x < W;
  float v[8];
  unpack8<__half>(__ldcg(reinterpret_cast<const int4*>(src) + (size_t)g * PR + kFront + P), v);      // rows past Ptot: the zero tail
  float lo = v[0], hi = v[0];
#pragma unroll
  for (int e = 1; e < 8; ++e) { lo = fminf(lo, v[e]); hi = fmaxf(hi, v[e]); }
  if (norm) {
    s_lo[g][lane] = lo; s_hi[g][lane] = hi;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) { lo = fminf(lo, s_lo[k][lane]); hi = fmaxf(hi, s_hi[k][lane]); }
  }
  if (!real) return;
  const float d = __fadd_rn(__fsub_rn(hi, lo), 1e-8f);
  const size_t cs = (size_t)H * W, base = (size_t)b * kC * cs + (size_t)y * W + x + (size_t)(g * 8) * cs;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    if (raw) raw[base + e * cs] = v[e];
    if (norm) norm[base + e * cs] = __fdiv_rn(__fsub_rn(v[e], lo), d);
  }
}

// The gradient with respect to a tower's output, as bf16 planes, from autograd's two pieces: g_raw = dL/d raw and
// g_norm = dL/d normalised (either may be missing).  With a = h - lo, d = hi - lo + 1e-8:
//   dh[c] = g_raw[c] + g_norm[c] / d + [c = argmin] (sum g_norm a / d^2 - sum g_norm / d) - [c = argmax] sum g_norm a / d^2
// (first index on ties, like a single min / max index of torch; tied minima are ReLU zeros whose gradient the tower's
// own ReLU mask removes anyway).  h is the tower's saved last activation.  Same block shape as tower_out_kernel; the
// row-wide quantities (lo, hi, their positions, the two sums) are combined over the 16 warps through shared memory.
__global__ void __launch_bounds__(kTowerIoThreads) tower_gradin_kernel(const float* __restrict__ g_raw, const float* __restrict__ g_norm,
                                                                       const uint16_t* __restrict__ h, uint16_t* __restrict__ dst,
                                                                       int Ptot, int PB, int Wp, int W, int H, int PR) {
  __shared__ float s_lo[16][33], s_hi[16][33], s_1[16][33], s_2[16][33];
  __shared__ int s_amin[16][33], s_amax[16][33];
  const int g = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int P = blockIdx.x * 32 + lane;
  const int b = P / PB, q = P - b * PB, y = q / Wp, x = q - y * Wp;
  const bool real = P < Ptot && y < H && x < W;
  const size_t cs = (size_t)H * W, base = real ? (size_t)b * kC * cs + (size_t)y * W + x + (size_t)(g * 8) * cs : 0;
  float o[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) o[e] = (real && g_raw) ? __ldg(g_raw + base + e * cs) : 0.0f;
  if (g_norm) {
    float v[8], gn[8];
    unpack8<__half>(__ldcg(reinterpret_cast<const int4*>(h) + (size_t)g * PR + kFront + P), v);
#pragma unroll
    for (int e = 0; e < 8; ++e) gn[e] = real ? __ldg(g_norm + base + e * cs) : 0.0f;
    float lo = v[0], hi = v[0];
    int amin = g * 8, amax = g * 8;
#pragma unroll
    for (int e = 1; e < 8; ++e) {
      if (v[e] < lo) { lo = v[e]; amin = g * 8 + e; }
      if (v[e] > hi) { hi = v[e]; amax = g * 8 + e; }
    }
    s_lo[g][lane] = lo; s_hi[g][lane] = hi; s_amin[g][lane] = amin; s_amax[g][lane] = amax;
    __syncthreads();
    lo = s_lo[0][lane]; hi = s_hi[0][lane]; amin = s_amin[0][lane]; amax = s_amax[0][lane];
#pragma unroll
    for (int k = 1; k < 16; ++k) {          // ascending groups, strict comparisons: the first index wins ties
      if (s_lo[k][lane] < lo) { lo = s_lo[k][lane]; amin = s_amin[k][lane]; }
      if (s_hi[k][lane] > hi) { hi = s_hi[k][lane]; amax = s_amax[k][lane]; }
    }
    float p1 = 0.0f, p2 = 0.0f;
#pragma unroll
    for (int e = 0; e < 8; ++e) { p1 += gn[e]; p2 += gn[e] * (v[e] - lo); }
    s_1[g][lane] = p1; s_2[g][lane] = p2;
    __syncthreads();
    float s1 = 0.0f, s2 = 0.0f;
#pragma unroll
    for (int k = 0; k < 16; ++k) { s1 += s_1[k][lane]; s2 += s_2[k][lane]; }
    const float d = __fadd_rn(__fsub_rn(hi, lo), 1e-8f);
    const float t = s2 / (d * d), dlo = t - s1 / d, dhi = -t;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int c = g * 8 + e;
      o[e] += gn[e] / d;
      if (c == amin) o[e] += dlo;
      if (c == amax) o[e] += dhi;
    }
  }
  if (P < Ptot) reinterpret_cast<int4*>(dst)[(size_t)g * PR + kFront + P] = real ? pack8<__nv_bfloat16>(o) : make_int4(0, 0, 0, 0);
}

// the action "planes" of DynamicsConvNet.forward (network.py:440-444, quirk C of DESIGN.md): flat element f of the
// [A*h*w] block is 1 iff f % A == action.  Written as channels 128.. of the dynamics' first-conv input (planes 16..31).
__global__ void action_planes_kernel(const int64_t* __restrict__ action, uint16_t* __restrict__ dst, uint16_t* __restrict__ dst_b, int A,
                                     int Ptot, int PB, int Wp, int W, int H, int PR) {
  const int g = blockIdx.y;                       // 0..15 -> plane 16 + g
  const int P = blockIdx.x * blockDim.x + threadIdx.x;
  if (P >= Ptot) return;
  const int b = P / PB, q = P - b * PB, y = q / Wp, x = q - y * Wp;
  const int a = (int)action[b];
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = g * 8 + e;
    float f = 0.0f;
    if (c < A && y < H && x < W) f = ((c * H * W + y * W + x) % A == a) ? 1.0f : 0.0f;
    v[e] = f;
  }
  reinterpret_cast<int4*>(dst)[(size_t)(16 + g) * PR + kFront + P] = pack8<__half>(v);
  reinterpret_cast<int4*>(dst_b)[(size_t)(16 + g) * PR + kFront + P] = pack8<__nv_bfloat16>(v);
}

// ---- weights ---------------------------------------------------------------------------------------------------
struct ConvDesc {
  const float* w;           // [128][ci_total][3][3]
  float* wgrad;
  uint16_t* wf;             // forward operand  [9][chunks][chunk_g][128 co][8 ci]
  uint16_t* wd;             // dgrad operand    [9][2][8][128 ci][8 co] (flipped taps) or nullptr
  float* partial;           // [ci_blocks][slices][9][N/4][128][4]
  int ci_total, cg_in, chunk_g, n_groups, ci_blocks, slices, tower;
};

__global__ void pack_weights_kernel(const ConvDesc* __restrict__ descs) {
  const ConvDesc d = descs[blockIdx.y];
  const int chunks = d.cg_in / d.chunk_g;
  const size_t nf = (size_t)9 * d.cg_in * kC * 8;
  const size_t nd = d.wd ? (size_t)9 * 16 * kC * 8 : 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nf + nd; i += (size_t)gridDim.x * blockDim.x) {
    if (i < nf) {
      const int e = (int)(i % 8);
      size_t r = i / 8;
      const int n = (int)(r % kC); r /= kC;
      const int gl = (int)(r % d.chunk_g); r /= d.chunk_g;
      const int ch = (int)(r % chunks);
      const int tap = (int)(r / chunks);
      const int c = (ch * d.chunk_g + gl) * 8 + e;
      const float v = c < d.ci_total ? d.w[((size_t)n * d.ci_total + c) * 9 + tap] : 0.0f;
      reinterpret_cast<__half*>(d.wf)[i] = __float2half_rn(fminf(fmaxf(v, -65504.0f), 65504.0f));
    } else {
      const size_t j = i - nf;
      const int e = (int)(j % 8);
      size_t r = j / 8;
      const int n = (int)(r % kC); r /= kC;          // ci
      const int gl = (int)(r % 8); r /= 8;
      const int ch = (int)(r % 2);
      const int tap = (int)(r / 2);
      const int co = (ch * 8 + gl) * 8 + e;
      reinterpret_cast<__nv_bfloat16*>(d.wd)[j] = __float2bfloat16_rn(d.w[((size_t)co * d.ci_total + n) * 9 + (8 - tap)]);
    }
  }
}

// the parameter's gradient [128][ci_total][3][3] += sum of the row-split partials
__global__ void wgrad_finalize_kernel(const ConvDesc* __restrict__ descs, int calls0, int calls1, int calls2) {
  const ConvDesc d = descs[blockIdx.y];
  const int used = (d.tower == 0 ? calls0 : (d.tower == 1 ? calls1 : calls2)) * kSplits;     // slices written in this step
  const int N = d.n_groups * 8;
  const size_t per_split = (size_t)9 * kC * N;
  const size_t total = (size_t)d.ci_blocks * per_split;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int blk = (int)(i / per_split);
    const size_t r = i - (size_t)blk * per_split;                   // partial layout [tap][N/4][co][4]
    const int e = (int)(r % 4), co = (int)((r / 4) % kC), q = (int)((r / (4 * kC)) % (N / 4)), tap = (int)(r / ((size_t)N * kC));
    const int n = q * 4 + e;
    const int ci = blk * kC + n;
    if (ci >= d.ci_total) continue;
    const float* src = d.partial + (size_t)blk * d.slices * per_split + r;
    float s = 0.0f;
    for (int k0 = 0; k0 < used; k0 += kSplits) {     // kSplits slices per call: that many loads in flight, then the adds
      float v[kSplits];
#pragma unroll
      for (int k = 0; k < kSplits; ++k) v[k] = __ldcs(src + (size_t)(k0 + k) * per_split);
#pragma unroll
      for (int k = 0; k < kSplits; ++k) s += v[k];
    }
    d.wgrad[((size_t)co * d.ci_total + ci) * 9 + tap] += s;     // autograd semantics: gradients accumulate
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
struct BnPtrs { float *gamma, *dgamma, *beta, *dbeta, *rmean, *rvar; };

}  // namespace
}  // namespace mz

using namespace mz;

struct mz_train {
  mz_train_config cfg;
  Geom g;
  int nconv;                               // convs: rep0, rep blocks (2 each), dyn0, dyn blocks, pred blocks
  int rep_first, dyn_first, pred_first;    // index of each tower's first conv
  std::vector<ConvDesc> convs;
  std::vector<BnPtrs> bn;
  std::vector<int> touched;                // wgrad partials written in this step
  ConvDesc* d_convs;
  bool bound;
  // arena carving
  unsigned char* arena;
  size_t arena_bytes;
  size_t plane_bytes;                      // one 16-bit plane
  uint16_t* grad_buf[4 + kDyRing];         // bf16 [16 planes]: four rotating gradient buffers, kDyRing dY buffers
  float* stats;                            // [slots][1280 floats]: fwd totals i64 [256] | saved (mean, invstd) f32 [256] | bwd totals i64 [256]
  size_t stats_floats;
  int stat_stride;
  int n_calls[3];
  // saved activations: slot(tower, call) -> X, then (Y, A) per layer
  std::vector<uint16_t*> slot_x, slot_xb;                    // xb / ab: bf16 copies for wgrad (ab == a for a tower's last layer: no copy)
  std::vector<std::vector<uint16_t*>> slot_y, slot_a, slot_ab;
  std::vector<std::vector<uint8_t*>> slot_m;                 // ReLU masks [R128][16] per layer
  // weight gradients run on streams of their own, beside the dgrad / BatchNorm chain (nothing on the chain reads them):
  // dY goes through a ring of buffers, ev_dy[k] = buffer k is written (main -> side), ev_wg[k] = its wgrad has read it
  // (side -> main, waited for only when the ring comes round to k again)
  int fwd_calls[3];                        // forward calls per tower in this step
  cudaStream_t side[kSideStreams];
  cudaEvent_t ev_dy[kDyRing], ev_wg[kDyRing];
  bool wg_pending[kDyRing];
  int dy_turn, side_turn;
  // Launch context of the tower call in progress: one forward call (n_sub = 1) or several calls of the prediction tower
  // stacked along the rows (the K unroll steps' predictions do not depend on one another: one launch chain over K * B
  // boards, every call keeping its own BatchNorm statistics)
  const Geom* cur_g;
  int cur_nsub, cur_sub_rows, cur_stat_sub;
  int num_sms;
  bool group_ok;                           // rows of one call are a multiple of 128 and of 16 * kSplits: tiles and weight-gradient splits never straddle calls
  Geom gg;                                 // geometry of the stacked buffers (plane stride for unroll_steps calls)
  uint16_t* ggrad_buf[4 + kDyRing];
  uint16_t *gslot_x, *gslot_xb;
  std::vector<uint16_t*> gslot_y, gslot_a, gslot_ab;
  std::vector<uint8_t*> gslot_m;
  std::vector<int> pred_stack_first;       // per prediction call of this step: first call of the stacked forward it ran in, or -1
  unsigned long long* timeline;           // MZ_TRAIN_TIMELINE=1: [kTimelineMax][10] stamps, one record per chain launch
  int tl_next;
};

namespace mz {
namespace {

int tower_layers(const mz_train* t, int tower) { return (tower == 2 ? 0 : 1) + 2 * t->cfg.num_res_blocks; }
int tower_first_conv(const mz_train* t, int tower) { return tower == 0 ? t->rep_first : (tower == 1 ? t->dyn_first : t->pred_first); }
int tower_in_groups(const mz_train* t, int tower) { return tower == 0 ? (t->cfg.in_channels + 15) / 16 * 2 : (tower == 1 ? 32 : 16); }
int slot_of(const mz_train* t, int tower, int call) {
  int s = 0;
  for (int k = 0; k < tower; ++k) s += t->n_calls[k];
  return s + call;
}
int stat_slot(const mz_train* t, int tower, int call, int layer) {
  int s = 0;
  for (int k = 0; k < tower; ++k) s += t->n_calls[k] * tower_layers(t, k);
  return s + call * tower_layers(t, tower) + layer;
}

size_t conv_smem_bytes(const Geom& g, int cg_in, int nbuf, int* stages_out, int* TP_out, int* TPs_out) {
  const int halo = g.Wp + 1;
  const int TP = 128 + 2 * halo, TPs = TP | 1;
  const int chunk_g = cg_in < 16 ? cg_in : 16;                     // a stage: one tap's weights for up to 128 input channels
  const size_t a = (((size_t)cg_in * TPs * 16) + 127) & ~(size_t)127;
  const size_t stage = (size_t)chunk_g * kC * 16;
  const size_t fixed = (size_t)nbuf * a + (2 * kConvStagesMax + 8) * 8 + 8 + 20 * kC * 4 + 64;
  int stages = (int)((220 * 1024 - fixed) / stage);
  const int need = 9 * (cg_in / chunk_g);
  if (stages > kConvStagesMax) stages = kConvStagesMax;
  if (stages > need) stages = need;
  if (stages_out) *stages_out = stages;
  if (TP_out) *TP_out = TP;
  if (TPs_out) *TPs_out = TPs;
  return fixed + (size_t)stages * stage;
}

size_t wgrad_smem_bytes(int n_groups) {
  const size_t dy = (size_t)16 * kWgStage * 16, x = ((size_t)n_groups * (kWgStage + 2) * 16 + 127) & ~(size_t)127;
  return kWgStages * (dy + x) + (2 * kWgStages + 2) * 8 + 16 + 64;
}

struct MaskArgs { const uint8_t* bits; const uint16_t* y; float* stat; };      // the layer whose ReLU / BatchNorm-backward sums a dgrad folds in

// The conv and BatchNorm kernels of a tower form a chain launched with programmatic dependent launch (launch_pdl): a
// kernel may start as soon as its predecessor has called griddepcontrol.launch_dependents (the chain kernels do so at
// once; after an ordinary kernel -- weight packing, layout conversion -- it starts when that kernel has completed);
// everything that touches the predecessor's data sits behind griddepcontrol.wait, what does not (barrier set-up, TMEM
// allocation, the weight ring's first fill) runs before it.

// forward: fp16 operands and output; dgrad: bf16
int launch_conv(mz_train* t, const uint16_t* in, int cg_in, const uint16_t* w, uint16_t* out, const uint16_t* add,
                float* stats, bool dgrad, cudaStream_t st, const MaskArgs* mask = nullptr) {
  TConvParams p;
  const Geom& g = *t->cur_g;
  p.sub_rows = t->cur_nsub > 1 ? t->cur_sub_rows : g.R128; p.stat_sub = t->cur_stat_sub;
  p.in = in; p.w = w; p.out = out; p.add = add; p.stats = reinterpret_cast<long long*>(stats);
  p.mask_bits = mask ? mask->bits : nullptr; p.mask_y = mask ? mask->y : nullptr;
  p.mask_saved = mask ? mask->stat + 512 : nullptr; p.mask_sums = mask ? reinterpret_cast<long long*>(mask->stat + 768) : nullptr;
  p.cg_in = cg_in; p.stage_g = cg_in < 16 ? cg_in : 16; p.chunks = cg_in / p.stage_g;
  p.Ptot = g.Ptot; p.PB = g.PB; p.Wp = g.Wp; p.W = g.W; p.H = g.H; p.PR = g.PR; p.R128 = g.R128;
  const int tiles = g.R128 / 128;
  p.nbuf = (tiles > t->num_sms && cg_in == 16) ? 2 : 1;
  const size_t smem = conv_smem_bytes(g, cg_in, p.nbuf, &p.stages, &p.TP, &p.TPs);
  p.idesc = idesc_of(128, kC, dgrad ? 1 : 0, dgrad ? 1 : 0, 0);
  p.dgrad = dgrad;
  p.tl = t->timeline && t->tl_next < kTimelineMax ? t->timeline + 10 * (size_t)t->tl_next++ : nullptr;
  void (*kern)(TConvParams) = p.stage_g == 16 ? (p.chunks == 1 ? tconv_kernel<1> : (p.chunks == 2 ? tconv_kernel<2> : tconv_kernel<0>)) : tconv_kernel<0>;
  cudaError_t e = launch_pdl(true, kern, dim3(p.nbuf == 2 ? t->num_sms : tiles), dim3(kTConvThreads), smem, st, p);
  if (e != cudaSuccess) { set_error("tconv_kernel launch: %s", cudaGetErrorString(e)); return MZ_ECUDA; }
  count_launch();
  return MZ_OK;
}

// dy = t->dy_buf[k] was just written on `st`: hand it to the side stream's weight-gradient kernel
int launch_wgrad(mz_train* t, int conv, int call, int k, const uint16_t* dy, const uint16_t* x, cudaStream_t st) {
  const ConvDesc& d = t->convs[conv];
  MZ_CUDA(cudaEventRecord(t->ev_dy[k], st));
  cudaStream_t side = t->side[t->side_turn];
  t->side_turn = (t->side_turn + 1) % kSideStreams;
  MZ_CUDA(cudaStreamWaitEvent(side, t->ev_dy[k], 0));
  st = side;
  TWgradParams p;
  const Geom& g = *t->cur_g;
  const int nsub = t->cur_nsub;
  p.dy = dy; p.x = x; p.partial = d.partial; p.n_groups = d.n_groups;
  // stacked calls: kSplits splits per call, each inside its call (cur_sub_rows is a multiple of 16 * kSplits)
  p.Rs = nsub > 1 ? t->cur_sub_rows / kSplits : ((g.Ptot + kSplits - 1) / kSplits + 15) / 16 * 16;
  p.Wp = g.Wp; p.PR = g.PR;
  p.slices = d.slices; p.slice0 = call * kSplits;
  p.idesc = idesc_of(128, (uint32_t)d.n_groups * 8, 1, 1, 1);
  p.tl = t->timeline && t->tl_next < kTimelineMax ? t->timeline + 10 * (size_t)t->tl_next++ : nullptr;
  twgrad_kernel<<<dim3(kSplits * nsub, 3, d.ci_blocks), kWgThreads, wgrad_smem_bytes(d.n_groups), st>>>(p);
  MZ_LAUNCH_CHECK("twgrad_kernel");
  MZ_CUDA(cudaEventRecord(t->ev_wg[k], st));
  t->wg_pending[k] = true;
  t->touched[conv] += nsub;
  return MZ_OK;
}

// next dY buffer; the main stream first waits until the weight-gradient kernel that last read it is done
int next_dy(mz_train* t, cudaStream_t st, int* k_out) {
  const int k = t->dy_turn;
  t->dy_turn = (k + 1) % kDyRing;
  if (t->wg_pending[k]) { MZ_CUDA(cudaStreamWaitEvent(st, t->ev_wg[k], 0)); t->wg_pending[k] = false; }
  *k_out = k;
  return MZ_OK;
}

dim3 ew_grid(const mz_train* t, int planes) {
  const int rows = t->cur_nsub > 1 ? t->cur_sub_rows : t->cur_g->Ptot;
  return dim3((rows + kEwThreads * kEwRows - 1) / (kEwThreads * kEwRows), planes, t->cur_nsub);
}

int launch_bn_fwd(mz_train* t, int conv, const uint16_t* y, const uint16_t* res, uint16_t* a, uint16_t* a_b, uint8_t* bits,
                  float* stat, cudaStream_t st) {
  const Geom& g = *t->cur_g;
  const BnPtrs& b = t->bn[conv];
  BnFwdParams p;
  p.n_sub = t->cur_nsub; p.sub_rows = t->cur_nsub > 1 ? t->cur_sub_rows : g.Ptot; p.stat_sub = t->cur_stat_sub;
  p.y = y; p.res = res; p.a = a; p.a_b = (a_b && a_b != a) ? a_b : nullptr; p.bits = bits; p.sums = reinterpret_cast<const long long*>(stat); p.saved = stat + 512;
  p.gamma = b.gamma; p.beta = b.beta; p.running_mean = b.rmean; p.running_var = b.rvar;
  p.Ptot = g.Ptot; p.PB = g.PB; p.Wp = g.Wp; p.W = g.W; p.H = g.H; p.PR = g.PR; p.R128 = g.R128;
  const double n = (double)g.B * g.H * g.W;
  p.inv_n = (float)(1.0 / n); p.unbias = (float)(n / (n - 1.0));
  p.tl = t->timeline && t->tl_next < kTimelineMax ? t->timeline + 10 * (size_t)t->tl_next++ : nullptr;
  cudaError_t e = launch_pdl(true, bn_fwd_kernel, ew_grid(t, 16), dim3(kEwThreads), 0, st, p);
  if (e != cudaSuccess) { set_error("bn_fwd_kernel launch: %s", cudaGetErrorString(e)); return MZ_ECUDA; }
  count_launch();
  return MZ_OK;
}

// a != nullptr: gin is dL/dA, the ReLU mask and the two sums are taken here (two launches; the top of a tower).
// a == nullptr: gin is already dZ and the sums were accumulated by the dgrad that produced it (one launch).
int launch_bn_bwd(mz_train* t, int conv, const uint16_t* gin, const uint16_t* a, const uint16_t* y, float* stat, uint16_t* dy,
                  uint16_t* dz, cudaStream_t st) {
  const Geom& g = *t->cur_g;
  const BnPtrs& b = t->bn[conv];
  BnBwdParams p;
  p.n_sub = t->cur_nsub; p.sub_rows = t->cur_nsub > 1 ? t->cur_sub_rows : g.Ptot; p.stat_sub = t->cur_stat_sub;
  p.g = gin; p.a = a; p.y = y; p.saved = stat + 512; p.sums = reinterpret_cast<long long*>(stat + 768); p.gamma = b.gamma; p.dgamma = b.dgamma; p.dbeta = b.dbeta;
  p.dy = dy; p.dz = dz;
  p.Ptot = g.Ptot; p.PB = g.PB; p.Wp = g.Wp; p.W = g.W; p.H = g.H; p.PR = g.PR;
  p.inv_n = (float)(1.0 / ((double)g.B * g.H * g.W));
  p.tl = nullptr;
  const int nchunk = 9;
  p.rows_per_cta = (p.sub_rows + nchunk - 1) / nchunk;
  if (a) {
    bn_bwd_reduce_kernel<<<dim3(nchunk, 16, t->cur_nsub), kEwThreads, 0, st>>>(p);
    MZ_LAUNCH_CHECK("bn_bwd_reduce_kernel");
  }
  p.tl = t->timeline && t->tl_next < kTimelineMax ? t->timeline + 10 * (size_t)t->tl_next++ : nullptr;
  cudaError_t e = launch_pdl(true, bn_bwd_apply_kernel, ew_grid(t, 16), dim3(kEwThreads), 0, st, p);
  if (e != cudaSuccess) { set_error("bn_bwd_apply_kernel launch: %s", cudaGetErrorString(e)); return MZ_ECUDA; }
  count_launch();
  return MZ_OK;
}

}  // namespace
}  // namespace mz

extern "C" {

static int train_layout(const mz_train_config* c, Geom* g, size_t* bytes, mz_train* t) {
  MZ_CHECK_ARG(c != nullptr, "mz_train: config is NULL");
  MZ_CHECK_ARG(c->num_planes == kC, "mz_train: the training kernels are built for num_planes = 128 (got %d)", c->num_planes);
  MZ_CHECK_ARG(c->board_h >= 2 && c->board_w >= 2 && c->board_w + 2 <= kFront, "mz_train: board %dx%d not supported", c->board_h, c->board_w);
  MZ_CHECK_ARG(c->in_channels >= 1 && c->in_channels <= 128, "mz_train: in_channels %d not supported", c->in_channels);
  MZ_CHECK_ARG(c->num_actions >= 1 && c->num_actions <= 128, "mz_train: num_actions %d not supported (<= 128)", c->num_actions);
  MZ_CHECK_ARG(c->num_res_blocks >= 1 && c->num_res_blocks <= 32, "mz_train: num_res_blocks %d not supported", c->num_res_blocks);
  MZ_CHECK_ARG(c->batch >= 2 && c->unroll_steps >= 1 && c->unroll_steps <= 16, "mz_train: batch %d / unroll_steps %d not supported", c->batch, c->unroll_steps);
  g->B = c->batch; g->H = c->board_h; g->W = c->board_w; g->Wp = g->W + 1; g->PB = (g->H + 1) * g->Wp;
  g->Ptot = g->B * g->PB; g->R128 = (g->Ptot + 127) / 128 * 128; g->PR = kFront + g->R128 + kTail;
  const size_t plane = (size_t)g->PR * 16;
  const int nb = c->num_res_blocks, T = c->unroll_steps;
  const int in_cg = (c->in_channels + 15) / 16 * 2;
  size_t total = 0;
  auto take = [&](size_t n) { const size_t off = total; total += align_up(n, 256); return off; };
  // operand copies of the weights + wgrad partials
  const int nconv = (1 + 2 * nb) + (1 + 2 * nb) + 2 * nb;
  if (t) { t->convs.resize(nconv); t->bn.resize(nconv); t->touched.assign(nconv, 0); t->nconv = nconv; }
  int idx = 0;
  for (int tower = 0; tower < 3; ++tower) {
    if (t) { if (tower == 0) t->rep_first = idx; else if (tower == 1) t->dyn_first = idx; else t->pred_first = idx; }
    const int layers = (tower == 2 ? 0 : 1) + 2 * nb;
    for (int l = 0; l < layers; ++l, ++idx) {
      const bool first = tower != 2 && l == 0;
      const int ci_total = first ? (tower == 0 ? c->in_channels : kC + c->num_actions) : kC;
      const int cg_in = first ? (tower == 0 ? in_cg : 32) : 16;
      const int chunk_g = cg_in < 8 ? cg_in : 8;
      const int n_groups = first && tower == 0 ? in_cg : 16;
      const int ci_blocks = first && tower == 1 ? 2 : 1;
      const size_t o_wf = take((size_t)9 * cg_in * kC * 16);
      const bool need_d = !(tower == 0 && l == 0);
      const size_t o_wd = need_d ? take((size_t)9 * 16 * kC * 16) : 0;
      const int slices = (tower == 0 ? 1 : T) * kSplits;
      const size_t o_p = take((size_t)ci_blocks * slices * 9 * kC * n_groups * 8 * 4);
      if (t) {
        ConvDesc& d = t->convs[idx];
        d.w = nullptr; d.wgrad = nullptr;
        d.wf = reinterpret_cast<uint16_t*>(t->arena + o_wf);
        d.wd = need_d ? reinterpret_cast<uint16_t*>(t->arena + o_wd) : nullptr;
        d.partial = reinterpret_cast<float*>(t->arena + o_p);
        d.ci_total = ci_total; d.cg_in = cg_in; d.chunk_g = chunk_g; d.n_groups = n_groups; d.ci_blocks = ci_blocks; d.slices = slices; d.tower = tower;
      }
    }
  }
  const size_t o_desc = take((size_t)nconv * sizeof(ConvDesc));
  if (t) t->d_convs = reinterpret_cast<ConvDesc*>(t->arena + o_desc);
  // gradient work buffers
  for (int k = 0; k < 4 + kDyRing; ++k) {
    const size_t o = take(16 * plane);
    if (t) t->grad_buf[k] = reinterpret_cast<uint16_t*>(t->arena + o);
  }
  // statistics
  const int calls[3] = {1, T, T};
  size_t nstat = 0;
  for (int tower = 0; tower < 3; ++tower) nstat += (size_t)calls[tower] * ((tower == 2 ? 0 : 1) + 2 * nb);
  const int stat_stride = 1280;
  const size_t o_stats = take(nstat * stat_stride * 4);
  if (t) {
    t->stats = reinterpret_cast<float*>(t->arena + o_stats); t->stats_floats = nstat * stat_stride; t->stat_stride = stat_stride;
    for (int k = 0; k < 3; ++k) t->n_calls[k] = calls[k];
    t->pred_stack_first.assign(T, -1);
  }
  // saved activations
  const int nslots = 1 + 2 * T;
  if (t) { t->slot_x.resize(nslots); t->slot_xb.resize(nslots); t->slot_y.resize(nslots); t->slot_a.resize(nslots); t->slot_ab.resize(nslots); t->slot_m.resize(nslots); }
  int s = 0;
  for (int tower = 0; tower < 3; ++tower)
    for (int call = 0; call < calls[tower]; ++call, ++s) {
      const int xg = tower == 0 ? in_cg : (tower == 1 ? 32 : 16);
      const size_t ox = take((size_t)xg * plane), oxb = take((size_t)xg * plane);
      if (t) { t->slot_x[s] = reinterpret_cast<uint16_t*>(t->arena + ox); t->slot_xb[s] = reinterpret_cast<uint16_t*>(t->arena + oxb); }
      const int layers = (tower == 2 ? 0 : 1) + 2 * nb;
      if (t) { t->slot_y[s].resize(layers); t->slot_a[s].resize(layers); t->slot_ab[s].resize(layers); t->slot_m[s].resize(layers); }
      for (int l = 0; l < layers; ++l) {
        const size_t oy = take(16 * plane), oa = take(16 * plane);
        // the tower's last activation feeds no convolution of this tower: no bf16 copy
        const size_t oab = l == layers - 1 ? oa : take(16 * plane);
        const size_t om = take((size_t)g->R128 * 16);
        if (t) {
          t->slot_m[s][l] = t->arena + om;
          t->slot_y[s][l] = reinterpret_cast<uint16_t*>(t->arena + oy); t->slot_a[s][l] = reinterpret_cast<uint16_t*>(t->arena + oa);
          t->slot_ab[s][l] = reinterpret_cast<uint16_t*>(t->arena + oab);
        }
      }
    }
  // stacked prediction calls: their own activation slots and gradient buffers with a plane stride for T calls
  const bool group_ok = T > 1 && g->Ptot % 128 == 0 && g->Ptot % (16 * kSplits) == 0;
  if (t) t->group_ok = group_ok;
  if (group_ok) {
    Geom gg = *g;
    gg.Ptot = T * g->Ptot; gg.R128 = gg.Ptot; gg.PR = kFront + gg.R128 + kTail;
    const size_t gplane = (size_t)gg.PR * 16;
    if (t) t->gg = gg;
    for (int k = 0; k < 4 + kDyRing; ++k) {
      const size_t o = take(16 * gplane);
      if (t) t->ggrad_buf[k] = reinterpret_cast<uint16_t*>(t->arena + o);
    }
    const int layers = 2 * nb;
    const size_t ox = take(16 * gplane), oxb = take(16 * gplane);
    if (t) {
      t->gslot_x = reinterpret_cast<uint16_t*>(t->arena + ox); t->gslot_xb = reinterpret_cast<uint16_t*>(t->arena + oxb);
      t->gslot_y.resize(layers); t->gslot_a.resize(layers); t->gslot_ab.resize(layers); t->gslot_m.resize(layers);
    }
    for (int l = 0; l < layers; ++l) {
      const size_t oy = take(16 * gplane), oa = take(16 * gplane);
      const size_t oab = l == layers - 1 ? oa : take(16 * gplane);
      const size_t om = take((size_t)gg.R128 * 16);
      if (t) {
        t->gslot_y[l] = reinterpret_cast<uint16_t*>(t->arena + oy); t->gslot_a[l] = reinterpret_cast<uint16_t*>(t->arena + oa);
        t->gslot_ab[l] = reinterpret_cast<uint16_t*>(t->arena + oab); t->gslot_m[l] = t->arena + om;
      }
    }
  }
  *bytes = total + 1024;
  return MZ_OK;
}

int mz_train_arena_bytes(const mz_train_config* cfg, size_t* bytes) {
  MZ_CHECK_ARG(bytes != nullptr, "mz_train_arena_bytes: bytes is NULL");
  Geom g;
  return train_layout(cfg, &g, bytes, nullptr);
}

int mz_train_create(const mz_train_config* cfg, void* arena_dev, size_t arena_bytes, mz_train** out) {
  MZ_CHECK_ARG(out != nullptr && arena_dev != nullptr, "mz_train_create: NULL argument");
  Geom g;
  size_t need = 0;
  int rc = train_layout(cfg, &g, &need, nullptr);
  if (rc) return rc;
  if (arena_bytes < need) { set_error("mz_train_create: arena of %zu bytes, %zu needed", arena_bytes, need); return MZ_ENOMEM; }
  mz_train* t = new mz_train();
  t->cfg = *cfg; t->g = g;
  t->arena = static_cast<unsigned char*>(arena_dev); t->arena_bytes = arena_bytes;
  t->plane_bytes = (size_t)g.PR * 16;
  t->bound = false;
  rc = train_layout(cfg, &t->g, &need, t);
  if (rc) { delete t; return rc; }
  // every plane's front / tail / halo rows must read as zero from the first use on: clear the arena once
  cudaError_t e = cudaMemset(arena_dev, 0, need);
  if (e != cudaSuccess) { delete t; set_error("cudaMemset: %s", cudaGetErrorString(e)); return MZ_ECUDA; }
  const int cgs[3] = {tower_in_groups(t, 0), 16, 32};
  size_t max_smem = 0;
  for (int k = 0; k < 3; ++k) { const size_t s = conv_smem_bytes(t->g, cgs[k], 1, nullptr, nullptr, nullptr); if (s > max_smem) max_smem = s; }
  { const size_t s = conv_smem_bytes(t->g, 16, 2, nullptr, nullptr, nullptr); if (s > max_smem) max_smem = s; }
  { int dev = 0, sms = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); t->num_sms = sms > 0 ? sms : 148; }
  e = cudaFuncSetAttribute(tconv_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_smem);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(tconv_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_smem);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(tconv_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_smem);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(twgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wgrad_smem_bytes(16));
  // The chain alternates kernels that need ~200 KB of shared memory with elementwise kernels that need none; left to
  // its defaults the driver re-partitions L1 / shared memory at every such boundary, which drains the SMs (measured:
  // 15 us per conv + BatchNorm pair with every instruction of the conv kernel ablated).  Everything asks for the
  // maximum carve-out instead.
  const void* ks[] = {(const void*)tconv_kernel<0>, (const void*)tconv_kernel<1>, (const void*)tconv_kernel<2>, (const void*)twgrad_kernel, (const void*)bn_fwd_kernel, (const void*)bn_bwd_apply_kernel,
                      (const void*)bn_bwd_reduce_kernel, (const void*)nchw_to_planes_kernel, (const void*)planes_to_nchw_kernel,
                      (const void*)action_planes_kernel};
  for (const void* k : ks)
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) { delete t; set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return MZ_ECUDA; }
  for (int k = 0; k < kSideStreams; ++k) t->side[k] = nullptr;
  for (int k = 0; k < kDyRing; ++k) { t->ev_dy[k] = nullptr; t->ev_wg[k] = nullptr; }
  e = cudaSuccess;
  for (int k = 0; k < kSideStreams && e == cudaSuccess; ++k) e = cudaStreamCreateWithFlags(&t->side[k], cudaStreamNonBlocking);
  for (int k = 0; k < kDyRing && e == cudaSuccess; ++k) {
    e = cudaEventCreateWithFlags(&t->ev_dy[k], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&t->ev_wg[k], cudaEventDisableTiming);
  }
  if (e != cudaSuccess) { delete t; set_error("mz_train_create: stream / event creation: %s", cudaGetErrorString(e)); return MZ_ECUDA; }
  t->dy_turn = 0; t->side_turn = 0;
  for (int k = 0; k < kDyRing; ++k) t->wg_pending[k] = false;
  t->timeline = nullptr; t->tl_next = 0;
  if (getenv("MZ_TRAIN_TIMELINE") && atoi(getenv("MZ_TRAIN_TIMELINE"))) {
    e = cudaMalloc(&t->timeline, (size_t)kTimelineMax * 10 * sizeof(unsigned long long));
    if (e != cudaSuccess) { delete t; set_error("mz_train_create: timeline buffer: %s", cudaGetErrorString(e)); return MZ_ECUDA; }
    cudaMemset(t->timeline, 0, (size_t)kTimelineMax * 10 * sizeof(unsigned long long));
  }
  *out = t;
  return MZ_OK;
}

int mz_train_destroy(mz_train* t) {
  if (t) {
    for (int k = 0; k < kSideStreams; ++k) if (t->side[k]) cudaStreamSynchronize(t->side[k]);
    for (int k = 0; k < kDyRing; ++k) { if (t->ev_dy[k]) cudaEventDestroy(t->ev_dy[k]); if (t->ev_wg[k]) cudaEventDestroy(t->ev_wg[k]); }
    for (int k = 0; k < kSideStreams; ++k) if (t->side[k]) cudaStreamDestroy(t->side[k]);
    if (t->timeline) cudaFree(t->timeline);
  }
  delete t;
  return MZ_OK;
}

int mz_train_bind(mz_train* t, void* const* ptrs, int32_t n, mz_stream stream) {
  MZ_CHECK_ARG(t != nullptr && ptrs != nullptr, "mz_train_bind: NULL argument");
  MZ_CHECK_ARG(n == 8 * t->nconv, "mz_train_bind: %d pointers, %d expected (8 per convolution)", n, 8 * t->nconv);
  for (int i = 0; i < t->nconv; ++i) {
    void* const* q = ptrs + 8 * i;
    for (int k = 0; k < 8; ++k) MZ_CHECK_ARG(q[k] != nullptr, "mz_train_bind: pointer %d of convolution %d is NULL", k, i);
    t->convs[i].w = static_cast<const float*>(q[0]); t->convs[i].wgrad = static_cast<float*>(q[1]);
    BnPtrs& b = t->bn[i];
    b.gamma = static_cast<float*>(q[2]); b.dgamma = static_cast<float*>(q[3]); b.beta = static_cast<float*>(q[4]);
    b.dbeta = static_cast<float*>(q[5]); b.rmean = static_cast<float*>(q[6]); b.rvar = static_cast<float*>(q[7]);
  }
  MZ_CUDA(cudaMemcpyAsync(t->d_convs, t->convs.data(), (size_t)t->nconv * sizeof(ConvDesc), cudaMemcpyHostToDevice,
                          static_cast<cudaStream_t>(stream)));
  MZ_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  t->bound = true;
  return MZ_OK;
}

int mz_train_begin_step(mz_train* t, mz_stream stream) {
  MZ_CHECK_ARG(t != nullptr, "mz_train_begin_step: NULL handle");
  if (!t->bound) { set_error("mz_train_begin_step: mz_train_bind has not been called"); return MZ_ESTATE; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  MZ_CUDA(cudaMemsetAsync(t->stats, 0, t->stats_floats * 4, st));
  pack_weights_kernel<<<dim3(32, t->nconv), 256, 0, st>>>(t->d_convs);
  MZ_LAUNCH_CHECK("pack_weights_kernel");
  std::fill(t->touched.begin(), t->touched.end(), 0);
  t->dy_turn = 0;                          // (pending weight-gradient launches keep their events: mz_train_join / next_dy wait for them)
  t->fwd_calls[0] = t->fwd_calls[1] = t->fwd_calls[2] = 0;
  std::fill(t->pred_stack_first.begin(), t->pred_stack_first.end(), -1);
  t->tl_next = 0;
  return MZ_OK;
}

// the buffers of one tower call (ncalls == 1) or of ncalls stacked prediction calls, and the launch context for them
struct CallBufs { uint16_t *x, *xb; uint16_t* const* y; uint16_t* const* a; uint16_t* const* ab; uint8_t* const* m; uint16_t** G; };

static int enter_calls(mz_train* t, const char* who, int32_t tower, int32_t call, int32_t ncalls, CallBufs* cb) {
  MZ_CHECK_ARG(tower >= 0 && tower < 3 && call >= 0 && ncalls >= 1 && call + ncalls <= t->n_calls[tower],
               "%s: tower %d calls %d..%d out of range", who, tower, call, call + ncalls - 1);
  t->cur_stat_sub = tower_layers(t, tower) * t->stat_stride;
  if (ncalls == 1) {
    const int sl = slot_of(t, tower, call);
    t->cur_g = &t->g; t->cur_nsub = 1; t->cur_sub_rows = t->g.Ptot;
    *cb = CallBufs{t->slot_x[sl], t->slot_xb[sl], t->slot_y[sl].data(), t->slot_a[sl].data(), t->slot_ab[sl].data(),
                   t->slot_m[sl].data(), t->grad_buf};
    return MZ_OK;
  }
  MZ_CHECK_ARG(tower == 2, "%s: only prediction-tower calls can be stacked (tower %d)", who, tower);
  if (!t->group_ok) { set_error("%s: stacked calls are not available for this shape (rows per call %d)", who, t->g.Ptot); return MZ_ESTATE; }
  t->gg.Ptot = ncalls * t->g.Ptot; t->gg.R128 = t->gg.Ptot;      // the plane stride gg.PR stays that of unroll_steps calls
  t->cur_g = &t->gg; t->cur_nsub = ncalls; t->cur_sub_rows = t->g.Ptot;
  *cb = CallBufs{t->gslot_x, t->gslot_xb, t->gslot_y.data(), t->gslot_a.data(), t->gslot_ab.data(), t->gslot_m.data(), t->ggrad_buf};
  return MZ_OK;
}

int mz_train_tower_forward_calls(mz_train* t, int32_t tower, int32_t call, int32_t ncalls, const float* x, const int64_t* action,
                                 float* out, float* out_norm, mz_stream stream) {
  MZ_CHECK_ARG(t != nullptr && x != nullptr && (out != nullptr || out_norm != nullptr), "mz_train_tower_forward: NULL argument");
  MZ_CHECK_ARG(tower != 1 || action != nullptr, "mz_train_tower_forward: the dynamics tower needs actions");
  if (!t->bound) { set_error("mz_train_tower_forward: mz_train_bind has not been called"); return MZ_ESTATE; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CallBufs cb;
  int rc0 = enter_calls(t, "mz_train_tower_forward", tower, call, ncalls, &cb);
  if (rc0) return rc0;
  const Geom& g = *t->cur_g;
  const int nb = t->cfg.num_res_blocks;
  if (call + ncalls > t->fwd_calls[tower]) t->fwd_calls[tower] = call + ncalls;
  if (tower == 2)                          // where mz_train_debug_view finds these calls' saved tensors
    for (int c = call; c < call + ncalls; ++c) t->pred_stack_first[c] = ncalls > 1 ? call : -1;
  const int xg = tower_in_groups(t, tower);
  const int c_in = tower == 0 ? t->cfg.in_channels : kC;
  const dim3 cgrid((g.Ptot + 255) / 256, tower == 1 ? 16 : xg);
  uint16_t* X = cb.x;
  nchw_to_planes_kernel<<<cgrid, 256, 0, st>>>(x, X, cb.xb, c_in, tower == 1 ? 16 : xg, g.Ptot, g.PB, g.Wp, g.W, g.H, g.PR);
  MZ_LAUNCH_CHECK("nchw_to_planes_kernel");
  if (tower == 1) {
    action_planes_kernel<<<dim3((g.Ptot + 255) / 256, 16), 256, 0, st>>>(action, X, cb.xb, t->cfg.num_actions, g.Ptot, g.PB, g.Wp,
                                                                       g.W, g.H, g.PR);
    MZ_LAUNCH_CHECK("action_planes_kernel");
  }
  int conv = tower_first_conv(t, tower), layer = 0, rc;
  const uint16_t* cur = X;
  auto stat = [&](int l) { return t->stats + (size_t)stat_slot(t, tower, call, l) * t->stat_stride; };
  if (tower != 2) {
    if ((rc = launch_conv(t, X, xg, t->convs[conv].wf, cb.y[0], nullptr, stat(0), false, st))) return rc;
    if ((rc = launch_bn_fwd(t, conv, cb.y[0], nullptr, cb.a[0], cb.ab[0], cb.m[0], stat(0), st))) return rc;
    cur = cb.a[0];
    ++conv; ++layer;
  }
  for (int b = 0; b < nb; ++b) {
    uint16_t *y1 = cb.y[layer], *a1 = cb.a[layer], *y2 = cb.y[layer + 1], *a2 = cb.a[layer + 1];
    if ((rc = launch_conv(t, cur, 16, t->convs[conv].wf, y1, nullptr, stat(layer), false, st))) return rc;
    if ((rc = launch_bn_fwd(t, conv, y1, nullptr, a1, cb.ab[layer], cb.m[layer], stat(layer), st))) return rc;
    if ((rc = launch_conv(t, a1, 16, t->convs[conv + 1].wf, y2, nullptr, stat(layer + 1), false, st))) return rc;
    if ((rc = launch_bn_fwd(t, conv + 1, y2, cur, a2, cb.ab[layer + 1], cb.m[layer + 1], stat(layer + 1), st))) return rc;
    cur = a2;
    conv += 2; layer += 2;
  }
  tower_out_kernel<<<dim3((g.Ptot + 31) / 32), kTowerIoThreads, 0, st>>>(cur, out, out_norm, g.Ptot, g.PB, g.Wp, g.W, g.H, g.PR);
  MZ_LAUNCH_CHECK("tower_out_kernel");
  return MZ_OK;
}

int mz_train_tower_forward(mz_train* t, int32_t tower, int32_t call, const float* x, const int64_t* action, float* out,
                           mz_stream stream) {
  return mz_train_tower_forward_calls(t, tower, call, 1, x, action, out, nullptr, stream);
}

int mz_train_tower_backward_calls(mz_train* t, int32_t tower, int32_t call, int32_t ncalls, const float* grad_out,
                                  const float* grad_norm, float* grad_in, mz_stream stream) {
  MZ_CHECK_ARG(t != nullptr && (grad_out != nullptr || grad_norm != nullptr), "mz_train_tower_backward: NULL argument");
  MZ_CHECK_ARG(tower == 0 || grad_in != nullptr, "mz_train_tower_backward: grad_in is NULL");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CallBufs cb;
  int rc0 = enter_calls(t, "mz_train_tower_backward", tower, call, ncalls, &cb);
  if (rc0) return rc0;
  const Geom& g = *t->cur_g;
  const int nb = t->cfg.num_res_blocks;
  const int first = tower != 2 ? 1 : 0;
  const int conv0 = tower_first_conv(t, tower);
  uint16_t** G = cb.G;                     // [0..3] rotate, [4..] the dY ring
  uint16_t** dYb = cb.G + 4;
  const dim3 cgrid((g.Ptot + 255) / 256, 16);
  auto stat = [&](int l) { return t->stats + (size_t)stat_slot(t, tower, call, l) * t->stat_stride; };
  // the gradient w.r.t. the current block output lives in G[cur]; `masked`: it already is dZ = dL/dA * (A > 0) and the
  // layer's BatchNorm-backward sums are in place (the dgrad that produced it folded both in)
  int cur = 0, k = 0, rc;
  bool masked = false;
  auto other = [&](int a, int b, int c) { for (int i = 0; i < 4; ++i) if (i != a && i != b && i != c) return i; return -1; };
  tower_gradin_kernel<<<dim3((g.Ptot + 31) / 32), kTowerIoThreads, 0, st>>>(grad_out, grad_norm, cb.a[first + 2 * nb - 1], G[cur], g.Ptot, g.PB,
                                                                  g.Wp, g.W, g.H, g.PR);
  MZ_LAUNCH_CHECK("tower_gradin_kernel");
  for (int b = nb - 1; b >= 0; --b) {
    const int l1 = first + 2 * b, l2 = l1 + 1;
    const int c1 = conv0 + l1, c2 = c1 + 1;
    const uint16_t* a_in_b = l1 > 0 ? cb.ab[l1 - 1] : cb.xb;
    // second conv of the block: out = relu(bn2(conv2(a1)) + a_in)
    if ((rc = next_dy(t, st, &k))) return rc;
    if (!masked) {
      const int f = other(cur, -1, -1);
      if ((rc = launch_bn_bwd(t, c2, G[cur], cb.a[l2], cb.y[l2], stat(l2), dYb[k], G[f], st))) return rc;
      cur = f;                             // the masked gradient: the skip connection's share
    } else {
      if ((rc = launch_bn_bwd(t, c2, G[cur], nullptr, cb.y[l2], stat(l2), dYb[k], nullptr, st))) return rc;
    }
    if ((rc = launch_wgrad(t, c2, call, k, dYb[k], cb.ab[l1], st))) return rc;
    const int f1 = other(cur, -1, -1);
    const MaskArgs m1{cb.m[l1], cb.y[l1], stat(l1)};
    if ((rc = launch_conv(t, dYb[k], 16, t->convs[c2].wd, G[f1], nullptr, nullptr, true, st, &m1))) return rc;
    // first conv: a1 = relu(bn1(conv1(a_in)))
    if ((rc = next_dy(t, st, &k))) return rc;
    if ((rc = launch_bn_bwd(t, c1, G[f1], nullptr, cb.y[l1], stat(l1), dYb[k], nullptr, st))) return rc;
    if ((rc = launch_wgrad(t, c1, call, k, dYb[k], a_in_b, st))) return rc;
    const int f2 = other(cur, f1, -1);
    if (l1 > 0) {                          // a_in is the output of layer l1 - 1 of this tower: fold its ReLU mask and sums in
      const MaskArgs m0{cb.m[l1 - 1], cb.y[l1 - 1], stat(l1 - 1)};
      if ((rc = launch_conv(t, dYb[k], 16, t->convs[c1].wd, G[f2], G[cur], nullptr, true, st, &m0))) return rc;
      masked = true;
    } else {                               // a_in is the tower's input: the plain gradient
      if ((rc = launch_conv(t, dYb[k], 16, t->convs[c1].wd, G[f2], G[cur], nullptr, true, st))) return rc;
      masked = false;
    }
    cur = f2;
  }
  if (first) {
    if ((rc = next_dy(t, st, &k))) return rc;
    if ((rc = launch_bn_bwd(t, conv0, G[cur], nullptr, cb.y[0], stat(0), dYb[k], nullptr, st))) return rc;
    if ((rc = launch_wgrad(t, conv0, call, k, dYb[k], cb.xb, st))) return rc;
    if (tower == 1) {
      const int f = other(cur, -1, -1);
      if ((rc = launch_conv(t, dYb[k], 16, t->convs[conv0].wd, G[f], nullptr, nullptr, true, st))) return rc;
      cur = f;
    }
  }
  if (tower != 0) {
    planes_to_nchw_kernel<<<cgrid, 256, 0, st>>>(G[cur], grad_in, kC, g.Ptot, g.PB, g.Wp, g.W, g.H, g.PR);
    MZ_LAUNCH_CHECK("planes_to_nchw_kernel");
  }
  return MZ_OK;
}

int mz_train_tower_backward(mz_train* t, int32_t tower, int32_t call, const float* grad_out, float* grad_in, mz_stream stream) {
  return mz_train_tower_backward_calls(t, tower, call, 1, grad_out, nullptr, grad_in, stream);
}

int mz_train_stacked_calls(mz_train* t, int32_t* max_calls) {
  MZ_CHECK_ARG(t != nullptr && max_calls != nullptr, "mz_train_stacked_calls: NULL argument");
  *max_calls = t->group_ok ? t->n_calls[2] : 1;
  return MZ_OK;
}

int mz_train_join(mz_train* t, mz_stream stream) {
  MZ_CHECK_ARG(t != nullptr, "mz_train_join: NULL handle");
  for (int k = 0; k < kDyRing; ++k)
    if (t->wg_pending[k]) { MZ_CUDA(cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), t->ev_wg[k], 0)); t->wg_pending[k] = false; }
  return MZ_OK;
}

int mz_train_end_step(mz_train* t, mz_stream stream) {
  MZ_CHECK_ARG(t != nullptr, "mz_train_end_step: NULL handle");
  // every tower call of the step must have gone through its backward: the finalize pass sums ALL slices of a tensor
  for (int i = 0; i < t->nconv; ++i) {
    const int want = t->fwd_calls[i < t->dyn_first ? 0 : (i < t->pred_first ? 1 : 2)];
    if (t->touched[i] != want) {
      set_error("mz_train_end_step: convolution %d has %d of %d weight-gradient passes (a tower backward is missing)", i, t->touched[i], want);
      return MZ_ESTATE;
    }
  }
  int rc = mz_train_join(t, stream);
  if (rc) return rc;
  wgrad_finalize_kernel<<<dim3(64, t->nconv), 256, 0, static_cast<cudaStream_t>(stream)>>>(t->d_convs, t->fwd_calls[0], t->fwd_calls[1],
                                                                                          t->fwd_calls[2]);
  MZ_LAUNCH_CHECK("wgrad_finalize_kernel");
  return MZ_OK;
}

int mz_train_debug_view(mz_train* t, int32_t tower, int32_t call, int32_t layer, int32_t which, void** ptr, size_t* bytes,
                        int32_t* plane_rows, int32_t* front_rows) {
  MZ_CHECK_ARG(t != nullptr && ptr != nullptr && bytes != nullptr, "mz_train_debug_view: NULL argument");
  MZ_CHECK_ARG(tower >= 0 && tower < 3 && call >= 0 && call < t->n_calls[tower], "mz_train_debug_view: tower %d call %d out of range", tower, call);
  const int slot = slot_of(t, tower, call);
  const int layers = tower_layers(t, tower);
  // a prediction call that ran stacked saved its tensors in the stacked buffers, at row (call - first) * Ptot of them
  const int first = tower == 2 ? t->pred_stack_first[call] : -1;
  const size_t plane_bytes = first >= 0 ? (size_t)t->gg.PR * 16 : t->plane_bytes;
  if (plane_rows) *plane_rows = first >= 0 ? t->gg.PR : t->g.PR;
  if (front_rows) *front_rows = kFront + (first >= 0 ? (call - first) * t->g.Ptot : 0);
  if (which == 4) {
    if (!t->timeline) { set_error("mz_train_debug_view: no timeline (MZ_TRAIN_TIMELINE=1 at creation)"); return MZ_ESTATE; }
    *ptr = t->timeline; *bytes = (size_t)t->tl_next * 10 * sizeof(unsigned long long);
    return MZ_OK;
  }
  if (which == 0) {
    *ptr = first >= 0 ? t->gslot_x : t->slot_x[slot];
    *bytes = (size_t)tower_in_groups(t, tower) * plane_bytes;
    return MZ_OK;
  }
  MZ_CHECK_ARG(layer >= 0 && layer < layers, "mz_train_debug_view: layer %d out of range", layer);
  if (which == 1) { *ptr = first >= 0 ? t->gslot_y[layer] : t->slot_y[slot][layer]; *bytes = 16 * plane_bytes; return MZ_OK; }
  if (which == 2) { *ptr = first >= 0 ? t->gslot_a[layer] : t->slot_a[slot][layer]; *bytes = 16 * plane_bytes; return MZ_OK; }
  if (which == 3) { *ptr = t->stats + (size_t)stat_slot(t, tower, call, layer) * t->stat_stride + 512; *bytes = 256 * 4; return MZ_OK; }
  set_error("mz_train_debug_view: unknown view %d", which);
  return MZ_EINVAL;
}

}  // extern "C"
