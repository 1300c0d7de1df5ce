// ResNet towers of MuZeroBoardGameNet / MuZeroAtariNet (network.py:273-574) on the
// Blackwell tensor cores (fp16 x fp16 -> fp32).
//
// Data layout ("channel-group planes"): a board is a grid of
//   PB = H*W positions,  position q = y*W + x.
// Flattening boards back to back (row P = b*PB + q) makes every 3x3 tap a constant row offset: tap (ky,kx) of
// output row P reads input row P + (ky-1)*W + (kx-1).  No row is padding: a tap whose neighbour lies across a board
// edge is switched off for that output row by the disable-output-lane vector of the tap's tcgen05.mma (edge masks
// per tile from the loader warp, centre tap first so that it initialises the accumulator).
// An activation tensor is stored as C/8 PLANES of [rows][8 channels] fp16 (16 bytes per row):
//   contiguous buffer:  element (P, c) at ((c/8) * plane_rows + P) * 8 + c%8
//   hidden-state slot:  element (q, c) of slot s at ((s * C/8 + c/8) * PB + q) * 8 + c%8
// which is exactly the no-swizzle K-major core-matrix layout tcgen05.mma reads from shared
// memory, so (a) a tile of 256 rows + W+1 rows either side is ONE contiguous run per plane and is fetched by
// 1-D bulk copies (TMA) with no per-element work, (b) the epilogue's stores (lane = row, 16
// bytes per plane) are fully coalesced.  Rows past the last board are never read by a valid output.
//
// Kernel: implicit GEMM, M = rows, N = C_out, K = 9 taps x C_in.
//   - the activation tile (256 rows + halo) is staged ONCE in shared memory; the 9 taps are 9
//     descriptor start addresses on that one tile (umma.cuh) -> activations are read once;
//   - folded conv+BatchNorm weights stream through an mbarrier ring of 1-D bulk copies,
//     pre-packed on the host side of mz_net_create in exactly the shared-memory layout;
//   - tcgen05.mma (M=128, N=C_out, K=16) accumulates in TMEM, two 128-row accumulators
//     per tile, double-buffered across tiles so that epilogue(i-1) and load(i+1)
//     overlap mma(i);
//   - warp roles: warp 0 weight producer, warps 1 and 3 MMA issuers (one per accumulator half:
//     a single warp cannot issue an M128 N128 MMA every 64 cycles), warp 2 tile loader (TMA),
//     warps 4-11 epilogue (bias / action-bias table / residual / ReLU / per-pixel channel
//     min-max normalisation of util.py:31-36 fused here).
#include "net.cuh"
#include "umma.cuh"
#include <cuda_fp16.h>
#include <cstdlib>

namespace mz {
using namespace umma;

// Activations and folded weights are IEEE fp16 (10-bit mantissa; the hidden state is min-max
// normalised to [0,1] and BatchNorm keeps tower activations O(1..100), far inside fp16 range;
// conversions saturate instead of overflowing).  Same tensor-core rate as bf16, 8x finer rounding.
typedef __half act_t;
typedef __half2 act2_t;

constexpr int kConvThreads = 384;   // w0 weights, w1 MMA (rows 0-127), w2 tile loader, w3 MMA (rows 128-255), w4-11 epilogue
constexpr int kEpiThreads = 256;
constexpr int kTileM = 256;     // rows per tile (two M=128 accumulators)
constexpr int kMaxStages = 6;
constexpr int kMaxPairStages = 12;   // SM-pair launches: a ring slot holds half a stage
constexpr int kPlaneSlack = 64; // rows allocated past the last tile of every plane (>= the widest halo)

constexpr int kMaxLayers = 34;   // one launch runs up to a whole recurrent inference: 1 + 16 + 16 convs
static_assert(kMaxLayers == MZ_DEBUG_MAX_LAYERS, "mz_debug_launch holds one entry per LayerDesc of a launch");

// One convolution layer of a launch.  Layers of a launch share geometry, channel counts and the
// persistent CTAs; layer l+1's tile t starts as soon as tiles t-1, t, t+1 of layer l are published
// (per-tile flags in global memory), so there is no per-layer launch, prologue or tail.
struct LayerDesc {
  const act_t* in;        // planes [Cin/8][plane_rows][8], or the slot array when in_slots is set
  const int32_t* in_index;        // slot input: board b lives in slot in_index[b] (nullptr: slot b)
  const act_t* w;         // packed [9][chunks][chunk_g][N][8]
  const act_t* w_pair;    // the same weights for SM-pair launches: [9][chunks][half][chunk_g][N/2][8]
  const float* bias;              // [N]
  const float* tab;               // [A][N/8][PB][8] per-action bias (dynamics conv0) or nullptr
  const int32_t* action;          // [B]
  const act_t* residual;  // contiguous planes or nullptr
  act_t* out;             // contiguous planes (relu'd) or nullptr
  act_t* out_norm;        // contiguous planes, min-max normalised, or nullptr
  act_t* out_slots;       // indexed slots, normalised, or nullptr
  const int32_t* out_index;
  int dep0, dep1;                 // layers of THIS launch that produce the input (-1: none / an earlier launch).  Two when
                                  // the producing conv ran as two 128-column passes (num_planes = 256)
  int fwd;                        // resident launches: 1 = the next layer reads this layer's `out`, 2 = its `out_norm`
  int res_layer;                  // layer of THIS launch that writes the residual buffer (-1: an earlier launch did)
  int in_slots;                   // input is an array of hidden-state slots, not a contiguous buffer
};

struct ConvParams {
  LayerDesc L[kMaxLayers];
  int num_layers;
  int rot;                        // tile t of layer l belongs to CTA (t + l*rot) % grid: rotates who gets the odd tile
  unsigned int* flags;            // [num_layers][num_tiles], zeroed before the launch (nullptr for one layer)
  int* err;                       // dependency wait timed out (should never happen)
  int Ptot, PB, W, H, B;
  int plane_rows;                 // rows per plane of the contiguous buffers of this launch
  int sub;                        // stride-2 layer: only rows with even (y, x) are stored, on the half-size grid
  int out_plane_rows, out_PB, out_W;    // geometry of the output buffer when sub is set
  int cg;                         // input channel groups of 8 (Cin_pad / 8), even
  int N;                          // output channels of one layer of this launch (multiple of 32, <= 128); wider convs
                                  // run as several 128-column passes, each its own LayerDesc
  int n_real;                     // channels < n_real are the network's; the rest pad num_planes up to 32 (zero weights)
                                  // and are left out of the min-max normalisation
  int tab_groups;                 // channel groups of a whole action-table entry / hidden-state slot (all passes)
  int relu;
  int num_tiles;
  int TP;                         // tile rows incl. halo, odd
  int stages;                     // weight ring depth (as many as shared memory allows, <= kMaxStages)
  long long* dbg;                 // optional per-CTA role timing (MZ_CONV_DEBUG), else nullptr
  int tile_stride;                // rows between the starts of consecutive tiles: kRows, or (resident) whole boards
  int khalf;                      // resident 256-row launches with two 64-channel K chunks: the K loop runs chunk by chunk
                                  // and the epilogue hands the low / high 64 channels of the next tile over separately
  int resident;                   // every CTA owns ONE board-aligned tile for all layers; activations stay in shared memory
};
// SM-pair launches (kPair: 256-row dataflow launches of more than one stride-1 layer) run as 2-CTA clusters.  The
// unit of work is a tile PAIR: pair item j of a layer is tiles 2j (even CTA) and 2j+1 (odd CTA; past the last tile it
// is a null tile whose rows are neither read nor written, nor published), and pair items rotate over the clusters
// per layer as tiles rotate over CTAs otherwise.  The even CTA issues tcgen05.mma.cta_group::2 M = 256 for both:
// each SM reads its own 128 activation rows and HALF of the weight operand (6 KB instead of 8 KB of shared memory
// per M128-equivalent MMA), and each SM streams only its half of every weight stage (half the ring fills and the L2
// weight traffic).  Arithmetic and summation order are those of the single-CTA form.

__device__ __forceinline__ void split_pos(int P, const ConvParams& p, int& b, int& q) {
  b = P / p.PB;
  q = P - b * p.PB;
}

__device__ __forceinline__ uint32_t pack2(float a, float b) {
  act2_t t = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}

__device__ __forceinline__ unsigned ld_acquire(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release(unsigned* p, unsigned v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// bias + residual + ReLU (+ fp16 saturation) of 32 accumulator columns -> four 16-byte plane rows
__device__ __forceinline__ void finish32(const uint32_t (&r)[32], const float* s_bias_c0, const int4 (&res)[4],
                                         float (&v)[32]) {
#pragma unroll
  for (int e = 0; e < 32; e += 4) {
    const float4 b4 = *reinterpret_cast<const float4*>(s_bias_c0 + e);
    v[e] = __uint_as_float(r[e]) + b4.x; v[e + 1] = __uint_as_float(r[e + 1]) + b4.y;
    v[e + 2] = __uint_as_float(r[e + 2]) + b4.z; v[e + 3] = __uint_as_float(r[e + 3]) + b4.w;
  }
#pragma unroll
  for (int e = 0; e < 32; e += 8) {
    const act2_t* h = reinterpret_cast<const act2_t*>(&res[e / 8]);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float2 f = __half22float2(h[u]);
      v[e + 2 * u] += f.x; v[e + 2 * u + 1] += f.y;
    }
  }
}
// ReLU + fp16 saturation + pack of two floats in ONE conversion (cvt.rn.relu.satfinite.f16x2.f32 d, hi, lo)
__device__ __forceinline__ uint32_t pack2_relu(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ int4 pack8_relu(const float* v) {
  return make_int4((int)pack2_relu(v[0], v[1]), (int)pack2_relu(v[2], v[3]), (int)pack2_relu(v[4], v[5]),
                   (int)pack2_relu(v[6], v[7]));
}
__device__ __forceinline__ int4 pack8(const float* v) {
  return make_int4((int)pack2(v[0], v[1]), (int)pack2(v[2], v[3]), (int)pack2(v[4], v[5]), (int)pack2(v[6], v[7]));
}

// kRows = 256: a tile is two 128-row accumulators, one per MMA warp (the throughput configuration).
// kRows = 128: a tile is ONE 128-row block whose K range is split between the two MMA warps (weight stages
// alternate between them; each accumulates into its own TMEM accumulator and the epilogue adds the two in a
// fixed order, so results stay deterministic).  Half the MMA time per tile: for launches with few tiles per SM
// the layer-to-layer dependency chain (load -> MMA -> epilogue -> publish) is the bound, not throughput.
// 64-thread named barrier 2 + quad with an IMMEDIATE id: with the id in a register ptxas must assume all 16
// hardware barriers are in use ("used 16 barriers"), and an SM whose 16 barriers are taken by the persistent conv CTA
// cannot host any other CTA that uses __syncthreads() -- the tree kernels of the other sub-batch then wait for
// the whole tower instead of running beside it (tools/coresident_probe.py).
__device__ __forceinline__ void quad_bar_sync(int quad) {
  switch (quad) {
    case 0: asm volatile("bar.sync 2, 64;" ::: "memory"); break;
    case 1: asm volatile("bar.sync 3, 64;" ::: "memory"); break;
    case 2: asm volatile("bar.sync 4, 64;" ::: "memory"); break;
    default: asm volatile("bar.sync 5, 64;" ::: "memory"); break;
  }
}

__device__ __forceinline__ void st_tile(uint32_t addr, const int4& v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __constant__ int kTapOrder[9] = {4, 0, 1, 2, 3, 5, 6, 7, 8};

template <int kN, int kRows, bool kPair = false>
__global__ void __maxnreg__(128) conv3x3_kernel(const __grid_constant__ ConvParams p) {
  static_assert(!kPair || kRows == 256, "SM-pair launches use 256-row tiles");
  constexpr bool kSplitK = (kRows == 128);
  constexpr int kRing = kPair ? kMaxPairStages : kMaxStages;
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int halo = p.W + 1;
  const int TP = p.TP;
  const int chunk_g = p.cg < 8 ? p.cg : 8;              // channel groups per weight stage
  const int chunks_tap = p.cg / chunk_g;                // weight stages per tap
  // a ring slot: the whole stage [chunk_g][N][8], or (pair) this CTA's half of its N rows, [chunk_g][N/2][8]
  const uint32_t half_rows = kPair ? (uint32_t)p.N / 2 : (uint32_t)p.N;
  const uint32_t stage_bytes = (uint32_t)chunk_g * half_rows * 16;
  const uint32_t a_bytes = (uint32_t)p.cg * TP * 16;
  // pair launches: this CTA's rank in its cluster; the even CTA (rank 0) issues the MMAs of both
  const uint32_t rank = kPair ? cluster_ctarank() : 0u;
  const bool resident = !kPair && p.resident, khalf = !kPair && p.khalf;

  unsigned char* sA = smem;                                              // [2][cg][TP][16]
  unsigned char* sW = smem + (((size_t)2 * a_bytes + 127) & ~(size_t)127);   // [kStages][stage_bytes]
  const uint32_t kStages = (uint32_t)p.stages;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sW + (size_t)kStages * stage_bytes);
  uint64_t* w_full = bars;                 // [kStages]
  uint64_t* w_empty = bars + kRing;        // [kStages]
  uint64_t* a_full = bars + 2 * kRing;     // [2]
  uint64_t* mma_done = a_full + 2;         // [2]
  uint64_t* acc_empty = mma_done + 2;      // [2]
  uint64_t* a_ready = acc_empty + 2;       // [2 tiles][low, high channels] resident launches: the epilogue has written
                                           // that half of the next layer's tile
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(a_ready + 4);
  float* s_bias = reinterpret_cast<float*>(tmem_holder + 4);            // [4][N] bias of layer l in slot l & 3, 16-byte aligned
  float2* s_mm = reinterpret_cast<float2*>(s_bias + 4 * p.N);           // [2][128] partial (min, max) per row
  uint32_t* s_mask = reinterpret_cast<uint32_t*>(s_mm + 2 * 128);       // [2 tiles][2 halves][left,right,top,bottom][4] edge rows

  if (tid == 0) {
    tmem_holder[2] = 0;
    // Arrival counts.  Pair launches: barriers the even CTA's MMAs wait on also take one arrival forwarded by the odd
    // CTA (its half of the weight stage / its tile has landed, its epilogue has drained its accumulator); the MMA
    // commits (w_empty, mma_done) are multicast to both CTAs, so those counts are the same in both.
    const uint32_t fwd = (kPair && rank == 0) ? 1u : 0u;
    for (uint32_t s = 0; s < kStages; ++s) {
      mbar_init(&w_full[s], 1 + fwd);                 // own producer (+ the odd CTA's forwarder)
      mbar_init(&w_empty[s], kSplitK ? 1 : 2);        // a commit per MMA warp that used the stage
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&a_full[b], 1 + fwd);                 // own tile loader (+ the odd CTA's forwarder)
      mbar_init(&mma_done[b], 2);                     // a commit per MMA warp
      mbar_init(&acc_empty[b], kEpiThreads + fwd);    // own epilogue threads (+ one arrival for the odd CTA's)
      mbar_init(&a_ready[2 * b], kEpiThreads); mbar_init(&a_ready[2 * b + 1], kEpiThreads);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    if (kPair) tmem_alloc_pair(tmem_holder, 512);
    else tmem_alloc(tmem_holder, 512);
  }
  tc_fence_before();
  if (kPair) cluster_sync();           // the peer's barriers are initialised before anything arrives on them
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_holder;
  // tmem_holder[2]: number of items whose RESIDUAL producer (layer res_layer, same tile, possibly another CTA) the
  // weight-producer lane has seen published (dataflow launches); read by the epilogue before it requests residual rows
  const uint32_t s_res_a = smem_u32(tmem_holder + 2);

  // every role walks the same (layer, unit) item sequence of this CTA; a unit is a tile, or (pair) a tile pair, and
  // BOTH CTAs of a pair walk the same sequence
  const int G = kPair ? (int)gridDim.x >> 1 : (int)gridDim.x;          // CTAs, or clusters
  const int me = kPair ? (int)blockIdx.x >> 1 : (int)blockIdx.x;
  const int num_units = kPair ? (p.num_tiles + 1) >> 1 : p.num_tiles;
  auto first_unit = [&](int l) { int t0 = (me - l * p.rot) % G; return t0 < 0 ? t0 + G : t0; };
  auto tile_of = [&](int u) { return kPair ? 2 * u + (int)rank : u; };
  const bool dbg = p.dbg != nullptr;
  // pair launches: the MMA-side role timing is the even CTA's
  const bool dbg_mma = dbg && (!kPair || rank == 0);

  if (warp == 0) {
    // ------------------------------------------------ weight producer
    if (lane == 0) {
      const int per_tile = 9 * chunks_tap;
      uint32_t it = 0, res_items = 0;
      long long t_wait = 0, t_gate = 0;
      const long long t_begin = clock64();
      // pair: a stage of the pair layout is two contiguous halves, this CTA's is at rank * stage_bytes
      const uint32_t full_stage = (uint32_t)chunk_g * p.N * 16, own = rank * stage_bytes;
      for (int l = 0; l < p.num_layers; ++l) {
        const unsigned char* wl = reinterpret_cast<const unsigned char*>(kPair ? p.L[l].w_pair : p.L[l].w);
        for (int u = first_unit(l); u < num_units; u += G) {
          const int tile = tile_of(u);
          if (!resident && p.flags) {
            const long long tg = dbg ? clock64() : 0;
            // The epilogue prefetches this item's residual rows (written by layer res_layer, same tile, in general by
            // ANOTHER CTA two layers ago) before its MMAs finish, i.e. possibly before this CTA's loader has acquired
            // the item's dependency flags -- nothing would order that write before the prefetch.  This lane, which
            // runs a few weight stages ahead of everything else, acquires the producer's flag (it is practically
            // always set already: 0 misses in 10^4 items measured) and publishes an item counter at CTA scope.
            const LayerDesc& Lr = p.L[l];
            if (Lr.residual && Lr.res_layer >= 0 && (!kPair || tile < p.num_tiles)) {
              const unsigned* f = p.flags + (size_t)Lr.res_layer * p.num_tiles + tile;
              unsigned spins = 0;
              while (ld_acquire(f) == 0u) {
                if (++spins > (1u << 26)) { if (p.err) atomicExch(p.err, 1); break; }
              }
            }
            ++res_items;
            if (dbg) t_gate += clock64() - tg;
            asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(s_res_a), "r"(res_items) : "memory");
          }
          for (int c = 0; c < per_tile; ++c, ++it) {
            const uint32_t s = it % kStages, ph = (it / kStages) & 1;
            const long long tw = dbg ? clock64() : 0;
            mbar_wait(&w_empty[s], ph ^ 1);
            if (dbg) t_wait += clock64() - tw;
            mbar_arrive_expect_tx(&w_full[s], stage_bytes);
            // taps are consumed centre first (kTapOrder): the centre tap is the one no edge mask applies to, so it is
            // the MMA that initialises every row of the accumulator
            // (khalf: all taps of the low 64 input channels first, then the high ones -- the order the MMA warps use)
            const int ti = khalf ? c % 9 : c / chunks_tap, chs = khalf ? c / 9 : c - ti * chunks_tap;
            const int src_stage = kTapOrder[ti] * chunks_tap + chs;
            bulk_g2s(sW + (size_t)s * stage_bytes, wl + (size_t)src_stage * full_stage + own, stage_bytes, &w_full[s]);
          }
        }
      }
      if (dbg) { long long* d = p.dbg + blockIdx.x * 16; d[0] = clock64() - t_begin; d[1] = t_wait; d[15] = t_gate; }
    }
  } else if (kPair && rank == 1 && (warp == 1 || warp == 3)) {
    // ------------------------------------------------ odd CTA of a pair: no MMAs to issue.  Its MMA warps forward the
    // completion of its own barriers to the even CTA, whose MMAs read this CTA's shared memory: a 1-D bulk copy can
    // only signal a barrier in the CTA it writes to.  Warp 1 forwards a_full once per item as a release at cluster
    // scope after the observed phase completion: besides TMA bytes it carries the edge masks the loader stored with
    // st.shared, which the even CTA reads with ld.shared::cluster after its cluster-scope acquire.  Warp 3 forwards
    // w_full once per weight stage as a RELAXED arrival: the only payload is bulk-copy bytes in this CTA's shared
    // memory, read by this SM's own tensor pipe, and they have landed when the local phase completes; the arrival is
    // issued only after that completion, and the MMA only after the even CTA sees the arrival.  A release at cluster
    // scope there compiles to MEMBAR.ALL.GPU per stage and measured 1.71 M instead of 1.03 M cycles per 33-layer
    // Gomoku launch.
    if (lane == 0) {
      const int per_tile = 9 * chunks_tap;
      uint32_t it = 0;
      int i = 0;
      for (int l = 0; l < p.num_layers; ++l)
        for (int u = first_unit(l); u < num_units; u += G, ++i) {
          if (warp == 1) {
            mbar_wait(&a_full[i & 1], (uint32_t)(i >> 1) & 1);
            mbar_arrive_remote(&a_full[i & 1], 0);
          } else {
            for (int c = 0; c < per_tile; ++c, ++it) {
              const uint32_t s = it % kStages, ph = (it / kStages) & 1;
              mbar_wait(&w_full[s], ph);
              mbar_arrive_remote_relaxed(&w_full[s], 0);
            }
          }
        }
    }
    __syncwarp();
  } else if (warp == 1 || warp == 3) {
    // ------------------------------------------------ MMA issuers: warp 1 drives accumulator 0 (tile rows 0-127),
    // warp 3 accumulator 1 (rows 128-255); a weight stage / a tile is released when BOTH have committed.
    // (Pair launches: the even CTA's warp 1 covers rows 0-127 of both CTAs' tiles, warp 3 rows 128-255.)
    // The WHOLE warp walks the loop and one lane is elected inside each tcgen05 asm statement, so
    // ptxas emits straight-line predicated UTCHMMAs (an `if (lane == 0)` around them costs a convergence
    // loop per MMA, ~100 cycles).  Descriptors are built once; only their 14-bit start-address field
    // (16-byte units) is stepped.
    const uint32_t mhalf = warp == 1 ? 0u : 1u;
    const uint32_t idesc = instr_desc_f16(kPair ? 256 : 128, (uint32_t)p.N);
    const uint64_t a_tmpl = smem_desc(0, (uint32_t)TP * 16, 128);
    const uint64_t b_tmpl = smem_desc(0, half_rows * 16, 128);
    const uint32_t a_hi = (uint32_t)(a_tmpl >> 32), a_lo0 = (uint32_t)a_tmpl;
    const uint32_t b_hi = (uint32_t)(b_tmpl >> 32), b_lo0 = (uint32_t)b_tmpl;
    const uint32_t a_kstep = 2u * (uint32_t)TP, b_kstep = 2u * half_rows;   // 16-byte units per K=16 step
    const uint32_t sA16 = smem_u32(sA) >> 4, sW16 = smem_u32(sW) >> 4, stage16 = stage_bytes >> 4;
    const int ksteps = chunk_g / 2;
    auto desc64 = [](uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; };
    // barriers that also count an arrival from the odd CTA are acquired at cluster scope
    auto wait_bar = [&](uint64_t* b, uint32_t ph) { if (kPair) mbar_wait_cluster(b, ph); else mbar_wait(b, ph); };
    uint32_t st = 0, st_ph = 0;                 // weight ring slot and its phase parity
    uint32_t b_slot = b_lo0 + sW16;             // descriptor low word of ring slot `st`
    const uint32_t b_first = b_slot;
    long long t_acc = 0, t_a = 0, t_w = 0, t_a_pos[3] = {0, 0, 0};
    const long long t_begin = clock64();
    int i = 0;
    for (int l = 0; l < p.num_layers; ++l)
    for (int u = first_unit(l); u < num_units; u += G, ++i) {
      const int buf = i & 1;
      const uint32_t uph = (i >> 1) & 1;
      const int pos_in_layer = (u - first_unit(l)) / G;
      long long tw = dbg ? clock64() : 0;
      wait_bar(&acc_empty[buf], uph ^ 1);
      long long tw2 = dbg ? clock64() : 0;
      t_acc += tw2 - tw;
      wait_bar(&a_full[buf], uph);
      // resident launch (item i == layer i): the tile of layer i >= 1 was written by the epilogue of layer i - 1
      const uint32_t rdy_ph = (uint32_t)(((i >> 1) - (buf == 0 ? 1 : 0)) & 1);
      if (resident && i > 0) {
        mbar_wait(&a_ready[2 * buf], rdy_ph);                         // low 64 channels of the tile
        if (!khalf) mbar_wait(&a_ready[2 * buf + 1], rdy_ph);         // khalf: the high half is awaited before its K chunk
      }
      if (dbg) { const long long dt = clock64() - tw2; t_a += dt; t_a_pos[pos_in_layer < 2 ? pos_in_layer : 2] += dt; }
      tc_fence_after();
      const uint32_t a_tile = a_lo0 + sA16 + (uint32_t)buf * (a_bytes >> 4) + (uint32_t)halo + (kSplitK ? 0u : 128u * mhalf);
      const uint32_t dacc = tmem + (uint32_t)(buf * 256) + 128u * mhalf;
      uint32_t acc = 0;
      uint32_t stage_no = 0;                    // weight stage within the tile (split-K: stage s belongs to warp s & 1)
      // rows of this accumulator that sit on a board edge (left / right column, top / bottom row), from the loader
      // (pair: also the odd CTA's, which its loader stored before the a_full arrival forwarded above)
      const uint4* em = reinterpret_cast<const uint4*>(s_mask + (buf * 2 + (kSplitK ? 0 : (int)mhalf)) * 16);
      const uint4 eL = em[0], eR = em[1], eT = em[2], eB = em[3];
      uint4 pL = make_uint4(0, 0, 0, 0), pR = pL, pT = pL, pB = pL;
      if (kPair) { pL = ld_shared_peer_v4(em, 1); pR = ld_shared_peer_v4(em + 1, 1); pT = ld_shared_peer_v4(em + 2, 1); pB = ld_shared_peer_v4(em + 3, 1); }
      // one weight stage (a 64-channel K chunk of one tap): wait for it, issue its MMAs, release it, step the ring
      auto run_stage = [&](uint32_t a_lo, const uint4& m, const uint4& pm) {
        if (kSplitK && (stage_no & 1u) != mhalf) {       // the other warp's stage: just step the ring
          ++stage_no;
          ++st; b_slot += stage16;
          if (st == kStages) { st = 0; st_ph ^= 1; b_slot = b_first; }
          return;
        }
        ++stage_no;
        const long long tws = (kPair && dbg) ? clock64() : 0;
        mbar_wait(&w_full[st], st_ph);      // see the odd CTA's w_full forwarder
        if (kPair && dbg) t_w += clock64() - tws;
        tc_fence_after();
        uint32_t b_lo = b_slot;
        if (kPair || ksteps == 4) {                       // pair launches always have 64-channel stages (flush)
          // the common case (64-channel stage) fully unrolled
          uint32_t al[4], bl[4];
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) { al[ks] = a_lo + (uint32_t)ks * a_kstep; bl[ks] = b_lo + (uint32_t)ks * b_kstep; }
          if (kPair)
            mma4_f16_pair_elect_masked(dacc, desc64(al[0], a_hi), desc64(al[1], a_hi), desc64(al[2], a_hi),
                                       desc64(al[3], a_hi), desc64(bl[0], b_hi), desc64(bl[1], b_hi), desc64(bl[2], b_hi),
                                       desc64(bl[3], b_hi), idesc, acc, m, pm);
          else
            mma4_f16_elect_masked(dacc, desc64(al[0], a_hi), desc64(al[1], a_hi), desc64(al[2], a_hi), desc64(al[3], a_hi),
                                  desc64(bl[0], b_hi), desc64(bl[1], b_hi), desc64(bl[2], b_hi), desc64(bl[3], b_hi), idesc,
                                  acc, m.x, m.y, m.z, m.w);
          acc = 1;
        } else {
          for (int ks = 0; ks < ksteps; ++ks) {
            mma_f16_elect_masked(dacc, desc64(a_lo, a_hi), desc64(b_lo, b_hi), idesc, acc, m.x, m.y, m.z, m.w);
            acc = 1;
            a_lo += a_kstep;
            b_lo += b_kstep;
          }
        }
        if (kPair) commit_pair_elect(&w_empty[st]);
        else commit_elect(&w_empty[st]);
        ++st; b_slot += stage16;
        if (st == kStages) { st = 0; st_ph ^= 1; b_slot = b_first; }
      };
      // taps centre first (kTapOrder); K chunks inside a tap -- or, khalf, all taps of the low 64 input channels, then
      // (once the epilogue of the previous layer has handed them over) all taps of the high 64
      const int outer = khalf ? 2 : 1;
      // output rows whose (y + ky - 1, x + kx - 1) neighbour is across a board edge take no part in a tap
      auto tap_mask = [](int ky, int kx, const uint4& L, const uint4& R, const uint4& T, const uint4& B) {
        auto w = [&](uint32_t l, uint32_t r, uint32_t t, uint32_t b) {
          return (kx == 0 ? l : 0u) | (kx == 2 ? r : 0u) | (ky == 0 ? t : 0u) | (ky == 2 ? b : 0u);
        };
        return make_uint4(w(L.x, R.x, T.x, B.x), w(L.y, R.y, T.y, B.y), w(L.z, R.z, T.z, B.z), w(L.w, R.w, T.w, B.w));
      };
      for (int ko = 0; ko < outer; ++ko) {
        if (khalf && ko == 1 && i > 0) { mbar_wait(&a_ready[2 * buf + 1], rdy_ph); tc_fence_after(); }
        for (int ti = 0; ti < 9; ++ti) {
          const int tap = ti == 0 ? 4 : (ti <= 4 ? ti - 1 : ti);
          const int ky = tap / 3, kx = tap - 3 * ky;
          const uint32_t a_tap = a_tile + (uint32_t)((ky - 1) * p.W + (kx - 1));   // wraps correctly: the shift may be negative
          const uint4 m = tap_mask(ky, kx, eL, eR, eT, eB);
          const uint4 pm = kPair ? tap_mask(ky, kx, pL, pR, pT, pB) : m;
          if (khalf) {
            run_stage(a_tap + (uint32_t)(ko * ksteps) * a_kstep, m, pm);
          } else {
            for (int ch = 0; ch < chunks_tap; ++ch) run_stage(a_tap + (uint32_t)(ch * ksteps) * a_kstep, m, pm);
          }
        }
      }
      if (kPair) commit_pair_elect(&mma_done[buf]);
      else commit_elect(&mma_done[buf]);
    }
    if (dbg_mma && lane == 0 && warp == 1) {
      long long* d = p.dbg + blockIdx.x * 16;
      d[2] = clock64() - t_begin; d[3] = t_acc; d[4] = t_a; d[5] = t_w; d[6] = i;
      d[12] = t_a_pos[0]; d[13] = t_a_pos[1]; d[14] = t_a_pos[2];
    }
  } else if (warp == 2) {
    // ------------------------------------------------ tile loader: activation rows -> shared memory by bulk copies.
    // A tile's rows are one contiguous run per channel-group plane (or one run per board and plane when the
    // input lives in indexed hidden-state slots), already in the shared-memory layout.
    const int cg = p.cg;
    long long t_wait = 0, t_dep = 0;
    const long long t_begin = clock64();
    int i = 0, bias_layer = -1;
    for (int l = 0; l < p.num_layers; ++l)
    for (int u = first_unit(l); u < num_units; u += G, ++i) {
      const int tile = tile_of(u);
      const LayerDesc& L = p.L[l];
      const int buf = i & 1;
      const int r0 = tile * p.tile_stride - halo, r1 = r0 + kRows + 2 * halo;       // tile rows [r0, r1)
      const bool handed_over = resident && l > 0;       // the epilogue of layer l - 1 writes this tile into shared memory
      // pair launches with an odd tile count: the odd CTA's last item is a null tile; it loads nothing but still
      // arrives, so that the pair's MMAs run (its accumulator rows are never stored)
      const bool null_tile = kPair && tile >= p.num_tiles;
      // dataflow dependency: the three tiles of the previous layer whose rows this tile reads
      long long tw = dbg ? clock64() : 0;
      if (L.dep0 >= 0 && !resident && !null_tile) {
        if (lane < 6) {
          const int tt = tile - 1 + lane % 3;
          const int dl = lane < 3 ? L.dep0 : L.dep1;
          if (dl >= 0 && tt >= 0 && tt < p.num_tiles) {
            const unsigned* f = p.flags + (size_t)dl * p.num_tiles + tt;
            unsigned spins = 0;
            while (ld_acquire(f) == 0u) {
              ++spins;
              if ((spins & 0xffffu) == 0 && p.err && *reinterpret_cast<volatile int*>(p.err)) break;   // sticky bail-out
              if (spins > (1u << 26)) { if (p.err) atomicExch(p.err, 1); break; }
            }
          }
        }
        __syncwarp();
        asm volatile("fence.proxy.async;" ::: "memory");   // other CTAs' (generic-proxy) stores -> our async-proxy reads
      }
      long long tw2 = dbg ? clock64() : 0;
      t_dep += tw2 - tw;
      // the buffer was last read by the MMAs of tile i-2
      if (i >= 2) mbar_wait(&mma_done[buf], (uint32_t)(((i - 2) >> 1) & 1));
      if (dbg) t_wait += clock64() - tw2;
      // this layer's bias vector -> slot l & 3 (the epilogue is at most two items behind, so a slot is not reused
      // while it is read; the write is ordered before the epilogue's reads by a_full -> MMA -> mma_done)
      if (l != bias_layer) {
        for (int c4 = lane; c4 * 4 < kN; c4 += 32)
          *reinterpret_cast<float4*>(s_bias + (l & 3) * kN + c4 * 4) = __ldg(reinterpret_cast<const float4*>(L.bias) + c4);
        bias_layer = l;
      }
      // which rows of this tile are a board's left / right column or top / bottom row: one ballot per 32 rows
      for (int h = 0; h < kRows / 128; ++h)
        for (int w = 0; w < 4; ++w) {
          const int P = tile * p.tile_stride + h * 128 + w * 32 + lane;
          const int q = P % p.PB, y = q / p.W, x = q - y * p.W;
          const unsigned mL = __ballot_sync(0xffffffffu, x == 0), mR = __ballot_sync(0xffffffffu, x == p.W - 1);
          const unsigned mT = __ballot_sync(0xffffffffu, y == 0), mB = __ballot_sync(0xffffffffu, y == p.H - 1);
          if (lane == 0) {
            uint32_t* m = s_mask + (buf * 2 + h) * 16;
            m[w] = mL; m[4 + w] = mR; m[8 + w] = mT; m[12 + w] = mB;
          }
        }
      const uint32_t dst0 = smem_u32(sA) + (uint32_t)buf * a_bytes;
      if (handed_over || null_tile) {   // nothing to load: bias and masks are staged, tell the MMA warps
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_full[buf]);
        continue;
      }
      // resident: exactly the tile's own boards (every tap that leaves them is masked); else the tile and its halo
      const int lo = resident ? tile * p.tile_stride : (r0 > 0 ? r0 : 0);
      int hi = L.in_slots ? p.Ptot : p.plane_rows;
      if (resident) { const int e = lo + p.tile_stride; hi = e < p.Ptot ? e : p.Ptot; }
      else hi = r1 < hi ? r1 : hi;
      if (r0 < 0 && !resident) {
        // rows before the first board are read by valid outputs (top-left taps of board 0): zeros
        const int nz = -r0;
        for (int k = lane; k < nz * cg; k += 32) {
          const int g = k / nz, q = k - g * nz;
          asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(dst0 + (uint32_t)(g * TP + q) * 16), "r"(0) : "memory");
        }
        fence_proxy_async();
      }
      __syncwarp();
      if (lane == 0) mbar_arrive_expect_tx(&a_full[buf], (uint32_t)(hi - lo) * 16u * (uint32_t)cg);
      __syncwarp();
      if (!L.in_slots) {
        for (int g = lane; g < cg; g += 32)
          bulk_g2s_u32(dst0 + (uint32_t)(g * TP + (lo - r0)) * 16, L.in + ((size_t)g * p.plane_rows + lo) * 8,
                       (uint32_t)(hi - lo) * 16u, &a_full[buf]);
      } else {
        const int b_lo = lo / p.PB, nb = (hi - 1) / p.PB - b_lo + 1;
        for (int k = lane; k < nb * cg; k += 32) {
          const int bi = k / cg, g = k - bi * cg, b = b_lo + bi;
          const int s0 = b * p.PB > lo ? b * p.PB : lo, s1 = (b + 1) * p.PB < hi ? (b + 1) * p.PB : hi;
          const size_t slot = L.in_index ? (size_t)L.in_index[b] : (size_t)b;
          bulk_g2s_u32(dst0 + (uint32_t)(g * TP + (s0 - r0)) * 16,
                       L.in + ((slot * cg + g) * p.PB + (size_t)(s0 - b * p.PB)) * 8, (uint32_t)(s1 - s0) * 16u,
                       &a_full[buf]);
        }
      }
    }
    if (dbg && lane == 0) {
      long long* d = p.dbg + blockIdx.x * 16;
      d[7] = clock64() - t_begin; d[8] = t_wait; d[9] = t_dep;
    }
  } else if (warp >= 4) {
    // ------------------------------------------------ epilogue (warps 4-11): TMEM -> registers -> global
    // warp w reads TMEM lanes 32*(w%4).. (its rows) and one half of the output columns
    const int quad = warp & 3, chalf = (warp - 4) >> 2;
    const int et = tid - 128;                // 0..255
    constexpr int NC = kN / 32;              // 32-column chunks of the accumulator
    constexpr int NCW = NC >= 2 ? NC / 2 : 1;     // chunks per warp
    const bool has_cols = chalf * NCW < NC;
    const size_t PR = (size_t)p.plane_rows;
    long long t_wait = 0;
    const long long t_begin = clock64();
    int k = 0;
    for (int l = 0; l < p.num_layers; ++l)
    for (int u = first_unit(l); u < num_units; u += G, ++k) {
      const int tile = tile_of(u);
      const LayerDesc& L = p.L[l];
      const bool norm = (L.out_norm != nullptr) || (L.out_slots != nullptr);
      const int buf = k & 1;
      const float* s_bias_l = s_bias + (l & 3) * kN;
      const bool fast = !norm && L.tab == nullptr && L.out != nullptr;
      // resident launch: this layer's output rows also go straight into the OTHER tile buffer in shared memory, in the
      // operand layout ([channel group][row][16 B], rows offset by the halo), where the next layer's MMAs read them
      const int hand = (resident && l + 1 < p.num_layers) ? L.fwd : 0;
      bool lo_done = false;
      const uint32_t next_a = smem_u32(sA) + (uint32_t)(buf ^ 1) * a_bytes + (uint32_t)halo * 16;
      const uint32_t tbase = tmem + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * 256);
      if (fast) {
        // Plain conv + bias (+ residual) + ReLU (30 of the 33 convs of a recurrent inference).  The steps of
        // this warp (2 row halves x NCW column chunks) form one unrolled sequence and the residual of step
        // t+2 is requested at step t (the first two before the MMAs even finish).
        constexpr int NJ = kRows / 128;      // 128-row blocks of a tile
        constexpr int STEPS = NJ * NCW;
        int Pj[2];
        size_t Dj[2];                        // destination row of the output buffer
        bool vj[2], inr[2];                  // row in range (of the batch and of this tile) / row that is stored
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          Pj[j] = tile * p.tile_stride + j * 128 + quad * 32 + lane;
          vj[j] = Pj[j] < p.Ptot && j * 128 + quad * 32 + lane < p.tile_stride;
          inr[j] = vj[j];
          Dj[j] = (size_t)Pj[j];
          int b, pos;                        // only used under p.sub; split here, ptxas then spills less at 128 registers
          split_pos(Pj[j], p, b, pos);
          if (p.sub) {
            // stride-2 convolution (padding 1) == the stride-1 result at the even positions: store those rows
            // on the half-size grid, drop the rest
            const int y = pos / p.W, x = pos - y * p.W;
            inr[j] = vj[j] && !((y | x) & 1);
            Dj[j] = (size_t)b * p.out_PB + (size_t)(y >> 1) * p.out_W + (x >> 1);
          }
        }
        const size_t PRo = p.sub ? (size_t)p.out_plane_rows : PR;
        const int4* resp = reinterpret_cast<const int4*>(L.residual);
        const bool has_res = resp != nullptr;
        int4 ring[3][4];
        // step t of this warp -> (row half j, 32-column chunk c).  khalf: low 64 channels (chunks 0, 1 across the two
        // column-half warps) of every row first, so that they can be handed to the next layer's first K chunk early
        const bool kh = khalf && NCW == 2;
        auto jof = [&](int t) { return kh ? t % NJ : t / NCW; };
        auto cof = [&](int t) { return kh ? 2 * (t / NJ) + chalf : chalf * NCW + t % NCW; };
        // j is a run-time value under khalf: select, do not index (indexing would move the arrays to local memory)
        auto pick = [&](const auto (&arr)[2], int j) { return (NJ > 1 && j) ? arr[NJ - 1] : arr[0]; };
        auto fetch = [&](int t, int4 (&dst)[4]) {
          const int j = jof(t), g0 = cof(t) * 4;
          const bool ld = has_res && pick(vj, j);
#pragma unroll
          for (int u = 0; u < 4; ++u) dst[u] = ld ? __ldcg(resp + (size_t)(g0 + u) * PR + pick(Pj, j)) : make_int4(0, 0, 0, 0);
        };
        if (!resident && has_res && p.flags && L.res_layer >= 0) {
          // ordered behind the residual producer's flag, see the weight-producer warp (a counter that is ahead of us)
          uint32_t seen;
          do { asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(seen) : "r"(s_res_a) : "memory"); } while (seen < (uint32_t)(k + 1));
        }
        if (has_cols) {
          fetch(0, ring[0]);
          if (STEPS > 1) fetch(1, ring[1]);
        }
        const long long tw = dbg ? clock64() : 0;
        mbar_wait(&mma_done[buf], (uint32_t)((k >> 1) & 1));
        if (dbg) t_wait += clock64() - tw;
        tc_fence_after();
        if (has_cols) {
          int4* outp = reinterpret_cast<int4*>(L.out);
#pragma unroll
          for (int t = 0; t < STEPS; ++t) {
            const int j = jof(t), c = cof(t), c0 = c * 32;
            if (t + 2 < STEPS) fetch(t + 2, ring[(t + 2) % 3]);
            uint32_t r[32];
            tmem_ld32(tbase + (uint32_t)(j * 128 + c0), r);
            if (kSplitK) {                     // second half of the K range lives in the other accumulator
              uint32_t r2[32];
              tmem_ld32(tbase + (uint32_t)(128 + c0), r2);
              tmem_ld_wait();
#pragma unroll
              for (int e = 0; e < 32; ++e) r[e] = __float_as_uint(__fadd_rn(__uint_as_float(r[e]), __uint_as_float(r2[e])));
            } else {
              tmem_ld_wait();
            }
            float v[32];
            finish32(r, s_bias_l + c0, ring[t % 3], v);
            // ReLU (every conv of these nets is followed by one) and fp16 saturation ride on the fp32 -> fp16
            // conversion
            if (pick(inr, j)) {
#pragma unroll
              for (int u = 0; u < 4; ++u) outp[(size_t)(c * 4 + u) * PRo + pick(Dj, j)] = pack8_relu(v + 8 * u);
            }
            if (hand == 1) {
#pragma unroll
              for (int u = 0; u < 4; ++u) st_tile(next_a + (uint32_t)((c * 4 + u) * TP + j * 128 + quad * 32 + lane) * 16,
                                                   pack8_relu(v + 8 * u));
              if (kh && t + 1 == NJ) {           // channels 0-63 of every row of this thread are in place
                fence_proxy_async();
                mbar_arrive(&a_ready[2 * (buf ^ 1)]);
                lo_done = true;
              }
            }
          }
        }
      } else {
        const long long tw = dbg ? clock64() : 0;
        mbar_wait(&mma_done[buf], (uint32_t)((k >> 1) & 1));
        if (dbg) t_wait += clock64() - tw;
        tc_fence_after();
#pragma unroll 1
        for (int j = 0; j < kRows / 128; ++j) {
          const int P = tile * p.tile_stride + j * 128 + quad * 32 + lane;
          int b = 0, pos = 0;
          const bool inrange = P < p.Ptot && j * 128 + quad * 32 + lane < p.tile_stride;
          if (inrange) split_pos(P, p, b, pos);
          const float* tab = (L.tab && inrange) ? L.tab + ((size_t)L.action[b] * p.tab_groups * p.PB + pos) * 8 : nullptr;
          const int4* resp = (L.residual && inrange) ? reinterpret_cast<const int4*>(L.residual) + P : nullptr;
          // conv + bias (+ table) (+ residual) + ReLU of one 32-column chunk of this row (one chunk live at a
          // time keeps the register count of the whole kernel low; the normalising layers read TMEM twice)
          auto chunk = [&](int c, float (&v)[32]) {
            int4 rres[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) rres[u] = resp ? __ldcg(resp + (size_t)(c * 4 + u) * PR) : make_int4(0, 0, 0, 0);
            uint32_t r[32];
            tmem_ld32(tbase + (uint32_t)(j * 128 + c * 32), r);
            if (kSplitK) {
              uint32_t r2[32];
              tmem_ld32(tbase + (uint32_t)(128 + c * 32), r2);
              tmem_ld_wait();
#pragma unroll
              for (int e = 0; e < 32; ++e) r[e] = __float_as_uint(__fadd_rn(__uint_as_float(r[e]), __uint_as_float(r2[e])));
            } else {
              tmem_ld_wait();
            }
            finish32(r, s_bias_l + c * 32, rres, v);
            if (tab) {
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const float4* t4 = reinterpret_cast<const float4*>(tab + (size_t)(c * 4 + u) * p.PB * 8);
                const float4 ta = t4[0], tb = t4[1];
                v[8 * u] += ta.x; v[8 * u + 1] += ta.y; v[8 * u + 2] += ta.z; v[8 * u + 3] += ta.w;
                v[8 * u + 4] += tb.x; v[8 * u + 5] += tb.y; v[8 * u + 6] += tb.z; v[8 * u + 7] += tb.w;
              }
            }
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = fminf(fmaxf(v[e], 0.0f), inrange ? 65504.0f : 0.0f);
          };
          float mn = INFINITY, mx = -INFINITY;
          int4* o = (L.out && inrange) ? reinterpret_cast<int4*>(L.out) + P : nullptr;
          if (has_cols) {
#pragma unroll 1
            for (int cc = 0; cc < NCW; ++cc) {
              const int c = chalf * NCW + cc;
              float v[32];
              chunk(c, v);
#pragma unroll
              for (int e = 0; e < 32; ++e)
                if (c * 32 + e < p.n_real) { mn = fminf(mn, v[e]); mx = fmaxf(mx, v[e]); }
              if (o) {
#pragma unroll
                for (int u = 0; u < 4; ++u) o[(size_t)(c * 4 + u) * PR] = pack8(v + 8 * u);
              }
              if (hand == 1) {
#pragma unroll
                for (int u = 0; u < 4; ++u) st_tile(next_a + (uint32_t)((c * 4 + u) * TP + j * 128 + quad * 32 + lane) * 16,
                                                     pack8(v + 8 * u));
              }
            }
          }
          if (norm) {
            // min/max over ALL channels of the row: combine with the warp holding the other column half
            s_mm[chalf * 128 + quad * 32 + lane] = make_float2(mn, mx);
            quad_bar_sync(quad);
            const float2 o = s_mm[(chalf ^ 1) * 128 + quad * 32 + lane];
            quad_bar_sync(quad);
            mn = fminf(mn, o.x); mx = fmaxf(mx, o.y);
            const float inv = inrange ? 1.0f / ((mx - mn) + 1e-8f) : 0.0f;
            if (has_cols) {             // warp-uniform: the TMEM loads inside chunk() are warp-collective
              int4* on = (L.out_norm && inrange) ? reinterpret_cast<int4*>(L.out_norm) + P : nullptr;
              int4* os = nullptr;
              if (L.out_slots && inrange) {
                const size_t slot = L.out_index ? (size_t)L.out_index[b] : (size_t)b;
                os = reinterpret_cast<int4*>(L.out_slots) + slot * p.tab_groups * p.PB + pos;
              }
#pragma unroll 1
              for (int cc = 0; cc < NCW; ++cc) {
                const int c = chalf * NCW + cc;
                float v[32];
                chunk(c, v);
#pragma unroll
                for (int e = 0; e < 32; ++e) v[e] = (c * 32 + e < p.n_real) ? (v[e] - mn) * inv : 0.0f;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  const int4 o4 = pack8(v + 8 * u);
                  if (on) on[(size_t)(c * 4 + u) * PR] = o4;
                  if (os) os[(size_t)(c * 4 + u) * p.PB] = o4;
                  if (hand == 2) st_tile(next_a + (uint32_t)((c * 4 + u) * TP + j * 128 + quad * 32 + lane) * 16, o4);
                }
              }
            }
          }
        }
      }
      if (hand) {
        fence_proxy_async();               // generic-proxy st.shared -> the MMAs' async-proxy reads
        if (!lo_done) mbar_arrive(&a_ready[2 * (buf ^ 1)]);
        mbar_arrive(&a_ready[2 * (buf ^ 1) + 1]);
      }
      tc_fence_before();
      if (!kPair || rank == 0) mbar_arrive(&acc_empty[buf]);
      if (kPair || p.flags) {
        // publish the tile: the barrier orders every epilogue thread's stores before thread 0, whose gpu-scope
        // release is cumulative over them (the CUTLASS semaphore pattern) -- no per-thread MEMBAR on the chain.
        // (A null tile publishes nothing.)  Pair launches: the odd CTA's accumulator is drained as well, which
        // thread 0 tells the even CTA's MMA warps with one cluster-scope arrival.
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (et == 0) {
          if (p.flags && (!kPair || tile < p.num_tiles)) st_release(p.flags + (size_t)l * p.num_tiles + tile, 1u);
          if (kPair && rank == 1) mbar_arrive_remote(&acc_empty[buf], 0);
        }
      }
    }
    if (dbg && et == 0) {
      long long* d = p.dbg + blockIdx.x * 16;
      d[10] = clock64() - t_begin; d[11] = t_wait;
    }
  }
  // pair launches: neither CTA leaves (or frees TMEM) while its peer may still arrive on its barriers, read its
  // shared memory or run MMAs into its TMEM
  tc_fence_before();
  if (kPair) cluster_sync();
  else __syncthreads();
  if (warp == 1) {
    if (kPair) tmem_dealloc_pair(tmem, 512);
    else tmem_dealloc(tmem, 512);
  }
  if (kPair) cluster_sync();
}

// ---------------------------------------------------------------------------
// small SIMT kernels: observation packing, heads, weight repacking
// ---------------------------------------------------------------------------
// obs f32 [B][C][H][W] -> fp16 planes [cpad/8][plane_rows][8] (zeros at padded channels)
__global__ void pack_obs_kernel(const float* __restrict__ obs, act_t* __restrict__ out, int B, int C, int H,
                                int W, int cpad, int plane_rows) {
  // one thread per (channel group, row): 8 plane reads that are each coalesced across the threads of a warp
  // (consecutive x), one 16-byte store
  const int PB = H * W;
  const size_t rows = (size_t)B * PB, n = rows * (cpad / 8);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t P = i % rows;
    const int g = (int)(i / rows);
    const int pos = (int)(P % PB), b = (int)(P / PB);
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int c = g * 8 + e;
      v[e] = c < C ? obs[((size_t)b * C + c) * PB + pos] : 0.0f;
      v[e] = fminf(fmaxf(v[e], -65504.0f), 65504.0f);
    }
    reinterpret_cast<int4*>(out)[(size_t)g * plane_rows + P] = pack8(v);
  }
}

// The same for an Atari observation handed over in its COMPACT form (gym_env.py:306-313: k uint8 frames cast to float32,
// then k constant action planes): frames u8 [B][K][H][W] + plane values f32 [B][K] -> the planes pack_obs_kernel would
// produce from the float32 [B][2K][H][W] observation (0..255 are exact in fp16), at a quarter of the bytes.
__global__ void pack_frames_kernel(const uint8_t* __restrict__ frames, const float* __restrict__ planes,
                                   act_t* __restrict__ out, int B, int K, int H, int W, int cpad, int plane_rows) {
  const int PB = H * W;
  const size_t rows = (size_t)B * PB, n = rows * (cpad / 8);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t P = i % rows;
    const int g = (int)(i / rows);
    const int pos = (int)(P % PB), b = (int)(P / PB);
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int c = g * 8 + e;
      float f = 0.0f;
      if (c < K) f = (float)frames[((size_t)b * K + c) * PB + pos];
      else if (c < 2 * K) f = fminf(fmaxf(planes[(size_t)b * K + (c - K)], -65504.0f), 65504.0f);
      v[e] = f;
    }
    reinterpret_cast<int4*>(out)[(size_t)g * plane_rows + P] = pack8(v);
  }
}

// 1x1 conv (C -> mid, BatchNorm folded) + ReLU + Flatten + Linear(mid*hw -> out) and the output
// transform: 0 = raw scalar (support 1), 1 = support->scalar (util.py:70-93), 2 = softmax.
// One CTA of 128 threads per board.
struct HeadParams {
  const act_t* act;   // contiguous planes [C/8][plane_rows][8]
  int plane_rows;
  const float* w1;            // [mid][C]  (scaled)
  const float* b1;            // [mid]
  const float* w2;            // [out][mid*hw]
  const float* b2;            // [out]
  float* dst;                 // [B] or [B][out]
  int C, H, W, mid, out, kind;
};

__device__ __forceinline__ float signed_parabolic_f(float x) {
  const float eps = 1e-3f;
  float z = __fadd_rn(1.0f, __fmul_rn(0.004f, __fadd_rn(1.001f, fabsf(x))));
  z = __fsqrt_rn(z);
  z = __fdiv_rn(__fdiv_rn(z, 2.0f), eps);
  z = __fsub_rn(z, 500.0f);
  const float r = __fsub_rn(__fmul_rn(z, z), 1.0f);
  return x > 0.0f ? r : (x < 0.0f ? -r : 0.0f);
}

constexpr int kMaxHeads = 3;
struct HeadsParams {
  HeadParams h[kMaxHeads];
  RootSetup root;             // mz_net_initial_search: the policy head's epilogue also prepares the search roots
};

// grid (boards, heads): all heads of one inference in ONE launch
__global__ void __launch_bounds__(128) head_kernel(const __grid_constant__ HeadsParams hp) {
  const HeadParams& p = hp.h[blockIdx.y];
  extern __shared__ float hs[];            // f[mid*hw] | logits[out]
  const int hw = p.H * p.W;
  float* f = hs;
  float* lg = hs + p.mid * hw;
  const int b = blockIdx.x;
  const int4* a = reinterpret_cast<const int4*>(p.act) + (size_t)b * hw;
  for (int i = threadIdx.x; i < p.mid * hw; i += blockDim.x) {
    const int m = i / hw, q = i % hw;
    const int4* row = a + q;
    const float* w = p.w1 + (size_t)m * p.C;
    float acc = 0.0f;
    for (int c = 0; c < p.C; c += 8) {
      const int4 r4 = row[(size_t)(c / 8) * p.plane_rows];
      const act2_t* h = reinterpret_cast<const act2_t*>(&r4);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float2 v = __half22float2(h[u]);
        acc = fmaf(v.x, w[c + 2 * u], acc);
        acc = fmaf(v.y, w[c + 2 * u + 1], acc);
      }
    }
    f[i] = fmaxf(acc + p.b1[m], 0.0f);     // index m*hw + y*W + x == nn.Flatten order
  }
  __syncthreads();
  const int K = p.mid * hw;
  {
    // Linear(mid*hw -> out): one warp per output, lanes split K (coalesced weight rows)
    const int wid = threadIdx.x >> 5, ln = threadIdx.x & 31;
    for (int o = wid; o < p.out; o += 4) {
      const float* w = p.w2 + (size_t)o * K;
      float acc = 0.0f;
      for (int k = ln; k < K; k += 32) acc = fmaf(f[k], w[k], acc);
#pragma unroll
      for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
      if (ln == 0) lg[o] = acc + p.b2[o];
    }
  }
  __syncthreads();
  if (p.kind == 0) {
    if (threadIdx.x == 0) p.dst[b] = lg[0];
    return;
  }
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    float m = -INFINITY;
    for (int i = lane; i < p.out; i += 32) m = fmaxf(m, lg[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float den = 0.0f, num = 0.0f;
    const int maxv = (p.out - 1) / 2;
    const float step = p.out > 1 ? (float)(2 * maxv) / (float)(p.out - 1) : 0.0f;
    for (int i = lane; i < p.out; i += 32) {
      const float e = expf(lg[i] - m);
      den += e;
      num += e * ((float)(-maxv) + step * (float)i);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      den += __shfl_xor_sync(0xffffffffu, den, o);
      num += __shfl_xor_sync(0xffffffffu, num, o);
    }
    if (p.kind == 1) {
      if (lane == 0) p.dst[b] = signed_parabolic_f(num / den);
    } else {
      for (int i = lane; i < p.out; i += 32) p.dst[(size_t)b * p.out + i] = expf(lg[i] - m) / den;
      // fused root preparation: board b is tree b; this lane wrote exactly the actions it reads back
      if (hp.root.enabled) root_setup_fused(hp.root, b, lane, p.dst + (size_t)b * p.out);
    }
  }
}

// BatchNorm (eval) folded into the preceding bias-free conv: scale = gamma / sqrt(var + eps)
__global__ void bn_fold_kernel(const float* g, const float* beta, const float* mean, const float* var, float* scale,
                               float* bias, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const float s = g[i] / sqrtf(var[i] + 1e-5f);
    scale[i] = s;
    bias[i] = beta[i] - mean[i] * s;
  }
}

// conv weight [N][cin_total][3][3] (first `cin` input channels) * scale[n] -> packed fp16
// [9 taps][chunks][chunk_g][N][8], or (pair) [9 taps][chunks][half][chunk_g][N/2][8]: each weight stage as two
// contiguous halves of its N rows, one per CTA of an SM pair
// (N rows packed; rows >= n_real are zero: the padding of num_planes up to 32, or past the end of a column pass)
__global__ void pack_conv_kernel(const float* __restrict__ w, const float* __restrict__ scale,
                                 act_t* __restrict__ out, int N, int n_real, int cin, int cin_total, int cg, int pair) {
  const int chunk_g = cg < 8 ? cg : 8;
  const int nh = pair ? N / 2 : N;
  const size_t total = (size_t)9 * cg * N * 8;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int e = (int)(i % 8);
    size_t r = i / 8;
    int n = (int)(r % nh); r /= nh;
    const int gl = (int)(r % chunk_g); r /= chunk_g;
    if (pair) { n += (int)(r % 2) * nh; r /= 2; }
    const int ch = (int)(r % (cg / chunk_g));
    const int tap = (int)(r / (cg / chunk_g));
    const int c = (ch * chunk_g + gl) * 8 + e;
    float v = 0.0f;
    if (c < cin && n < n_real) v = w[(((size_t)n * cin_total + c) * 3 + tap / 3) * 3 + tap % 3] * scale[n];
    out[i] = __float2half_rn(fminf(fmaxf(v, -65504.0f), 65504.0f));
  }
}

// 1x1 head conv weight [mid][C][1][1] * scale[mid] -> f32 [mid][C]
__global__ void scale_rows_kernel(const float* w, const float* scale, float* out, int rows, int cols) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < rows * cols) out[i] = w[i] * scale[i / cols];
}

// per-action bias table of the dynamics' first conv: the A extra input planes are a fixed
// 0/1 pattern per action (QUIRK C, network.py:440-444: flat element f of the [A*h*w] block is
// 1 iff f % A == action), so their contribution is tab[a][pos][n] = scale[n] * sum over
// (plane c, tap) of w[n][C + c][tap] * E_a[c][y+ky-1][x+kx-1].
__global__ void action_table_kernel(const float* __restrict__ w, const float* __restrict__ scale,
                                    float* __restrict__ tab, int A, int C, int N, int n_real, int H, int W) {
  const int PB = H * W;
  const size_t total = (size_t)A * PB * N;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    // table layout [A][N/8][PB][8]: the epilogue (lane = row) reads 32 contiguous bytes per channel group
    const int e = (int)(i % 8);
    const int pos = (int)((i / 8) % PB);
    const int g = (int)((i / ((size_t)8 * PB)) % (N / 8));
    const int a = (int)(i / ((size_t)N * PB));
    const int n = g * 8 + e;
    const int y = pos / W, x = pos % W;
    float acc = 0.0f;
    if (n < n_real) {
      for (int c = 0; c < A; ++c)
        for (int ky = 0; ky < 3; ++ky)
          for (int kx = 0; kx < 3; ++kx) {
            const int yy = y + ky - 1, xx = x + kx - 1;
            if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
            const int fidx = c * PB + yy * W + xx;
            if (fidx % A == a) acc += w[(((size_t)n * (C + A) + C + c) * 3 + ky) * 3 + kx];
          }
      acc *= scale[n];
    }
    tab[i] = acc;
  }
}

// ---------------------------------------------------------------------------
// MuZeroAtariNet representation extras (network.py:312-353): two stride-2 3x3 convs (no
// BatchNorm, ReLU) and two 3x3/stride-2 average pools, once per search.  The stride-2 convs run on
// the tcgen05 kernel above as stride-1 convs whose epilogue keeps the even positions (4x the
// flops, still 3-4x faster than a SIMT kernel); the pools are plain SIMT kernels; the residual
// blocks between them go through the tcgen05 kernel at 48x48 / 24x24 / 12x12.
// ---------------------------------------------------------------------------
// AvgPool2d(3, stride 2, padding 1), count_include_pad (divide by 9), C = 128 or 256: one warp per output
// position, 4 channels per lane and 128-channel block.  Optionally min-max normalises over ALL channels
// (util.py:31-36) and also writes the result to indexed hidden-state slots.
__global__ void __launch_bounds__(256) avgpool_kernel(const act_t* __restrict__ in, act_t* __restrict__ out,
                                                      act_t* __restrict__ slots, const int32_t* __restrict__ out_index,
                                                      int B, int Hi, int Wi, int normalise, int rows_in, int rows_out,
                                                      int C) {
  const int Ho = Hi / 2, Wo = Wi / 2, PBi = Hi * Wi, PBo = Ho * Wo;
  const int lane = threadIdx.x & 31;
  const int g0 = lane >> 1, off = (lane & 1) * 4;     // channel-group plane and offset of this lane's 4 channels
  const int nblk = C / 128;                           // 128-channel blocks (<= 2)
  const long long total = (long long)B * PBo;
  for (long long i = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); i < total; i += (long long)gridDim.x * 8) {
    const int b = (int)(i / PBo), pos = (int)(i % PBo), oy = pos / Wo, ox = pos % Wo;
    float s[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx) {
        const int iy = 2 * oy + ky - 1, ix = 2 * ox + kx - 1;
        if (iy < 0 || iy >= Hi || ix < 0 || ix >= Wi) continue;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          if (k >= nblk) break;
          const int g = g0 + 16 * k;
          const uint2 v = *reinterpret_cast<const uint2*>(in + ((size_t)g * rows_in + (size_t)b * PBi + (size_t)iy * Wi + ix) * 8 + off);
          const float2 f0 = __half22float2(*reinterpret_cast<const act2_t*>(&v.x));
          const float2 f1 = __half22float2(*reinterpret_cast<const act2_t*>(&v.y));
          s[k][0] += f0.x; s[k][1] += f0.y; s[k][2] += f1.x; s[k][3] += f1.y;
        }
      }
#pragma unroll
    for (int k = 0; k < 2; ++k)
#pragma unroll
      for (int j = 0; j < 4; ++j) s[k][j] *= (1.0f / 9.0f);
    if (normalise) {
      float mn = INFINITY, mx = -INFINITY;
#pragma unroll
      for (int k = 0; k < 2; ++k)
        if (k < nblk)
#pragma unroll
          for (int j = 0; j < 4; ++j) { mn = fminf(mn, s[k][j]); mx = fmaxf(mx, s[k][j]); }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      }
      const float inv = 1.0f / ((mx - mn) + 1e-8f);
#pragma unroll
      for (int k = 0; k < 2; ++k)
#pragma unroll
        for (int j = 0; j < 4; ++j) s[k][j] = (s[k][j] - mn) * inv;
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (k >= nblk) break;
      const int g = g0 + 16 * k;
      uint2 pk;
      pk.x = pack2(s[k][0], s[k][1]);
      pk.y = pack2(s[k][2], s[k][3]);
      if (out) *reinterpret_cast<uint2*>(out + ((size_t)g * rows_out + (size_t)b * PBo + pos) * 8 + off) = pk;
      if (slots) {
        const size_t board = out_index ? (size_t)out_index[b] : (size_t)b;
        *reinterpret_cast<uint2*>(slots + ((board * (C / 8) + g) * PBo + pos) * 8 + off) = pk;
      }
    }
  }
}

// Per-position min-max normalisation over ALL channels (util.py:31-36) of a contiguous planar buffer, for convs wider
// than one 128-column pass (their halves are written by different layers of a launch, so the normalising epilogue of
// conv3x3_kernel cannot see the whole row): raw planes -> normalised planes and / or indexed hidden-state slots.
// One thread per row; the row's 16-byte plane entries are re-read from L1/L2 in the second pass.
__global__ void normalise_rows_kernel(const act_t* __restrict__ raw, act_t* __restrict__ out, act_t* __restrict__ slots,
                                      const int32_t* __restrict__ out_index, int Ptot, int PB, int groups, int plane_rows) {
  const int P = blockIdx.x * blockDim.x + threadIdx.x;
  if (P >= Ptot) return;
  const int4* src = reinterpret_cast<const int4*>(raw) + P;
  float mn = INFINITY, mx = -INFINITY;
  for (int g = 0; g < groups; ++g) {
    const int4 r4 = src[(size_t)g * plane_rows];
    const act2_t* h = reinterpret_cast<const act2_t*>(&r4);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float2 v = __half22float2(h[u]);
      mn = fminf(mn, fminf(v.x, v.y)); mx = fmaxf(mx, fmaxf(v.x, v.y));
    }
  }
  const float inv = 1.0f / ((mx - mn) + 1e-8f);
  const int b = P / PB, pos = P - b * PB;
  int4* on = out ? reinterpret_cast<int4*>(out) + P : nullptr;
  int4* os = nullptr;
  if (slots) {
    const size_t slot = out_index ? (size_t)out_index[b] : (size_t)b;
    os = reinterpret_cast<int4*>(slots) + slot * groups * PB + pos;
  }
  for (int g = 0; g < groups; ++g) {
    const int4 r4 = src[(size_t)g * plane_rows];
    const act2_t* h = reinterpret_cast<const act2_t*>(&r4);
    float v[8];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float2 f = __half22float2(h[u]);
      v[2 * u] = (f.x - mn) * inv; v[2 * u + 1] = (f.y - mn) * inv;
    }
    const int4 o4 = pack8(v);
    if (on) on[(size_t)g * plane_rows] = o4;
    if (os) os[(size_t)g * PB] = o4;
  }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
struct ConvLayer {
  const act_t* w[2];      // packed weights per 128-column pass
  const act_t* w_pair;    // single-pass convs of >= 64 channels in and out: the pair layout (SM-pair launches), else null
  const float* bias[2];
  int cg;                 // input channel groups of 8 (padded)
  int n_out;              // output channels incl. padding: 32, 64, 128 or 256
  int n_real;             // the network's output channels (< n_out only for num_planes = 16)
  int passes() const { return n_out > 128 ? 2 : 1; }
  int n_pass() const { return n_out > 128 ? 128 : n_out; }
};
struct Head {
  const float *w1, *b1, *w2, *b2;
  int mid, out, kind;
};
// A board grid: H*W rows per board (the layout at the top of this file).
struct Geo {
  int H, W;
  int PB() const { return H * W; }
};
// channels as the kernels see them: num_planes rounded up to a multiple of 32 (the reference's ResNet Tic-Tac-Toe
// variant has 16, config.py:126-127); the extra channels have zero weights and zero bias everywhere
static int padded_planes(int n) { return n < 32 ? 32 : (n + 31) / 32 * 32; }

struct ConvNet : NetImpl {
  mz_net_config cfg;
  Geo lat;                          // latent grid: the board (board games) or 6x6 (Atari)
  int C;                            // tower channels incl. padding (hidden-state slots hold C channels)
  int Creal;                        // the network's num_planes
  int A, blocks, max_batch, num_sms;
  bool atari;
  int in_cg;                        // channel groups of the packed observation
  ConvLayer rep0, dyn0;
  ConvLayer rep_blocks[64], dyn_blocks[64], pred_blocks[64];   // 2 per block
  // Atari representation: conv_1 (s2) -> 2 blocks @48 -> conv_2 (s2) -> 2 blocks @24 -> pool -> 2 blocks @12 -> pool
  ConvLayer s2_1, s2_2;             // the two stride-2 convs (no BatchNorm): stride-1 on tcgen05, even rows kept
  ConvLayer at_blocks[3][4];
  const float* tab;
  Head h_reward, h_policy, h_value;
  act_t *xobs, *b0, *b1, *b2, *b3, *b4;
  unsigned* flags;
  size_t flags_cap;
  int* err_flag;
  // 2-CTA clusters of conv3x3_kernel<128 / 64, 256, true> the device can hold at once (at the largest shared memory a
  // launch may ask for, so a bound for every launch)
  int pair_clusters[2] = {0, 0};

  // ---- test aid (mz_net_debug_capture): every conv / pool output of a call in a region of its own ----
  char* cap_buf = nullptr;
  size_t cap_size = 0, cap_used = 0;
  int cap_stage = 0, cap_conv = 0, cap_pool = 0;
  std::vector<mz_debug_tensor> cap_tensors;
  std::vector<mz_debug_launch> cap_launches;
  bool capturing() const { return cap_buf != nullptr; }
  void cap_begin() { cap_used = 0; cap_tensors.clear(); cap_launches.clear(); cap_set_stage(0); }
  void cap_set_stage(int s) { cap_stage = s; cap_conv = 0; cap_pool = 0; }
  size_t act_bytes(int batch) const {
    auto rows = [&](size_t pb) { return ((size_t)batch * pb + kTileM - 1) / kTileM * kTileM + kPlaneSlack; };
    const size_t mid_pb = atari ? (size_t)(cfg.in_h / 4 + 1) * (cfg.in_w / 4 + 1) : (size_t)lat.PB();
    const size_t big_pb = atari ? (size_t)(cfg.in_h / 2 + 1) * (cfg.in_w / 2 + 1) : (size_t)lat.PB();
    size_t a = rows(mid_pb) * C * 2;
    if (atari && rows(big_pb) * 128 * 2 > a) a = rows(big_pb) * 128 * 2;
    return align_up(a, 256);
  }
  // index of the recorded tensor whose planes contain p (a column pass points inside its conv's tensor), -1: none
  int cap_find(const void* p) const {
    for (size_t i = 0; i < cap_tensors.size(); ++i) {
      const mz_debug_tensor& t = cap_tensors[i];
      const char* b = (const char*)t.ptr;
      if ((const char*)p >= b && (const char*)p < b + (size_t)t.plane_rows * t.groups * 16) return (int)i;
    }
    return -1;
  }
  int cap_add(void* ptr, int kind, const Geo& g, int batch, int groups, int src, int residual) {
    mz_debug_tensor t;
    t.ptr = ptr; t.kind = kind; t.stage = cap_stage;
    t.index = kind == MZ_DEBUG_CONV ? cap_conv++ : (kind == MZ_DEBUG_POOL ? cap_pool++ : 0);
    t.plane_rows = plane_rows_of(g, batch); t.groups = groups; t.h = g.H; t.w = g.W; t.batch = batch;
    t.src = src; t.residual = residual;
    cap_tensors.push_back(t);
    return (int)cap_tensors.size() - 1;
  }
  // a fresh region of the capture buffer for a conv / pool output (nullptr: the buffer is full, error set)
  act_t* cap_take(int kind, const Geo& g, int batch, int groups, const void* src, const void* residual) {
    const size_t bytes = align_up((size_t)plane_rows_of(g, batch) * groups * 16, 256);
    if (cap_used + bytes > cap_size) {
      // the call fails here: drop the layers it already queued, which point into this call's buffers
      reset_pending();
      num_pend_heads = 0; pend_heads_smem = 0;
      set_error("mz_net_debug_capture: buffer of %zu bytes too small", cap_size);
      return nullptr;
    }
    act_t* r = (act_t*)(cap_buf + cap_used);
    cap_used += bytes;
    cap_add(r, kind, g, batch, groups, src ? cap_find(src) : -1, residual ? cap_find(residual) : -1);
    return r;
  }
  int debug_capture_bytes(int batch, size_t* bytes) override {
    // more regions than any call takes: board 1 + 4 blocks convs, Atari 14 + 2 blocks convs and one pool
    *bytes = (size_t)(16 + 4 * blocks) * act_bytes(batch);
    return MZ_OK;
  }
  int debug_capture(void* buf, size_t bytes) override {
    reset_pending();                 // every call flushes what it queued; nothing of an earlier buffer may stay queued
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

  static int tp_of(const Geo& g, int rows = kTileM) { return (rows + 2 * (g.W + 1)) | 1; }
  // rows of one channel-group plane of a contiguous activation buffer holding `batch` boards of grid g
  static int plane_rows_of(const Geo& g, int batch) {
    return (batch * g.PB() + kTileM - 1) / kTileM * kTileM + kPlaneSlack;
  }
  // n = output channels of one pass (the width of a weight stage and of the bias slots)
  // pair: SM-pair launch, whose ring slots hold half a weight stage
  static size_t conv_fixed_smem(const Geo& g, int cg, int n, int rows, bool pair = false) {
    const int TP = tp_of(g, rows);
    size_t a = (((size_t)2 * cg * TP * 16) + 127) & ~(size_t)127;
    return a + (2 * (pair ? kMaxPairStages : kMaxStages) + 10) * 8 + 16 + (size_t)4 * n * 4 + 2048 + 256 + 64;
  }
  static size_t slot_bytes(int cg, int n, bool pair) { return (size_t)(cg < 8 ? cg : 8) * (pair ? n / 2 : n) * 16; }
  // Ring depth: as many slots as shared memory holds, at most kMaxStages (kMaxPairStages).  A pair launch's half-size
  // slots double what fits: the Gomoku tower (9x9, 128 channels) goes from 5 x 16 KB to 10 x 8 KB, i.e. the same
  // bytes in flight ahead of the MMAs, but in finer steps; the 48x48 Atari blocks go from 2 to 5 slots.
  static int conv_stages(const Geo& g, int cg, int n, int rows, bool pair = false) {
    const size_t stage = slot_bytes(cg, n, pair);
    const size_t fixed = conv_fixed_smem(g, cg, n, rows, pair);
    if (fixed + 2 * stage > 227 * 1024) return 0;
    const int s = (int)((227 * 1024 - fixed) / stage), cap = pair ? kMaxPairStages : kMaxStages;
    return s > cap ? cap : s;
  }
  static size_t conv_smem(const Geo& g, int cg, int n, int rows, bool pair = false) {
    return conv_fixed_smem(g, cg, n, rows, pair) + (size_t)conv_stages(g, cg, n, rows, pair) * slot_bytes(cg, n, pair);
  }
  // tile rows a conv with `cg` input groups can use at all: 256-row tiles need 2 x cg x TP x 16 bytes of activations
  static bool fits(const Geo& g, int cg, int n, int rows) { return conv_stages(g, cg, n, rows) >= 2; }

  // ---- layer batching: consecutive convs on the same grid become ONE dataflow launch ----
  ConvParams pend;                 // layers collected so far
  Geo pend_geo{0, 0};
  int pend_cg = 0, pend_batch = 0;
  bool pend_sub = false;           // the (single) pending conv is a stride-2 conv writing the half-size grid
  int pend_prev_first = -1, pend_prev_count = 0;     // LayerDescs of the previous conv of the pending launch
  const act_t* pend_out_base[kMaxLayers];            // un-offset `out` / `out_norm` of each pending layer + its pass
  const act_t* pend_norm_base[kMaxLayers];
  int pend_pass[kMaxLayers];

  // One convolution = L.passes() LayerDescs (128 output columns each).  `sub`: stride-2 conv, the epilogue keeps the
  // even positions on the half-size grid (the caller flushes right after it).
  int add_conv(const ConvLayer& L, const Geo& g, const act_t* in, const int32_t* in_index, bool in_slots, int batch,
               const float* tab_, const int32_t* action, const act_t* residual, act_t* out, act_t* out_norm,
               act_t* out_slots, const int32_t* out_index, cudaStream_t st, bool sub = false) {
    const int np = L.passes();
    // channels of a pass that take part in the min-max normalisation (all of them unless num_planes was padded)
    const int eff_real = L.n_real < L.n_out ? L.n_real : L.n_pass();
    if (pend.num_layers > 0 && (pend_cg != L.cg || pend_geo.H != g.H || pend_geo.W != g.W || pend_batch != batch ||
                                pend.N != L.n_pass() || pend.n_real != eff_real || pend.tab_groups != L.n_out / 8 ||
                                pend.num_layers + np > kMaxLayers || sub || pend_sub)) {
      int rc = flush(st);
      if (rc) return rc;
    }
    if (np > 1 && (out_norm || out_slots)) {
      set_error("internal: a conv wider than one column pass cannot normalise in its epilogue");
      return MZ_EINVAL;
    }
    const size_t PR = (size_t)plane_rows_of(g, batch);
    const Geo go{g.H / 2, g.W / 2};
    const size_t PRo = sub ? (size_t)plane_rows_of(go, batch) : PR;
    const int first = pend.num_layers;
    for (int h = 0; h < np; ++h) {
      LayerDesc& d = pend.L[pend.num_layers];
      const size_t goff = (size_t)h * 16;                    // channel groups before this pass
      d.in = in; d.in_index = in_index; d.w = L.w[h]; d.w_pair = L.w_pair; d.bias = L.bias[h];
      d.tab = tab_ ? tab_ + goff * g.PB() * 8 : nullptr;
      d.action = action;
      d.residual = residual ? residual + goff * PR * 8 : nullptr;
      d.out = out ? out + goff * PRo * 8 : nullptr;
      d.out_norm = out_norm; d.out_slots = out_slots; d.out_index = out_index;
      d.dep0 = pend_prev_count > 0 ? pend_prev_first : -1;
      d.dep1 = pend_prev_count > 1 ? pend_prev_first + 1 : -1;
      d.fwd = 0;
      d.res_layer = -1;
      d.in_slots = in_slots ? 1 : 0;
      pend_out_base[pend.num_layers] = out; pend_norm_base[pend.num_layers] = out_norm; pend_pass[pend.num_layers] = h;
      if (residual)                                          // which pending layer wrote this column half of the residual
        for (int j = pend.num_layers - 1; j >= 0; --j)
          if (pend_pass[j] == h && (pend_out_base[j] == residual || pend_norm_base[j] == residual)) { d.res_layer = j; break; }
      ++pend.num_layers;
    }
    pend_prev_first = first; pend_prev_count = np;
    pend_geo = g; pend_cg = L.cg; pend_batch = batch; pend_sub = sub;
    pend.N = L.n_pass(); pend.n_real = eff_real; pend.tab_groups = L.n_out / 8;
    return MZ_OK;
  }

  void reset_pending() { pend.num_layers = 0; pend_prev_first = -1; pend_prev_count = 0; pend_sub = false; }

  int flush(cudaStream_t st) {
    if (pend.num_layers == 0) return MZ_OK;
    ConvParams& p = pend;
    const Geo g = pend_geo;
    const int batch = pend_batch, cg = pend_cg, nl = p.num_layers, N = p.N;
    const bool multi_pass = p.tab_groups * 8 > 128;
    p.PB = g.PB(); p.W = g.W; p.H = g.H; p.B = batch;
    p.Ptot = batch * p.PB;
    p.plane_rows = plane_rows_of(g, batch);
    p.sub = pend_sub ? 1 : 0;
    {
      const Geo go{g.H / 2, g.W / 2};
      p.out_plane_rows = plane_rows_of(go, batch); p.out_PB = go.PB(); p.out_W = go.W;
    }
    p.cg = cg; p.relu = 1;
    // Few tiles per SM (small batches / small grids): a multi-layer launch is bound by the dependency chain between
    // layers, so use 128-row tiles whose K range is split over the two MMA warps (half the MMA time per tile).
    // Otherwise 256-row tiles (half the weight traffic per row).
    const char* force_env = getenv("MZ_CONV_TILE_ROWS");          // tests force either variant at any size
    const int force_rows = force_env ? atoi(force_env) : 0;
    int rows = (nl > 1 && (p.Ptot + kTileM - 1) / kTileM < 2 * num_sms) ? 128 : kTileM;
    if (force_rows == 128 || force_rows == 256) rows = force_rows;
    // split-K tiles give the second MMA warp the odd weight stages; with one stage per tap its first MMA would be a
    // masked (non-centre) tap and could not initialise its accumulator
    if (cg <= 8) rows = kTileM;
    // 256 input channels: two 256-row activation buffers do not fit shared memory
    if (!fits(g, cg, N, rows)) rows = rows == kTileM ? 128 : kTileM;
    // RESIDENT launch: when every CTA can own one tile of whole boards for all layers, nothing a tile needs comes from
    // another tile (every tap that leaves a board is masked), so the layers of a tower hand their activations over
    // in shared memory -- no tile flags, no tile loads, no waiting for neighbours after layer 0.
    // This is the regime of small batches and small grids (single-tree searches, the 6x6 Atari latent), where a
    // launch is bound by the chain flag -> load -> MMA -> epilogue -> publish of every layer, not by throughput.
    const int sm_cap0 = (cta_limit > 0 && cta_limit < num_sms) ? cta_limit : num_sms;
    p.resident = 0;
    p.khalf = 0;
    p.tile_stride = rows;
    if (nl > 1 && !p.sub && !multi_pass) {
      bool chain = true;
      for (int i = 0; i + 1 < nl && chain; ++i) {
        LayerDesc& a = pend.L[i];
        const LayerDesc& b = pend.L[i + 1];
        a.fwd = (b.in_slots == 0 && b.in == a.out && a.out) ? 1 : ((b.in_slots == 0 && b.in == a.out_norm && a.out_norm) ? 2 : 0);
        chain = a.fwd != 0;
      }
      if (chain) {
        const int cand[2] = {128, kTileM};
        for (int ci = 0; ci < 2 && !p.resident; ++ci) {
          const int rr = cand[ci];
          if (force_rows && force_rows != rr) continue;
          if (rr == 128 && cg <= 8) continue;
          if (!fits(g, cg, N, rr)) continue;
          const int bpt = rr / p.PB;                               // whole boards per tile
          if (bpt < 1) continue;
          if ((batch + bpt - 1) / bpt > sm_cap0) continue;
          p.resident = 1; rows = rr; p.tile_stride = bpt * p.PB;
          p.khalf = (rr == kTileM && cg == 16) ? 1 : 0;
        }
      }
    }
    p.num_tiles = p.resident ? (p.Ptot + p.tile_stride - 1) / p.tile_stride : (p.Ptot + rows - 1) / rows;
    p.TP = tp_of(g, rows);
    const int sm_cap = (cta_limit > 0 && cta_limit < num_sms) ? cta_limit : num_sms;
    // SM-pair launch (see kPair): the 256-row dataflow launch of several stride-1 single-pass layers with 64-channel
    // weight stages.  Pairs rotate over pair items as CTAs rotate over tiles; as many pairs as there are pair items,
    // as fit beside whatever else holds SMs (cta_limit, rounded down to an even CTA count) and as the device can
    // place at once.  No pair fits (cta_limit 1): the single-CTA form.
    const int units = (p.num_tiles + 1) / 2;
    int pairs = 0;
    bool pair_w = true;
    for (int i = 0; i < nl; ++i) pair_w = pair_w && p.L[i].w_pair != nullptr;
    if (rows == kTileM && nl > 1 && !p.resident && !p.sub && !multi_pass && pair_w) {
      pairs = units < sm_cap / 2 ? units : sm_cap / 2;
      const int mc = pair_clusters[N == 128 ? 0 : 1];
      if (pairs > mc) pairs = mc;
    }
    const bool pair = pairs > 0;
    p.stages = conv_stages(g, cg, N, rows, pair);
    p.err = err_flag;
    if (p.stages < 2) { reset_pending(); set_error("conv tile does not fit shared memory for a %dx%d grid", g.H, g.W); return MZ_EINVAL; }
    const size_t smem = conv_smem(g, cg, N, rows, pair);
    const int grid = pair ? 2 * pairs : (p.num_tiles < sm_cap ? p.num_tiles : sm_cap);
    p.rot = nl > 1 ? (pair ? units % pairs : p.num_tiles % grid) : 0;
    p.flags = nullptr;
    if (nl > 1 && !p.resident) {
      if ((size_t)nl * p.num_tiles > flags_cap) { reset_pending(); set_error("internal: flag buffer too small"); return MZ_EINVAL; }
      p.flags = flags;
      cudaError_t e = cudaMemsetAsync(flags, 0, (size_t)nl * p.num_tiles * sizeof(unsigned), st);
      if (e != cudaSuccess) { reset_pending(); set_error("cudaMemsetAsync: %s", cudaGetErrorString(e)); return MZ_ECUDA; }
    }
    p.dbg = nullptr;
    static const bool debug = getenv("MZ_CONV_DEBUG") != nullptr;
    if (debug) cudaMalloc(&p.dbg, (size_t)grid * 16 * sizeof(long long));
    prof_mark(kProfConv, st, multi_pass ? (nl + 1) / 2 : nl);       // counted in convolutions, not passes
    {
      // Layers of a launch wait on each other's tiles, so every CTA must be resident: a cooperative launch
      // makes the hardware place the grid all at once (two such grids of different streams could otherwise
      // each grab part of the SMs and wait for the rest forever).
      cudaLaunchConfig_t lc = {};
      lc.gridDim = dim3((unsigned)grid); lc.blockDim = dim3(kConvThreads); lc.dynamicSmemBytes = smem; lc.stream = st;
      cudaLaunchAttribute at[2];
      at[0].id = cudaLaunchAttributeCooperative;
      at[0].val.cooperative = nl > 1 ? 1 : 0;
      at[1].id = cudaLaunchAttributeClusterDimension;
      at[1].val.clusterDim.x = 2; at[1].val.clusterDim.y = 1; at[1].val.clusterDim.z = 1;
      lc.attrs = at; lc.numAttrs = pair ? 2 : 1;
      cudaError_t le;
      if (pair) {
        if (N == 128) le = cudaLaunchKernelEx(&lc, conv3x3_kernel<128, 256, true>, p);
        else le = cudaLaunchKernelEx(&lc, conv3x3_kernel<64, 256, true>, p);
      } else if (rows == 256) {
        if (N == 128) le = cudaLaunchKernelEx(&lc, conv3x3_kernel<128, 256>, p);
        else if (N == 64) le = cudaLaunchKernelEx(&lc, conv3x3_kernel<64, 256>, p);
        else le = cudaLaunchKernelEx(&lc, conv3x3_kernel<32, 256>, p);
      } else {
        if (N == 128) le = cudaLaunchKernelEx(&lc, conv3x3_kernel<128, 128>, p);
        else if (N == 64) le = cudaLaunchKernelEx(&lc, conv3x3_kernel<64, 128>, p);
        else le = cudaLaunchKernelEx(&lc, conv3x3_kernel<32, 128>, p);
      }
      if (le != cudaSuccess) { reset_pending(); set_error("conv3x3_kernel launch: %s", cudaGetErrorString(le)); cudaGetLastError(); return MZ_ECUDA; }
    }
    if (capturing()) {
      mz_debug_launch r = {};
      r.num_layers = nl; r.tile_rows = rows; r.resident = p.resident; r.khalf = p.khalf; r.pair = pairs; r.sub = p.sub;
      r.multi_pass = multi_pass ? 1 : 0; r.grid = grid; r.num_tiles = p.num_tiles; r.cg = cg; r.n = N; r.h = g.H;
      r.w = g.W; r.batch = batch;
      for (int i = 0; i < nl; ++i) {
        const LayerDesc& d = p.L[i];
        r.out[i] = d.out ? cap_find(d.out) : -1;
        r.pass[i] = pend_pass[i];
        r.flags[i] = (d.out_norm ? 1 : 0) | (d.out_slots ? 2 : 0) | (d.tab ? 4 : 0);
        r.dep0[i] = d.dep0; r.res_layer[i] = d.res_layer; r.fwd[i] = d.fwd;
      }
      cap_launches.push_back(r);
    }
    prof_mark(-1, st);
    reset_pending();
    MZ_LAUNCH_CHECK("conv3x3_kernel");
    if (debug) {   // measurement aid: per-role cycle accounting, averaged over CTAs
      cudaDeviceSynchronize();
      std::vector<long long> h((size_t)grid * 16);
      cudaMemcpy(h.data(), p.dbg, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
      cudaFree(p.dbg);
      // the MMA fields (2-6, 12-14) of a pair launch are written by the even CTAs only; items/cta is then per pair
      double a[16] = {0};
      const bool mma_field[16] = {0, 0, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 1, 1, 1, 0};
      for (int c = 0; c < grid; ++c)
        for (int k = 0; k < 16; ++k) a[k] += (double)h[(size_t)c * 16 + k] / (pair && mma_field[k] ? grid / 2 : grid);
      fprintf(stderr, "[conv dbg] %dx%d cg=%d layers=%d %s items/cta=%.1f | producer total %.0f wait_empty %.0f "
              "residual_gate %.0f | mma total %.0f wait_acc %.0f wait_a %.0f (1st / 2nd / 3rd tile of a layer: %.0f / %.0f / "
              "%.0f) wait_w %.0f | loader total %.0f wait_mma %.0f wait_dep %.0f | epilogue total %.0f wait_mma %.0f\n",
              g.H, g.W, cg, nl, pair ? "pair" : "single", a[6], a[0], a[1], a[15], a[2], a[3], a[4], a[12], a[13], a[14],
              a[5], a[7], a[8], a[9], a[10], a[11]);
    }
    return MZ_OK;
  }
  // heads of one inference, launched together
  HeadsParams pend_heads;
  int num_pend_heads = 0;
  size_t pend_heads_smem = 0;
  void add_head(const Head& h, const act_t* act, int batch, float* dst) {
    HeadParams& p = pend_heads.h[num_pend_heads++];
    p.act = act; p.w1 = h.w1; p.b1 = h.b1; p.w2 = h.w2; p.b2 = h.b2; p.dst = dst;
    p.plane_rows = plane_rows_of(lat, batch);
    p.C = Creal; p.H = lat.H; p.W = lat.W; p.mid = h.mid; p.out = h.out; p.kind = h.kind;
    const size_t smem = ((size_t)h.mid * lat.H * lat.W + h.out) * 4;
    if (smem > pend_heads_smem) pend_heads_smem = smem;
  }
  int launch_heads(int batch, cudaStream_t st) {
    if (num_pend_heads == 0) return MZ_OK;
    if (pending_root) pend_heads.root = *pending_root; else pend_heads.root.enabled = 0;
    prof_mark(kProfHead, st);
    head_kernel<<<dim3(batch, num_pend_heads), 128, pend_heads_smem, st>>>(pend_heads);
    prof_mark(-1, st);
    num_pend_heads = 0;
    pend_heads_smem = 0;
    MZ_LAUNCH_CHECK("head_kernel");
    return MZ_OK;
  }

  // [first conv] -> nblk residual blocks on grid g; the LAST layer optionally also emits the min-max
  // normalised state (contiguous copy and/or indexed slots).  *final_buf = buffer holding the raw
  // (ReLU'd) tower output, unless want_raw is false and the last layer normalises.
  int tower(const ConvLayer* first, const ConvLayer* blk, int nblk, const Geo& g, const act_t* in,
            const int32_t* in_index, bool in_slots, const float* tab_, const int32_t* action, int batch, bool want_raw,
            act_t* norm_out, act_t* slots, const int32_t* out_index, cudaStream_t st, act_t** final_buf,
            act_t* raw_dst = nullptr) {
    const act_t* cur = in;
    const int32_t* cur_index = in_index;
    bool cur_slots = in_slots;
    act_t* pp[2] = {b0, b1};
    int which = (in == b0) ? 1 : 0, rc;
    const bool normalise = (norm_out != nullptr) || (slots != nullptr);
    // convs wider than one column pass cannot normalise in their epilogue: the last layer writes the raw output and
    // normalise_rows_kernel follows
    const ConvLayer& last_layer = nblk > 0 ? blk[2 * nblk - 1] : *first;
    const bool late_norm = normalise && last_layer.passes() > 1;
    const bool keep_raw = want_raw || late_norm;
    // Capture (mz_net_debug_capture): every conv writes a region of its own instead of b0 / b1 / b2 / raw_dst, and the
    // last layer of a normalising tower also stores its raw output.  The launches stay as they are: add_conv groups
    // convs on (cg, grid, N, n_real, batch, layer count, sub) only, flush() chooses the form from those, `fits()` and
    // cta_limit, and the pointer tests it makes still hold -- each layer reads its producer's `out` (or the `out_norm`
    // b3, which is not moved) so the resident hand-over `fwd` is the same, and a residual is still the `out` / `out_norm`
    // of the layer that res_layer names.  Only the in-place block output (over its input) becomes a separate store.
    const bool cap = capturing();
    if (first) {
      const bool last = (nblk == 0);
      act_t* dst = (last && raw_dst) ? raw_dst : pp[which];
      act_t* out = (last && normalise && !keep_raw) ? nullptr : dst;
      if (cap && !(dst = out = cap_take(MZ_DEBUG_CONV, g, batch, first->n_out / 8, cur_slots ? nullptr : cur, nullptr)))
        return MZ_ENOMEM;
      rc = add_conv(*first, g, cur, cur_index, cur_slots, batch, tab_, action, nullptr, out,
                    (last && !late_norm) ? norm_out : nullptr, (last && !late_norm) ? slots : nullptr, out_index, st);
      if (rc) return rc;
      cur = dst; cur_index = nullptr; cur_slots = false; which ^= 1;
    }
    for (int i = 0; i < nblk; ++i) {
      const bool last = (i == nblk - 1);
      act_t* mid = b2;
      if (cap && !(mid = cap_take(MZ_DEBUG_CONV, g, batch, blk[2 * i].n_out / 8, cur_slots ? nullptr : cur, nullptr)))
        return MZ_ENOMEM;
      rc = add_conv(blk[2 * i], g, cur, cur_index, cur_slots, batch, nullptr, nullptr, nullptr, mid, nullptr, nullptr, nullptr, st);
      if (rc) return rc;
      if (cur_slots) { set_error("internal: residual input must be contiguous"); return MZ_EINVAL; }
      // The block's output goes back INTO the buffer its input came from: element (row, channel) of the residual is read
      // by the very thread that writes the output there, earlier in program order, and every other reader of the old
      // contents (the block's first conv, tiles t-1..t+1) has published before this tile starts.  Two live buffers per
      // tower instead of three: two engines' activations (2 x 2 x 21 MB for 1024 Gomoku boards) then fit the 126 MB L2,
      // where three per engine (126 MB + weights + trees) were evicted to DRAM between a layer's write and its rewrite.
      act_t* dst = pp[which];
      if (dst == cur) dst = pp[which ^ 1];
      if (cur == b0 || cur == b1 || cur == b3) dst = const_cast<act_t*>(cur);
      if (last && raw_dst) dst = raw_dst;
      act_t* out = (last && normalise && !keep_raw) ? nullptr : dst;
      if (cap && !(dst = out = cap_take(MZ_DEBUG_CONV, g, batch, blk[2 * i + 1].n_out / 8, mid, cur))) return MZ_ENOMEM;
      rc = add_conv(blk[2 * i + 1], g, mid, nullptr, false, batch, nullptr, nullptr, cur, out,
                    (last && !late_norm) ? norm_out : nullptr, (last && !late_norm) ? slots : nullptr, out_index, st);
      if (rc) return rc;
      cur = dst; which ^= 1;
    }
    // the normalised state the next tower reads (b3 is not moved): one more tensor of the record
    if (cap && norm_out) cap_add(norm_out, MZ_DEBUG_NORM, g, batch, C / 8, cap_find(cur), -1);
    if (late_norm) {
      if ((rc = flush(st))) return rc;
      const int Ptot = batch * g.PB();
      prof_mark(kProfPack, st);
      normalise_rows_kernel<<<(Ptot + 127) / 128, 128, 0, st>>>(cur, norm_out, slots, out_index, Ptot, g.PB(),
                                                               last_layer.n_out / 8, plane_rows_of(g, batch));
      prof_mark(-1, st);
      MZ_LAUNCH_CHECK("normalise_rows_kernel");
    }
    *final_buf = const_cast<act_t*>(cur);
    return MZ_OK;
  }

  int represent_atari(int batch, const float* obs, const uint8_t* frames, const float* plane_values, act_t* slots,
                      const int32_t* dst_index, cudaStream_t st) {
    const int Hin = cfg.in_h, Win = cfg.in_w;
    const Geo g0{Hin, Win}, g1{Hin / 2, Win / 2}, g2{Hin / 4, Win / 4}, g3{Hin / 8, Win / 8};
    prof_mark(kProfPack, st);
    if (frames)
      pack_frames_kernel<<<num_sms * 8, 256, 0, st>>>(frames, plane_values, xobs, batch, cfg.in_channels / 2, Hin, Win, 16,
                                                      plane_rows_of(g0, batch));
    else
      pack_obs_kernel<<<num_sms * 8, 256, 0, st>>>(obs, xobs, batch, cfg.in_channels, Hin, Win, 16, plane_rows_of(g0, batch));
    prof_mark(-1, st);
    MZ_LAUNCH_CHECK("pack_obs_kernel");
    if (capturing()) cap_add(xobs, MZ_DEBUG_OBS, g0, batch, 2, -1, -1);
    // stride-2 conv + ReLU: one tcgen05 launch at the input resolution whose epilogue stores the even positions on
    // the half-size grid
    // under capture the stride-2 convs and the first pool write a region of their own: `out` returns where
    auto s2 = [&](const ConvLayer& L, const act_t* in, act_t*& out, const Geo& gi) -> int {
      if (capturing() && !(out = cap_take(MZ_DEBUG_CONV, Geo{gi.H / 2, gi.W / 2}, batch, L.n_out / 8, in, nullptr)))
        return MZ_ENOMEM;
      int rc2 = add_conv(L, gi, in, nullptr, false, batch, nullptr, nullptr, nullptr, out, nullptr, nullptr, nullptr, st, true);
      if (rc2) return rc2;
      return flush(st);
    };
    auto pool = [&](const act_t* in, act_t*& out, act_t* sl, const int32_t* idx, const Geo& gi, const Geo& go, int norm) -> int {
      if (capturing()) {
        if (out == b3) cap_add(out, MZ_DEBUG_POOL, go, batch, C / 8, cap_find(in), -1);   // the normalised state
        else if (!(out = cap_take(MZ_DEBUG_POOL, go, batch, C / 8, in, nullptr))) return MZ_ENOMEM;
      }
      prof_mark(kProfPack, st);
      avgpool_kernel<<<num_sms * 8, 256, 0, st>>>(in, out, sl, idx, batch, gi.H, gi.W, norm, plane_rows_of(gi, batch),
                                                  plane_rows_of(go, batch), C);
      prof_mark(-1, st);
      MZ_LAUNCH_CHECK("avgpool_kernel");
      return MZ_OK;
    };
    act_t* fin;
    int rc;
    // every writer writes every row of the grid it produces, so grids of different sizes can reuse the same buffers
    act_t* c1 = b0;
    if ((rc = s2(s2_1, xobs, c1, g0))) return rc;                                              // relu(conv_1)
    if ((rc = tower(nullptr, at_blocks[0], 2, g1, c1, nullptr, false, nullptr, nullptr, batch, true, nullptr, nullptr,
                    nullptr, st, &fin))) return rc;
    if ((rc = flush(st))) return rc;
    act_t* nxt = (fin == b0) ? b1 : b0;
    if ((rc = s2(s2_2, fin, nxt, g1))) return rc;                                              // relu(conv_2)
    if ((rc = tower(nullptr, at_blocks[1], 2, g2, nxt, nullptr, false, nullptr, nullptr, batch, true, nullptr, nullptr,
                    nullptr, st, &fin))) return rc;
    if ((rc = flush(st))) return rc;
    nxt = (fin == b0) ? b1 : b0;
    if ((rc = pool(fin, nxt, nullptr, nullptr, g2, g3, 0))) return rc;                         // avg_pool_1
    if ((rc = tower(nullptr, at_blocks[2], 2, g3, nxt, nullptr, false, nullptr, nullptr, batch, true, nullptr, nullptr,
                    nullptr, st, &fin))) return rc;
    if ((rc = flush(st))) return rc;
    act_t* norm = b3;
    return pool(fin, norm, slots, dst_index, g3, lat, 1);                                      // avg_pool_2 + normalise
  }

  int initial(int batch, const float* obs, void* hidden_out, const int32_t* dst_index, float* pi_probs, float* value,
              cudaStream_t st) override {
    int rc;
    if (capturing()) cap_begin();
    if (atari) {
      rc = represent_atari(batch, obs, nullptr, nullptr, (act_t*)hidden_out, dst_index, st);
    } else {
      prof_mark(kProfPack, st);
      pack_obs_kernel<<<num_sms * 4, 256, 0, st>>>(obs, xobs, batch, cfg.in_channels, lat.H, lat.W, in_cg * 8,
                                                   plane_rows_of(lat, batch));
      prof_mark(-1, st);
      MZ_LAUNCH_CHECK("pack_obs_kernel");
      if (capturing()) cap_add(xobs, MZ_DEBUG_OBS, lat, batch, in_cg, -1, -1);
      act_t* fin;
      // representation: raw output is not needed, normalised goes to b3 (for the prediction tower) and the slots
      rc = tower(&rep0, rep_blocks, blocks, lat, xobs, nullptr, false, nullptr, nullptr, batch, false, b3,
                 (act_t*)hidden_out, dst_index, st, &fin);
    }
    if (rc) return rc;
    if ((rc = predict(batch, pi_probs, value, st))) return rc;
    return launch_heads(batch, st);
  }

  int initial_frames(int batch, const uint8_t* frames, const float* plane_values, void* hidden_out,
                     const int32_t* dst_index, float* pi_probs, float* value, cudaStream_t st) override {
    if (!atari || (cfg.in_channels & 1)) {
      set_error("mz_net_initial_frames: compact (uint8 frames + action planes) observations are the MuZeroAtariNet format "
                "with an even number of stacked planes");
      return MZ_EINVAL;
    }
    if (capturing()) cap_begin();
    int rc = represent_atari(batch, nullptr, frames, plane_values, (act_t*)hidden_out, dst_index, st);
    if (rc) return rc;
    if ((rc = predict(batch, pi_probs, value, st))) return rc;
    return launch_heads(batch, st);
  }

  int predict(int batch, float* pi_probs, float* value, cudaStream_t st) {
    act_t* fin;
    if (capturing()) cap_set_stage(2);
    int rc = tower(nullptr, pred_blocks, blocks, lat, b3, nullptr, false, nullptr, nullptr, batch, true, nullptr, nullptr,
                   nullptr, st, &fin);
    if (rc) return rc;
    if ((rc = flush(st))) return rc;
    if (pi_probs) add_head(h_policy, fin, batch, pi_probs);
    add_head(h_value, fin, batch, value);
    return MZ_OK;     // the caller launches the collected heads
  }

  int recurrent(int batch, const void* hidden_in, const int32_t* src_index, const int32_t* action, void* hidden_out,
                const int32_t* dst_index, float* reward_out, float* value_out, float* pi_probs,
                cudaStream_t st) override {
    act_t* fin;
    if (capturing()) { cap_begin(); cap_set_stage(1); }
    // dynamics: raw output (for the reward head) in a ping-pong buffer, normalised copy in b3 + the slots
    // The dynamics tower and the prediction tower run as ONE launch; the dynamics' raw output goes to b4,
    // which the prediction tower never touches, so the reward head can read it afterwards.
    int rc = tower(&dyn0, dyn_blocks, blocks, lat, (const act_t*)hidden_in, src_index, true, tab, action, batch, true, b3,
                   (act_t*)hidden_out, dst_index, st, &fin, b4);
    if (rc) return rc;
    rc = predict(batch, pi_probs, value_out, st);
    if (rc) return rc;
    add_head(h_reward, fin, batch, reward_out);                 // reward head reads the UN-normalised state
    return launch_heads(batch, st);
  }
};

static int conv_geometry(const mz_net_config& c, int* H, int* W) {
  MZ_CHECK_ARG(c.num_planes == 16 || c.num_planes == 32 || c.num_planes == 64 || c.num_planes == 128 || c.num_planes == 256,
               "conv nets need num_planes in {16, 32, 64, 128, 256}, got %d", c.num_planes);
  MZ_CHECK_ARG(c.num_res_blocks >= 0 && c.num_res_blocks <= 32, "num_res_blocks out of range");
  if (c.kind == MZ_NET_BOARD) {
    MZ_CHECK_ARG(c.in_channels > 0 && c.in_channels <= 64, "board nets take 1..64 observation planes, got %d",
                 c.in_channels);
    *H = c.in_h; *W = c.in_w;
    MZ_CHECK_ARG(*H > 0 && *W > 0 && *W <= 40, "unsupported board size %dx%d", *H, *W);
  } else {
    // network.py:516-519 hard-wires the 6x6 latent, i.e. 96x96 frames (gym_env.py:373-374); the first
    // residual stage is 128 wide whatever num_planes says (network.py:324-327)
    MZ_CHECK_ARG(c.in_h == 96 && c.in_w == 96, "MuZeroAtariNet needs 96x96 observations (6x6 latent), got %dx%d",
                 c.in_h, c.in_w);
    MZ_CHECK_ARG(c.num_planes == 128 || c.num_planes == 256, "MuZeroAtariNet is built for num_planes 128 or 256, got %d",
                 c.num_planes);
    MZ_CHECK_ARG(c.in_channels > 0 && c.in_channels <= 16, "MuZeroAtariNet takes 1..16 stacked planes, got %d",
                 c.in_channels);
    *H = 6; *W = 6;
  }
  return MZ_OK;
}

int conv_hidden_bytes(const mz_net_config& c, int32_t* bytes) {
  int H, W;
  int rc = conv_geometry(c, &H, &W);
  if (rc) return rc;
  *bytes = H * W * padded_planes(c.num_planes) * 2;
  return MZ_OK;
}

static size_t conv_w_bytes(int cg, int N) { return align_up((size_t)9 * cg * N * 16, 256); }
// convs that can run in SM-pair launches (64-channel weight stages, one pass of >= 64 columns) also keep their weights
// in the pair layout
static bool pair_layout(int cg, int n_out) { return cg >= 8 && n_out >= 64 && n_out <= 128; }
static int obs_cg(int cin) { return ((cin + 15) / 16) * 2; }

// An upper bound on what conv_create takes: its grids are sized (H+1)(W+1), more than the H*W rows a board uses.
int conv_arena_bytes(const mz_net_config& c, int max_batch, size_t* bytes) {
  int H, W;
  int rc = conv_geometry(c, &H, &W);
  if (rc) return rc;
  const bool atari = c.kind == MZ_NET_ATARI;
  const int N = padded_planes(c.num_planes), PB = (H + 1) * (W + 1), A = c.num_actions, hw = H * W;
  size_t t = 0;
  const int nconv_main = 1 + 6 * c.num_res_blocks + (atari ? 12 : 0);   // dyn0 + 2 per block x 3 towers (+ Atari rep)
  t += conv_w_bytes(obs_cg(c.in_channels), N) + (size_t)nconv_main * (conv_w_bytes(N / 8, N) + 512);
  t += (size_t)(nconv_main + 1) * conv_w_bytes(N / 8, N);                             // pair layouts (+ rep0)
  t += (size_t)(2 + 6 * c.num_res_blocks + 12) * 2 * align_up((size_t)N * 4, 256);     // scale + bias per conv
  t += 2 * align_up((size_t)9 * 128 * 256 * 2, 256);                                    // stride-2 conv weights
  t += align_up((size_t)A * PB * N * 4, 256);                                           // action table
  t += 3 * (align_up((size_t)2 * N * 4, 256) + 2 * 256 + 256);                          // head 1x1 weights/bias/scale
  t += align_up((size_t)c.reward_support * hw * 4, 256) + align_up((size_t)A * 2 * hw * 4, 256) +
       align_up((size_t)c.value_support * hw * 4, 256) + 3 * align_up((size_t)(A + c.value_support + c.reward_support) * 4, 256);
  const size_t big_pb = atari ? (size_t)(c.in_h / 2 + 1) * (c.in_w / 2 + 1) : (size_t)PB;   // largest activation grid
  const size_t obs_pb = atari ? (size_t)(c.in_h + 1) * (c.in_w + 1) : (size_t)PB;
  auto rows = [&](size_t pb) { return ((size_t)max_batch * pb + kTileM - 1) / kTileM * kTileM + kPlaneSlack; };
  // activation buffers: the largest (grid, channels) product any stage of the net produces (Atari: 128 channels at
  // 48x48, num_planes at 24x24)
  const size_t mid_pb = atari ? (size_t)(c.in_h / 4 + 1) * (c.in_w / 4 + 1) : (size_t)PB;
  size_t act_bytes = rows(mid_pb) * N * 2;
  if (atari && rows(big_pb) * 128 * 2 > act_bytes) act_bytes = rows(big_pb) * 128 * 2;
  t += align_up(rows(obs_pb) * (atari ? 2 : obs_cg(c.in_channels)) * 16, 256);           // packed observations
  t += 3 * align_up(act_bytes, 256);                                                     // b0..b2
  t += 2 * align_up(rows(PB) * N * 2, 256);                                              // b3, b4 (latent grid only)
  t += align_up((size_t)kMaxLayers * (((size_t)max_batch * big_pb + 127) / 128) * 4, 256) + 256;   // tile flags (128-row tiles)
  *bytes = t + 8192;
  return MZ_OK;
}

int conv_create(const mz_net_config& c, const float* const* w, int nw, int max_batch, void* arena, size_t arena_bytes,
                NetImpl** out) {
  int H, W;
  int rc = conv_geometry(c, &H, &W);
  if (rc) return rc;
  const bool atari = c.kind == MZ_NET_ATARI;
  const int Nreal = c.num_planes, N = padded_planes(Nreal), A = c.num_actions, hw = H * W, blocks = c.num_res_blocks;
  const int rep_tensors = atari ? (1 + 20 + 1 + 20 + 20) : (5 + 10 * blocks);
  const int expect = rep_tensors + (5 + 10 * blocks + 7) + (10 * blocks + 14);
  MZ_CHECK_ARG(nw == expect, "%s with %d blocks has %d state_dict tensors, got %d",
               atari ? "MuZeroAtariNet" : "MuZeroBoardGameNet", blocks, expect, nw);
  size_t need;
  conv_arena_bytes(c, max_batch, &need);
  if (arena_bytes < need) { set_error("net arena too small: %zu < %zu", arena_bytes, need); return MZ_ENOMEM; }

  ConvNet* net = new ConvNet();
  net->cfg = c; net->lat = Geo{H, W}; net->C = N; net->Creal = Nreal; net->A = A; net->atari = atari;
  net->blocks = blocks; net->max_batch = max_batch;
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&net->num_sms, cudaDevAttrMultiProcessorCount, dev);
  net->in_cg = obs_cg(c.in_channels);
  const int PB = net->lat.PB();

  char* p = (char*)arena;
  auto take = [&](size_t bytes) { char* r = p; p += align_up(bytes, 256); return r; };
  int cur = 0;
  auto next = [&]() { return w[cur++]; };

  // pack the (scaled) weights of a conv with n_real output channels (cin of cin_total input channels, the first ones)
  // as one block of n_out rows per 128-column pass
  auto pack_passes = [&](const float* cw, const float* scale, const float* bias, int n_real, int n_out, int cin,
                         int cin_total, int cg, ConvLayer* L) -> int {
    L->cg = cg; L->n_out = n_out; L->n_real = n_real;
    const int np = L->passes(), npass = L->n_pass();
    for (int h = 0; h < np; ++h) {
      act_t* wp = (act_t*)take((size_t)9 * cg * npass * 16);
      const int rows_real = n_real - h * 128 < npass ? n_real - h * 128 : npass;
      pack_conv_kernel<<<256, 256>>>(cw + (size_t)h * 128 * cin_total * 9, scale + h * 128, wp, npass, rows_real, cin,
                                     cin_total, cg, 0);
      MZ_LAUNCH_CHECK("pack_conv_kernel");
      L->w[h] = wp; L->bias[h] = bias + h * 128;
    }
    L->w_pair = nullptr;
    if (pair_layout(cg, n_out)) {
      act_t* wp = (act_t*)take((size_t)9 * cg * n_out * 16);
      pack_conv_kernel<<<256, 256>>>(cw, scale, wp, n_out, n_real, cin, cin_total, cg, 1);
      MZ_LAUNCH_CHECK("pack_conv_kernel");
      L->w_pair = wp;
    }
    return MZ_OK;
  };
  // conv (no bias) + BatchNorm -> packed fp16 weights + fp32 bias; n_real real output channels padded to n_out
  auto fold_conv = [&](int cin, int cin_total, int cg, int n_real, int n_out, ConvLayer* L, float** scale_out) -> int {
    const float* cw = next();
    const float *g = next(), *beta = next(), *mean = next(), *var = next();
    float* scale = (float*)take((size_t)n_out * 4);
    float* bias = (float*)take((size_t)n_out * 4);
    MZ_CUDA(cudaMemset(scale, 0, (size_t)n_out * 4));
    MZ_CUDA(cudaMemset(bias, 0, (size_t)n_out * 4));
    bn_fold_kernel<<<(n_real + 127) / 128, 128>>>(g, beta, mean, var, scale, bias, n_real);
    MZ_LAUNCH_CHECK("bn_fold_kernel");
    if (scale_out) *scale_out = scale;
    return pack_passes(cw, scale, bias, n_real, n_out, cin, cin_total, cg, L);
  };
  // conv without BatchNorm or bias (the Atari stride-2 convs): scale 1, bias 0
  float* ones = (float*)take((size_t)256 * 4);
  float* zeros = (float*)take((size_t)256 * 4);
  {
    std::vector<float> h1((size_t)256, 1.0f);
    MZ_CUDA(cudaMemcpy(ones, h1.data(), (size_t)256 * 4, cudaMemcpyHostToDevice));
    MZ_CUDA(cudaMemset(zeros, 0, (size_t)256 * 4));
  }
  auto plain_conv = [&](int cin, int cg, int n_out, ConvLayer* L) -> int {
    const float* cw = next();
    return pack_passes(cw, ones, zeros, n_out, n_out, cin, cin, cg, L);
  };
  auto fold_head = [&](int mid, int outn, int kind, Head* h) -> int {
    const float* cw = next();
    const float *g = next(), *beta = next(), *mean = next(), *var = next();
    float* scale = (float*)take(256);
    float* bias = (float*)take(256);
    bn_fold_kernel<<<1, 32>>>(g, beta, mean, var, scale, bias, mid);
    MZ_LAUNCH_CHECK("bn_fold_kernel");
    float* w1 = (float*)take((size_t)mid * Nreal * 4);
    scale_rows_kernel<<<(mid * Nreal + 255) / 256, 256>>>(cw, scale, w1, mid, Nreal);
    MZ_LAUNCH_CHECK("scale_rows_kernel");
    const float* lw = next();
    const float* lb = next();
    float* w2 = (float*)take((size_t)outn * mid * hw * 4);
    float* b2 = (float*)take((size_t)outn * 4);
    MZ_CUDA(cudaMemcpy(w2, lw, (size_t)outn * mid * hw * 4, cudaMemcpyDeviceToDevice));
    MZ_CUDA(cudaMemcpy(b2, lb, (size_t)outn * 4, cudaMemcpyDeviceToDevice));
    h->w1 = w1; h->b1 = bias; h->w2 = w2; h->b2 = b2; h->mid = mid; h->out = outn; h->kind = kind;
    return MZ_OK;
  };
#define MZ_TRY(x) do { int rc__ = (x); if (rc__) { delete net; return rc__; } } while (0)

  if (atari) {
    // representation (network.py:312-353): conv_1 (-> 128), res_blocks_1 x2 @128, conv_2 (128 -> num_planes),
    // res_blocks_2 x2, res_blocks_3 x2
    MZ_TRY(plain_conv(c.in_channels, 2, 128, &net->s2_1));
    for (int i = 0; i < 4; ++i) MZ_TRY(fold_conv(128, 128, 16, 128, 128, &net->at_blocks[0][i], nullptr));
    MZ_TRY(plain_conv(128, 16, N, &net->s2_2));
    for (int i = 0; i < 4; ++i) MZ_TRY(fold_conv(N, N, N / 8, N, N, &net->at_blocks[1][i], nullptr));
    for (int i = 0; i < 4; ++i) MZ_TRY(fold_conv(N, N, N / 8, N, N, &net->at_blocks[2][i], nullptr));
  } else {
    // representation (network.py:356-393)
    MZ_TRY(fold_conv(c.in_channels, c.in_channels, net->in_cg, Nreal, N, &net->rep0, nullptr));
    for (int i = 0; i < 2 * blocks; ++i) MZ_TRY(fold_conv(Nreal, Nreal, N / 8, Nreal, N, &net->rep_blocks[i], nullptr));
  }
  // dynamics (network.py:396-449): first conv sees C + A channels; the A action planes become a table
  {
    const float* dyn_w = w[cur];
    float* scale = nullptr;
    MZ_TRY(fold_conv(Nreal, Nreal + A, N / 8, Nreal, N, &net->dyn0, &scale));
    float* tab = (float*)take((size_t)A * PB * N * 4);
    action_table_kernel<<<512, 256>>>(dyn_w, scale, tab, A, Nreal, N, Nreal, H, W);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("action_table_kernel: %s", cudaGetErrorString(e)); delete net; return MZ_ECUDA; }
    count_launch();
    net->tab = tab;
  }
  for (int i = 0; i < 2 * blocks; ++i) MZ_TRY(fold_conv(Nreal, Nreal, N / 8, Nreal, N, &net->dyn_blocks[i], nullptr));
  MZ_TRY(fold_head(1, c.reward_support, c.reward_support == 1 ? 0 : 1, &net->h_reward));
  // prediction (network.py:452-498)
  for (int i = 0; i < 2 * blocks; ++i) MZ_TRY(fold_conv(Nreal, Nreal, N / 8, Nreal, N, &net->pred_blocks[i], nullptr));
  MZ_TRY(fold_head(2, A, 2, &net->h_policy));
  MZ_TRY(fold_head(1, c.value_support, c.value_support == 1 ? 0 : 1, &net->h_value));
#undef MZ_TRY
  const size_t big_pb = atari ? (size_t)(c.in_h / 2 + 1) * (c.in_w / 2 + 1) : (size_t)PB;
  const size_t mid_pb = atari ? (size_t)(c.in_h / 4 + 1) * (c.in_w / 4 + 1) : (size_t)PB;
  const size_t obs_pb = atari ? (size_t)(c.in_h + 1) * (c.in_w + 1) : (size_t)PB;
  auto rows = [&](size_t pb) { return ((size_t)max_batch * pb + kTileM - 1) / kTileM * kTileM + kPlaneSlack; };
  net->xobs = (act_t*)take(rows(obs_pb) * (atari ? 2 : net->in_cg) * 16);
  size_t act_bytes = rows(mid_pb) * N * 2;
  if (atari && rows(big_pb) * 128 * 2 > act_bytes) act_bytes = rows(big_pb) * 128 * 2;
  net->b0 = (act_t*)take(act_bytes);
  net->b1 = (act_t*)take(act_bytes);
  net->b2 = (act_t*)take(act_bytes);
  net->b3 = (act_t*)take(rows(PB) * N * 2);
  net->b4 = (act_t*)take(rows(PB) * N * 2);
  net->flags_cap = (size_t)kMaxLayers * (((size_t)max_batch * big_pb + 127) / 128);
  net->flags = (unsigned*)take(net->flags_cap * 4);
  net->err_flag = (int*)take(256);
  cudaMemset(net->err_flag, 0, 4);
  net->reset_pending();
  if ((size_t)(p - (char*)arena) > arena_bytes) {
    set_error("internal: net arena overrun (%zu > %zu)", (size_t)(p - (char*)arena), arena_bytes);
    delete net;
    return MZ_ENOMEM;
  }
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { set_error("weight repacking failed: %s", cudaGetErrorString(e)); delete net; return MZ_ECUDA; }
  {
    // every (grid, input groups) combination of this net must fit one of the two tile shapes
    const int npass = N > 128 ? 128 : N;
    auto ok = [&](const Geo& g, int cg, int n) { return ConvNet::fits(g, cg, n, kTileM) || ConvNet::fits(g, cg, n, 128); };
    bool fit = ok(net->lat, N / 8, npass) && (atari || ok(net->lat, net->in_cg, npass));
    if (atari)
      fit = fit && ok(Geo{c.in_h, c.in_w}, 2, 128) && ok(Geo{c.in_h / 2, c.in_w / 2}, 16, 128) &&
            ok(Geo{c.in_h / 4, c.in_w / 4}, N / 8, npass);
    if (!fit) {
      set_error("conv tile does not fit shared memory (grid too wide)");
      delete net;
      return MZ_EINVAL;
    }
  }
  const int smem_max = 227 * 1024;
  e = cudaFuncSetAttribute(conv3x3_kernel<128, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3x3_kernel<64, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3x3_kernel<32, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3x3_kernel<128, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3x3_kernel<64, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3x3_kernel<32, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3x3_kernel<128, 256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv3x3_kernel<64, 256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(head_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); delete net; return MZ_ECUDA; }
  {
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3(2 * (unsigned)net->num_sms); lc.blockDim = dim3(kConvThreads); lc.dynamicSmemBytes = smem_max;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    lc.attrs = at; lc.numAttrs = 1;
    e = cudaOccupancyMaxActiveClusters(&net->pair_clusters[0], conv3x3_kernel<128, 256, true>, &lc);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveClusters(&net->pair_clusters[1], conv3x3_kernel<64, 256, true>, &lc);
    if (e != cudaSuccess) { set_error("cudaOccupancyMaxActiveClusters: %s", cudaGetErrorString(e)); delete net; return MZ_ECUDA; }
  }
  *out = net;
  return MZ_OK;
}

}  // namespace mz
