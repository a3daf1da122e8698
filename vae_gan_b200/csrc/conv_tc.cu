// tcgen05 / TMEM / TMA implicit-GEMM convolution kernels for sm_100a (bf16 in, fp32 accumulate).
//
// One kernel family covers every dense contraction of the reference's hot path (SURVEY.md K1-K3,
// K5): Conv2d 3x3 / 1x1 at stride 1 and 2, ConvTranspose2d 4x4 stride 2, forward and dgrad
// (tc_conv_kernel, "tap table" form) and all their weight gradients (tc_wgrad_kernel).
//
// tc_conv_kernel: D[128 pixels][BN channels] = sum over taps t, 64-channel chunks kc of
//     A_t,kc[128 pixels][64]  .  W_t,kc[BN][64]^T
//   * A tile = ONE TMA box {64 ch, TW, TH, TN} of the NHWC activation at the tap's (dx,dy) shift;
//     out-of-bounds coordinates are zero-filled by TMA, which is exactly the convolution padding.
//     A box lands as 128 rows x 128 B with the 128B swizzle = the canonical K-major UMMA layout.
//   * stride-2 gathers read one of four "parity" tensor maps (even/odd rows x even/odd columns
//     of the fine tensor), so every load is still a dense unit-stride box;
//   * stride-2 scatters (ConvTranspose2d forward, Conv2d-s2 dgrad) are decomposed into the four
//     output sub-pixel phases (blockIdx.z), each a small stride-1 convolution - no zero insertion.
//   * warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane), warp 2 = TMEM allocator,
//     warps 4.. = epilogue (tcgen05.ld -> bias / Dropout2d column scale -> bf16|f32 -> global).
//   Three forms, chosen per layer by tc_conv_run: one-shot CTAs (tc_conv_kernel, small problems and split-K),
//   persistent CTAs with a double-buffered TMEM accumulator (tc_conv_persist_kernel), and persistent CTA
//   pairs issuing M=256 cta_group::2 MMAs (tc_conv_pair_kernel, 128/256-wide tiles).  The persist and pair
//   kernels are one body (conv_persistent, CTAs per MMA as a template argument), and all three forms run each
//   work item through the same producer, MMA and epilogue pieces (load_item, mma_item, drain_tile).  Every
//   tcgen05 kernel, tc_wgrad_kernel included, takes its shared-memory layout from TcSmem (the host reads the
//   launch size from the same type) and shares tc_prologue / tc_teardown.
//
// tc_wgrad_kernel: dW[128 = 2 x 64 (tap, c_s chunk)][BN = c_u tile] += S^T . U over a range of
//   64-pixel boxes (split-K across CTAs, fp32 atomics into the torch-layout gradient).  Both
//   operands are MN-major (channels contiguous, pixels along K) straight from the same TMA boxes.
#include <algorithm>
#include <array>
#include <map>
#include <mutex>
#include <vector>
#include "vg_common.cuh"
#include "sm100_ptx.cuh"

namespace vg {

// ------------------------------------------------------------------------------------------
// parameter blocks (passed by value as __grid_constant__)
// ------------------------------------------------------------------------------------------
struct TcTap {
  int8_t map, dy, dx, pad_;
  int32_t wrow;   // row offset of this tap's slab in the weight tensor map (= tap * n_out)
};
struct TcPhase {
  int32_t ntaps, oy_off, ox_off, pad_;
  TcTap taps[16];
};
struct alignas(64) TcConvParams {
  CUtensorMap in_maps[4];
  CUtensorMap w_map;
  TcPhase phases[4];
  int tiles_x, tiles_y, tiles_n;
  int tw_log2, th_log2, TW, TH, TN;
  int gw, gh, gn;        // GEMM pixel grid of one phase
  int k_chunks;          // reduction channels / 64
  int n_out;             // output channels
  int n_store;           // columns actually stored per N tile (== BN except for single-channel outputs)
  int OH, OW, os;        // output tensor spatial dims and phase stride
  int out_f32;
  int ksplit, k_per_split;   // split-K over blockIdx.z (only with a single phase, fp32 atomics)
  void* out;
  const float* bias;
  const float* colscale;
  const float* sigma;    // nullable: the accumulator is multiplied by 1 / sigma[group] (spectral norm applied in the epilogue,
  int sigma_group_n;     //   so the packed weights stay valid across forwards); group = sample / sigma_group_n (0: one group)
  // inference epilogue (BatchNorm-folded sampling path, bf16 outputs only; see VgConvEpilogue in the header)
  float act_slope;       // LeakyReLU slope of the stored output (1 = none)
  const void* residual;  // nullable: same shape/dtype as out, added (after rounding the accumulator to bf16) before the activation
  void* out2;            // nullable second output: leaky_relu(post_scale[c] * out + post_shift[c], post_slope)
  const float* post_scale;
  const float* post_shift;
  float post_slope;
  CUtensorMap out_maps[4];  // bf16 output as {32 channels, bx, by, bn} boxes (64-byte swizzle = the staging buffer's XOR
                            // pattern); one per output phase: a stride-2 scatter writes four interleaved sub-grids
  int tma_store;         // 1: the staged 32 x 32 output chunks leave through cp.async.bulk.tensor stores (out_map)
  int* det_locks;        // deterministic mode, split-K: one turn counter per output tile (the splits add in split order)
  long long det_split_stride;  // deterministic mode, split-K: != 0 -> split z STORES its partial tile at out + z * stride (scratch);
                               //   ordered_reduce_f32 adds the splits in order afterwards (no serialisation, no atomics)
};

struct alignas(64) TcWgradParams {
  CUtensorMap s_maps[4];
  CUtensorMap u_map;
  TcTap taps[16];
  int ntaps, cs_chunks, cs, cu;
  int tiles_x, tiles_y, tiles_n, TW, TH, TN;
  int n_boxes, boxes_per_split;
  int packed;    // 1: dw is the packed scratch [tap][c_s][c_u] (vector reductions); 0: torch layout [c_u][c_s][tap]
  float* dw;
  int* det_locks;  // deterministic mode: one turn counter per (slab pair, c_u tile); the pixel splits add in split order
  long long det_split_stride;  // deterministic mode: != 0 -> split z STORES its partial sums at dw + z * stride (scratch)
};

constexpr int kTcThreads = 256;
constexpr int kABytes = 128 * 128;   // 128 rows x 64 bf16
constexpr int kStageBytes = 32 * 64;  // per epilogue warp: 32 rows x 32 bf16 of one output chunk (coalescing transpose)

// Dynamic shared memory of a tcgen05 kernel; the host takes kBytes for the launch, the kernel takes the pointers.
// At a 1024-byte boundary (the 128-byte swizzle atoms): a STAGES-deep ring of A stages (A_BYTES) and B stages (B_BYTES),
// the ring's full[STAGES] / empty[STAGES] mbarriers, NACC accumulator mbarriers, the TMEM address slot and EW per-warp
// epilogue staging buffers.  The staging buffers are 512-byte aligned: their XOR pattern is then exactly TMA's 64-byte
// swizzle (absolute address bits).
template <int STAGES, int A_BYTES, int B_BYTES, int NACC, int EW>
struct TcSmem {
  static constexpr int kStages = STAGES, kA = A_BYTES, kB = B_BYTES;
  static constexpr int kBytes =
      1024 + STAGES * (A_BYTES + B_BYTES) + (2 * STAGES + NACC) * 8 + 16 + (EW > 0 ? 16 + 512 + EW * kStageBytes : 0);
  uint8_t* a;
  uint8_t* b;
  uint64_t* full;
  uint64_t* empty;
  uint64_t* acc;
  uint32_t* tmem_slot;
  uint8_t* stage;
  __device__ explicit TcSmem(uint8_t* raw) {
    a = raw + ((1024u - (ptx::smem_u32(raw) & 1023u)) & 1023u);
    b = a + STAGES * A_BYTES;
    full = reinterpret_cast<uint64_t*>(b + STAGES * B_BYTES);
    empty = full + STAGES;
    acc = empty + STAGES;
    tmem_slot = reinterpret_cast<uint32_t*>(acc + NACC);
    stage = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 511) & ~(uintptr_t)511);
  }
};

// one-shot form: one accumulator barrier, four epilogue warps
template <int BN, int STAGES>
using ConvSmem = TcSmem<STAGES, kABytes, BN * 128, 1, 4>;
// persistent forms: MT pixel tiles per A stage, a CTA of a pair (CTAS = 2) stages half of the weight tile; acc_full[2], acc_empty[2]
template <int CTAS, int BN, int MT, int STAGES, int EW>
using ConvPersistSmem = TcSmem<STAGES, MT * kABytes, (BN / CTAS) * 128, 4, EW>;
// weight gradient: one stage = two S boxes and NB U boxes of 8 KB
template <int NB, int STAGES>
using WgradSmem = TcSmem<STAGES, (2 + NB) * 8192, 0, 1, 0>;

// Set-up of every tcgen05 kernel: warp 0 prefetches two tensor-map descriptors, warp 1 initialises the ring barriers and
// (init_acc) the accumulator barriers, warp 2 allocates TMEM_COLS TMEM columns (for both CTAs of a pair when CTAS == 2).
// The CTA - or the pair - then synchronises, so every barrier of both CTAs exists before anyone signals it.  All of this
// overlaps the previous kernel's tail: it runs before pdl_entry() and touches no global memory.  Returns the TMEM base.
template <int CTAS, int TMEM_COLS, class Smem, class InitAcc>
__device__ __forceinline__ uint32_t tc_prologue(const Smem& sm, const CUtensorMap* map0, const CUtensorMap* map1, InitAcc init_acc) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(map0);
    ptx::prefetch_tmap(map1);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < Smem::kStages; ++s) {
      ptx::mbar_init(&sm.full[s], 1);
      ptx::mbar_init(&sm.empty[s], 1);
    }
    init_acc();
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    if constexpr (CTAS == 2) ptx::tmem_alloc_pair<TMEM_COLS>(sm.tmem_slot);
    else ptx::tmem_alloc<TMEM_COLS>(sm.tmem_slot);
  }
  ptx::tc_fence_before();
  if constexpr (CTAS == 2) ptx::cluster_sync();
  else __syncthreads();
  ptx::tc_fence_after();
  vg::pdl_entry();
  return *sm.tmem_slot;
}

// Neither the CTA's warps nor the pair's other CTA may still use its TMEM, signal its barriers or read its shared memory
// when it frees the TMEM and retires.
template <int CTAS, int TMEM_COLS>
__device__ __forceinline__ void tc_teardown(uint32_t tmem_base) {
  ptx::tc_fence_before();
  if constexpr (CTAS == 2) ptx::cluster_sync();
  else __syncthreads();
  if ((threadIdx.x >> 5) == 2) {
    if constexpr (CTAS == 2) ptx::tmem_dealloc_pair<TMEM_COLS>(tmem_base);
    else ptx::tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

// origin of pixel tile t (a TW x TH x TN box of the GEMM pixel grid; x fastest, then y, then image)
struct Tile { int x0, y0, n0; };
template <class P>
__device__ __forceinline__ Tile tile_origin(const P& p, int t) {
  const int tx = t % p.tiles_x; t /= p.tiles_x;
  const int ty = t % p.tiles_y;
  const int tn = t / p.tiles_y;
  return Tile{tx * p.TW, ty * p.TH, tn * p.TN};
}

// a role warp's position in the operand ring
template <class Smem>
struct RingPos {
  int stage = 0;
  uint32_t phase = 0;
  __device__ __forceinline__ bool next() {     // true when the ring wraps
    if (++stage < Smem::kStages) return false;
    stage = 0;
    phase ^= 1u;
    return true;
  }
};

// Finishes one 32-column chunk of one accumulator row per thread: 1/sigma, bias, Dropout2d column scale, store
// (bf16 / fp32 / split-K vector reductions / single channel).  z is the work item's output phase, or its k-split when
// p.ksplit > 1 (the bias is added by split 0 only).
//
// bf16 outputs go through `stage` (a 2 KB per-warp shared-memory buffer) when it is given: lane = pixel row holds 64 B of
// consecutive channels, so a direct 16-byte store per lane touches 32 different 128-byte lines per instruction - the
// store path, not the issue rate, bounded the epilogue (8 epilogue warps instead of 4 changed nothing on the 64-wide
// layers).  The warp writes its 32 x 64 B block into shared memory (XOR-swizzled 16-byte units, conflict-free both ways),
// reads it back transposed and stores with FOUR consecutive lanes covering one row's 64 bytes: 8 lines per instruction.
template <bool INF>
__device__ __forceinline__ void epilogue_chunk(const TcConvParams& p, const uint32_t (&r)[32], bool valid, long long opix, int gn,
                                               int ncol, bool first_chunk, uint8_t* stage, int sx, int sy, int sn, int z) {
  const int lane = threadIdx.x & 31;
  const bool add_bias = p.ksplit <= 1 || z == 0;
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
  if (p.sigma != nullptr && valid) {
    const float inv = 1.0f / __ldg(p.sigma + (p.sigma_group_n > 0 ? gn / p.sigma_group_n : 0));
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] *= inv;
  }
  if (p.bias != nullptr && add_bias) {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (ncol + j < p.n_out) v[j] += __ldg(p.bias + ncol + j);
  }
  if (p.colscale != nullptr && valid) {
    const float* cs = p.colscale + (long long)gn * p.n_out + ncol;
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] *= __ldg(cs + j);
  }
  const bool staged = stage != nullptr && !p.out_f32 && p.ksplit <= 1 && p.n_store != 1;
  if (staged) {
    if (INF && p.act_slope != 1.0f && p.residual == nullptr) {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = v[j] > 0.f ? v[j] : v[j] * p.act_slope;
    }
    uint32_t w[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    const bool tma_out = !INF && p.tma_store != 0;
    if (tma_out) {
      // the previous chunk's bulk store must have READ the staging buffer before it is overwritten
      if (lane == 0) ptx::bulk_wait_group_read0();
      __syncwarp();
    }
    uint4* srow = reinterpret_cast<uint4*>(stage + lane * 64);
    const int sw = (lane >> 1) & 3;
#pragma unroll
    for (int q = 0; q < 4; ++q) srow[q ^ sw] = make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
    if (tma_out) {
      // TMA-store epilogue: the warp's 32 pixels are a {bx, by, bn} sub-box of the tile starting at (sx, sy, sn); pixels
      // outside the tensor are clipped by the TMA unit (= the `valid` mask of the manual path)
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        ptx::tma_store_4d(&p.out_maps[z], stage, ncol, sx, sy, sn);
        ptx::bulk_commit_group();
      }
      __syncwarp();
    } else {
    __syncwarp();
    __nv_bfloat16* ob = reinterpret_cast<__nv_bfloat16*>(p.out);
    const bool post = INF && (p.residual != nullptr || p.out2 != nullptr);       // kernel-uniform; compiled out of the training kernels
    float ps[8], pt[8];
    if (INF && p.out2 != nullptr) {
      const int c0 = ncol + (lane & 3) * 8;       // this lane's 8 channels are the same for all four row groups
#pragma unroll
      for (int j = 0; j < 8; ++j) { ps[j] = __ldg(p.post_scale + c0 + j); pt[j] = __ldg(p.post_shift + c0 + j); }
    }
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int row = it * 8 + (lane >> 2), q = lane & 3;
      uint4 val = *reinterpret_cast<const uint4*>(stage + row * 64 + ((q ^ ((row >> 1) & 3)) << 4));
      const long long op = __shfl_sync(0xffffffffu, opix, row);
      const int ok = __shfl_sync(0xffffffffu, (int)valid, row);
      if (ok) {
        const long long e = op * p.n_out + ncol + q * 8;
        if (INF && post) {
          float f[8];
          const uint32_t wv[4] = {val.x, val.y, val.z, val.w};
#pragma unroll
          for (int i = 0; i < 4; ++i) { f[2 * i] = __uint_as_float(wv[i] << 16); f[2 * i + 1] = __uint_as_float(wv[i] & 0xffff0000u); }
          if (p.residual != nullptr) {
            const uint4 rr = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.residual) + e);
            const uint32_t rv[4] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) { f[2 * i] += __uint_as_float(rv[i] << 16); f[2 * i + 1] += __uint_as_float(rv[i] & 0xffff0000u); }
            if (p.act_slope != 1.0f) {
#pragma unroll
              for (int j = 0; j < 8; ++j) f[j] = f[j] > 0.f ? f[j] : f[j] * p.act_slope;
            }
            uint32_t o[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
              o[i] = *reinterpret_cast<uint32_t*>(&h);
              // the second output is computed from the value AS STORED (what a separate elementwise pass would read)
              f[2 * i] = __uint_as_float(o[i] << 16);
              f[2 * i + 1] = __uint_as_float(o[i] & 0xffff0000u);
            }
            val = make_uint4(o[0], o[1], o[2], o[3]);
          }
          if (p.out2 != nullptr) {
            uint32_t o2[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              float a0 = fmaf(ps[2 * i], f[2 * i], pt[2 * i]), a1 = fmaf(ps[2 * i + 1], f[2 * i + 1], pt[2 * i + 1]);
              a0 = a0 > 0.f ? a0 : a0 * p.post_slope;
              a1 = a1 > 0.f ? a1 : a1 * p.post_slope;
              __nv_bfloat162 h = __floats2bfloat162_rn(a0, a1);
              o2[i] = *reinterpret_cast<uint32_t*>(&h);
            }
            *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out2) + e) = make_uint4(o2[0], o2[1], o2[2], o2[3]);
          }
        }
        *reinterpret_cast<uint4*>(ob + e) = val;
      }
    }
    __syncwarp();                      // the buffer is rewritten by this warp's next chunk
    }
  } else if (valid) {
    if (p.n_store == 1) {
      // single-channel output (Conv2d C->1 forward / Conv2d 1->C dgrad): only column 0 is real
      // (static register index - a dynamic one would push v[] into local memory)
      if (first_chunk) {
        if (p.out_f32) reinterpret_cast<float*>(p.out)[opix] = v[0];
        else reinterpret_cast<__nv_bfloat16*>(p.out)[opix] = __float2bfloat16_rn(v[0]);
      }
    } else if (p.ksplit > 1) {
      // split-K partial sums: 16-byte vector reductions (a quarter of the RED instructions of scalar atomics - the
      // Linear layers' one-shot CTAs spent most of their time issuing them; n_out % 64 == 0 keeps them aligned)
      float* o = reinterpret_cast<float*>(p.out) + opix * p.n_out + ncol;
      if (p.det_split_stride != 0) {
        // deterministic mode: this split's partial tile goes to its own scratch slab
        o += (long long)z * p.det_split_stride;
#pragma unroll
        for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
      } else {
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          asm volatile("red.global.v4.f32.add [%0], {%1, %2, %3, %4};" ::"l"(o + j), "f"(v[j]), "f"(v[j + 1]), "f"(v[j + 2]), "f"(v[j + 3])
                       : "memory");
      }
    } else if (p.out_f32) {
      float* o = reinterpret_cast<float*>(p.out) + opix * p.n_out + ncol;
#pragma unroll
      for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    } else {
      __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.out) + opix * p.n_out + ncol;
#pragma unroll
      for (int j = 0; j < 32; j += 8) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          __nv_bfloat162 h = __floats2bfloat162_rn(v[j + 2 * i], v[j + 2 * i + 1]);
          w[i] = *reinterpret_cast<uint32_t*>(&h);
        }
        *reinterpret_cast<uint4*>(o + j) = make_uint4(w[0], w[1], w[2], w[3]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// forward / dgrad implicit GEMM
// ------------------------------------------------------------------------------------------
// NOTES (measured on B200, round 1; microbenchmarks in scripts/microbench/, numbers in DESIGN.md section 3):
//  * a tcgen05.mma (M=128, K=16, SS mode) takes max(N/2, 32 + N/4) cycles - the operands are re-read from
//    shared memory at 128 B/cycle - so N=64 tiles cap at 67 % of the tensor peak, N>=128 can reach it;
//  * the tensor pipe queues only ~1-2 instructions and every mbarrier wait stalls the issuing thread for
//    ~105 cycles: one wait per k-block costs a ~135-cycle bubble unless the queued MMAs are N=256 wide;
//    sharing one full/empty barrier pair between two k-blocks halves those waits but measured nothing in the
//    real kernel and cost the 256-wide tiles 8 % (coarser refill granularity; DESIGN.md 3.3 item 2);
//  * under a divergent `lane == 0` branch nvcc wraps each UTCHMMA/UTMALDG in an elect-and-retry loop and
//    rebuilding 64-bit descriptors costs ~14 uniform instructions per MMA: the role warps therefore run
//    warp-uniformly, elect only around the issue, and advance 32-bit descriptor halves by adds;
//  * the chip is power-capped under tensor load (SM clock 1.3-1.5 GHz), so removing loads, stores or waits
//    buys cycles but little time; what pays is fewer shared-memory/L2 bytes per FLOP (CTA pairs below).
//
// The three forms share the per-item pieces below: conv_slice (which k-blocks an item reduces), load_item (producer warp),
// mma_item (MMA warp) and drain_tile (epilogue warps).

// k-blocks [kb0, kb1) of slice z - an output phase, or a k-split when p.ksplit > 1 - and the tap table they read
__device__ __forceinline__ const TcPhase& conv_slice(const TcConvParams& p, int z, int& kb0, int& kb1) {
  const TcPhase& ph = p.phases[p.ksplit > 1 ? 0 : z];
  const int total = ph.ntaps * p.k_chunks;
  if (p.ksplit > 1) { kb0 = z * p.k_per_split; kb1 = min(total, kb0 + p.k_per_split); }
  else { kb0 = 0; kb1 = total; }
  if (kb1 < kb0) kb1 = kb0;
  return ph;
}

// Producer warp, one work item: k-blocks [kb0, kb1) into the ring.  A k-block is the A boxes of the first `nvalid` of the
// CTA's MT pixel tiles (at the tap's shift) and the weight tile from row tap.wrow + wrow0.  In a CTA pair (CTAS == 2) both
// CTAs count their bytes on the leader's full barrier, which the leader (rank 0) arms for both.
template <int CTAS, int MT, class Smem>
__device__ __forceinline__ void load_item(const TcConvParams& p, const TcPhase& ph, int kb0, int kb1, const Tile (&t)[MT], int nvalid,
                                          int wrow0, uint32_t rank, const Smem& sm, RingPos<Smem>& pos) {
  int tp = kb0 / p.k_chunks, kc = kb0 % p.k_chunks;
  for (int i = kb0; i < kb1; ++i) {
    const TcTap tap = ph.taps[tp];
    const CUtensorMap* im = &p.in_maps[tap.map];
    ptx::mbar_wait(&sm.empty[pos.stage], pos.phase ^ 1u);
    if (ptx::elect_one()) {
      uint8_t* a = sm.a + pos.stage * Smem::kA;
      uint8_t* b = sm.b + pos.stage * Smem::kB;
      if constexpr (CTAS == 2) {
        if (rank == 0) ptx::mbar_arrive_expect_tx(&sm.full[pos.stage], 2 * (Smem::kA + Smem::kB));
        const uint32_t bar = ptx::mapa(ptx::smem_u32(&sm.full[pos.stage]), 0);
#pragma unroll
        for (int m = 0; m < MT; ++m)
          ptx::tma_load_4d_pair(a + m * kABytes, im, bar, kc * 64, t[m].x0 + tap.dx, t[m].y0 + tap.dy, t[m].n0);
        ptx::tma_load_2d_pair(b, &p.w_map, bar, kc * 64, tap.wrow + wrow0);
      } else {
        ptx::mbar_arrive_expect_tx(&sm.full[pos.stage], nvalid * kABytes + Smem::kB);
#pragma unroll
        for (int m = 0; m < MT; ++m)
          if (m < nvalid)
            ptx::tma_load_4d(a + m * kABytes, im, &sm.full[pos.stage], kc * 64, t[m].x0 + tap.dx, t[m].y0 + tap.dy, t[m].n0);
        ptx::tma_load_2d(b, &p.w_map, &sm.full[pos.stage], kc * 64, tap.wrow + wrow0);
      }
    }
    __syncwarp();
    pos.next();
    if (++kc == p.k_chunks) { kc = 0; ++tp; }
  }
}

// tcgen05.commit to `bar` (of both CTAs of a pair) once the MMAs issued so far have completed
template <int CTAS>
__device__ __forceinline__ void commit_to(uint64_t* bar) {
  if constexpr (CTAS == 2) ptx::mma_commit_pair(bar, 3);
  else ptx::mma_commit(bar);
}

// MMA warp, one work item: num_k k-blocks from the ring into the accumulator at TMEM address `acc` (pixel tile m at column
// m * BN; M = 256 over both CTAs of a pair, issued by the leader alone), releasing each stage as its MMAs complete.
// a_lo / b_lo are the descriptor low words of the ring position's stage (a_lo0 / b_lo0: stage 0).
template <int CTAS, int BN, int MT, class Smem>
__device__ __forceinline__ void mma_item(uint32_t acc, int num_k, int nvalid, const Smem& sm, RingPos<Smem>& pos, uint32_t a_lo0,
                                         uint32_t b_lo0, uint32_t& a_lo, uint32_t& b_lo) {
  constexpr uint32_t idesc = ptx::make_idesc_bf16(128 * CTAS, BN, 0, 0);
  constexpr uint32_t kDescHi = ptx::smem_desc_hi(1024);
  for (int i = 0; i < num_k; ++i) {
    ptx::mbar_wait(&sm.full[pos.stage], pos.phase);
    ptx::tc_fence_after();
    if (ptx::elect_one()) {
#pragma unroll
      for (int m = 0; m < MT; ++m) {
        if (m < nvalid) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint32_t d = acc + (uint32_t)(m * BN), a = a_lo + (uint32_t)((m * kABytes + k * 32) >> 4),
                           b = b_lo + (uint32_t)((k * 32) >> 4);
            if constexpr (CTAS == 2) ptx::mma_bf16_ss_pair_lohi(d, a, b, kDescHi, idesc, (i | k) != 0);
            else ptx::mma_bf16_ss_lohi(d, a, b, kDescHi, idesc, (i | k) != 0);
          }
        }
      }
      commit_to<CTAS>(&sm.empty[pos.stage]);
    }
    __syncwarp();
    if (pos.next()) { a_lo = a_lo0; b_lo = b_lo0; }
    else { a_lo += (uint32_t)(Smem::kA >> 4); b_lo += (uint32_t)(Smem::kB >> 4); }
  }
}

// An epilogue warp's share of every tile: warp ew + 4 reads TMEM lane quarter q, i.e. tile rows q * 32 + lane.  Warp w may
// only touch TMEM lanes 32*(w%4)..+31, so with EW = 8 two warps share each lane quarter and split the 32-column chunks
// between them (chunk group cgrp); that doubles the epilogue throughput.
struct EpiWarp {
  int ew, q, cgrp;
  int xl, yl, nl;      // this thread's row in the tile
  int xl0, yl0, nl0;   // the quarter's first row: origin of its TMA-store sub-box
  __device__ explicit EpiWarp(const TcConvParams& p) {
    ew = (int)(threadIdx.x >> 5) - 4;
    q = ew & 3;
    cgrp = ew >> 2;
    const int row = q * 32 + (threadIdx.x & 31), row0 = q * 32;
    xl = row & (p.TW - 1);
    yl = (row >> p.tw_log2) & (p.TH - 1);
    nl = row >> (p.tw_log2 + p.th_log2);
    xl0 = row0 & (p.TW - 1), yl0 = (row0 >> p.tw_log2) & (p.TH - 1), nl0 = row0 >> (p.tw_log2 + p.th_log2);
  }
};

// Epilogue warp, one 128-pixel tile at origin t: its lane quarter of the accumulator at TMEM address `acc` (zeros when the
// item has no k-blocks), chunk by chunk through epilogue_chunk; pixels outside the grid, or all of them when !live, store
// nothing.
template <int BN, int EW, bool INF>
__device__ __forceinline__ void drain_tile(const TcConvParams& p, const TcPhase& ph, const EpiWarp& e, uint32_t acc, bool has_k, Tile t,
                                           bool live, int ncol0, int z, uint8_t* stage_base) {
  const int gx = t.x0 + e.xl, gy = t.y0 + e.yl, gn = t.n0 + e.nl;
  const bool valid = gx < p.gw && gy < p.gh && gn < p.gn && live;
  const long long opix = ((long long)gn * p.OH + (long long)gy * p.os + ph.oy_off) * p.OW + (long long)gx * p.os + ph.ox_off;
#pragma unroll(EW == 4 ? BN / 32 : 1)
  for (int i = 0; i < BN / EW / 8; ++i) {     // this warp's chunks
    const int c = EW == 4 ? i : i * (EW / 4) + e.cgrp;
    const int c0 = c * 32;
    uint32_t r[32];
    if (has_k) {
      ptx::tmem_ld_32x32(acc + ((uint32_t)(e.q * 32) << 16) + (uint32_t)c0, r);
      ptx::tmem_ld_wait();
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) r[j] = 0u;
    }
    epilogue_chunk<INF>(p, r, valid, opix, gn, ncol0 + c0, c == 0, stage_base + e.ew * kStageBytes, t.x0 + e.xl0, t.y0 + e.yl0,
                        t.n0 + e.nl0, z);
  }
}

// One-shot form: one CTA per (128-pixel tile, N tile, phase | k-split), two CTAs per SM.
// warp 0 = TMA producer, warp 1 = MMA issuer, warp 2 = TMEM allocator, warps 4-7 = epilogue.
template <int BN, int STAGES, bool INF>
__global__ void __launch_bounds__(kTcThreads) tc_conv_kernel(const __grid_constant__ TcConvParams p) {
  using Smem = ConvSmem<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  const Smem sm(smem_raw);
  uint64_t* const tmem_full = sm.acc;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int z = (int)blockIdx.z;
  int kb0, kb1;
  const TcPhase& ph = conv_slice(p, z, kb0, kb1);
  const bool has_k = kb1 > kb0;
  const Tile t = tile_origin(p, (int)blockIdx.x);
  const int ncol0 = blockIdx.y * BN;
  const uint32_t tmem_base = tc_prologue<1, BN>(sm, &p.w_map, &p.in_maps[0], [&] { ptx::mbar_init(tmem_full, 1); });

  if (has_k) {
    RingPos<Smem> pos;
    if (warp == 0) {
      const Tile ts[1] = {t};
      load_item<1, 1>(p, ph, kb0, kb1, ts, 1, ncol0, 0, sm, pos);
    } else if (warp == 1) {
      const uint32_t a_lo0 = ptx::smem_desc_lo(ptx::smem_u32(sm.a), 16), b_lo0 = ptx::smem_desc_lo(ptx::smem_u32(sm.b), 16);
      uint32_t a_lo = a_lo0, b_lo = b_lo0;
      mma_item<1, BN, 1>(tmem_base, kb1 - kb0, 1, sm, pos, a_lo0, b_lo0, a_lo, b_lo);
      if (ptx::elect_one()) ptx::mma_commit(tmem_full);
      __syncwarp();
    }
  }

  if (warp >= 4) {
    if (has_k) {
      ptx::mbar_wait(tmem_full, 0);
      ptx::tc_fence_after();
    }
    // deterministic split-K: this split's reductions go after those of split z - 1 of the same output tile
    int* const det_lock = (p.det_locks != nullptr && p.ksplit > 1) ? p.det_locks + (blockIdx.y * gridDim.x + blockIdx.x) : nullptr;
    if (det_lock) {
      if (lane == 0) det_wait_turn(det_lock, z);
      __syncwarp();
    }
    // an empty k-split adds nothing, but with per-split slabs it stores its zeros
    const bool live = !(p.ksplit > 1 && !has_k && p.det_split_stride == 0);
    drain_tile<BN, 4, INF>(p, ph, EpiWarp(p), tmem_base, has_k, t, live, ncol0, z, sm.stage);
    if (det_lock) {
      __threadfence();
      asm volatile("bar.sync 2, 128;" ::: "memory");      // the four epilogue warps
      if (warp == 4 && lane == 0) det_publish_turn(det_lock, z + 1 == p.ksplit ? 0 : z + 1);
    }
    if (!INF && p.tma_store && lane == 0) ptx::bulk_wait_group0();      // this warp's bulk stores have landed
  }
  tc_teardown<1, BN>(tmem_base);
}

// Persistent forms: one CTA per SM (CTAS = 1, tc_conv_persist_kernel) or one CTA pair per two SMs (CTAS = 2,
// tc_conv_pair_kernel) loops over work items (phase | k-split, N tile, group of CTAS x MT pixel tiles).  The TMEM accumulator
// is double-buffered so the epilogue of item i overlaps the main loop of item i+1, and the MT pixel tiles of a CTA share
// every staged weight tile.  Warps as in the one-shot form, with EW epilogue warps (4 or 8).
//
// CTA pairs (cta_group::2): the two CTAs of a cluster - two SMs - issue ONE M=256 MMA.  Each CTA stages its own MT pixel
// tiles (A, 128 rows each) and HALF of the weight tile (B, BN/2 rows); the tensor core of each SM reads its own A and both
// halves of B, so the per-SM shared-memory reads per MMA drop from (4 KB + BN*32 B) to (4 KB + BN*16 B) and the staged weight
// bytes halve as well.  Protocol (leader = cluster rank 0):
//   * producer warp in BOTH CTAs: waits its own empty[s] (multicast commit), issues its TMA loads with the completion bytes
//     counted on the LEADER's full[s]; the leader arms full[s] with the bytes of both CTAs;
//   * MMA warp in the leader only; tcgen05.commit multicasts to empty[s] / acc_full[a] of both CTAs;
//   * epilogue warps in both CTAs drain their own TMEM and arrive (cluster scope) on the leader's acc_empty[a], which
//     therefore counts 2*EW arrivals.
// Requires total pixel tiles % (2*MT) == 0 (the host falls back to the single-CTA kernel otherwise).
template <int CTAS, int BN, int MT, int STAGES, int EW, bool INF>
__device__ __forceinline__ void conv_persistent(const TcConvParams& p, int n_ntiles, int n_groups, int n_work) {
  static_assert(EW == 4 || EW == 8, "4 or 8 epilogue warps");
  constexpr int kAccCols = MT * BN;
  constexpr int kTmemCols = 2 * kAccCols;
  static_assert(kTmemCols <= 512 && kTmemCols >= 32, "TMEM budget");
  using Smem = ConvPersistSmem<CTAS, BN, MT, STAGES, EW>;
  extern __shared__ uint8_t smem_raw[];
  const Smem sm(smem_raw);
  uint64_t* const acc_full = sm.acc;        // [2]
  uint64_t* const acc_empty = sm.acc + 2;   // [2]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = CTAS == 2 ? ptx::cluster_ctarank() : 0u;
  const int w_first = blockIdx.x / CTAS, w_step = gridDim.x / CTAS;
  const int total_tiles = p.tiles_x * p.tiles_y * p.tiles_n;
  const uint32_t tmem_base = tc_prologue<CTAS, kTmemCols>(sm, &p.w_map, &p.in_maps[0], [&] {
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&acc_full[a], 1);
      ptx::mbar_init(&acc_empty[a], CTAS * EW);     // one arrival per epilogue warp of the CTA (of both CTAs of a pair)
    }
  });

  // work item -> (z, n tile, pixel-tile group); groups vary fastest so that concurrently running
  // CTAs stream the same weight tile (L2 reuse) over neighbouring pixels
  auto decode = [&](int w, int& z, int& nt, int& g) {
    const int per_z = n_ntiles * n_groups;
    z = w / per_z;
    const int r = w - z * per_z;
    nt = r / n_groups;
    g = r - nt * n_groups;
  };
  // this CTA's first pixel tile of group g, and how many of its MT tiles exist (all of them in a pair)
  auto tiles_of = [&](int g, int& tile0, int& nvalid) {
    tile0 = (g * CTAS + (int)rank) * MT;
    nvalid = CTAS == 2 ? MT : min(MT, total_tiles - tile0);
  };

  if (warp == 0) {
    RingPos<Smem> pos;
    for (int w = w_first; w < n_work; w += w_step) {
      int z, nt, g, kb0, kb1, tile0, nvalid;
      decode(w, z, nt, g);
      const TcPhase& ph = conv_slice(p, z, kb0, kb1);
      if (kb1 == kb0) continue;
      tiles_of(g, tile0, nvalid);
      Tile t[MT];
#pragma unroll
      for (int m = 0; m < MT; ++m) t[m] = tile_origin(p, tile0 + m);
      load_item<CTAS, MT>(p, ph, kb0, kb1, t, nvalid, nt * BN + (int)rank * (BN / CTAS), rank, sm, pos);
    }
  } else if (warp == 1) {
    if (rank == 0) {
      const uint32_t a_lo0 = ptx::smem_desc_lo(ptx::smem_u32(sm.a), 16), b_lo0 = ptx::smem_desc_lo(ptx::smem_u32(sm.b), 16);
      uint32_t a_lo = a_lo0, b_lo = b_lo0;
      RingPos<Smem> pos;
      int it = 0;                       // number of accumulator uses so far
      for (int w = w_first; w < n_work; w += w_step) {
        int z, nt, g, kb0, kb1, tile0, nvalid;
        decode(w, z, nt, g);
        conv_slice(p, z, kb0, kb1);
        if (kb1 == kb0) continue;
        tiles_of(g, tile0, nvalid);
        const int as = it & 1;
        ptx::mbar_wait(&acc_empty[as], (uint32_t)(((it >> 1) & 1) ^ 1));
        ptx::tc_fence_after();
        mma_item<CTAS, BN, MT>(tmem_base + (uint32_t)(as * kAccCols), kb1 - kb0, nvalid, sm, pos, a_lo0, b_lo0, a_lo, b_lo);
        if (ptx::elect_one()) commit_to<CTAS>(&acc_full[as]);
        __syncwarp();
        ++it;
      }
    }
  } else if (warp >= 4) {
    const EpiWarp e(p);
    int it = 0;
    for (int w = w_first; w < n_work; w += w_step) {
      int z, nt, g, kb0, kb1, tile0, nvalid;
      decode(w, z, nt, g);
      const TcPhase& ph = conv_slice(p, z, kb0, kb1);
      const bool has_k = kb1 > kb0;
      if (!has_k && p.ksplit > 1) continue;          // empty k-split: contributes nothing
      tiles_of(g, tile0, nvalid);
      const int as = it & 1;
      if (has_k) {
        ptx::mbar_wait(&acc_full[as], (uint32_t)((it >> 1) & 1));
        ptx::tc_fence_after();
      }
#pragma unroll 1
      for (int m = 0; m < nvalid; ++m)
        drain_tile<BN, EW, INF>(p, ph, e, tmem_base + (uint32_t)(as * kAccCols + m * BN), has_k, tile_origin(p, tile0 + m), true, nt * BN,
                                z, sm.stage);
      if (has_k) {
        // this warp is done reading accumulator stage `as`: hand it back to the MMA warp (of the leader)
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (CTAS == 2) ptx::mbar_arrive_cluster(ptx::mapa(ptx::smem_u32(&acc_empty[as]), 0));
          else ptx::mbar_arrive(&acc_empty[as]);
        }
        ++it;
      }
    }
    if (!INF && p.tma_store && lane == 0) ptx::bulk_wait_group0();      // this warp's bulk stores have landed
  }
  tc_teardown<CTAS, kTmemCols>(tmem_base);
}

template <int BN, int MT, int STAGES, int EW, bool INF>
__global__ void __launch_bounds__(128 + 32 * EW, 1)
    tc_conv_persist_kernel(const __grid_constant__ TcConvParams p, int n_ntiles, int n_groups, int n_work) {
  conv_persistent<1, BN, MT, STAGES, EW, INF>(p, n_ntiles, n_groups, n_work);
}

template <int BN, int MT, int STAGES, int EW, bool INF>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128 + 32 * EW, 1)
    tc_conv_pair_kernel(const __grid_constant__ TcConvParams p, int n_ntiles, int n_groups, int n_work) {
  conv_persistent<2, BN, MT, STAGES, EW, INF>(p, n_ntiles, n_groups, n_work);
}

// ------------------------------------------------------------------------------------------
// weight gradient
// ------------------------------------------------------------------------------------------
template <int NB, int STAGES>
__global__ void __launch_bounds__(kTcThreads) tc_wgrad_kernel(const __grid_constant__ TcWgradParams p) {
  using Smem = WgradSmem<NB, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  constexpr int BN = NB * 64;
  constexpr int kStageBytes = Smem::kA;
  const Smem sm(smem_raw);
  uint8_t* const smem = sm.a;
  uint64_t* const full = sm.full;
  uint64_t* const empty = sm.empty;
  uint64_t* const tmem_full = sm.acc;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_slabs = p.ntaps * p.cs_chunks;
  const int slab0 = blockIdx.x * 2;
  const bool has2 = slab0 + 1 < n_slabs;
  const int slab1 = has2 ? slab0 + 1 : slab0;
  const int box_begin = blockIdx.z * p.boxes_per_split;
  const int box_end = min(p.n_boxes, box_begin + p.boxes_per_split);
  const int num_k = max(0, box_end - box_begin);

  const uint32_t tmem_base = tc_prologue<1, BN>(sm, &p.u_map, &p.s_maps[0], [&] { ptx::mbar_init(tmem_full, 1); });

  if (num_k > 0) {
    // role warps loop warp-uniformly; one elected lane issues the TMA / MMA instructions (NOTES above)
    if (warp == 0) {
      const int tapA = slab0 / p.cs_chunks, chA = slab0 % p.cs_chunks;
      const int tapB = slab1 / p.cs_chunks, chB = slab1 % p.cs_chunks;
      const TcTap ta = p.taps[tapA], tb = p.taps[tapB];
      int stage = 0;
      uint32_t phase = 0;
      for (int b = box_begin; b < box_end; ++b) {
        const Tile t = tile_origin(p, b);
        const int x0 = t.x0, y0 = t.y0, n0 = t.n0;
        ptx::mbar_wait(&empty[stage], phase ^ 1u);
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx(&full[stage], kStageBytes);
          uint8_t* st = smem + stage * kStageBytes;
          ptx::tma_load_4d(st, &p.s_maps[ta.map], &full[stage], chA * 64, x0 + ta.dx, y0 + ta.dy, n0);
          ptx::tma_load_4d(st + 8192, &p.s_maps[tb.map], &full[stage], chB * 64, x0 + tb.dx, y0 + tb.dy, n0);
#pragma unroll
          for (int j = 0; j < NB; ++j)
            ptx::tma_load_4d(st + (2 + j) * 8192, &p.u_map, &full[stage], (blockIdx.y * NB + j) * 64, x0, y0, n0);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    } else if (warp == 1) {
      constexpr uint32_t idesc = ptx::make_idesc_bf16(128, BN, 1, 1);
      constexpr uint32_t kDescHi = ptx::smem_desc_hi(1024);
      const uint32_t a_lo0 = ptx::smem_desc_lo(ptx::smem_u32(smem), 8192);   // MN-major: LBO = 64-channel slab stride
      uint32_t a_lo = a_lo0;
      int stage = 0;
      uint32_t phase = 0;
      for (int i = 0; i < num_k; ++i) {
        ptx::mbar_wait(&full[stage], phase);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k)     // 16 pixels (two 8-row atoms) per MMA
            ptx::mma_bf16_ss_lohi(tmem_base, a_lo + (uint32_t)((k * 2048) >> 4), a_lo + (uint32_t)((2 * 8192 + k * 2048) >> 4), kDescHi,
                                  idesc, (i | k) != 0);
          ptx::mma_commit(&empty[stage]);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; a_lo = a_lo0; }
        else a_lo += (uint32_t)(kStageBytes >> 4);
      }
      if (ptx::elect_one()) ptx::mma_commit(tmem_full);
      __syncwarp();
    }
  }

  int* const det_lock = p.det_locks != nullptr ? p.det_locks + (blockIdx.y * gridDim.x + blockIdx.x) : nullptr;
  if (warp >= 4 && det_lock) {
    if (lane == 0) det_wait_turn(det_lock, (int)blockIdx.z);
    __syncwarp();
  }
  if (warp >= 4 && num_k > 0) {
    const int q = warp - 4;
    const int row = q * 32 + lane;
    const int slab = (row < 64) ? slab0 : slab1;
    const bool row_valid = (row < 64) || has2;
    const int tap = slab / p.cs_chunks, chunk = slab % p.cs_chunks;
    const int cs = chunk * 64 + (row & 63);
    ptx::mbar_wait(tmem_full, 0);
    ptx::tc_fence_after();
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t r[32];
      ptx::tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, r);
      ptx::tmem_ld_wait();
      if (row_valid) {
        const int cu0 = blockIdx.y * BN + c0;
        if (p.packed) {
          // 32 consecutive c_u of one (tap, c_s) row: eight 16-byte vector reductions
          float* dst = p.dw + (long long)blockIdx.z * p.det_split_stride + ((long long)tap * p.cs + cs) * p.cu + cu0;
          if (p.det_split_stride != 0) {
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              *reinterpret_cast<float4*>(dst + j) = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]),
                                                                __uint_as_float(r[j + 3]));
          } else {
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              asm volatile("red.global.v4.f32.add [%0], {%1, %2, %3, %4};" ::"l"(dst + j), "f"(__uint_as_float(r[j])),
                           "f"(__uint_as_float(r[j + 1])), "f"(__uint_as_float(r[j + 2])), "f"(__uint_as_float(r[j + 3]))
                           : "memory");
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            float* dst = p.dw + (long long)blockIdx.z * p.det_split_stride + ((long long)(cu0 + j) * p.cs + cs) * p.ntaps + tap;
            if (p.det_split_stride != 0) *dst = __uint_as_float(r[j]);
            else atomicAdd(dst, __uint_as_float(r[j]));
          }
        }
      }
    }
  }
  if (warp >= 4 && det_lock) {
    __threadfence();
    asm volatile("bar.sync 2, 128;" ::: "memory");        // the four epilogue warps
    if (warp == 4 && lane == 0) det_publish_turn(det_lock, blockIdx.z + 1 == gridDim.z ? 0 : (int)blockIdx.z + 1);
  }
  tc_teardown<1, BN>(tmem_base);
}

// dw[cu][cs][tap] += ws[tap][cs][cu]  (32x32 smem-tile transpose between cu and r = cs*taps+tap)
__global__ void __launch_bounds__(256) wgrad_unpack_kernel(const float* __restrict__ ws, int cu_n, int cs_n, int taps, float* __restrict__ dw) {
  vg::pdl_entry();
  __shared__ float tile[32][33];
  const int R = cs_n * taps;
  const int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int i = ty; i < 32; i += 8) {
    const int r = r0 + i, cu = c0 + tx;
    float v = 0.f;
    if (r < R && cu < cu_n) {
      const int cs = r / taps, tap = r - cs * taps;
      v = ws[((long long)tap * cs_n + cs) * cu_n + cu];
    }
    tile[i][tx] = v;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int cu = c0 + i, r = r0 + tx;
    if (cu < cu_n && r < R) dw[(long long)cu * R + r] += tile[tx][i];
  }
}

// ==========================================================================================
// host side: tensor maps, tap tables, launch
// ==========================================================================================
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static std::once_flag g_encode_once;

// cuTensorMapEncodeTiled is a DRIVER entry point and needs a current context on the calling
// thread.  torch's autograd worker threads only select a runtime device; a (cheap, once per
// thread) runtime call binds the primary context before the first encode.
static void bind_context_once() {
  static thread_local bool done = false;
  if (!done) {
    cudaFree(0);
    done = true;
  }
}

static EncodeTiledFn get_encode() {
  std::call_once(g_encode_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  });
  return g_encode;
}

// cuTensorMapEncodeTiled of a bf16 tensor with `rank` dimensions (dims, byte strides and box innermost first); `what` names the
// tensor in the error message
static int encode_map(CUtensorMap* m, const char* what, int rank, const void* base, const cuuint64_t* dims, const cuuint64_t* strides,
                      const cuuint32_t* box, CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled entry point unavailable");
    return VG_ECUDA;
  }
  bind_context_once();
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char shape[128];
    int len = 0;
    for (int i = 0; i < rank; ++i)
      len += snprintf(shape + len, sizeof(shape) - len, " %llu/%u", (unsigned long long)dims[i], (unsigned)box[i]);
    set_error("cuTensorMapEncodeTiled(%s) failed: %d (dim/box:%s)", what, (int)r, shape);
    return VG_ECUDA;
  }
  return VG_OK;
}

// NHWC bf16 activation [n][h][w][c]; parity (py,px) with step `s` selects rows py, py+s, ... and
// columns px, px+s, ...  Box = {64, TW, TH, TN}.
static int make_act_map(CUtensorMap* m, const void* base, int n, int h, int w, int c, int s, int py, int px, int TW, int TH,
                        int TN) {
  const int hs = (h - py + s - 1) / s, ws = (w - px + s - 1) / s;
  const cuuint64_t dims[4] = {(cuuint64_t)c, (cuuint64_t)std::max(ws, 1), (cuuint64_t)std::max(hs, 1), (cuuint64_t)n};
  const cuuint64_t strides[3] = {(cuuint64_t)s * c * 2, (cuuint64_t)s * w * c * 2, (cuuint64_t)h * w * c * 2};
  const cuuint32_t box[4] = {64, (cuuint32_t)TW, (cuuint32_t)TH, (cuuint32_t)TN};
  return encode_map(m, "activation", 4, (const char*)base + ((size_t)py * w + px) * c * 2, dims, strides, box,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
}

// bf16 output tensor (N, OH, OW, C) as {32 channels, bx, by, bn} boxes with the 64-byte swizzle (TMA-store epilogue)
// (s, py, px): the sub-grid of output pixels (py + s*i, px + s*j) a scatter phase writes (s = 1: the whole tensor)
static int make_out_map(CUtensorMap* m, void* base, int n, int h, int w, int c, int bx, int by, int bn, int s, int py, int px) {
  const int hs = (h - py + s - 1) / s, ws = (w - px + s - 1) / s;
  const cuuint64_t dims[4] = {(cuuint64_t)c, (cuuint64_t)std::max(ws, 1), (cuuint64_t)std::max(hs, 1), (cuuint64_t)n};
  const cuuint64_t strides[3] = {(cuuint64_t)s * c * 2, (cuuint64_t)s * w * c * 2, (cuuint64_t)h * w * c * 2};
  const cuuint32_t box[4] = {32, (cuuint32_t)bx, (cuuint32_t)by, (cuuint32_t)bn};
  return encode_map(m, "output", 4, (char*)base + ((size_t)py * w + px) * c * 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B,
                    CU_TENSOR_MAP_L2_PROMOTION_NONE);
}

static int make_weight_map(CUtensorMap* m, const void* base, long long rows, int k, int box_rows) {
  const cuuint64_t dims[2] = {(cuuint64_t)k, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)k * 2};
  const cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  return encode_map(m, "weights", 2, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
}

static int ilog2(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}

// choose a {TW,TH,TN} box of `pixels` (power of two) GEMM rows minimising padded work
static void choose_box(int gw, int gh, int gn, int pixels, int* TW, int* TH, int* TN) {
  double best = 1e30;
  int bw = 1, bh = 1;
  for (int tw = 1; tw <= pixels; tw *= 2)
    for (int th = 1; tw * th <= pixels; th *= 2) {
      int tn = pixels / (tw * th);
      if (tw > 256 || th > 256 || tn > 256) continue;
      double padded = (double)cdiv(gw, tw) * tw * (double)cdiv(gh, th) * th * (double)cdiv(gn, tn) * tn;
      double score = padded - 1e-3 * tw - 1e-6 * th;   // ties: prefer wide boxes (longer contiguous runs)
      if (score < best) { best = score; bw = tw; bh = th; }
    }
  *TW = bw; *TH = bh; *TN = pixels / (bw * bh);
}

// what the forward / dgrad and the weight-gradient kernels both need: bf16 activations, stride 1 or 2, a square kernel of at
// most 16 taps, even fine grids at stride 2 (parity maps / scatter phases), and the tensor-map encoder
static bool tc_common_supported(const VgConvDesc* d) {
  if (g_force_simt) return false;
  if (d->act_dtype != VG_BF16) return false;
  if (d->stride != 1 && d->stride != 2) return false;
  if (d->kh != d->kw || d->kh * d->kw > 16) return false;
  if (d->stride == 2 && ((d->transposed ? d->h_out : d->h_in) % 2 != 0 || (d->transposed ? d->w_out : d->w_in) % 2 != 0)) return false;
  return get_encode() != nullptr;
}

bool tc_conv_supported(const VgConvDesc* d, bool dgrad) {
  const int c_red = dgrad ? d->c_out : d->c_in;
  const int n_out = dgrad ? d->c_in : d->c_out;
  // n_out == 1: the N tile is filled with the neighbouring taps' weight rows (finite garbage) and only
  // column 0 is stored - the reduction over 64+ input channels still runs on the tensor cores
  return c_red % 64 == 0 && (n_out % 64 == 0 || n_out == 1) && tc_common_supported(d);
}

bool tc_wgrad_supported(const VgConvDesc* d) {
  return d->c_in % 64 == 0 && d->c_out % 64 == 0 && tc_common_supported(d);
}

// Launches one kernel instance with `smem` bytes of dynamic shared memory; the first launch of the instance raises its
// shared-memory limit (once: autograd worker threads call in concurrently).
template <auto Kernel, class... Args>
static int launch(dim3 grid, int threads, int smem, cudaStream_t s, const Args&... args) {
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [smem] { attr_err = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); });
  VG_CUDA(attr_err);
  vg::Launch(grid, threads, smem, s)(Kernel, args...);
  VG_LAUNCHED();
  return VG_OK;
}

// Build the tap table(s).  `gather` : out grid coarse (or same), input fine via parity maps when
// stride 2.  `scatter`: out grid fine, decomposed into s*s phases over the coarse input grid.
// flip=false: weight slab index = ky*kw+kx.
static void build_gather_taps(TcPhase* ph, int k, int stride, int pad, int n_out) {
  ph->ntaps = 0; ph->oy_off = 0; ph->ox_off = 0;
  for (int ky = 0; ky < k; ++ky)
    for (int kx = 0; kx < k; ++kx) {
      TcTap& t = ph->taps[ph->ntaps++];
      const int ty = ky - pad, tx = kx - pad;
      if (stride == 1) {
        t.map = 0; t.dy = (int8_t)ty; t.dx = (int8_t)tx;
      } else {
        const int py = ((ty % 2) + 2) % 2, px = ((tx % 2) + 2) % 2;
        t.map = (int8_t)(py * 2 + px);
        t.dy = (int8_t)((ty - py) / 2);
        t.dx = (int8_t)((tx - px) / 2);
      }
      t.pad_ = 0;
      t.wrow = (ky * k + kx) * n_out;
    }
}
static void build_scatter_phase(TcPhase* ph, int k, int stride, int pad, int n_out, int phy, int phx) {
  ph->ntaps = 0; ph->oy_off = phy; ph->ox_off = phx;
  for (int ky = 0; ky < k; ++ky) {
    if (((phy + pad - ky) % stride + stride) % stride != 0) continue;
    for (int kx = 0; kx < k; ++kx) {
      if (((phx + pad - kx) % stride + stride) % stride != 0) continue;
      TcTap& t = ph->taps[ph->ntaps++];
      t.map = 0;
      // input index = q + (ph + pad - k)/stride (exact division, may be negative)
      t.dy = (int8_t)((phy + pad - ky) / stride);
      t.dx = (int8_t)((phx + pad - kx) / stride);
      t.pad_ = 0;
      t.wrow = (ky * k + kx) * n_out;
    }
  }
}

// ---- tile table (SURVEY.md section 8f N4): per (layer shape, batch, direction) the N tile and the kernel form that an
// autotune run measured fastest (vae_gan_b200/tune.py fills it through vg_conv_tune_set; vae_gan_b200/tile_table.json is the
// table measured on B200 for the BASELINE configurations).  Shapes without an entry use the heuristics below.
enum TuneForm { kFormAuto = 0, kFormOneShot = 1, kFormPersist = 2, kFormPair = 3 };
using TuneKey = std::array<int, 10>;   // dgrad, n, h_in, w_in, c_in, c_out, k, stride, pad, transposed
struct TuneVal { int bn, form; };
static std::map<TuneKey, TuneVal> g_tune;
static std::vector<TuneKey> g_tune_seen;
static bool g_tune_record = false;
static std::mutex g_tune_mu;
static TuneKey tune_key(const VgConvDesc* d, bool dgrad) {
  return TuneKey{dgrad ? 1 : 0, d->n, d->h_in, d->w_in, d->c_in, d->c_out, d->kh, d->stride, d->pad, d->transposed ? 1 : 0};
}
static TuneVal tune_lookup(const VgConvDesc* d, bool dgrad) {
  std::lock_guard<std::mutex> lk(g_tune_mu);
  const TuneKey k = tune_key(d, dgrad);
  if (g_tune_record && std::find(g_tune_seen.begin(), g_tune_seen.end(), k) == g_tune_seen.end()) g_tune_seen.push_back(k);
  auto it = g_tune.find(k);
  return it == g_tune.end() ? TuneVal{0, kFormAuto} : it->second;
}
int tc_tune_set(const VgConvDesc* d, int dgrad, int bn, int form) {
  VG_CHECK_ARG(d != nullptr, "null descriptor");
  VG_CHECK_ARG(bn == 0 || bn == 64 || bn == 128 || bn == 256, "N tile must be 0 (heuristic), 64, 128 or 256 (got %d)", bn);
  VG_CHECK_ARG(form >= kFormAuto && form <= kFormPair, "kernel form must be 0..3 (got %d)", form);
  std::lock_guard<std::mutex> lk(g_tune_mu);
  if (bn == 0 && form == kFormAuto) g_tune.erase(tune_key(d, dgrad != 0));
  else g_tune[tune_key(d, dgrad != 0)] = TuneVal{bn, form};
  return VG_OK;
}
void tc_tune_clear() {
  std::lock_guard<std::mutex> lk(g_tune_mu);
  g_tune.clear();
}
void tc_tune_record(int on) {
  std::lock_guard<std::mutex> lk(g_tune_mu);
  g_tune_record = on != 0;
  if (on) g_tune_seen.clear();
}
int tc_tune_seen(int* keys, int max_keys) {
  std::lock_guard<std::mutex> lk(g_tune_mu);
  const int n = (int)std::min<size_t>(g_tune_seen.size(), (size_t)std::max(0, max_keys));
  for (int i = 0; i < n && keys != nullptr; ++i)
    for (int j = 0; j < 10; ++j) keys[i * 10 + j] = g_tune_seen[i][j];
  return (int)g_tune_seen.size();
}

static int pick_bn(int n_out) {
  if (n_out % 256 == 0) return 256;
  if (n_out % 128 == 0) return 128;
  return 64;
}

// kernel-form heuristic of tc_conv_run (a tile-table form overrides it)
constexpr int kPersistMinItemsPerSm64 = 6;   // 64-wide tiles go persistent from this many work items per SM on
constexpr int kPairMinBN = 128;              // CTA pairs for 128- and 256-wide tiles; 64-wide tiles gain nothing (DESIGN.md 3.1)

// persistent forms: (n_groups x N tiles x phases | k-splits) work items over at most one CTA per SM (CTAS = 2: one pair per
// two SMs; the caller checked grid.x % (2 * MT) == 0)
template <int CTAS, int BN, int MT, int STAGES, int EW, bool INF>
static int launch_persistent(const TcConvParams& p, dim3 grid, cudaStream_t s) {
  const int n_groups = (int)cdiv(grid.x, CTAS * MT);
  const int n_work = (int)((long long)n_groups * grid.y * grid.z);
  const int ctas = CTAS * std::min(n_work, num_sms() / CTAS);
  const int threads = 128 + 32 * EW, smem = ConvPersistSmem<CTAS, BN, MT, STAGES, EW>::kBytes;
  if constexpr (CTAS == 2)
    return launch<tc_conv_pair_kernel<BN, MT, STAGES, EW, INF>>(ctas, threads, smem, s, p, (int)grid.y, n_groups, n_work);
  else
    return launch<tc_conv_persist_kernel<BN, MT, STAGES, EW, INF>>(ctas, threads, smem, s, p, (int)grid.y, n_groups, n_work);
}

// the kernel instance of each (form, N tile).  The inference epilogue (activation / residual / second output) lives in its
// OWN instantiations (INF): compiled into the training kernels it cost them 12 % (b256 step 59.8 -> 67.3 ms: registers at
// the launch-bound cap, spills in the epilogue).
// 64-wide tiles are EPILOGUE-bound (9 k-blocks of N=64 MMAs per 128 x 64 outputs).  Eight epilogue warps instead of four
// (<64,2,4,8>) measured NO gain on B200 (64->64 @96: 74.4 vs 74.9 us) and were removed: the bound was the store path
// (32 lines per store instruction), addressed by the staged, coalesced stores of epilogue_chunk.
template <bool INF>
static int launch_conv(int form, int BN, const TcConvParams& p, dim3 grid, cudaStream_t s) {
  switch (form * 1000 + BN) {
    case kFormOneShot * 1000 + 64: return launch<tc_conv_kernel<64, 4, INF>>(grid, kTcThreads, ConvSmem<64, 4>::kBytes, s, p);
    case kFormOneShot * 1000 + 128: return launch<tc_conv_kernel<128, 3, INF>>(grid, kTcThreads, ConvSmem<128, 3>::kBytes, s, p);
    case kFormOneShot * 1000 + 256: return launch<tc_conv_kernel<256, 4, INF>>(grid, kTcThreads, ConvSmem<256, 4>::kBytes, s, p);
    case kFormPersist * 1000 + 64: return launch_persistent<1, 64, 4, 3, 4, INF>(p, grid, s);
    case kFormPersist * 1000 + 128: return launch_persistent<1, 128, 2, 4, 8, INF>(p, grid, s);
    case kFormPersist * 1000 + 256: return launch_persistent<1, 256, 1, 4, 8, INF>(p, grid, s);
    case kFormPair * 1000 + 64: return launch_persistent<2, 64, 4, 3, 4, INF>(p, grid, s);
    case kFormPair * 1000 + 128: return launch_persistent<2, 128, 2, 4, 8, INF>(p, grid, s);
    case kFormPair * 1000 + 256: return launch_persistent<2, 256, 1, 6, 8, INF>(p, grid, s);
    default: set_error("unsupported BN %d", BN); return VG_EUNSUPPORTED;
  }
}

// dgrad=false: y = conv(x).  dgrad=true: dx from dy.  `in` is the tensor being read.
int tc_conv_run(const VgConvDesc* d, bool dgrad, const void* in, const void* wpack, const float* bias, const float* colscale,
                const float* sigma, int sigma_group_n, void* out, int out_dtype, cudaStream_t s, const VgConvEpilogue* ep) {
  TcConvParams p;
  memset(&p, 0, sizeof(p));
  // pattern: which side is the coarse grid
  //   Conv2d fwd           : gather  (in = x fine, out = y coarse)
  //   Conv2d dgrad         : scatter (in = dy coarse, out = dx fine)
  //   ConvTranspose2d fwd  : scatter (in = x coarse, out = y fine)
  //   ConvTranspose2d dgrad: gather  (in = dy fine, out = dx coarse)
  const bool gather = (d->transposed != 0) == dgrad;
  const int in_h = dgrad ? d->h_out : d->h_in, in_w = dgrad ? d->w_out : d->w_in, in_c = dgrad ? d->c_out : d->c_in;
  const int out_h = dgrad ? d->h_in : d->h_out, out_w = dgrad ? d->w_in : d->w_out, n_out = dgrad ? d->c_in : d->c_out;
  const int k = d->kh, st = d->stride, pad = d->pad;
  p.k_chunks = in_c / 64;
  p.n_out = n_out;
  p.OH = out_h; p.OW = out_w;
  p.out = out; p.out_f32 = out_dtype == VG_F32;
  p.bias = bias; p.colscale = colscale;
  p.sigma = sigma; p.sigma_group_n = sigma_group_n;
  p.act_slope = 1.0f; p.post_slope = 1.0f;
  if (ep != nullptr) {
    p.act_slope = ep->act_slope; p.residual = ep->residual; p.out2 = ep->y2;
    p.post_scale = ep->post_scale; p.post_shift = ep->post_shift; p.post_slope = ep->post_slope;
  }
  int nphase = 1;
  if (gather) {
    p.gw = out_w; p.gh = out_h; p.gn = d->n; p.os = 1;
    build_gather_taps(&p.phases[0], k, st, pad, n_out);
  } else {
    p.os = st;
    nphase = st * st;
    p.gw = (out_w + st - 1) / st; p.gh = (out_h + st - 1) / st; p.gn = d->n;
    for (int phy = 0; phy < st; ++phy)
      for (int phx = 0; phx < st; ++phx) build_scatter_phase(&p.phases[phy * st + phx], k, st, pad, n_out, phy, phx);
  }
  choose_box(p.gw, p.gh, p.gn, 128, &p.TW, &p.TH, &p.TN);
  p.tw_log2 = ilog2(p.TW); p.th_log2 = ilog2(p.TH);
  p.tiles_x = (int)cdiv(p.gw, p.TW); p.tiles_y = (int)cdiv(p.gh, p.TH); p.tiles_n = (int)cdiv(p.gn, p.TN);
  int rc;
  if (gather && st == 2) {
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px)
        if ((rc = make_act_map(&p.in_maps[py * 2 + px], in, d->n, in_h, in_w, in_c, 2, py, px, p.TW, p.TH, p.TN))) return rc;
  } else {
    if ((rc = make_act_map(&p.in_maps[0], in, d->n, in_h, in_w, in_c, 1, 0, 0, p.TW, p.TH, p.TN))) return rc;
    p.in_maps[1] = p.in_maps[2] = p.in_maps[3] = p.in_maps[0];
  }
  const TuneVal tuned = tune_lookup(d, dgrad);
  const int BN = (n_out == 1) ? 64 : ((tuned.bn != 0 && n_out % tuned.bn == 0) ? tuned.bn : pick_bn(n_out));
  p.n_store = (n_out == 1) ? 1 : BN;
  if ((rc = make_weight_map(&p.w_map, wpack, (long long)k * k * n_out, in_c, BN))) return rc;
  dim3 grid((unsigned)(p.tiles_x * p.tiles_y * p.tiles_n), (unsigned)std::max(1, n_out / BN), (unsigned)nphase);
  if (grid.x == 0) return VG_OK;
  if (ep != nullptr && (ep->act_slope != 1.0f || ep->residual != nullptr || ep->y2 != nullptr) && (p.out_f32 || p.n_store == 1)) {
    set_error("the activation / residual / second-output epilogue needs a bf16 output with c_out %% 64 == 0");
    return VG_EUNSUPPORTED;
  }
  p.ksplit = 1;
  p.k_per_split = p.phases[0].ntaps * p.k_chunks;
  {
    // few output tiles but a long reduction (the discriminator's Linear layers run here as 1x1
    // convolutions on [B,1,1,C] tensors): split K over blockIdx.z, fp32 atomics into a zeroed output
    const long long ctas = (long long)grid.x * grid.y;
    const int total_kb = p.phases[0].ntaps * p.k_chunks;
    if (nphase == 1 && p.out_f32 && colscale == nullptr && ctas * 2 <= num_sms() && total_kb >= 16) {
      int ks = (int)std::min<long long>(cdiv(2LL * num_sms(), ctas), total_kb / 4);
      if (ks > 1) {
        p.k_per_split = (int)cdiv(total_kb, ks);
        p.ksplit = (int)cdiv(total_kb, p.k_per_split);
        grid.z = (unsigned)p.ksplit;
        const size_t out_elems = (size_t)d->n * out_h * out_w * n_out;
        VG_CUDA(cudaMemsetAsync(out, 0, out_elems * sizeof(float), s));
        if (g_det.on) {
          // deterministic mode: every split stores its partial tile into its own scratch slab and ordered_reduce_f32 adds
          // the slabs in split order (below); if the caller's scratch is too small the splits take turns instead
          if ((size_t)p.ksplit * out_elems * sizeof(float) <= g_det.scratch_bytes) {
            p.out = g_det.scratch;
            p.det_split_stride = (long long)out_elems;
          } else if (!(p.det_locks = det_locks(ctas))) {
            return VG_EINVAL;
          }
        }
      }
    }
  }
  // kernel variant: persistent CTAs (double-buffered accumulator, MT pixel tiles share each staged weight
  // tile) when there is enough work; one-shot CTAs (two resident per SM) for small problems and split-K.
  // Measured on B200 (scripts/sweep_conv.py): a persistent single-tile CTA loses to two co-resident
  // one-shot CTAs, and one-shot CTAs of two pixel tiles (no double-buffered accumulator) were slower still
  // (128->128 @96: 897 -> 769 TFLOP/s) and were removed.
  // TMA-store epilogue (VG_TC_TMA_STORE, default 2): bf16 outputs without split-K and without the inference epilogue leave
  // the staging buffers as cp.async.bulk.tensor stores - 1: gather-type launches only (output on the GEMM's own pixel grid),
  // 2: also the scatter launches (one strided output map per phase), 0: the manual coalesced stores.  Measured on B200
  // (profiles/r2_tma_store_ab.txt): 60.2 -> 59.2 ms/step at batch 256, 10.58 -> 10.36 at 32; 64->64 @96 74 -> 67 us,
  // 64->128 @96 110 -> 97 us, 1x1 stride-2 51 -> 43 us; the scatter phases add another 0.3 %.
  static int tma_store = -1;
  if (tma_store < 0) { const char* e = getenv("VG_TC_TMA_STORE"); tma_store = e ? atoi(e) : 2; }
  if (tma_store && !p.out_f32 && p.ksplit == 1 && p.n_store != 1 && (p.os == 1 || tma_store >= 2) &&
      p.act_slope == 1.0f && p.residual == nullptr && p.out2 == nullptr) {
    const int bx = std::min(p.TW, 32), by = std::min(p.TH, 32 / bx), bn = 32 / (bx * by);
    // a scatter launch (ConvTranspose2d forward, stride-2 dgrad) writes st x st interleaved sub-grids, one per phase (grid.z)
    for (int ph = 0; ph < nphase; ++ph)
      if ((rc = make_out_map(&p.out_maps[ph], out, d->n, out_h, out_w, n_out, bx, by, bn, p.os, p.phases[ph].oy_off, p.phases[ph].ox_off)))
        return rc;
    p.tma_store = 1;
  }
  const long long ctas1 = (long long)grid.x * grid.y * grid.z;
  // 256-wide tiles go persistent as soon as there is more than one work item per SM (288 tiles of the 24x24 layers at
  // batch 64 ran as one-shot CTAs without epilogue overlap: 38-85 us for 31 us of tensor work)
  const bool heur_persist = !(g_det.on && p.ksplit > 1) &&       // deterministic split-K: the one-shot kernel takes turns
                            ((BN == 256 && ctas1 > (long long)num_sms()) ||
                             // 128-wide: the CTA-pair kernel (1000+ TFLOP/s) from two work items per pair on; below 6 x SMs tiles
                             // these layers ran as one-shot CTAs (G 128->128 @48 at 32 images: 496 TFLOP/s)
                             (BN == 128 && ctas1 >= 2LL * num_sms()) ||
                             (BN == 64 && ctas1 >= (long long)kPersistMinItemsPerSm64 * num_sms()));
  // a tile-table entry overrides the form (split-K launches keep the heuristic: only the one-shot kernel was tuned for them)
  const int form = p.ksplit > 1 ? kFormAuto : tuned.form;
  const bool use_persist = form == kFormAuto ? heur_persist : (form != kFormOneShot);
  // CTA pairs (cta_group::2) halve the per-SM shared-memory operand reads that bound the narrow tiles
  int run_form = use_persist ? kFormPersist : kFormOneShot;
  if (use_persist && p.n_store != 1 && (form == kFormPair || (form == kFormAuto && BN >= kPairMinBN))) {
    const int mt = BN == 64 ? 4 : (BN == 128 ? 2 : 1);
    if (grid.x % (2 * mt) == 0) {
      if ((rc = make_weight_map(&p.w_map, wpack, (long long)k * k * n_out, in_c, BN / 2))) return rc;
      run_form = kFormPair;
    }
  }
  const bool inf = p.act_slope != 1.0f || p.residual != nullptr || p.out2 != nullptr;
  rc = inf ? launch_conv<true>(run_form, BN, p, grid, s) : launch_conv<false>(run_form, BN, p, grid, s);
  if (rc == VG_OK && p.det_split_stride != 0)
    rc = ordered_reduce_f32((const float*)p.out, p.ksplit, p.det_split_stride, (float*)out, s);
  return rc;
}

// acc_only: leave the result in `workspace` - packed [tap][c_s][c_u] for k > 1, torch layout [c_u][c_s] for k = 1 (the
// caller zeroed it and consumes it itself: vg_conv_wgrad_sn) - instead of adding it into dw
int tc_wgrad_run(const VgConvDesc* d, const void* x, const void* dy, float* dw, float* workspace, cudaStream_t s, bool acc_only) {
  TcWgradParams p;
  memset(&p, 0, sizeof(p));
  // dw[cu][cs][tap] += sum_q U[q][cu] * S[q*stride - pad + k][cs]
  const void *U, *S;
  int hu, wu, cu, hs, ws, cs;
  if (!d->transposed) { U = dy; hu = d->h_out; wu = d->w_out; cu = d->c_out; S = x; hs = d->h_in; ws = d->w_in; cs = d->c_in; }
  else                { U = x;  hu = d->h_in;  wu = d->w_in;  cu = d->c_in;  S = dy; hs = d->h_out; ws = d->w_out; cs = d->c_out; }
  const int k = d->kh, st = d->stride, pad = d->pad;
  TcPhase tmp;
  build_gather_taps(&tmp, k, st, pad, 0);
  p.ntaps = tmp.ntaps;
  for (int i = 0; i < tmp.ntaps; ++i) p.taps[i] = tmp.taps[i];
  p.cs_chunks = cs / 64; p.cs = cs; p.cu = cu;
  choose_box(wu, hu, d->n, 64, &p.TW, &p.TH, &p.TN);
  p.tiles_x = (int)cdiv(wu, p.TW); p.tiles_y = (int)cdiv(hu, p.TH); p.tiles_n = (int)cdiv(d->n, p.TN);
  p.n_boxes = p.tiles_x * p.tiles_y * p.tiles_n;
  // 1x1 convolutions / Linear layers: torch layout [c_u][c_s] already has c_s contiguous, so the epilogue's per-lane
  // reductions are coalesced (32 lanes = 32 consecutive c_s) and the scratch + memset + unpack round trip is skipped
  p.packed = workspace != nullptr && tmp.ntaps > 1;
  p.dw = (p.packed || acc_only) ? workspace : dw;
  const size_t welems = (size_t)k * k * cs * cu;
  if (p.packed && !acc_only) VG_CUDA(cudaMemsetAsync(workspace, 0, welems * sizeof(float), s));
  int rc;
  if (st == 2) {
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px)
        if ((rc = make_act_map(&p.s_maps[py * 2 + px], S, d->n, hs, ws, cs, 2, py, px, p.TW, p.TH, p.TN))) return rc;
  } else {
    if ((rc = make_act_map(&p.s_maps[0], S, d->n, hs, ws, cs, 1, 0, 0, p.TW, p.TH, p.TN))) return rc;
    p.s_maps[1] = p.s_maps[2] = p.s_maps[3] = p.s_maps[0];
  }
  if ((rc = make_act_map(&p.u_map, U, d->n, hu, wu, cu, 1, 0, 0, p.TW, p.TH, p.TN))) return rc;
  const int NB = (cu % 256 == 0) ? 4 : ((cu % 128 == 0) ? 2 : 1);
  const int m_tiles = (p.ntaps * p.cs_chunks + 1) / 2;
  const int n_tiles = cu / (NB * 64);
  if (p.n_boxes == 0) return VG_OK;
  // one CTA per SM (160-192 KB of smem): pick the split count that fills whole waves
  const long long tiles = (long long)m_tiles * n_tiles;
  long long splits = 1;
  {
    double best = -1.0;
    const long long max_splits = std::max<long long>(1, p.n_boxes / 4);
    for (long long waves = 1; waves <= 4; ++waves) {
      long long sp = std::max<long long>(1, std::min<long long>((waves * num_sms()) / tiles, max_splits));
      long long bps = cdiv(p.n_boxes, sp);
      sp = cdiv(p.n_boxes, bps);
      const long long ctas = tiles * sp;
      const double eff = (double)ctas / (double)(cdiv(ctas, num_sms()) * num_sms());   // wave quantisation
      const double score = eff - 0.02 * (double)sp / (double)max_splits - (ctas < num_sms() ? 0.5 : 0.0);
      if (score > best) { best = score; splits = sp; }
    }
  }
  p.boxes_per_split = (int)cdiv(p.n_boxes, splits);
  splits = cdiv(p.n_boxes, p.boxes_per_split);
  dim3 grid((unsigned)m_tiles, (unsigned)n_tiles, (unsigned)splits);
  float* const wgrad_dst = p.dw;
  if (g_det.on && splits > 1) {
    // deterministic mode: per-split scratch slabs + ordered reduce (see the forward's split-K), turn-taking as the fallback
    if ((size_t)splits * welems * sizeof(float) <= g_det.scratch_bytes) {
      p.dw = (float*)g_det.scratch;
      p.det_split_stride = (long long)welems;
    } else if (!(p.det_locks = det_locks(tiles))) {
      return VG_EINVAL;
    }
  }
  switch (NB) {
    case 1: rc = launch<tc_wgrad_kernel<1, 6>>(grid, kTcThreads, WgradSmem<1, 6>::kBytes, s, p); break;
    case 2: rc = launch<tc_wgrad_kernel<2, 5>>(grid, kTcThreads, WgradSmem<2, 5>::kBytes, s, p); break;
    default: rc = launch<tc_wgrad_kernel<4, 4>>(grid, kTcThreads, WgradSmem<4, 4>::kBytes, s, p); break;
  }
  if (rc == VG_OK && p.det_split_stride != 0) rc = ordered_reduce_f32(p.dw, (int)splits, p.det_split_stride, wgrad_dst, s);
  if (rc || !p.packed || acc_only) return rc;
  dim3 ug((unsigned)cdiv((long long)cs * p.ntaps, 32), (unsigned)cdiv(cu, 32));
  vg::Launch(ug, 256, 0, s)(wgrad_unpack_kernel, workspace, cu, cs, p.ntaps, dw);
  VG_LAUNCHED();
  return VG_OK;
}

}  // namespace vg
