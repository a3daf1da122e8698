// BatchNorm2d-family STREAMING kernels (round 2): the memory-bound passes of the step - statistics,
// BN + LeakyReLU + dropout apply, backward reduce / apply, residual add - as persistent CTAs fed by a
// bulk-copy (TMA, cp.async.bulk) pipeline.  Replaces nn.BatchNorm2d / nn.LeakyReLU / nn.Dropout /
// `out += shortcut(x)` of the reference (README.md:143-197, 376-419, 442, 466-468).
//
// Why: the register-staged kernels of bn.cu keep only 16-32 KB of loads in flight per SM (one 256-thread
// block of 116-147 registers per SM), while HBM3e at 6.5 TB/s needs ~40 KB per SM in flight: they measured
// 64-81 % of the copy bandwidth.  Here ONE producer warp issues 8-16 KB bulk copies per input stream into a
// 3-4 stage shared-memory ring (full/empty mbarriers, 64-96 KB per CTA, two CTAs per SM), so the bytes in
// flight no longer depend on registers or occupancy; eight consumer warps read the staged tile with
// conflict-free 16-byte shared loads, do the arithmetic in fp32 and store 16 B per thread, coalesced.
//
// Work decomposition: the NHWC tensor is a flat array of "vectors" (8 consecutive channels = 16 B of bf16).
// A tile is KT * tpb consecutive vectors, tpb = (256 / cg) * cg, cg = C / 8, so consumer thread `tid` always
// owns channel group tid % cg and keeps that group's per-channel constants in registers for its whole life.
//
// Folded-in small kernels (each was a separate 3-5 us launch, ~130 per training step):
//   * finalize: the consumers derive (mean, rstd) themselves from the fp64 sums (or from the running
//     statistics in eval mode); block 0 also writes mean_rstd for the backward and updates the running
//     statistics (torch semantics: momentum, unbiased variance);
//   * parameter gradients: block 0 of the backward-apply adds dgamma / dbeta from the sums.
#include <algorithm>
#include <mutex>
#include "vg_common.cuh"
#include "sm100_ptx.cuh"

namespace vg {

namespace bs {

constexpr int kConsumers = 256;
constexpr int kThreads = kConsumers + 32;      // + one producer warp

enum Mode { kStats = 0, kFwd = 1, kBwdReduce = 2, kBwdApply = 3, kBwdApplyAdd = 4, kAdd = 5, kAddStats = 6, kAddDual = 7 };

// how a kernel obtains (mean, rstd) of one BatchNorm: kind -1 none (identity), 0 read mean_rstd, 1 finalize
// from the fp64 sums (training), 2 from the running statistics (eval)
struct Chan {
  const float* mean_rstd;
  const double* sums;
  const float* gamma;
  const float* beta;
  float* running_mean;
  float* running_var;
  float* mean_rstd_out;
  double count;
  float eps, momentum;
  int kind;
};

struct Args {
  const void* in0;
  const void* in1;
  const void* in2;
  void* out;
  long long nvec;        // total 8-element vectors
  long long ntiles;
  int c;                 // channels of the tensor (1 when folded)
  int cg;                // channel groups per row (c / 8; 1 when folded)
  int tpb;               // consumer threads in use = (256 / cg) * cg
  int fold;              // single-channel tensor viewed as [rows / 8][8]
  // L2 reuse between consecutive passes over the same tensor: a producer (convolution, previous pass) leaves the END of
  // the tensor it wrote / read last in the 126 MB L2.  The reduction-type passes (statistics, backward reduce, residual
  // add) therefore walk the tensor backwards (reverse = 1) - they start on the freshest lines - and the apply passes that
  // follow them walk forwards, starting on what the reduction touched last.
  int reverse;
  int hw;
  Chan A, B;
  // reductions
  double* sums_out;
  double* partials;      // deterministic mode: per-block partial sums [grid][2 * c] instead of atomics on sums_out
  // backward apply
  const double* sums_in;
  double count;
  const float* out_colscale;
  float* dgamma;
  float* dbeta;
  float param_scale;
  // kAddDual (eval / sampling path): second output = leaky_relu(post_scale[c] * out + post_shift[c], post_slope)
  void* out2;
  const float* post_scale;
  const float* post_shift;
  float post_slope;
  // activation / dropout
  float slope, drop_scale;
  uint32_t thr16;
  unsigned long long seed, offset;
  const unsigned long long* step_ptr;
  unsigned long long vbase;     // Philox block index of vector 0 = sample_offset * hw * c / 8
  int training;
};

template <int MODE> struct ModeTraits {
  static constexpr int NIN = (MODE == kStats || MODE == kFwd) ? 1 : (MODE == kBwdApplyAdd ? 3 : 2);
  static constexpr bool kReduce = MODE == kStats || MODE == kBwdReduce || MODE == kAddStats;
  static constexpr bool kStore = MODE == kFwd || MODE == kBwdApply || MODE == kBwdApplyAdd || MODE == kAdd || MODE == kAddStats || MODE == kAddDual;
};

template <typename T, int MODE> struct Geo {
  static constexpr int NIN = ModeTraits<MODE>::NIN;
  static constexpr int VB = 8 * (int)sizeof(T);                                 // bytes per vector
  static constexpr int KT = ((sizeof(T) == 2) ? 4 : 2) / (NIN == 3 ? 2 : 1);     // vectors per thread per tile
  static constexpr int ST = (NIN == 2) ? 3 : 4;                                  // pipeline stages
  static constexpr int kInBytes = KT * kConsumers * VB;                          // one input stream of one stage
  static constexpr int kStageBytes = NIN * kInBytes;
  static constexpr int kRingBytes = ST * kStageBytes;
  static constexpr int kSmemBytes = kRingBytes + 2 * ST * 8 + 128;               // + barriers + alignment slack
  static_assert(kRingBytes >= 2 * 8 * kConsumers * 4, "the reduction scratch reuses the ring");
};

__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(ptx::smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(ptx::smem_u32(bar))
               : "memory");
}
// barrier over the 256 consumer threads only (the producer warp runs its own loop)
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

__device__ __forceinline__ void chan_stats(const Chan& ch, int c, int idx, float& mean, float& rstd) {
  if (ch.kind == 1) {
    const double m = ch.sums[idx] / ch.count;
    double var = ch.sums[c + idx] / ch.count - m * m;
    if (var < 0.0) var = 0.0;
    mean = (float)m;
    rstd = (float)(1.0 / sqrt(var + (double)ch.eps));
  } else if (ch.kind == 2) {
    mean = ch.running_mean[idx];
    rstd = (float)(1.0 / sqrt((double)ch.running_var[idx] + (double)ch.eps));
  } else {
    mean = ch.mean_rstd[idx];
    rstd = ch.mean_rstd[c + idx];
  }
}

// executed by ONE thread per channel of block 0: what vg_bn_finalize / vg_bn_eval_stats did in their own launch
__device__ __forceinline__ void chan_side_effects(const Chan& ch, int c, int idx) {
  if (ch.kind == 1) {
    const double m = ch.sums[idx] / ch.count;
    double var = ch.sums[c + idx] / ch.count - m * m;
    if (var < 0.0) var = 0.0;
    if (ch.mean_rstd_out != nullptr) {
      ch.mean_rstd_out[idx] = (float)m;
      ch.mean_rstd_out[c + idx] = (float)(1.0 / sqrt(var + (double)ch.eps));
    }
    if (ch.running_mean != nullptr) {
      const double unbiased = ch.count > 1.0 ? var * ch.count / (ch.count - 1.0) : var;
      ch.running_mean[idx] = (float)((1.0 - ch.momentum) * (double)ch.running_mean[idx] + ch.momentum * m);
      ch.running_var[idx] = (float)((1.0 - ch.momentum) * (double)ch.running_var[idx] + ch.momentum * unbiased);
    }
  } else if (ch.kind == 2 && ch.mean_rstd_out != nullptr) {
    ch.mean_rstd_out[idx] = ch.running_mean[idx];
    ch.mean_rstd_out[c + idx] = (float)(1.0 / sqrt((double)ch.running_var[idx] + (double)ch.eps));
  }
}

// 16-bit Philox keep decisions for the 8 elements of vector `vec` (same stream layout as bn.cu / the oracle)
__device__ __forceinline__ void keep8(const Philox& ph, unsigned long long vec, uint32_t thr16, bool keep[8]) {
  const uint4 r = ph.block(vec);
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    keep[2 * i] = (w[i] & 0xffffu) >= thr16;
    keep[2 * i + 1] = (w[i] >> 16) >= thr16;
  }
}

template <typename T, int MODE, bool DROP>
__global__ void __launch_bounds__(kThreads, 2) bn_stream_kernel(const __grid_constant__ Args a) {
  using G = Geo<T, MODE>;
  constexpr int NIN = G::NIN, VB = G::VB, KT = G::KT, ST = G::ST;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  uint8_t* ring = smem_raw + ((128u - (raw_addr & 127u)) & 127u);
  uint64_t* full = reinterpret_cast<uint64_t*>(ring + G::kRingBytes);
  uint64_t* empty = full + ST;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < ST; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], kConsumers / 32);
    }
    ptx::fence_barrier_init();
  }
  __syncthreads();
  vg::pdl_entry();   // the barrier set-up above overlaps the previous kernel's tail; everything below reads global memory

  const int tile_vecs = KT * a.tpb;

  if (warp == kConsumers / 32) {
    // ------------------------------ producer warp ------------------------------
    int stage = 0;
    uint32_t phase = 0;
    for (long long tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
      ptx::mbar_wait(&empty[stage], phase ^ 1u);
      if (ptx::elect_one()) {
        const long long v0 = (a.reverse ? a.ntiles - 1 - tile : tile) * tile_vecs;
        const long long nv = min((long long)tile_vecs, a.nvec - v0);
        const uint32_t bytes = (uint32_t)(nv * VB);
        ptx::mbar_arrive_expect_tx(&full[stage], bytes * NIN);
        uint8_t* dst = ring + (size_t)stage * G::kStageBytes;
        bulk_load(dst, reinterpret_cast<const uint8_t*>(a.in0) + v0 * VB, bytes, &full[stage]);
        if (NIN >= 2) bulk_load(dst + G::kInBytes, reinterpret_cast<const uint8_t*>(a.in1) + v0 * VB, bytes, &full[stage]);
        if (NIN >= 3) bulk_load(dst + 2 * G::kInBytes, reinterpret_cast<const uint8_t*>(a.in2) + v0 * VB, bytes, &full[stage]);
      }
      __syncwarp();
      if (++stage == ST) { stage = 0; phase ^= 1u; }
    }
    return;
  }

  // ------------------------------ consumer warps ------------------------------
  const bool active = tid < a.tpb;
  const int g = tid % a.cg;
  const int c = a.c;
  // per-channel constants of this thread's 8 channels
  float ca[8], cb[8];            // pre-activation = ca * x + cb   (BatchNorm A folded with its affine)
  float cm[8], cr[8];            // mean, rstd (reduce) | mean, c1 (apply) | scale, shift of operand B (add)
  float c0[8];                   // apply: -a * mean(g)
  float acc[2][8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { ca[j] = 1.f; cb[j] = 0.f; cm[j] = 0.f; cr[j] = 1.f; c0[j] = 0.f; acc[0][j] = 0.f; acc[1][j] = 0.f; }
  if (active && MODE != kStats) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int ch = a.fold ? 0 : g * 8 + j;
      if (a.A.kind >= 0) {
        float mean, rstd;
        chan_stats(a.A, c, ch, mean, rstd);
        const float aa = a.A.gamma[ch] * rstd;
        ca[j] = aa;
        cb[j] = a.A.beta[ch] - mean * aa;
        if (MODE == kBwdReduce) { cm[j] = mean; cr[j] = rstd; }
        if (MODE == kBwdApply || MODE == kBwdApplyAdd) {
          float k1 = 0.f, k2 = 0.f;
          if (a.training) {
            k1 = (float)(a.sums_in[ch] / a.count);
            k2 = (float)(a.sums_in[c + ch] / a.count);
          }
          cm[j] = mean;
          cr[j] = -aa * k2 * rstd;        // dx = a*g - a*k1 - a*k2*xhat = a*g + c0 + c1*(x - mean)
          c0[j] = -aa * k1;
        }
      }
      if (MODE == kAddDual) {
        c0[j] = a.post_scale[ch];               // (the add itself is plain: both operands identity)
        cm[j] = a.post_shift[ch];
      }
      if (MODE == kAdd || MODE == kAddStats) {
        if (a.B.kind >= 0) {
          float mean, rstd;
          chan_stats(a.B, c, ch, mean, rstd);
          const float bb = a.B.gamma[ch] * rstd;
          cm[j] = bb;
          cr[j] = a.B.beta[ch] - mean * bb;
        } else {
          cm[j] = 1.f;
          cr[j] = 0.f;
        }
      }
    }
  }
  // block 0: the side effects of the folded finalize / parameter-gradient kernels, one thread per channel
  if (blockIdx.x == 0 && active && (a.fold ? tid == 0 : tid < a.cg)) {
    const int nch = a.fold ? 1 : 8;
    for (int j = 0; j < nch; ++j) {
      const int ch = a.fold ? 0 : g * 8 + j;
      if (MODE == kFwd || MODE == kAdd || MODE == kAddStats) {
        if (a.A.kind >= 1) chan_side_effects(a.A, c, ch);
        if ((MODE == kAdd || MODE == kAddStats) && a.B.kind >= 1) chan_side_effects(a.B, c, ch);
      }
      if (MODE == kBwdApply || MODE == kBwdApplyAdd) {
        if (a.dbeta != nullptr && a.sums_in != nullptr) a.dbeta[ch] += (float)(a.sums_in[ch] * (double)a.param_scale);
        if (a.dgamma != nullptr && a.sums_in != nullptr) a.dgamma[ch] += (float)(a.sums_in[c + ch] * (double)a.param_scale);
      }
    }
  }

  unsigned long long eoff = a.offset;
  if (DROP && a.step_ptr != nullptr) eoff += 65536ull * (*a.step_ptr);
  const Philox ph(a.seed, eoff);
  const unsigned long long vbase = a.vbase;

  int stage = 0;
  uint32_t phase = 0;
  for (long long tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
    ptx::mbar_wait(&full[stage], phase);
    if (active) {
      const uint8_t* sb = ring + (size_t)stage * G::kStageBytes;
#pragma unroll
      for (int k = 0; k < KT; ++k) {
        const int lv = tid + k * a.tpb;
        const long long v = (a.reverse ? a.ntiles - 1 - tile : tile) * tile_vecs + lv;
        if (v < a.nvec) {
          Vec8<T> x0, x1;
          x0.load(reinterpret_cast<const T*>(sb + (size_t)lv * VB));
          if (NIN >= 2) x1.load(reinterpret_cast<const T*>(sb + G::kInBytes + (size_t)lv * VB));
          bool kp[8];
          if (DROP) keep8(ph, vbase + (unsigned long long)v, a.thr16, kp);
          if (MODE == kStats) {
#pragma unroll
            for (int j = 0; j < 8; ++j) { acc[0][j] += x0.v[j]; acc[1][j] = fmaf(x0.v[j], x0.v[j], acc[1][j]); }
          } else if (MODE == kFwd) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float t = fmaf(ca[j], x0.v[j], cb[j]);
              t = t > 0.f ? t : t * a.slope;
              if (DROP) t = kp[j] ? t * a.drop_scale : 0.f;
              x0.v[j] = t;
            }
            x0.store(reinterpret_cast<T*>(a.out) + v * 8);
          } else if (MODE == kBwdReduce) {
            // in0 = dy, in1 = x
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float pre = fmaf(ca[j], x1.v[j], cb[j]);
              float gg = x0.v[j] * (pre > 0.f ? 1.f : a.slope);
              if (DROP) gg = kp[j] ? gg * a.drop_scale : 0.f;
              const float xh = (x1.v[j] - cm[j]) * cr[j];
              acc[0][j] += gg;
              acc[1][j] = fmaf(gg, xh, acc[1][j]);
            }
          } else if (MODE == kBwdApply || MODE == kBwdApplyAdd) {
            // in0 = dy, in1 = x, in2 = addend
            float cs[8];
            if (a.out_colscale != nullptr) {
              const long long n = (v / a.cg) / a.hw;
              const float4* p = reinterpret_cast<const float4*>(a.out_colscale + n * c + g * 8);
              const float4 p0 = __ldg(p), p1 = __ldg(p + 1);
              cs[0] = p0.x; cs[1] = p0.y; cs[2] = p0.z; cs[3] = p0.w; cs[4] = p1.x; cs[5] = p1.y; cs[6] = p1.z; cs[7] = p1.w;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float pre = fmaf(ca[j], x1.v[j], cb[j]);
              float gg = x0.v[j] * (pre > 0.f ? 1.f : a.slope);
              if (DROP) gg = kp[j] ? gg * a.drop_scale : 0.f;
              float r = fmaf(cr[j], x1.v[j] - cm[j], fmaf(ca[j], gg, c0[j]));
              if (a.out_colscale != nullptr) r *= cs[j];
              x0.v[j] = r;
            }
            if (MODE == kBwdApplyAdd) {
              Vec8<T> ad;
              ad.load(reinterpret_cast<const T*>(sb + 2 * G::kInBytes + (size_t)lv * VB));
#pragma unroll
              for (int j = 0; j < 8; ++j) x0.v[j] += ad.v[j];
            }
            x0.store(reinterpret_cast<T*>(a.out) + v * 8);
          } else if (MODE == kAddDual) {
            // out = in0 + in1 ; out2 = lrelu(post_scale * out + post_shift) computed from out AS STORED
            Vec8<T> y2;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float t = x0.v[j] + x1.v[j];
              t = t > 0.f ? t : t * a.slope;
              x0.v[j] = t;
              const float r = sizeof(T) == 2 ? to_f32(from_f32<T>(t)) : t;
              float u = fmaf(c0[j], r, cm[j]);
              y2.v[j] = u > 0.f ? u : u * a.post_slope;
            }
            x0.store(reinterpret_cast<T*>(a.out) + v * 8);
            y2.store(reinterpret_cast<T*>(a.out2) + v * 8);
          } else {
            // kAdd / kAddStats: out = lrelu(bnA(in0) + bnB(in1))
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float t = fmaf(ca[j], x0.v[j], cb[j]) + fmaf(cm[j], x1.v[j], cr[j]);
              t = t > 0.f ? t : t * a.slope;
              x0.v[j] = t;
            }
            x0.store(reinterpret_cast<T*>(a.out) + v * 8);
            if (MODE == kAddStats) {
              // statistics of the values as STORED (bf16-rounded on the bf16 path)
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float r = sizeof(T) == 2 ? to_f32(from_f32<T>(x0.v[j])) : x0.v[j];
                acc[0][j] += r;
                acc[1][j] = fmaf(r, r, acc[1][j]);
              }
            }
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&empty[stage]);
    if (++stage == ST) { stage = 0; phase ^= 1u; }
  }

  if (ModeTraits<MODE>::kReduce) {
    // per-channel block reduction through the (now idle) ring, then one fp64 atomic per (block, channel, quantity)
    consumer_sync();
    float* red = reinterpret_cast<float*>(ring);        // [2 * 8][256]
#pragma unroll
    for (int q = 0; q < 2; ++q)
#pragma unroll
      for (int j = 0; j < 8; ++j) red[(q * 8 + j) * kConsumers + tid] = active ? acc[q][j] : 0.f;
    consumer_sync();
    if (a.fold) {
      // every (thread, lane) value belongs to channel 0
      for (int q = 0; q < 2; ++q) {
        double s = 0.0;
        for (int i = tid; i < 8 * kConsumers; i += kConsumers) s += (double)red[q * 8 * kConsumers + i];
        s = warp_sum(s);
        // fold: c == 1; the 8 consumer warps each own a slot in deterministic mode
        if (lane == 0) {
          if (a.partials) a.partials[((size_t)blockIdx.x * 2 + q) * (kConsumers / 32) + warp] = s;
          else atomicAdd(&a.sums_out[q * c], s);
        }
      }
    } else {
      const int rpb = a.tpb / a.cg;
      for (int idx = tid; idx < 2 * c; idx += kConsumers) {
        const int q = idx / c, ch = idx - q * c;
        const int gg = ch >> 3, j = ch & 7;
        double s = 0.0;
        for (int r = 0; r < rpb; ++r) s += (double)red[(q * 8 + j) * kConsumers + r * a.cg + gg];
        if (a.partials) a.partials[(size_t)blockIdx.x * 2 * c + idx] = s;
        else atomicAdd(&a.sums_out[q * c + ch], s);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
constexpr int kCtasPerSm = 2;

// folded (single-channel) tensors in deterministic mode: partials[block][q][warp] -> sums_out[q * c] (c == 1), one thread
// per quantity walking blocks and warps in order (a few thousand fp64 adds)
__global__ void ordered_reduce_fold_kernel(const double* __restrict__ partials, int nblocks, int c, double* __restrict__ out) {
  vg::pdl_entry();
  const int q = threadIdx.x;
  if (q >= 2) return;
  constexpr int W = kConsumers / 32;
  double s = 0.0;
  for (int b = 0; b < nblocks; ++b)
    for (int w = 0; w < W; ++w) s += partials[((size_t)b * 2 + q) * W + w];
  out[q * c] += s;
}
static int ordered_reduce_fold(const double* partials, int nblocks, double* out, int c, cudaStream_t s) {
  vg::Launch(1, 32, 0, s)(ordered_reduce_fold_kernel, partials, nblocks, c, out);
  VG_LAUNCHED();
  return VG_OK;
}

template <typename T, int MODE, bool DROP>
static int launch(const Args& a, cudaStream_t s) {
  using G = Geo<T, MODE>;
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [] {
    attr_err = cudaFuncSetAttribute(bn_stream_kernel<T, MODE, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, G::kSmemBytes);
  });
  VG_CUDA(attr_err);
  const long long cap = (long long)num_sms() * kCtasPerSm;
  const int grid = (int)std::max<long long>(1, std::min<long long>(a.ntiles, cap));
  if (ModeTraits<MODE>::kReduce && g_det.on) {
    // deterministic mode: per-block partial sums, added in block order by a second tiny kernel.  A folded single-channel
    // tensor has 2 quantities x 8 warp slots per block, reduced as [grid * 8 "blocks"][2]... laid out [block][q][warp].
    Args b = a;
    const size_t per_block = a.fold ? (size_t)2 * (kConsumers / 32) : (size_t)2 * a.c;
    b.partials = (double*)det_scratch((size_t)grid * per_block * sizeof(double));
    if (!b.partials) return VG_EINVAL;
    vg::Launch(grid, kThreads, G::kSmemBytes, s)(bn_stream_kernel<T, MODE, DROP>, b);
    VG_LAUNCHED();
    if (a.fold) return ordered_reduce_fold(b.partials, grid, a.sums_out, a.c, s);
    return ordered_reduce_f64(b.partials, grid, 2LL * a.c, a.sums_out, s);
  }
  vg::Launch(grid, kThreads, G::kSmemBytes, s)(bn_stream_kernel<T, MODE, DROP>, a);
  VG_LAUNCHED();
  return VG_OK;
}

template <typename T, int MODE>
static int launch_drop(const Args& a, cudaStream_t s) {
  if (a.thr16 != 0) {
    if constexpr (MODE == kFwd || MODE == kBwdReduce || MODE == kBwdApply || MODE == kBwdApplyAdd) return launch<T, MODE, true>(a, s);
  }
  return launch<T, MODE, false>(a, s);
}

}  // namespace bs

// can the streaming kernels take this tensor?  (vector path: C % 8 == 0 and C / 8 <= 256; folded path: C == 1 and
// rows % 8 == 0; every streamed pointer 16-byte aligned)
bool bn_stream_ok(const VgBnDesc* d, const void* p0, const void* p1, const void* p2, const void* p3) {
  if (d->rows <= 0) return false;
  const bool vec = d->c % 8 == 0 && d->c / 8 <= bs::kConsumers;
  const bool fold = d->c == 1 && d->rows % 8 == 0;
  if (!vec && !fold) return false;
  const void* ps[4] = {p0, p1, p2, p3};
  for (const void* p : ps)
    if (p != nullptr && (reinterpret_cast<uintptr_t>(p) & 15u) != 0) return false;
  // the dropout stream is indexed by 8-element Philox blocks: the tensor's first element must start one
  if (d->drop_p > 0.f && ((unsigned long long)d->sample_offset * (unsigned long long)d->hw * (unsigned long long)d->c) % 8ull != 0) return false;
  return true;
}

static uint32_t thr16_of_p(float p) {
  const double t = (double)p * 65536.0;
  return t >= 65535.0 ? 65535u : (uint32_t)t;
}

static void fill_common(bs::Args& a, const VgBnDesc* d) {
  memset(&a, 0, sizeof(a));
  const bool fold = !(d->c % 8 == 0 && d->c / 8 <= bs::kConsumers);
  a.fold = fold ? 1 : 0;
  a.c = d->c;
  a.cg = fold ? 1 : d->c / 8;
  a.tpb = (bs::kConsumers / a.cg) * a.cg;
  a.nvec = fold ? d->rows / 8 : d->rows * (long long)a.cg;
  a.hw = d->hw;
  a.A.kind = -1;
  a.B.kind = -1;
  a.slope = d->slope;
  a.drop_scale = d->drop_p > 0.f ? 1.0f / (1.0f - d->drop_p) : 1.0f;
  a.thr16 = d->drop_p > 0.f ? thr16_of_p(d->drop_p) : 0u;
  a.seed = d->seed;
  a.offset = d->offset;
  a.step_ptr = d->step_ptr;
  a.vbase = ((unsigned long long)d->sample_offset * (unsigned long long)d->hw * (unsigned long long)d->c) >> 3;
  a.training = d->training;
}

template <int MODE>
static int dispatch(bs::Args& a, const VgBnDesc* d, cudaStream_t s) {
  // the tile count depends on KT, a compile-time property of (dtype, mode)
  if (d->dtype == VG_BF16) {
    a.ntiles = cdiv(a.nvec, (long long)bs::Geo<__nv_bfloat16, MODE>::KT * a.tpb);
    return bs::launch_drop<__nv_bfloat16, MODE>(a, s);
  }
  a.ntiles = cdiv(a.nvec, (long long)bs::Geo<float, MODE>::KT * a.tpb);
  return bs::launch_drop<float, MODE>(a, s);
}

static void set_chan(bs::Chan& ch, const VgBnChannel* p, int training) {
  memset(&ch, 0, sizeof(ch));
  if (p == nullptr) { ch.kind = -1; return; }
  ch.gamma = p->gamma;
  ch.beta = p->beta;
  ch.mean_rstd = p->mean_rstd_in;
  ch.sums = p->sums;
  ch.count = p->count;
  ch.running_mean = p->running_mean;
  ch.running_var = p->running_var;
  ch.mean_rstd_out = p->mean_rstd_out;
  ch.eps = p->eps;
  ch.momentum = p->momentum;
  if (p->mean_rstd_in != nullptr) ch.kind = 0;
  else if (training && p->sums != nullptr) ch.kind = 1;
  else ch.kind = 2;
}

// ---- entry points used by bn.cu's C ABI -------------------------------------------------------
int bn_stream_stats(const void* x, const VgBnDesc* d, double* sums, cudaStream_t s) {
  bs::Args a;
  fill_common(a, d);
  a.in0 = x;
  a.sums_out = sums;
  a.thr16 = 0;
  a.reverse = 1;
  return dispatch<bs::kStats>(a, d, s);
}

int bn_stream_act_forward(const void* x, const VgBnChannel* bn, const VgBnDesc* d, void* y, cudaStream_t s) {
  bs::Args a;
  fill_common(a, d);
  a.in0 = x;
  a.out = y;
  set_chan(a.A, bn, d->training);
  return dispatch<bs::kFwd>(a, d, s);
}

int bn_stream_bwd_reduce(const void* dy, const void* x, const float* mean_rstd, const float* gamma, const float* beta,
                         const VgBnDesc* d, double* sums, cudaStream_t s) {
  bs::Args a;
  fill_common(a, d);
  a.in0 = dy;
  a.in1 = x;
  a.A.kind = 0;
  a.A.mean_rstd = mean_rstd;
  a.A.gamma = gamma;
  a.A.beta = beta;
  a.sums_out = sums;
  a.reverse = 1;
  return dispatch<bs::kBwdReduce>(a, d, s);
}

int bn_stream_bwd_apply(const void* dy, const void* x, const float* mean_rstd, const float* gamma, const float* beta,
                        const double* sums, double count, const VgBnDesc* d, const float* out_colscale, const void* addend,
                        void* dx, float* dgamma, float* dbeta, float param_scale, cudaStream_t s) {
  bs::Args a;
  fill_common(a, d);
  a.in0 = dy;
  a.in1 = x;
  a.in2 = addend;
  a.out = dx;
  a.A.kind = 0;
  a.A.mean_rstd = mean_rstd;
  a.A.gamma = gamma;
  a.A.beta = beta;
  a.sums_in = sums;
  a.count = count;
  a.out_colscale = out_colscale;
  a.dgamma = dgamma;
  a.dbeta = dbeta;
  a.param_scale = param_scale;
  if (addend != nullptr) return dispatch<bs::kBwdApplyAdd>(a, d, s);
  return dispatch<bs::kBwdApply>(a, d, s);
}

int bn_stream_add_dual(const void* x0, const void* x1, const float* post_scale, const float* post_shift, float post_slope,
                       const VgBnDesc* d, void* out, void* out2, cudaStream_t s) {
  bs::Args a;
  fill_common(a, d);
  a.in0 = x0;
  a.in1 = x1;
  a.out = out;
  a.out2 = out2;
  a.post_scale = post_scale;
  a.post_shift = post_shift;
  a.post_slope = post_slope;
  a.thr16 = 0;
  return dispatch<bs::kAddDual>(a, d, s);
}

int bn_stream_add(const void* x0, const VgBnChannel* bn_a, const void* x1, const VgBnChannel* bn_b, const VgBnDesc* d, void* out,
                  double* stats, cudaStream_t s) {
  bs::Args a;
  fill_common(a, d);
  a.in0 = x0;
  a.in1 = x1;
  a.out = out;
  set_chan(a.A, bn_a, d->training);
  set_chan(a.B, bn_b, d->training);
  a.sums_out = stats;
  a.thr16 = 0;
  a.reverse = 1;
  if (stats != nullptr) return dispatch<bs::kAddStats>(a, d, s);
  return dispatch<bs::kAdd>(a, d, s);
}

}  // namespace vg
