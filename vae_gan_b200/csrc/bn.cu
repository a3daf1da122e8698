// BatchNorm2d-family memory-bound kernels (NHWC): statistics, apply + LeakyReLU + Philox dropout,
// backward reduce / apply, residual add.  Replaces nn.BatchNorm2d / nn.LeakyReLU / nn.Dropout /
// `out += shortcut(x)` of the reference (README.md:143-197, 376-419, 442, 466-468).
//
// Thread mapping (vector path, C % 8 == 0): a thread owns ONE group of 8 consecutive channels
// for its whole life (per-channel constants live in registers) and walks rows with a grid
// stride; consecutive threads touch consecutive 16 B (bf16) / 32 B (f32) chunks, so every warp
// access is fully coalesced.  Per-channel reductions: registers -> shared -> one fp64
// atomicAdd per (block, channel).  C == 1 tensors are folded into an [rows/8][8] view.
// Anything else takes the scalar path.
#include <algorithm>
#include <mutex>
#include "vg_common.cuh"

namespace vg {

constexpr int kBnThreads = 256;
constexpr int kUnroll = 4;
// loads in flight per thread for the kernels that only READ activations or write one tensor (statistics,
// forward apply, backward reduction): measured on B200 at 128 channels x 96^2 x 64, 8 vs 4: stats 37.4 -> 35.3 us,
// act_fwd 62.2 -> 57.8 us, bwd reduce 68.3 -> 56.5 us; the backward APPLY (two loads + one store) is
// fastest at 4 (98.8 us vs 119.3 us at 8).
constexpr int kUnrollWide = 8;

struct RowMap {
  int cg;        // channel groups per row (C/8)
  int tpb;       // threads per block actually used = (256/cg)*cg
  int rpb;       // rows per block iteration
};

__host__ __device__ inline RowMap make_rowmap(int c) {
  RowMap m;
  m.cg = c / 8;
  m.rpb = kBnThreads / m.cg;
  m.tpb = m.rpb * m.cg;
  return m;
}

static inline bool vec_ok(int c) { return c % 8 == 0 && c / 8 <= kBnThreads; }

static inline int grid_for(long long rows, int rpb, int iters_target = kUnroll * 2, int blocks_per_sm = 8) {
  long long blocks = cdiv(rows, (long long)rpb * iters_target);
  long long cap = (long long)num_sms() * blocks_per_sm;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}
// kernels that end in a per-channel reduction: every block issues 2C same-address fp64 atomics, which
// serialise in L2 - keep the block count at a small multiple of the SM count and give each block
// more rows instead.
constexpr int kReduceBlocksPerSm = 3;
constexpr int kApplyBlocksPerSm = 4;

// 16-bit Philox keep decisions for 8 consecutive elements starting at linear index e0 (e0 % 8 == 0)
__device__ __forceinline__ void keep8(const Philox& ph, unsigned long long e0, uint32_t thr16, bool keep[8]) {
  uint4 r = ph.block(e0 >> 3);
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    keep[2 * i] = (w[i] & 0xffffu) >= thr16;
    keep[2 * i + 1] = (w[i] >> 16) >= thr16;
  }
}
__device__ __forceinline__ bool keep1(const Philox& ph, unsigned long long e, uint32_t thr16) {
  uint4 r = ph.block(e >> 3);
  uint32_t j = (uint32_t)e & 7u;
  uint32_t w = (j >> 1) == 0 ? r.x : ((j >> 1) == 1 ? r.y : ((j >> 1) == 2 ? r.z : r.w));
  uint32_t h = (j & 1u) ? (w >> 16) : (w & 0xffffu);
  return h >= thr16;
}
__host__ __device__ inline uint32_t thr16_of(float p) {
  double t = (double)p * 65536.0;
  return t >= 65535.0 ? 65535u : (uint32_t)t;
}

// block-level per-channel reduction of NV values per thread-channel, then fp64 atomics.
// acc[v][8]: v-th quantity for the thread's 8 channels.  `fold`: all 8 lanes are channel 0.
template <int NV>
__device__ __forceinline__ void block_reduce_to_global(float (&acc)[NV][8], const RowMap& m, int c, bool fold,
                                                       double* out /* [NV][c] */, float* smem,
                                                       double* partials = nullptr /* deterministic mode: [grid][NV][c] */) {
  const int tid = threadIdx.x;
  // smem layout [NV*8][kBnThreads]
#pragma unroll
  for (int v = 0; v < NV; ++v)
#pragma unroll
    for (int j = 0; j < 8; ++j) smem[(v * 8 + j) * kBnThreads + tid] = (tid < m.tpb) ? acc[v][j] : 0.f;
  __syncthreads();
  if (fold) {
    // every (thread, lane) belongs to channel 0
    for (int v = 0; v < NV; ++v) {
      double s = 0.0;
      for (int i = tid; i < 8 * kBnThreads; i += kBnThreads) s += (double)smem[v * 8 * kBnThreads + i];
      s = warp_sum(s);
      __shared__ double wsum[kBnThreads / 32];
      if ((tid & 31) == 0) wsum[tid >> 5] = s;
      __syncthreads();
      if (tid == 0) {
        double t = 0.0;
        for (int w = 0; w < kBnThreads / 32; ++w) t += wsum[w];
        if (partials) partials[(size_t)blockIdx.x * NV * c + v * c] = t;
        else atomicAdd(&out[v * c], t);
      }
      __syncthreads();
    }
    return;
  }
  // channel ch = g*8 + j is handled by thread index (g*8+j) over NV values
  for (int idx = tid; idx < NV * c; idx += kBnThreads) {
    int v = idx / c, ch = idx - v * c;
    int g = ch >> 3, j = ch & 7;
    double s = 0.0;
    for (int r = 0; r < m.rpb; ++r) s += (double)smem[(v * 8 + j) * kBnThreads + r * m.cg + g];
    if (partials) partials[(size_t)blockIdx.x * NV * c + idx] = s;
    else atomicAdd(&out[v * c + ch], s);
  }
}

// ------------------------------------------------------------------------------------------
// statistics
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kBnThreads) bn_stats_vec_kernel(const T* __restrict__ x, long long rows, int c,
                                                                   bool fold, double* __restrict__ sums, double* __restrict__ partials) {
  vg::pdl_entry();
  extern __shared__ float smem[];
  const int cv = fold ? 8 : c;
  const RowMap m = make_rowmap(cv);
  const int tid = threadIdx.x;
  const int g = tid % m.cg, r0 = tid / m.cg;
  float acc[2][8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[0][j] = acc[1][j] = 0.f;
  if (tid < m.tpb) {
    const long long stride = (long long)gridDim.x * m.rpb;
    long long row = (long long)blockIdx.x * m.rpb + r0;
    for (; row + (kUnrollWide - 1) * stride < rows; row += kUnrollWide * stride) {
      Vec8<T> v[kUnrollWide];
#pragma unroll
      for (int u = 0; u < kUnrollWide; ++u) v[u].load(x + (row + u * stride) * cv + g * 8);
#pragma unroll
      for (int u = 0; u < kUnrollWide; ++u)
#pragma unroll
        for (int j = 0; j < 8; ++j) { acc[0][j] += v[u].v[j]; acc[1][j] += v[u].v[j] * v[u].v[j]; }
    }
    for (; row < rows; row += stride) {
      Vec8<T> v;
      v.load(x + row * cv + g * 8);
#pragma unroll
      for (int j = 0; j < 8; ++j) { acc[0][j] += v.v[j]; acc[1][j] += v.v[j] * v.v[j]; }
    }
  }
  block_reduce_to_global<2>(acc, m, c, fold, sums, smem, partials);
}

template <typename T>
__global__ void bn_stats_scalar_kernel(const T* __restrict__ x, long long total, int c, double* __restrict__ sums) {
  vg::pdl_entry();
  extern __shared__ double dsm[];  // [2*c]
  for (int i = threadIdx.x; i < 2 * c; i += blockDim.x) dsm[i] = 0.0;
  __syncthreads();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    float v = to_f32(x[i]);
    int ch = (int)(i % c);
    atomicAdd(&dsm[ch], (double)v);
    atomicAdd(&dsm[c + ch], (double)v * v);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * c; i += blockDim.x) atomicAdd(&sums[i], dsm[i]);
}

__global__ void bn_finalize_kernel(const double* __restrict__ sums, double count, int c, float eps, float momentum,
                                   float* running_mean, float* running_var, float* __restrict__ mean_rstd) {
  vg::pdl_entry();
  int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  double mean = sums[ch] / count;
  double var = sums[c + ch] / count - mean * mean;
  if (var < 0.0) var = 0.0;
  mean_rstd[ch] = (float)mean;
  mean_rstd[c + ch] = (float)(1.0 / sqrt(var + (double)eps));
  if (running_mean != nullptr) {
    double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
    running_mean[ch] = (float)((1.0 - momentum) * (double)running_mean[ch] + momentum * mean);
    running_var[ch] = (float)((1.0 - momentum) * (double)running_var[ch] + momentum * unbiased);
  }
}

__global__ void bn_eval_stats_kernel(const float* __restrict__ rm, const float* __restrict__ rv, int c, float eps,
                                     float* __restrict__ mean_rstd) {
  vg::pdl_entry();
  int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  mean_rstd[ch] = rm[ch];
  mean_rstd[c + ch] = (float)(1.0 / sqrt((double)rv[ch] + (double)eps));
}

__global__ void bn_param_grads_kernel(const double* __restrict__ sums, int c, double scale, float* dgamma, float* dbeta) {
  vg::pdl_entry();
  int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  if (dbeta) dbeta[ch] += (float)(sums[ch] * scale);
  if (dgamma) dgamma[ch] += (float)(sums[c + ch] * scale);
}

// ------------------------------------------------------------------------------------------
// forward apply: y = drop(lrelu(a*x + b)),  a = gamma*rstd, b = beta - mean*a
// ------------------------------------------------------------------------------------------
struct BnK {
  long long rows;
  int c, hw;
  float slope, drop_scale;
  uint32_t thr16;
  unsigned long long seed, offset;
  const unsigned long long* step_ptr;
  long long sample_offset;
  int training;
  bool fold;
};
__device__ __forceinline__ unsigned long long eff_offset(unsigned long long offset, const unsigned long long* step_ptr) {
  return step_ptr ? offset + 65536ull * (*step_ptr) : offset;
}

static inline BnK make_bnk(const VgBnDesc* d) {
  BnK k;
  k.rows = d->rows; k.c = d->c; k.hw = d->hw; k.slope = d->slope;
  k.drop_scale = d->drop_p > 0.f ? 1.0f / (1.0f - d->drop_p) : 1.0f;
  k.thr16 = d->drop_p > 0.f ? thr16_of(d->drop_p) : 0u;
  k.seed = d->seed; k.offset = d->offset; k.step_ptr = d->step_ptr; k.sample_offset = d->sample_offset; k.training = d->training;
  k.fold = false;
  return k;
}

template <typename T, bool DROP>
__global__ void __launch_bounds__(kBnThreads) bn_act_fwd_vec_kernel(const T* __restrict__ x, const float* __restrict__ mean_rstd,
                                                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                     BnK k, T* __restrict__ y) {
  vg::pdl_entry();
  const int cv = k.fold ? 8 : k.c;
  const RowMap m = make_rowmap(cv);
  const int tid = threadIdx.x;
  if (tid >= m.tpb) return;
  const int g = tid % m.cg, r0 = tid / m.cg;
  float a[8], b[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    int ch = k.fold ? 0 : g * 8 + j;
    float aa = gamma[ch] * mean_rstd[k.c + ch];
    a[j] = aa;
    b[j] = beta[ch] - mean_rstd[ch] * aa;
  }
  Philox ph(k.seed, eff_offset(k.offset, k.step_ptr));
  const unsigned long long ebase = (unsigned long long)k.sample_offset * (unsigned long long)k.hw * (unsigned long long)k.c;
  const long long stride = (long long)gridDim.x * m.rpb;
  long long row = (long long)blockIdx.x * m.rpb + r0;
  auto body = [&](Vec8<T>& v, long long rw) {
    bool kp[8];
    if (DROP) keep8(ph, ebase + (unsigned long long)rw * cv + g * 8, k.thr16, kp);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float t = fmaf(a[j], v.v[j], b[j]);
      t = t > 0.f ? t : t * k.slope;
      if (DROP) t = kp[j] ? t * k.drop_scale : 0.f;
      v.v[j] = t;
    }
  };
  for (; row + (kUnrollWide - 1) * stride < k.rows; row += kUnrollWide * stride) {
    Vec8<T> v[kUnrollWide];
#pragma unroll
    for (int u = 0; u < kUnrollWide; ++u) v[u].load(x + (row + u * stride) * cv + g * 8);
#pragma unroll
    for (int u = 0; u < kUnrollWide; ++u) {
      body(v[u], row + u * stride);
      v[u].store(y + (row + u * stride) * cv + g * 8);
    }
  }
  for (; row < k.rows; row += stride) {
    Vec8<T> v;
    v.load(x + row * cv + g * 8);
    body(v, row);
    v.store(y + row * cv + g * 8);
  }
}

template <typename T>
__global__ void bn_act_fwd_scalar_kernel(const T* __restrict__ x, const float* __restrict__ mean_rstd,
                                         const float* __restrict__ gamma, const float* __restrict__ beta, BnK k,
                                         T* __restrict__ y) {
  vg::pdl_entry();
  Philox ph(k.seed, eff_offset(k.offset, k.step_ptr));
  const unsigned long long ebase = (unsigned long long)k.sample_offset * (unsigned long long)k.hw * (unsigned long long)k.c;
  const long long total = k.rows * k.c;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int ch = (int)(i % k.c);
    float aa = gamma[ch] * mean_rstd[k.c + ch];
    float t = fmaf(aa, to_f32(x[i]), beta[ch] - mean_rstd[ch] * aa);
    t = t > 0.f ? t : t * k.slope;
    if (k.thr16) t = keep1(ph, ebase + (unsigned long long)i, k.thr16) ? t * k.drop_scale : 0.f;
    y[i] = from_f32<T>(t);
  }
}

// ------------------------------------------------------------------------------------------
// backward: g = dy * drop' * lrelu'(a*x+b);  reduce: sum g, sum g*xhat;  apply: dx
// ------------------------------------------------------------------------------------------
template <typename T, bool DROP, bool APPLY>
__global__ void __launch_bounds__(kBnThreads, APPLY ? 1 : 3) bn_act_bwd_vec_kernel(const T* __restrict__ dy, const T* __restrict__ x,
                                                                     const float* __restrict__ mean_rstd,
                                                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                     BnK k, double* __restrict__ sums_out /* reduce */,
                                                                     double* __restrict__ partials /* reduce, deterministic mode */,
                                                                     const double* __restrict__ sums_in /* apply */, double count,
                                                                     const float* __restrict__ out_colscale,
                                                                     const T* __restrict__ addend, T* __restrict__ dx) {
  vg::pdl_entry();
  extern __shared__ float smem[];
  const int cv = k.fold ? 8 : k.c;
  const RowMap m = make_rowmap(cv);
  const int tid = threadIdx.x;
  const int g = tid % m.cg, r0 = tid / m.cg;
  float acc[2][8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[0][j] = acc[1][j] = 0.f;
  if (tid < m.tpb) {
    float a[8], b[8], mean[8], rstd[8], k1[8], k2[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int ch = k.fold ? 0 : g * 8 + j;
      mean[j] = mean_rstd[ch];
      rstd[j] = mean_rstd[k.c + ch];
      a[j] = gamma[ch] * rstd[j];
      b[j] = beta[ch] - mean[j] * a[j];
      if (APPLY) {
        if (k.training) {
          k1[j] = (float)(sums_in[ch] / count);
          k2[j] = (float)(sums_in[k.c + ch] / count);
        } else {
          k1[j] = 0.f; k2[j] = 0.f;
        }
      }
    }
    Philox ph(k.seed, eff_offset(k.offset, k.step_ptr));
    const unsigned long long ebase = (unsigned long long)k.sample_offset * (unsigned long long)k.hw * (unsigned long long)k.c;
    const long long stride = (long long)gridDim.x * m.rpb;
    long long row = (long long)blockIdx.x * m.rpb + r0;
    auto body = [&](Vec8<T>& vdy, const Vec8<T>& vx, long long rw) {
      bool kp[8];
      if (DROP) keep8(ph, ebase + (unsigned long long)rw * cv + g * 8, k.thr16, kp);
      float cs[8];
      if (APPLY && out_colscale != nullptr) {
        long long n = rw / k.hw;
        const float* p = out_colscale + n * k.c + g * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) cs[j] = p[j];
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float pre = fmaf(a[j], vx.v[j], b[j]);
        float gg = vdy.v[j] * (pre > 0.f ? 1.f : k.slope);
        if (DROP) gg = kp[j] ? gg * k.drop_scale : 0.f;
        float xh = (vx.v[j] - mean[j]) * rstd[j];
        if (APPLY) {
          float r = a[j] * (gg - k1[j] - xh * k2[j]);
          if (out_colscale != nullptr) r *= cs[j];
          vdy.v[j] = r;
        } else {
          acc[0][j] += gg;
          acc[1][j] += gg * xh;
        }
      }
    };
    constexpr int U = APPLY ? kUnroll / 2 : kUnrollWide / 2;      // (dy, x) pairs in flight
    for (; row + (U - 1) * stride < k.rows; row += U * stride) {
      Vec8<T> vd[U], vx[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        vd[u].load(dy + (row + u * stride) * cv + g * 8);
        vx[u].load(x + (row + u * stride) * cv + g * 8);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        body(vd[u], vx[u], row + u * stride);
        if (APPLY) {
          if (addend != nullptr) {
            Vec8<T> ad;
            ad.load(addend + (row + u * stride) * cv + g * 8);
#pragma unroll
            for (int j = 0; j < 8; ++j) vd[u].v[j] += ad.v[j];
          }
          vd[u].store(dx + (row + u * stride) * cv + g * 8);
        }
      }
    }
    for (; row < k.rows; row += stride) {
      Vec8<T> vd, vx;
      vd.load(dy + row * cv + g * 8);
      vx.load(x + row * cv + g * 8);
      body(vd, vx, row);
      if (APPLY) {
        if (addend != nullptr) {
          Vec8<T> ad;
          ad.load(addend + row * cv + g * 8);
#pragma unroll
          for (int j = 0; j < 8; ++j) vd.v[j] += ad.v[j];
        }
        vd.store(dx + row * cv + g * 8);
      }
    }
  }
  if (!APPLY) block_reduce_to_global<2>(acc, m, k.c, k.fold, sums_out, smem, partials);
}

// ------------------------------------------------------------------------------------------
// second-order backward (gradient penalty, README.md:717-739): derivative of the BatchNorm(+LeakyReLU)
// input gradient  dx = gamma*rstd*(dyb - mean(dyb) - xh*mean(dyb*xh)) * cs,  dyb = dy*m,  with respect to
// dy, x (given G = dL/d(dx)); `cs` is the Dropout2d column scale of the producing convolution (nullable).
//   REDUCE: sums[5][C] = sum dyb, sum dyb*xh, sum G', sum G'*xh, sum G'*dyb     (G' = G*cs)
//   APPLY : g_dy = gamma*rstd*(G' - mean(G') - xh*mean(G'*xh))*m
//           g_x  = cs*( rstd*(Q - mean(Q) - xh*mean(Q*xh)) - rstd^2*gamma*S1/M * xh ),
//                  Q = -gamma*rstd*(b*G' + c*dyb),  S1 = sum G'*dyb - a*sum G' - b*sum G'*xh
// (closed form derived and checked against autograd in vae_gan_b200/gp.py:bn_double_backward)
// ------------------------------------------------------------------------------------------
template <typename T, bool APPLY>
__global__ void __launch_bounds__(kBnThreads) bn_dbl_bwd_vec_kernel(const T* __restrict__ dy, const T* __restrict__ x,
                                                                    const T* __restrict__ G, const float* __restrict__ mean_rstd,
                                                                    const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                    BnK k, const float* __restrict__ colscale,
                                                                    double* __restrict__ sums_out, double* __restrict__ partials,
                                                                    const double* __restrict__ sums_in,
                                                                    double count, T* __restrict__ g_dy, T* __restrict__ g_x) {
  vg::pdl_entry();
  extern __shared__ float smem[];
  const int cv = k.c;
  const RowMap m = make_rowmap(cv);
  const int tid = threadIdx.x;
  const int g = tid % m.cg, r0 = tid / m.cg;
  float acc[5][8];
#pragma unroll
  for (int v = 0; v < 5; ++v)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[v][j] = 0.f;
  if (tid < m.tpb) {
    float ga[8], be[8], mean[8], rstd[8];
    float c_a[8], c_b[8], c_c[8], c_mg[8], c_k[8];   // APPLY: mean(dyb), mean(dyb*xh), mean(G'xh), mean(G'), rstd*gamma*S1/M
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int ch = g * 8 + j;
      mean[j] = mean_rstd[ch];
      rstd[j] = mean_rstd[k.c + ch];
      ga[j] = gamma[ch];
      be[j] = beta[ch];
      if (APPLY) {
        const double s_dyb = sums_in[ch], s_dybx = sums_in[k.c + ch], s_g = sums_in[2 * k.c + ch], s_gx = sums_in[3 * k.c + ch],
                     s_gdyb = sums_in[4 * k.c + ch];
        const double a = s_dyb / count, b = s_dybx / count;
        c_a[j] = (float)a; c_b[j] = (float)b; c_c[j] = (float)(s_gx / count); c_mg[j] = (float)(s_g / count);
        c_k[j] = (float)((double)rstd[j] * ga[j] * (s_gdyb - a * s_g - b * s_gx) / count);
      }
    }
    const long long stride = (long long)gridDim.x * m.rpb;
    for (long long row = (long long)blockIdx.x * m.rpb + r0; row < k.rows; row += stride) {
      Vec8<T> vd, vx, vg;
      const long long off = row * cv + g * 8;
      vd.load(dy + off);
      vx.load(x + off);
      vg.load(G + off);
      float cs[8];
      if (colscale != nullptr) {
        const float* p = colscale + (row / k.hw) * k.c + g * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) cs[j] = p[j];
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) cs[j] = 1.f;
      }
      Vec8<T> o_dy, o_x;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float xh = (vx.v[j] - mean[j]) * rstd[j];
        const float mk = fmaf(ga[j], xh, be[j]) > 0.f ? 1.f : k.slope;
        const float dyb = vd.v[j] * mk;
        const float gg = vg.v[j] * cs[j];
        if (!APPLY) {
          acc[0][j] += dyb;
          acc[1][j] += dyb * xh;
          acc[2][j] += gg;
          acc[3][j] += gg * xh;
          acc[4][j] += gg * dyb;
        } else {
          const float gr = ga[j] * rstd[j];
          o_dy.v[j] = gr * (gg - c_mg[j] - xh * c_c[j]) * mk;
          const float q = -gr * (c_b[j] * gg + c_c[j] * dyb);
          const float mq = -gr * (c_b[j] * c_mg[j] + c_c[j] * c_a[j]);
          const float mqx = -2.f * gr * c_b[j] * c_c[j];
          o_x.v[j] = (rstd[j] * (q - mq - xh * mqx) - rstd[j] * c_k[j] * xh) * cs[j];
        }
      }
      if (APPLY) {
        o_dy.store(g_dy + off);
        o_x.store(g_x + off);
      }
    }
  }
  if (!APPLY) block_reduce_to_global<5>(acc, m, k.c, false, sums_out, smem, partials);
}

template <typename T, bool APPLY>
__global__ void bn_act_bwd_scalar_kernel(const T* __restrict__ dy, const T* __restrict__ x, const float* __restrict__ mean_rstd,
                                         const float* __restrict__ gamma, const float* __restrict__ beta, BnK k,
                                         double* __restrict__ sums_out, const double* __restrict__ sums_in, double count,
                                         const float* __restrict__ out_colscale, const T* __restrict__ addend,
                                         T* __restrict__ dx) {
  vg::pdl_entry();
  extern __shared__ double dsm[];
  if (!APPLY) {
    for (int i = threadIdx.x; i < 2 * k.c; i += blockDim.x) dsm[i] = 0.0;
    __syncthreads();
  }
  Philox ph(k.seed, eff_offset(k.offset, k.step_ptr));
  const unsigned long long ebase = (unsigned long long)k.sample_offset * (unsigned long long)k.hw * (unsigned long long)k.c;
  const long long total = k.rows * k.c;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int ch = (int)(i % k.c);
    float mean = mean_rstd[ch], rstd = mean_rstd[k.c + ch];
    float aa = gamma[ch] * rstd;
    float xv = to_f32(x[i]);
    float pre = fmaf(aa, xv, beta[ch] - mean * aa);
    float gg = to_f32(dy[i]) * (pre > 0.f ? 1.f : k.slope);
    if (k.thr16) gg = keep1(ph, ebase + (unsigned long long)i, k.thr16) ? gg * k.drop_scale : 0.f;
    float xh = (xv - mean) * rstd;
    if (APPLY) {
      float k1 = k.training ? (float)(sums_in[ch] / count) : 0.f;
      float k2 = k.training ? (float)(sums_in[k.c + ch] / count) : 0.f;
      float r = aa * (gg - k1 - xh * k2);
      if (out_colscale != nullptr) r *= out_colscale[(i / k.c / k.hw) * k.c + ch];
      if (addend != nullptr) r += to_f32(addend[i]);
      dx[i] = from_f32<T>(r);
    } else {
      atomicAdd(&dsm[ch], (double)gg);
      atomicAdd(&dsm[k.c + ch], (double)gg * xh);
    }
  }
  if (!APPLY) {
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * k.c; i += blockDim.x) atomicAdd(&sums_out[i], dsm[i]);
  }
}

// ------------------------------------------------------------------------------------------
// residual add: out = lrelu(bnA(a) + bnB(b)) (+ stats of out)
// ------------------------------------------------------------------------------------------
template <typename T, bool STATS>
__global__ void __launch_bounds__(kBnThreads, 3) bn_add_vec_kernel(const T* __restrict__ A, const float* __restrict__ mrA,
                                                                 const float* __restrict__ gA, const float* __restrict__ bA,
                                                                 const T* __restrict__ B, const float* __restrict__ mrB,
                                                                 const float* __restrict__ gB, const float* __restrict__ bB, BnK k,
                                                                 T* __restrict__ out, double* __restrict__ stats,
                                                                 double* __restrict__ partials) {
  vg::pdl_entry();
  extern __shared__ float smem[];
  const int cv = k.fold ? 8 : k.c;
  const RowMap m = make_rowmap(cv);
  const int tid = threadIdx.x;
  const int g = tid % m.cg, r0 = tid / m.cg;
  float acc[2][8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[0][j] = acc[1][j] = 0.f;
  if (tid < m.tpb) {
    float sa[8], ta[8], sb[8], tb[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int ch = k.fold ? 0 : g * 8 + j;
      if (mrA) { sa[j] = gA[ch] * mrA[k.c + ch]; ta[j] = bA[ch] - mrA[ch] * sa[j]; } else { sa[j] = 1.f; ta[j] = 0.f; }
      if (mrB) { sb[j] = gB[ch] * mrB[k.c + ch]; tb[j] = bB[ch] - mrB[ch] * sb[j]; } else { sb[j] = 1.f; tb[j] = 0.f; }
    }
    const long long stride = (long long)gridDim.x * m.rpb;
    for (long long row = (long long)blockIdx.x * m.rpb + r0; row < k.rows; row += 2 * stride) {
      Vec8<T> va[2], vb[2];
      bool has2 = row + stride < k.rows;
      va[0].load(A + row * cv + g * 8);
      vb[0].load(B + row * cv + g * 8);
      if (has2) {
        va[1].load(A + (row + stride) * cv + g * 8);
        vb[1].load(B + (row + stride) * cv + g * 8);
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (u == 1 && !has2) break;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float t = fmaf(sa[j], va[u].v[j], ta[j]) + fmaf(sb[j], vb[u].v[j], tb[j]);
          t = t > 0.f ? t : t * k.slope;
          va[u].v[j] = t;
        }
        va[u].store(out + (row + u * stride) * cv + g * 8);
        if (STATS) {
          // statistics are taken on the values as STORED (bf16-rounded on the bf16 path)
          Vec8<T> rb;
          rb = va[u];
          if (sizeof(T) == 2) {
#pragma unroll
            for (int j = 0; j < 8; ++j) rb.v[j] = to_f32(from_f32<T>(rb.v[j]));
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) { acc[0][j] += rb.v[j]; acc[1][j] += rb.v[j] * rb.v[j]; }
        }
      }
    }
  }
  if (STATS) block_reduce_to_global<2>(acc, m, k.c, k.fold, stats, smem, partials);
}

template <typename T>
__global__ void bn_add_scalar_kernel(const T* __restrict__ A, const float* __restrict__ mrA, const float* __restrict__ gA,
                                     const float* __restrict__ bA, const T* __restrict__ B, const float* __restrict__ mrB,
                                     const float* __restrict__ gB, const float* __restrict__ bB, BnK k, T* __restrict__ out,
                                     double* __restrict__ stats) {
  vg::pdl_entry();
  extern __shared__ double dsm[];
  if (stats) {
    for (int i = threadIdx.x; i < 2 * k.c; i += blockDim.x) dsm[i] = 0.0;
    __syncthreads();
  }
  const long long total = k.rows * k.c;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int ch = (int)(i % k.c);
    float va = to_f32(A[i]), vb = to_f32(B[i]);
    if (mrA) { float s = gA[ch] * mrA[k.c + ch]; va = fmaf(s, va, bA[ch] - mrA[ch] * s); }
    if (mrB) { float s = gB[ch] * mrB[k.c + ch]; vb = fmaf(s, vb, bB[ch] - mrB[ch] * s); }
    float t = va + vb;
    t = t > 0.f ? t : t * k.slope;
    T o = from_f32<T>(t);
    out[i] = o;
    if (stats) {
      float r = to_f32(o);
      atomicAdd(&dsm[ch], (double)r);
      atomicAdd(&dsm[k.c + ch], (double)r * r);
    }
  }
  if (stats) {
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * k.c; i += blockDim.x) atomicAdd(&stats[i], dsm[i]);
  }
}

// elementwise helpers -----------------------------------------------------------------------
template <typename T>
__global__ void lrelu_bwd_kernel(const T* __restrict__ dy, const T* __restrict__ yref, long long n, float slope, T* __restrict__ dx) {
  vg::pdl_entry();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    dx[i] = from_f32<T>(to_f32(dy[i]) * (to_f32(yref[i]) > 0.f ? 1.f : slope));
}
template <typename T>
__global__ void add_kernel(const T* __restrict__ a, const T* __restrict__ b, long long n, T* __restrict__ out) {
  vg::pdl_entry();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = from_f32<T>(to_f32(a[i]) + to_f32(b[i]));
}
template <typename T>
__global__ void add_vec_kernel(const T* __restrict__ a, const T* __restrict__ b, long long nvec, T* __restrict__ out) {
  vg::pdl_entry();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    Vec8<T> va, vb;
    va.load(a + i * 8);
    vb.load(b + i * 8);
#pragma unroll
    for (int j = 0; j < 8; ++j) va.v[j] += vb.v[j];
    va.store(out + i * 8);
  }
}

__global__ void dropout_mask_kernel(BnK k, uint8_t* __restrict__ mask) {
  vg::pdl_entry();
  Philox ph(k.seed, eff_offset(k.offset, k.step_ptr));
  const unsigned long long ebase = (unsigned long long)k.sample_offset * (unsigned long long)k.hw * (unsigned long long)k.c;
  const long long total = k.rows * k.c;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
    mask[i] = k.thr16 ? (keep1(ph, ebase + (unsigned long long)i, k.thr16) ? 1 : 0) : 1;
}

__global__ void dropout2d_scale_kernel(float* __restrict__ scale, long long total, int c, float p, unsigned long long seed,
                                       unsigned long long offset, const unsigned long long* step_ptr, long long sample_offset) {
  vg::pdl_entry();
  Philox ph(seed, eff_offset(offset, step_ptr));
  uint32_t thr = drop_threshold(p);
  float sc = 1.0f / (1.0f - p);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    unsigned long long e = (unsigned long long)sample_offset * c + (unsigned long long)i;
    scale[i] = (p <= 0.f) ? 1.f : (ph.word(e) >= thr ? sc : 0.f);
  }
}

__global__ void philox_normal_kernel(float* __restrict__ out, long long n, unsigned long long seed, unsigned long long offset,
                                     const unsigned long long* step_ptr, long long start) {
  vg::pdl_entry();
  Philox ph(seed, eff_offset(offset, step_ptr));
  const long long nblk = (n + 3) / 4;
  for (long long bidx = (long long)blockIdx.x * blockDim.x + threadIdx.x; bidx < nblk; bidx += (long long)gridDim.x * blockDim.x) {
    // element e = start + 4*bidx + l uses block (e >> 2) only when start % 4 == 0 (enforced by the host)
    uint4 r = ph.block((unsigned long long)(start / 4 + bidx));
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
    float z[4];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float u1 = ((float)w[2 * h] + 0.5f) * 2.3283064365386963e-10f;  // (0,1]
      float u2 = ((float)w[2 * h + 1] + 0.5f) * 2.3283064365386963e-10f;
      u1 = fminf(fmaxf(u1, 1e-12f), 1.0f);
      float rad = sqrtf(-2.0f * logf(u1));
      float s, c;
      sincospif(2.0f * u2, &s, &c);
      z[2 * h] = rad * c;
      z[2 * h + 1] = rad * s;
    }
#pragma unroll
    for (int l = 0; l < 4; ++l)
      if (4 * bidx + l < n) out[4 * bidx + l] = z[l];
  }
}

// u[i] = (word(start + i) >> 8) * 2^-24 in [0, 1): the gradient-penalty interpolation weights (README.md:719)
__global__ void philox_uniform_kernel(float* __restrict__ out, long long n, unsigned long long seed, unsigned long long offset,
                                      const unsigned long long* step_ptr, long long start) {
  vg::pdl_entry();
  Philox ph(seed, eff_offset(offset, step_ptr));
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const unsigned long long e = (unsigned long long)(start + i);
    uint4 r = ph.block(e >> 2);
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
    out[i] = (float)(w[e & 3] >> 8) * 5.9604644775390625e-08f;
  }
}

}  // namespace vg

// ==========================================================================================
// C ABI
// ==========================================================================================
using namespace vg;

namespace vg {
// bn_stream.cu: the bulk-copy pipelined implementations (default whenever the tensor qualifies)
bool bn_stream_ok(const VgBnDesc* d, const void* p0, const void* p1, const void* p2, const void* p3);
int bn_stream_stats(const void* x, const VgBnDesc* d, double* sums, cudaStream_t s);
int bn_stream_act_forward(const void* x, const VgBnChannel* bn, const VgBnDesc* d, void* y, cudaStream_t s);
int bn_stream_bwd_reduce(const void* dy, const void* x, const float* mean_rstd, const float* gamma, const float* beta,
                         const VgBnDesc* d, double* sums, cudaStream_t s);
int bn_stream_bwd_apply(const void* dy, const void* x, const float* mean_rstd, const float* gamma, const float* beta,
                        const double* sums, double count, const VgBnDesc* d, const float* out_colscale, const void* addend,
                        void* dx, float* dgamma, float* dbeta, float param_scale, cudaStream_t s);
int bn_stream_add(const void* x0, const VgBnChannel* bn_a, const void* x1, const VgBnChannel* bn_b, const VgBnDesc* d, void* out,
                  double* stats, cudaStream_t s);
int bn_stream_add_dual(const void* x0, const void* x1, const float* post_scale, const float* post_shift, float post_slope,
                       const VgBnDesc* d, void* out, void* out2, cudaStream_t s);
}  // namespace vg

static int check_desc(const VgBnDesc* d) {
  VG_CHECK_ARG(d != nullptr, "VgBnDesc is null");
  VG_CHECK_ARG(d->rows >= 0 && d->c > 0 && d->hw > 0, "bad VgBnDesc dims rows=%lld c=%d hw=%d", d->rows, d->c, d->hw);
  VG_CHECK_ARG(d->dtype == VG_F32 || d->dtype == VG_BF16, "bad dtype %d", d->dtype);
  VG_CHECK_ARG(d->drop_p >= 0.f && d->drop_p < 1.f, "bad dropout p %f", d->drop_p);
  return VG_OK;
}

// decide the mapping: 0 scalar, 1 vector, 2 folded single channel
static inline int path_for(const VgBnDesc* d) {
  if (vec_ok(d->c)) return 1;
  if (d->c == 1 && d->rows % 8 == 0 && d->rows > 0) return 2;
  return 0;
}
static inline size_t vec_smem() { return (size_t)2 * 8 * kBnThreads * sizeof(float); }

extern "C" int vg_bn_stats(const void* x, const VgBnDesc* d, double* sums, vg_stream_t stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  VG_CHECK_ARG(x && sums, "null pointer");
  if (d->rows == 0) return VG_OK;
  cudaStream_t s = as_stream(stream);
  {
    VgBnDesc dd = *d;
    dd.drop_p = 0.f;                 // statistics never draw dropout bits
    if (bn_stream_ok(&dd, x, nullptr, nullptr, nullptr)) return bn_stream_stats(x, &dd, sums, s);
  }
  int path = path_for(d);
  if (path) {
    bool fold = path == 2;
    long long rows = fold ? d->rows / 8 : d->rows;
    int cv = fold ? 8 : d->c;
    RowMap m = make_rowmap(cv);
    int grid = grid_for(rows, m.rpb, kUnrollWide * 2, kReduceBlocksPerSm);
    double* part = nullptr;
    if (g_det.on && !(part = (double*)det_scratch((size_t)grid * 2 * d->c * sizeof(double)))) return VG_EINVAL;
    if (d->dtype == VG_BF16)
      vg::Launch(grid, kBnThreads, vec_smem(), s)(bn_stats_vec_kernel<__nv_bfloat16>, (const __nv_bfloat16*)x, rows, d->c, fold, sums, part);
    else
      vg::Launch(grid, kBnThreads, vec_smem(), s)(bn_stats_vec_kernel<float>, (const float*)x, rows, d->c, fold, sums, part);
    if (part) {
      VG_LAUNCHED();
      return ordered_reduce_f64(part, grid, 2LL * d->c, sums, s);
    }
  } else {
    VG_DET_UNSUPPORTED("BatchNorm statistics with C % 8 != 0");
    long long total = d->rows * d->c;
    int grid = (int)std::min<long long>(cdiv(total, 256 * 8), (long long)num_sms() * 4);
    size_t sm = (size_t)2 * d->c * sizeof(double);
    VG_CHECK_ARG(sm <= 48 * 1024, "scalar BN path supports c <= 3072 (c=%d)", d->c);
    if (d->dtype == VG_BF16)
      vg::Launch(grid, 256, sm, s)(bn_stats_scalar_kernel<__nv_bfloat16>, (const __nv_bfloat16*)x, total, d->c, sums);
    else
      vg::Launch(grid, 256, sm, s)(bn_stats_scalar_kernel<float>, (const float*)x, total, d->c, sums);
  }
  VG_LAUNCHED();
  return VG_OK;
}

extern "C" int vg_bn_finalize(const double* sums, double count, int c, float eps, float momentum, float* running_mean,
                              float* running_var, float* mean_rstd, vg_stream_t stream) {
  VG_CHECK_ARG(sums && mean_rstd && c > 0 && count > 0, "bad args");
  VG_CHECK_ARG((running_mean == nullptr) == (running_var == nullptr), "running_mean/var must both be given or both null");
  vg::Launch((c + 127) / 128, 128, 0, as_stream(stream))(bn_finalize_kernel, sums, count, c, eps, momentum, running_mean, running_var, mean_rstd);
  VG_LAUNCHED();
  return VG_OK;
}

extern "C" int vg_bn_eval_stats(const float* running_mean, const float* running_var, int c, float eps, float* mean_rstd,
                                vg_stream_t stream) {
  VG_CHECK_ARG(running_mean && running_var && mean_rstd && c > 0, "bad args");
  vg::Launch((c + 127) / 128, 128, 0, as_stream(stream))(bn_eval_stats_kernel, running_mean, running_var, c, eps, mean_rstd);
  VG_LAUNCHED();
  return VG_OK;
}

extern "C" int vg_bn_param_grads_scaled(const double* sums, int c, float scale, float* dgamma, float* dbeta, vg_stream_t stream) {
  VG_CHECK_ARG(sums && c > 0, "bad args");
  vg::Launch((c + 127) / 128, 128, 0, as_stream(stream))(bn_param_grads_kernel, sums, c, (double)scale, dgamma, dbeta);
  VG_LAUNCHED();
  return VG_OK;
}

extern "C" int vg_bn_param_grads(const double* sums, int c, float* dgamma, float* dbeta, vg_stream_t stream) {
  return vg_bn_param_grads_scaled(sums, c, 1.0f, dgamma, dbeta, stream);
}

template <typename T>
static int bn_act_forward_t(const T* x, const float* mr, const float* gamma, const float* beta, const VgBnDesc* d, T* y,
                            cudaStream_t s) {
  BnK k = make_bnk(d);
  int path = path_for(d);
  if (path) {
    k.fold = path == 2;
    long long rows = k.fold ? d->rows / 8 : d->rows;
    k.rows = rows;
    RowMap m = make_rowmap(k.fold ? 8 : d->c);
    int grid = grid_for(rows, m.rpb, kUnrollWide * 2);
    if (k.thr16)
      vg::Launch(grid, kBnThreads, 0, s)(bn_act_fwd_vec_kernel<T, true>, x, mr, gamma, beta, k, y);
    else
      vg::Launch(grid, kBnThreads, 0, s)(bn_act_fwd_vec_kernel<T, false>, x, mr, gamma, beta, k, y);
  } else {
    long long total = d->rows * d->c;
    int grid = (int)std::min<long long>(cdiv(total, 256 * 4), (long long)num_sms() * 8);
    vg::Launch(grid, 256, 0, s)(bn_act_fwd_scalar_kernel<T>, x, mr, gamma, beta, k, y);
  }
  VG_LAUNCHED();
  return VG_OK;
}

extern "C" int vg_bn_act_forward(const void* x, const float* mean_rstd, const float* gamma, const float* beta,
                                 const VgBnDesc* d, void* y, vg_stream_t stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  VG_CHECK_ARG(x && mean_rstd && gamma && beta && y, "null pointer");
  if (d->rows == 0) return VG_OK;
  if (bn_stream_ok(d, x, y, nullptr, nullptr)) {
    VgBnChannel ch{};
    ch.gamma = gamma; ch.beta = beta; ch.mean_rstd_in = mean_rstd;
    return bn_stream_act_forward(x, &ch, d, y, as_stream(stream));
  }
  if (d->dtype == VG_BF16)
    return bn_act_forward_t<__nv_bfloat16>((const __nv_bfloat16*)x, mean_rstd, gamma, beta, d, (__nv_bfloat16*)y, as_stream(stream));
  return bn_act_forward_t<float>((const float*)x, mean_rstd, gamma, beta, d, (float*)y, as_stream(stream));
}

// (mean, rstd) of a VgBnChannel through the stand-alone finalize / eval-stats kernels: the composed path for tensors
// the streaming kernels do not take (odd channel counts, misaligned views)
static int channel_mean_rstd(const VgBnChannel* bn, const VgBnDesc* d, const float** mr, vg_stream_t stream) {
  if (bn->mean_rstd_in != nullptr) { *mr = bn->mean_rstd_in; return VG_OK; }
  VG_CHECK_ARG(bn->mean_rstd_out != nullptr, "mean_rstd_out is required when (mean, rstd) are not given");
  *mr = bn->mean_rstd_out;
  if (d->training && bn->sums != nullptr)
    return vg_bn_finalize(bn->sums, bn->count, d->c, bn->eps, bn->momentum, bn->running_mean, bn->running_var, bn->mean_rstd_out, stream);
  VG_CHECK_ARG(bn->running_mean && bn->running_var, "eval-mode BatchNorm needs running statistics");
  return vg_bn_eval_stats(bn->running_mean, bn->running_var, d->c, bn->eps, bn->mean_rstd_out, stream);
}
static int check_channel(const VgBnChannel* bn, const VgBnDesc* d) {
  VG_CHECK_ARG(bn->gamma && bn->beta, "BatchNorm needs gamma / beta");
  if (bn->mean_rstd_in == nullptr) {
    if (d->training && bn->sums != nullptr) {
      VG_CHECK_ARG(bn->count > 0, "count must be positive");
      VG_CHECK_ARG((bn->running_mean == nullptr) == (bn->running_var == nullptr), "running_mean/var must both be given or both null");
    } else {
      VG_CHECK_ARG(bn->running_mean && bn->running_var, "eval-mode BatchNorm needs running statistics");
    }
  }
  return VG_OK;
}

extern "C" int vg_bn_act_forward_fused(const void* x, const VgBnChannel* bn, const VgBnDesc* d, void* y, vg_stream_t stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  VG_CHECK_ARG(x && bn && y, "null pointer");
  if ((rc = check_channel(bn, d))) return rc;
  if (d->rows == 0) return VG_OK;
  if (bn_stream_ok(d, x, y, nullptr, nullptr)) return bn_stream_act_forward(x, bn, d, y, as_stream(stream));
  const float* mr = nullptr;
  if ((rc = channel_mean_rstd(bn, d, &mr, stream))) return rc;
  return vg_bn_act_forward(x, mr, bn->gamma, bn->beta, d, y, stream);
}

template <typename T, bool APPLY>
static int bn_act_backward_t(const T* dy, const T* x, const float* mr, const float* gamma, const float* beta, const VgBnDesc* d,
                             double* sums_out, const double* sums_in, double count, const float* ocs, const T* addend, T* dx,
                             cudaStream_t s) {
  BnK k = make_bnk(d);
  int path = path_for(d);
  if (path == 2 && ocs != nullptr) path = 0;  // per-sample colscale needs real row indices
  if (path) {
    k.fold = path == 2;
    long long rows = k.fold ? d->rows / 8 : d->rows;
    k.rows = rows;
    RowMap m = make_rowmap(k.fold ? 8 : d->c);
    int grid = grid_for(rows, m.rpb, APPLY ? kUnroll : kUnrollWide, APPLY ? kApplyBlocksPerSm : kReduceBlocksPerSm);
    size_t sm = APPLY ? 0 : vec_smem();
    double* part = nullptr;
    if (!APPLY && g_det.on && !(part = (double*)det_scratch((size_t)grid * 2 * d->c * sizeof(double)))) return VG_EINVAL;
    if (k.thr16)
      vg::Launch(grid, kBnThreads, sm, s)(bn_act_bwd_vec_kernel<T, true, APPLY>, dy, x, mr, gamma, beta, k, sums_out, part, sums_in, count, ocs, addend, dx);
    else
      vg::Launch(grid, kBnThreads, sm, s)(bn_act_bwd_vec_kernel<T, false, APPLY>, dy, x, mr, gamma, beta, k, sums_out, part, sums_in, count, ocs, addend, dx);
    if (part) {
      VG_LAUNCHED();
      return ordered_reduce_f64(part, grid, 2LL * d->c, sums_out, s);
    }
  } else {
    if (!APPLY) VG_DET_UNSUPPORTED("BatchNorm backward with C % 8 != 0");
    long long total = d->rows * d->c;
    int grid = (int)std::min<long long>(cdiv(total, 256 * 4), (long long)num_sms() * 8);
    size_t sm = APPLY ? 0 : (size_t)2 * d->c * sizeof(double);
    VG_CHECK_ARG(sm <= 48 * 1024, "scalar BN path supports c <= 3072 (c=%d)", d->c);
    vg::Launch(grid, 256, sm, s)(bn_act_bwd_scalar_kernel<T, APPLY>, dy, x, mr, gamma, beta, k, sums_out, sums_in, count, ocs, addend, dx);
  }
  VG_LAUNCHED();
  return VG_OK;
}

extern "C" int vg_bn_act_backward_reduce(const void* dy, const void* x, const float* mean_rstd, const float* gamma,
                                         const float* beta, const VgBnDesc* d, double* sums, vg_stream_t stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  VG_CHECK_ARG(dy && x && mean_rstd && gamma && beta && sums, "null pointer");
  if (d->rows == 0) return VG_OK;
  if (bn_stream_ok(d, dy, x, nullptr, nullptr)) return bn_stream_bwd_reduce(dy, x, mean_rstd, gamma, beta, d, sums, as_stream(stream));
  if (d->dtype == VG_BF16)
    return bn_act_backward_t<__nv_bfloat16, false>((const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, mean_rstd, gamma, beta, d, sums,
                                                   nullptr, 1.0, nullptr, nullptr, nullptr, as_stream(stream));
  return bn_act_backward_t<float, false>((const float*)dy, (const float*)x, mean_rstd, gamma, beta, d, sums, nullptr, 1.0, nullptr,
                                         nullptr, nullptr, as_stream(stream));
}

extern "C" int vg_bn_act_backward_apply_fused(const void* dy, const void* x, const float* mean_rstd, const float* gamma,
                                              const float* beta, const double* sums, double count, const VgBnDesc* d,
                                              const float* out_colscale, const void* addend, void* dx, float* dgamma,
                                              float* dbeta, float param_scale, vg_stream_t stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  VG_CHECK_ARG(dy && x && mean_rstd && gamma && beta && dx, "null pointer");
  VG_CHECK_ARG(!d->training || (sums != nullptr && count > 0), "training-mode BN backward needs sums and count");
  VG_CHECK_ARG((dgamma == nullptr && dbeta == nullptr) || sums != nullptr, "parameter gradients need the sums");
  if (d->rows == 0) return VG_OK;
  const bool fold_cs = (d->c == 1 && out_colscale != nullptr);      // per-sample scale needs real row indices
  if (!fold_cs && bn_stream_ok(d, dy, x, addend, dx))
    return bn_stream_bwd_apply(dy, x, mean_rstd, gamma, beta, sums, count, d, out_colscale, addend, dx, dgamma, dbeta, param_scale,
                               as_stream(stream));
  rc = vg_bn_act_backward_apply(dy, x, mean_rstd, gamma, beta, sums, count, d, out_colscale, addend, dx, stream);
  if (rc) return rc;
  if (dgamma != nullptr || dbeta != nullptr) rc = vg_bn_param_grads_scaled(sums, d->c, param_scale, dgamma, dbeta, stream);
  return rc;
}

extern "C" int vg_bn_act_backward_apply(const void* dy, const void* x, const float* mean_rstd, const float* gamma,
                                        const float* beta, const double* sums, double count, const VgBnDesc* d,
                                        const float* out_colscale, const void* addend, void* dx, vg_stream_t stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  VG_CHECK_ARG(dy && x && mean_rstd && gamma && beta && dx, "null pointer");
  VG_CHECK_ARG(!d->training || (sums != nullptr && count > 0), "training-mode BN backward needs sums and count");
  if (d->rows == 0) return VG_OK;
  if (!(d->c == 1 && out_colscale != nullptr) && bn_stream_ok(d, dy, x, addend, dx))
    return bn_stream_bwd_apply(dy, x, mean_rstd, gamma, beta, sums, count, d, out_colscale, addend, dx, nullptr, nullptr, 1.f,
                               as_stream(stream));
  if (d->dtype == VG_BF16)
    return bn_act_backward_t<__nv_bfloat16, true>((const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, mean_rstd, gamma, beta, d, nullptr,
                                                  sums, count, out_colscale, (const __nv_bfloat16*)addend, (__nv_bfloat16*)dx,
                                                  as_stream(stream));
  return bn_act_backward_t<float, true>((const float*)dy, (const float*)x, mean_rstd, gamma, beta, d, nullptr, sums, count,
                                        out_colscale, (const float*)addend, (float*)dx, as_stream(stream));
}

template <typename T, bool APPLY>
static int bn_dbl_bwd_t(const T* dy, const T* x, const T* G, const float* mean_rstd, const float* gamma, const float* beta,
                        const VgBnDesc* d, const float* colscale, double* sums_out, const double* sums_in, double count, T* g_dy,
                        T* g_x, cudaStream_t s) {
  BnK k = make_bnk(d);
  RowMap m = make_rowmap(d->c);
  int grid = grid_for(d->rows, m.rpb, kUnroll, APPLY ? kApplyBlocksPerSm : kReduceBlocksPerSm);
  const size_t smem = APPLY ? 0 : (size_t)5 * 8 * kBnThreads * sizeof(float);
  double* part = nullptr;
  if (!APPLY && g_det.on && !(part = (double*)det_scratch((size_t)grid * 5 * d->c * sizeof(double)))) return VG_EINVAL;
  vg::Launch(grid, kBnThreads, smem, s)(bn_dbl_bwd_vec_kernel<T, APPLY>, dy, x, G, mean_rstd, gamma, beta, k, colscale, sums_out, part, sums_in,
                                        count, g_dy, g_x);
  VG_LAUNCHED();
  if (part) return ordered_reduce_f64(part, grid, 5LL * d->c, sums_out, s);
  return VG_OK;
}

extern "C" int vg_bn_act_double_backward_reduce(const void* dy, const void* x, const void* G, const float* mean_rstd,
                                                const float* gamma, const float* beta, const VgBnDesc* d, const float* colscale,
                                                double* sums5, vg_stream_t stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  VG_CHECK_ARG(dy && x && G && mean_rstd && gamma && beta && sums5, "null pointer");
  VG_CHECK_ARG(vec_ok(d->c) && d->training && d->drop_p == 0.f, "needs training-mode BatchNorm, channels % 8 == 0 and <= 2048, no dropout");
  if (d->rows == 0) return VG_OK;
  if (d->dtype == VG_BF16) {
    static std::once_flag once;
    static cudaError_t attr_err = cudaSuccess;
    std::call_once(once, [] { attr_err = cudaFuncSetAttribute(bn_dbl_bwd_vec_kernel<__nv_bfloat16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 48 * 1024); });
    VG_CUDA(attr_err);
    return bn_dbl_bwd_t<__nv_bfloat16, false>((const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, (const __nv_bfloat16*)G, mean_rstd, gamma, beta,
                                              d, colscale, sums5, nullptr, 1.0, nullptr, nullptr, as_stream(stream));
  }
  return bn_dbl_bwd_t<float, false>((const float*)dy, (const float*)x, (const float*)G, mean_rstd, gamma, beta, d, colscale, sums5, nullptr,
                                    1.0, nullptr, nullptr, as_stream(stream));
}

extern "C" int vg_bn_act_double_backward_apply(const void* dy, const void* x, const void* G, const float* mean_rstd,
                                               const float* gamma, const float* beta, const double* sums5, double count,
                                               const VgBnDesc* d, const float* colscale, void* g_dy, void* g_x, vg_stream_t stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  VG_CHECK_ARG(dy && x && G && mean_rstd && gamma && beta && sums5 && g_dy && g_x && count > 0, "bad args");
  VG_CHECK_ARG(vec_ok(d->c) && d->training && d->drop_p == 0.f, "needs training-mode BatchNorm, channels % 8 == 0 and <= 2048, no dropout");
  if (d->rows == 0) return VG_OK;
  if (d->dtype == VG_BF16)
    return bn_dbl_bwd_t<__nv_bfloat16, true>((const __nv_bfloat16*)dy, (const __nv_bfloat16*)x, (const __nv_bfloat16*)G, mean_rstd, gamma, beta,
                                             d, colscale, nullptr, sums5, count, (__nv_bfloat16*)g_dy, (__nv_bfloat16*)g_x, as_stream(stream));
  return bn_dbl_bwd_t<float, true>((const float*)dy, (const float*)x, (const float*)G, mean_rstd, gamma, beta, d, colscale, nullptr, sums5,
                                   count, (float*)g_dy, (float*)g_x, as_stream(stream));
}

template <typename T>
static int bn_add_t(const T* a, const float* mra, const float* ga, const float* ba, const T* b, const float* mrb, const float* gb,
                    const float* bb, const VgBnDesc* d, T* out, double* stats, cudaStream_t s) {
  BnK k = make_bnk(d);
  int path = path_for(d);
  if (path) {
    k.fold = path == 2;
    long long rows = k.fold ? d->rows / 8 : d->rows;
    k.rows = rows;
    RowMap m = make_rowmap(k.fold ? 8 : d->c);
    int grid = grid_for(rows, m.rpb, kUnroll, stats ? kReduceBlocksPerSm : kApplyBlocksPerSm);
    double* part = nullptr;
    if (stats && g_det.on && !(part = (double*)det_scratch((size_t)grid * 2 * d->c * sizeof(double)))) return VG_EINVAL;
    if (stats)
      vg::Launch(grid, kBnThreads, vec_smem(), s)(bn_add_vec_kernel<T, true>, a, mra, ga, ba, b, mrb, gb, bb, k, out, stats, part);
    else
      vg::Launch(grid, kBnThreads, 0, s)(bn_add_vec_kernel<T, false>, a, mra, ga, ba, b, mrb, gb, bb, k, out, stats, part);
    if (part) {
      VG_LAUNCHED();
      return ordered_reduce_f64(part, grid, 2LL * d->c, stats, s);
    }
  } else {
    if (stats) VG_DET_UNSUPPORTED("residual add + statistics with C % 8 != 0");
    long long total = d->rows * d->c;
    int grid = (int)std::min<long long>(cdiv(total, 256 * 4), (long long)num_sms() * 8);
    size_t sm = stats ? (size_t)2 * d->c * sizeof(double) : 0;
    VG_CHECK_ARG(sm <= 48 * 1024, "scalar BN path supports c <= 3072 (c=%d)", d->c);
    vg::Launch(grid, 256, sm, s)(bn_add_scalar_kernel<T>, a, mra, ga, ba, b, mrb, gb, bb, k, out, stats);
  }
  VG_LAUNCHED();
  return VG_OK;
}

extern "C" int vg_bn_add_forward(const void* a, const float* mean_rstd_a, const float* gamma_a, const float* beta_a,
                                 const void* b, const float* mean_rstd_b, const float* gamma_b, const float* beta_b,
                                 const VgBnDesc* d, void* out, double* stats, vg_stream_t stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  VG_CHECK_ARG(a && b && out, "null pointer");
  VG_CHECK_ARG(!mean_rstd_a || (gamma_a && beta_a), "bnA needs gamma/beta");
  VG_CHECK_ARG(!mean_rstd_b || (gamma_b && beta_b), "bnB needs gamma/beta");
  if (d->rows == 0) return VG_OK;
  if (bn_stream_ok(d, a, b, out, nullptr)) {
    VgBnChannel ca{}, cb{};
    ca.gamma = gamma_a; ca.beta = beta_a; ca.mean_rstd_in = mean_rstd_a;
    cb.gamma = gamma_b; cb.beta = beta_b; cb.mean_rstd_in = mean_rstd_b;
    return bn_stream_add(a, mean_rstd_a ? &ca : nullptr, b, mean_rstd_b ? &cb : nullptr, d, out, stats, as_stream(stream));
  }
  if (d->dtype == VG_BF16)
    return bn_add_t<__nv_bfloat16>((const __nv_bfloat16*)a, mean_rstd_a, gamma_a, beta_a, (const __nv_bfloat16*)b, mean_rstd_b, gamma_b,
                                   beta_b, d, (__nv_bfloat16*)out, stats, as_stream(stream));
  return bn_add_t<float>((const float*)a, mean_rstd_a, gamma_a, beta_a, (const float*)b, mean_rstd_b, gamma_b, beta_b, d, (float*)out,
                         stats, as_stream(stream));
}

extern "C" int vg_bn_add_forward_fused(const void* a, const VgBnChannel* bn_a, const void* b, const VgBnChannel* bn_b,
                                       const VgBnDesc* d, void* out, double* stats, vg_stream_t stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  VG_CHECK_ARG(a && b && out, "null pointer");
  if (bn_a != nullptr && (rc = check_channel(bn_a, d))) return rc;
  if (bn_b != nullptr && (rc = check_channel(bn_b, d))) return rc;
  if (d->rows == 0) return VG_OK;
  if (bn_stream_ok(d, a, b, out, nullptr)) return bn_stream_add(a, bn_a, b, bn_b, d, out, stats, as_stream(stream));
  const float *mra = nullptr, *mrb = nullptr;
  if (bn_a != nullptr && (rc = channel_mean_rstd(bn_a, d, &mra, stream))) return rc;
  if (bn_b != nullptr && (rc = channel_mean_rstd(bn_b, d, &mrb, stream))) return rc;
  return vg_bn_add_forward(a, mra, bn_a ? bn_a->gamma : nullptr, bn_a ? bn_a->beta : nullptr, b, mrb, bn_b ? bn_b->gamma : nullptr,
                           bn_b ? bn_b->beta : nullptr, d, out, stats, stream);
}

extern "C" int vg_add_dual_forward(const void* a, const void* b, const float* post_scale, const float* post_shift, float post_slope,
                                   const VgBnDesc* d, void* out, void* out2, vg_stream_t stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  VG_CHECK_ARG(a && b && out && out2 && post_scale && post_shift, "null pointer");
  if (d->rows == 0) return VG_OK;
  VgBnDesc dd = *d;
  dd.drop_p = 0.f;
  if (!bn_stream_ok(&dd, a, b, out, out2) || d->c % 8 != 0) {
    set_error("vg_add_dual_forward needs channels %% 8 == 0 (<= 2048) and 16-byte aligned tensors");
    return VG_EUNSUPPORTED;
  }
  return bn_stream_add_dual(a, b, post_scale, post_shift, post_slope, &dd, out, out2, as_stream(stream));
}

extern "C" int vg_lrelu_backward(const void* dy, const void* y_ref, long long n, int dtype, float slope, void* dx,
                                 vg_stream_t stream) {
  VG_CHECK_ARG(dy && y_ref && dx && n >= 0, "bad args");
  if (n == 0) return VG_OK;
  int grid = (int)std::min<long long>(cdiv(n, 256 * 4), (long long)num_sms() * 8);
  if (dtype == VG_BF16)
    vg::Launch(grid, 256, 0, as_stream(stream))(lrelu_bwd_kernel<__nv_bfloat16>, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)y_ref, n, slope,
                                                                         (__nv_bfloat16*)dx);
  else
    vg::Launch(grid, 256, 0, as_stream(stream))(lrelu_bwd_kernel<float>, (const float*)dy, (const float*)y_ref, n, slope, (float*)dx);
  VG_LAUNCHED();
  return VG_OK;
}

extern "C" int vg_add(const void* a, const void* b, long long n, int dtype, void* out, vg_stream_t stream) {
  VG_CHECK_ARG(a && b && out && n >= 0, "bad args");
  if (n == 0) return VG_OK;
  cudaStream_t s = as_stream(stream);
  bool aligned = ((uintptr_t)a % 32 == 0) && ((uintptr_t)b % 32 == 0) && ((uintptr_t)out % 32 == 0) && (n % 8 == 0);
  if (aligned) {
    long long nv = n / 8;
    int grid = (int)std::min<long long>(cdiv(nv, 256 * 2), (long long)num_sms() * 8);
    if (dtype == VG_BF16)
      vg::Launch(grid, 256, 0, s)(add_vec_kernel<__nv_bfloat16>, (const __nv_bfloat16*)a, (const __nv_bfloat16*)b, nv, (__nv_bfloat16*)out);
    else
      vg::Launch(grid, 256, 0, s)(add_vec_kernel<float>, (const float*)a, (const float*)b, nv, (float*)out);
  } else {
    int grid = (int)std::min<long long>(cdiv(n, 256 * 4), (long long)num_sms() * 8);
    if (dtype == VG_BF16)
      vg::Launch(grid, 256, 0, s)(add_kernel<__nv_bfloat16>, (const __nv_bfloat16*)a, (const __nv_bfloat16*)b, n, (__nv_bfloat16*)out);
    else
      vg::Launch(grid, 256, 0, s)(add_kernel<float>, (const float*)a, (const float*)b, n, (float*)out);
  }
  VG_LAUNCHED();
  return VG_OK;
}

extern "C" int vg_dropout_mask(const VgBnDesc* d, uint8_t* mask, vg_stream_t stream) {
  int rc = check_desc(d);
  if (rc) return rc;
  VG_CHECK_ARG(mask, "null pointer");
  if (d->rows == 0) return VG_OK;
  BnK k = make_bnk(d);
  long long total = d->rows * d->c;
  int grid = (int)std::min<long long>(cdiv(total, 256 * 4), (long long)num_sms() * 8);
  vg::Launch(grid, 256, 0, as_stream(stream))(dropout_mask_kernel, k, mask);
  VG_LAUNCHED();
  return VG_OK;
}

extern "C" int vg_dropout2d_scale(float* scale, int n, int c, float p, unsigned long long seed, unsigned long long offset,
                                  const unsigned long long* step_ptr, long long sample_offset, vg_stream_t stream) {
  VG_CHECK_ARG(scale && n >= 0 && c > 0 && p >= 0.f && p < 1.f, "bad args");
  long long total = (long long)n * c;
  if (total == 0) return VG_OK;
  int grid = (int)std::min<long long>(cdiv(total, 256), (long long)num_sms() * 4);
  vg::Launch(grid, 256, 0, as_stream(stream))(dropout2d_scale_kernel, scale, total, c, p, seed, offset, step_ptr, sample_offset);
  VG_LAUNCHED();
  return VG_OK;
}

__global__ void counter_add_kernel(unsigned long long* c, unsigned long long inc) {
  vg::pdl_entry(); *c += inc; }

extern "C" int vg_counter_add(unsigned long long* counter, unsigned long long inc, vg_stream_t stream) {
  VG_CHECK_ARG(counter, "null pointer");
  vg::Launch(1, 1, 0, as_stream(stream))(counter_add_kernel, counter, inc);
  VG_LAUNCHED();
  return VG_OK;
}

extern "C" int vg_philox_uniform(float* out, long long n, unsigned long long seed, unsigned long long offset,
                                 const unsigned long long* step_ptr, long long start, vg_stream_t stream) {
  VG_CHECK_ARG(out && n >= 0 && start >= 0, "bad args");
  if (n == 0) return VG_OK;
  int grid = (int)std::min<long long>(cdiv(n, 256), (long long)num_sms() * 8);
  vg::Launch(grid, 256, 0, as_stream(stream))(philox_uniform_kernel, out, n, seed, offset, step_ptr, start);
  VG_LAUNCHED();
  return VG_OK;
}

extern "C" int vg_philox_normal(float* out, long long n, unsigned long long seed, unsigned long long offset,
                                const unsigned long long* step_ptr, long long start, vg_stream_t stream) {
  VG_CHECK_ARG(out && n >= 0 && start >= 0 && start % 4 == 0, "bad args (start must be a multiple of 4)");
  if (n == 0) return VG_OK;
  long long nblk = (n + 3) / 4;
  int grid = (int)std::min<long long>(cdiv(nblk, 256), (long long)num_sms() * 8);
  vg::Launch(grid, 256, 0, as_stream(stream))(philox_normal_kernel, out, n, seed, offset, step_ptr, start);
  VG_LAUNCHED();
  return VG_OK;
}
