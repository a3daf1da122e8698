// CUDA-core convolution kernels (NHWC): the fp32 parity path, and the product path for the
// degenerate layers (c_in == 1 or c_out == 1, README.md:230,289,441) that are memory-bound and
// have no GEMM shape worth a tensor-core tile.  Also the weight re-layout ("pack") kernel.
//
// Two index patterns cover Conv2d and ConvTranspose2d, forward and dgrad:
//   gather : out[o]  = sum_k in[o*s - p + k] . W_k        (Conv2d fwd, ConvTranspose2d dgrad)
//   scatter: out[j]  = sum_{k : (j+p-k) % s == 0} in[(j+p-k)/s] . W_k
//                                                          (ConvTranspose2d fwd, Conv2d dgrad)
// W_k is [tap][c_red][c_out'] with c_out' contiguous, so a thread owning 8 output channels
// reads 8 contiguous weights per (tap, c_red).
#include <algorithm>
#include <string.h>
#include "vg_common.cuh"

namespace vg {

struct ConvGeom {
  int n, hi, wi, cr;   // input of THIS kernel (reduction channels cr)
  int ho, wo, co;      // output of this kernel
  int kh, kw, stride, pad;
};

// ---- weight pack ---------------------------------------------------------------------------
template <typename T>
__global__ void pack_weights_kernel(const float* __restrict__ w, const float* __restrict__ sigma, int c_out, int c_in, int taps,
                                    int transposed, T* __restrict__ pack_kn, T* __restrict__ pack_nk) {
  vg::pdl_entry();
  const long long total = (long long)taps * c_out * c_in;
  const float inv = sigma ? 1.0f / *sigma : 1.0f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    // i enumerates the torch layout so the read is coalesced
    int tap = (int)(i % taps);
    long long r = i / taps;
    int co, ci;
    if (transposed) { co = (int)(r % c_out); ci = (int)(r / c_out); }   // [ci][co][tap]
    else            { ci = (int)(r % c_in);  co = (int)(r / c_in); }    // [co][ci][tap]
    T v = from_f32<T>(w[i] * inv);
    if (pack_kn) pack_kn[((long long)tap * c_out + co) * c_in + ci] = v;
    if (pack_nk) pack_nk[((long long)tap * c_in + ci) * c_out + co] = v;
  }
}

// Tiled variant for the layer sizes the tensor-core path uses: a block stages a 16 x 32 x TAPS tile of the
// torch weight [r0][r1][tap] in shared memory (coalesced reads) and writes BOTH packed layouts in runs
// of 16 / 32 consecutive elements, i.e. whole 32-byte sectors; the element-wise kernel above scatters 2-byte
// writes with a stride of c_out*c_in elements.  TAPS is a template parameter and the loops are nested so that
// no thread divides by a run-time value (those divisions made a 16-block launch take 15 us).
constexpr int kPackR0 = 16, kPackR1 = 32;
template <typename T, int TAPS>
__global__ void __launch_bounds__(256) pack_weights_tiled_kernel(const float* __restrict__ w, const float* __restrict__ sigma, int n0, int n1,
                                                                 int transposed, T* __restrict__ pack_kn, T* __restrict__ pack_nk) {
  vg::pdl_entry();
  constexpr int TP = TAPS | 1;                      // odd strides: no bank conflicts
  constexpr int ROW = kPackR1 * TP + 1;
  __shared__ float tile[kPackR0 * ROW];
  const float inv = sigma ? 1.0f / *sigma : 1.0f;
  const int r0b = blockIdx.y * kPackR0, r1b = blockIdx.x * kPackR1;
  const int n1t = min(kPackR1, n1 - r1b), n0t = min(kPackR0, n0 - r0b);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // load: for each r0 the (r1, tap) block is contiguous in the torch layout; warp w takes rows w, w+8
  const int run = n1t * TAPS;
  for (int a = warp; a < n0t; a += 8) {
    const float* src = w + ((long long)(r0b + a) * n1 + r1b) * TAPS;
    for (int b = lane; b < run; b += 32) {
      const int r1l = b / TAPS, tap = b - r1l * TAPS;
      tile[a * ROW + r1l * TP + tap] = src[b] * inv;
    }
  }
  __syncthreads();
  // torch layout: Conv2d [co][ci][tap] (r0 = co, r1 = ci), ConvTranspose2d [ci][co][tap] (r0 = ci, r1 = co)
  T* along_r1 = transposed ? pack_nk : pack_kn;   // rows indexed by (tap, r0), consecutive r1
  T* along_r0 = transposed ? pack_kn : pack_nk;   // rows indexed by (tap, r1), consecutive r0
  if (along_r1 != nullptr && lane < n1t) {
    for (int row = warp; row < TAPS * n0t; row += 8) {          // row = tap * n0t + a, lane = r1
      const int tap = row / n0t, a = row - tap * n0t;
      along_r1[((long long)tap * n0 + r0b + a) * n1 + r1b + lane] = from_f32<T>(tile[a * ROW + lane * TP + tap]);
    }
  }
  if (along_r0 != nullptr) {
    const int a = lane & 15, half = lane >> 4;                  // 16 consecutive r0 per row, two rows per warp pass
    if (a < n0t) {
      for (int row = warp * 2 + half; row < TAPS * n1t; row += 16) {   // row = tap * n1t + b
        const int tap = row / n1t, b = row - tap * n1t;
        along_r0[((long long)tap * n1 + r1b + b) * n0 + r0b + a] = from_f32<T>(tile[a * ROW + b * TP + tap]);
      }
    }
  }
}

// taps == 1 (1x1 convolutions and the discriminator's Linear layers, up to 18.9 M elements): pack_kn is a cast
// copy, pack_nk a transpose; 32 x 32 tiles, 128-byte coalesced reads, 64-byte coalesced writes.
template <typename T>
__global__ void __launch_bounds__(256) pack_weights_1x1_kernel(const float* __restrict__ w, const float* __restrict__ sigma, int n0, int n1,
                                                               T* __restrict__ same, T* __restrict__ transp) {
  vg::pdl_entry();
  __shared__ float tile[32][33];
  const float inv = sigma ? 1.0f / *sigma : 1.0f;
  const int r0b = blockIdx.y * 32, r1b = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int a = ty + 8 * i;
    float v = 0.f;
    if (r0b + a < n0 && r1b + tx < n1) {
      v = w[(long long)(r0b + a) * n1 + r1b + tx] * inv;
      if (same != nullptr) same[(long long)(r0b + a) * n1 + r1b + tx] = from_f32<T>(v);
    }
    tile[a][tx] = v;
  }
  __syncthreads();
  if (transp == nullptr) return;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int b = ty + 8 * i;
    if (r1b + b < n1 && r0b + tx < n0) transp[(long long)(r1b + b) * n0 + r0b + tx] = from_f32<T>(tile[tx][b]);
  }
}


// ---- batched weight pack: EVERY conv / Linear weight of a network in one launch -----------------------------------
// The per-layer pack kernels above are 8-10 us launches with a few blocks each (~50 of them per training iteration).
// Here a block finds its (weight, tile) in a by-value table and runs the same tile bodies; no sigma - the spectral
// norm is applied in the convolution epilogue (vg_conv_forward_scaled), so a pack stays valid until the optimizer step.
struct PackTable {
  VgPackItem it[VG_PACK_MAX];
  int first_block[VG_PACK_MAX + 1];
  int n;
};

template <typename T, int TAPS>
__device__ __forceinline__ void pack_tile_body(float* tile, const float* __restrict__ w, int n0, int n1, int transposed, T* __restrict__ pack_kn,
                                               T* __restrict__ pack_nk, int bx, int by) {
  constexpr int TP = TAPS | 1;
  constexpr int ROW = kPackR1 * TP + 1;
  const int r0b = by * kPackR0, r1b = bx * kPackR1;
  const int n1t = min(kPackR1, n1 - r1b), n0t = min(kPackR0, n0 - r0b);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int run = n1t * TAPS;
  for (int a = warp; a < n0t; a += 8) {
    const float* src = w + ((long long)(r0b + a) * n1 + r1b) * TAPS;
    for (int b = lane; b < run; b += 32) {
      const int r1l = b / TAPS, tap = b - r1l * TAPS;
      tile[a * ROW + r1l * TP + tap] = src[b];
    }
  }
  __syncthreads();
  T* along_r1 = transposed ? pack_nk : pack_kn;
  T* along_r0 = transposed ? pack_kn : pack_nk;
  if (along_r1 != nullptr && lane < n1t) {
    for (int row = warp; row < TAPS * n0t; row += 8) {
      const int tap = row / n0t, a = row - tap * n0t;
      along_r1[((long long)tap * n0 + r0b + a) * n1 + r1b + lane] = from_f32<T>(tile[a * ROW + lane * TP + tap]);
    }
  }
  if (along_r0 != nullptr) {
    const int a = lane & 15, half = lane >> 4;
    if (a < n0t) {
      for (int row = warp * 2 + half; row < TAPS * n1t; row += 16) {
        const int tap = row / n1t, b = row - tap * n1t;
        along_r0[((long long)tap * n1 + r1b + b) * n0 + r0b + a] = from_f32<T>(tile[a * ROW + b * TP + tap]);
      }
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(256) pack_weights_batched_kernel(const __grid_constant__ PackTable tb) {
  vg::pdl_entry();
  __shared__ float tile[kPackR0 * (kPackR1 * 17 + 1)];      // sized for TAPS = 16; the 1x1 body uses it as [32][33]
  int i = 0;
  while (i + 1 < tb.n && (int)blockIdx.x >= tb.first_block[i + 1]) ++i;
  const VgPackItem& it = tb.it[i];
  const int lb = (int)blockIdx.x - tb.first_block[i];
  const float* w = it.w;
  T* kn = reinterpret_cast<T*>(it.pack_kn);
  T* nk = reinterpret_cast<T*>(it.pack_nk);
  const int n0 = it.n0, n1 = it.n1;
  if (it.taps == 1) {
    // [r0][r1] -> same layout (cast copy) + transpose; 32 x 32 tiles
    T* same = it.transposed ? nk : kn;
    T* transp = it.transposed ? kn : nk;
    const int tiles_x = (n1 + 31) / 32;
    const int r0b = (lb / tiles_x) * 32, r1b = (lb % tiles_x) * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    float (*t2)[33] = reinterpret_cast<float (*)[33]>(tile);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int a = ty + 8 * q;
      float v = 0.f;
      if (r0b + a < n0 && r1b + tx < n1) {
        v = w[(long long)(r0b + a) * n1 + r1b + tx];
        if (same != nullptr) same[(long long)(r0b + a) * n1 + r1b + tx] = from_f32<T>(v);
      }
      t2[a][tx] = v;
    }
    __syncthreads();
    if (transp == nullptr) return;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int b = ty + 8 * q;
      if (r1b + b < n1 && r0b + tx < n0) transp[(long long)(r1b + b) * n0 + r0b + tx] = from_f32<T>(t2[tx][b]);
    }
    return;
  }
  const int tiles_x = (n1 + kPackR1 - 1) / kPackR1;
  const int bx = lb % tiles_x, by = lb / tiles_x;
  if (it.taps == 9) pack_tile_body<T, 9>(tile, w, n0, n1, it.transposed, kn, nk, bx, by);
  else if (it.taps == 16) pack_tile_body<T, 16>(tile, w, n0, n1, it.transposed, kn, nk, bx, by);
  else {
    // generic tap count: element-wise over this block's 16 x 32 x taps chunk of the torch layout
    const int r0b = by * kPackR0, r1b = bx * kPackR1;
    const int n0t = min(kPackR0, n0 - r0b), n1t = min(kPackR1, n1 - r1b);
    const int taps = it.taps;
    const int c_out = it.transposed ? n1 : n0, c_in = it.transposed ? n0 : n1;
    for (int e = threadIdx.x; e < n0t * n1t * taps; e += blockDim.x) {
      const int tap = e % taps;
      const int r = e / taps;
      const int b = r % n1t, a = r / n1t;
      const float v = w[((long long)(r0b + a) * n1 + r1b + b) * taps + tap];
      const int co = it.transposed ? r1b + b : r0b + a, ci = it.transposed ? r0b + a : r1b + b;
      if (kn) kn[((long long)tap * c_out + co) * c_in + ci] = from_f32<T>(v);
      if (nk) nk[((long long)tap * c_in + ci) * c_out + co] = from_f32<T>(v);
    }
  }
}

int simt_pack_weights_batched(const VgPackItem* items, int n_items, int dtype, cudaStream_t s) {
  for (int base = 0; base < n_items; base += VG_PACK_MAX) {
    PackTable tb;
    memset(&tb, 0, sizeof(tb));
    tb.n = std::min(VG_PACK_MAX, n_items - base);
    int blocks = 0;
    for (int i = 0; i < tb.n; ++i) {
      const VgPackItem& it = items[base + i];
      VG_CHECK_ARG(it.w && (it.pack_kn || it.pack_nk) && it.n0 > 0 && it.n1 > 0 && it.taps > 0, "bad pack item %d", base + i);
      tb.it[i] = it;
      tb.first_block[i] = blocks;
      if (it.taps == 1) blocks += (int)(cdiv(it.n1, 32) * cdiv(it.n0, 32));
      else blocks += (int)(cdiv(it.n1, kPackR1) * cdiv(it.n0, kPackR0));
    }
    tb.first_block[tb.n] = blocks;
    if (blocks == 0) continue;
    if (dtype == VG_BF16) vg::Launch(blocks, 256, 0, s)(pack_weights_batched_kernel<__nv_bfloat16>, tb);
    else vg::Launch(blocks, 256, 0, s)(pack_weights_batched_kernel<float>, tb);
    VG_LAUNCHED();
  }
  return VG_OK;
}

// ---- generic direct convolution --------------------------------------------------------------
// thread -> (output pixel, group of CO_T output channels)
template <typename TI, typename TO, bool SCATTER, int CO_T>
__global__ void __launch_bounds__(256) conv_direct_kernel(const TI* __restrict__ in, const TI* __restrict__ W,
                                                          const float* __restrict__ bias, const float* __restrict__ colscale,
                                                          const float* __restrict__ sigma, int sigma_group_n,
                                                          ConvGeom g, TO* __restrict__ out) {
  vg::pdl_entry();
  const unsigned cog = (unsigned)(g.co / CO_T);
  const unsigned total = (unsigned)g.n * g.ho * g.wo * cog;      // host guarantees < 2^31
  for (unsigned idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int cg = (int)(idx % cog);
    const unsigned pix = idx / cog;
    const int ox = (int)(pix % (unsigned)g.wo);
    const unsigned t = pix / (unsigned)g.wo;
    const int oy = (int)(t % (unsigned)g.ho);
    const int n = (int)(t / (unsigned)g.ho);
    const int co0 = cg * CO_T;
    float acc[CO_T];
#pragma unroll
    for (int j = 0; j < CO_T; ++j) acc[j] = 0.f;
    for (int ky = 0; ky < g.kh; ++ky) {
      int iy;
      if (SCATTER) {
        int ty = oy + g.pad - ky;
        if (ty < 0 || ty % g.stride != 0) continue;
        iy = ty / g.stride;
      } else {
        iy = oy * g.stride - g.pad + ky;
      }
      if (iy < 0 || iy >= g.hi) continue;
      for (int kx = 0; kx < g.kw; ++kx) {
        int ix;
        if (SCATTER) {
          int tx = ox + g.pad - kx;
          if (tx < 0 || tx % g.stride != 0) continue;
          ix = tx / g.stride;
        } else {
          ix = ox * g.stride - g.pad + kx;
        }
        if (ix < 0 || ix >= g.wi) continue;
        const TI* ip = in + (((long long)n * g.hi + iy) * g.wi + ix) * g.cr;
        const TI* wp = W + (long long)(ky * g.kw + kx) * g.cr * g.co + co0;
        int c = 0;
        if ((g.cr & 7) == 0) {
          for (; c < g.cr; c += 8) {
            Vec8<TI> xv;
            xv.load(ip + c);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              if (CO_T == 8) {
                Vec8<TI> wv;
                wv.load(wp + (long long)(c + q) * g.co);
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[j] = fmaf(xv.v[q], wv.v[j], acc[j]);
              } else {
#pragma unroll
                for (int j = 0; j < CO_T; ++j) acc[j] = fmaf(xv.v[q], to_f32(wp[(long long)(c + q) * g.co + j]), acc[j]);
              }
            }
          }
        }
        for (; c < g.cr; ++c) {
          float xs = to_f32(ip[c]);
          if (CO_T == 8) {
            Vec8<TI> wv;
            wv.load(wp + (long long)c * g.co);
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] = fmaf(xs, wv.v[j], acc[j]);
          } else {
#pragma unroll
            for (int j = 0; j < CO_T; ++j) acc[j] = fmaf(xs, to_f32(wp[(long long)c * g.co + j]), acc[j]);
          }
        }
      }
    }
    TO* op = out + (long long)pix * g.co + co0;
    // spectral norm applied here (1 / sigma of the sample's group) so that the packed weights stay valid across forwards
    const float inv_sigma = sigma ? 1.0f / sigma[sigma_group_n > 0 ? n / sigma_group_n : 0] : 1.0f;
#pragma unroll
    for (int j = 0; j < CO_T; ++j) {
      float v = acc[j] * inv_sigma;
      if (bias) v += bias[co0 + j];
      if (colscale) v *= colscale[(long long)n * g.co + co0 + j];
      acc[j] = v;
    }
    if (CO_T == 8) {
      Vec8<TO> ov;
#pragma unroll
      for (int j = 0; j < 8; ++j) ov.v[j] = acc[j];
      ov.store(op);
    } else {
#pragma unroll
      for (int j = 0; j < CO_T; ++j) op[j] = from_f32<TO>(acc[j]);
    }
  }
}

// ---- degenerate layers (one side has a single channel) --------------------------------------
// reduce1: out[p] = sum_taps sum_c in[p (+) tap][c] * W[tap][c]     (Conv2d C->1 forward, Conv2d 1->C dgrad)
// 8 threads cooperate on one output pixel, each owning 8 channels of every tap; the weights of
// a thread (taps x 8) live in registers for the whole kernel.  cr == 64 only (8 lanes x 8 ch).
template <typename TI, typename TO, bool SCATTER, int TAPS>
__global__ void __launch_bounds__(256) conv_reduce1_kernel(const TI* __restrict__ in, const TI* __restrict__ W,
                                                           const float* __restrict__ bias, ConvGeom g, TO* __restrict__ out) {
  vg::pdl_entry();
  const int sub = threadIdx.x & 7;            // channel group within the pixel
  float w[TAPS][8];
#pragma unroll
  for (int t = 0; t < TAPS; ++t) {
    Vec8<TI> wv;
    wv.load(W + (long long)t * g.cr + sub * 8);   // W is [tap][cr][1]
#pragma unroll
    for (int j = 0; j < 8; ++j) w[t][j] = wv.v[j];
  }
  const unsigned npix = (unsigned)g.n * g.ho * g.wo;
  for (unsigned pix = (blockIdx.x * blockDim.x + threadIdx.x) >> 3; pix < npix; pix += (gridDim.x * blockDim.x) >> 3) {
    const int ox = (int)(pix % (unsigned)g.wo);
    const unsigned t0 = pix / (unsigned)g.wo;
    const int oy = (int)(t0 % (unsigned)g.ho);
    const int n = (int)(t0 / (unsigned)g.ho);
    float acc = 0.f;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      if (ky >= g.kh) break;
      int iy;
      if (SCATTER) { int ty = oy + g.pad - ky; if (ty < 0 || ty % g.stride != 0) continue; iy = ty / g.stride; }
      else iy = oy * g.stride - g.pad + ky;
      if (iy < 0 || iy >= g.hi) continue;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        if (kx >= g.kw) break;
        int ix;
        if (SCATTER) { int tx = ox + g.pad - kx; if (tx < 0 || tx % g.stride != 0) continue; ix = tx / g.stride; }
        else ix = ox * g.stride - g.pad + kx;
        if (ix < 0 || ix >= g.wi) continue;
        Vec8<TI> xv;
        xv.load(in + (((long long)n * g.hi + iy) * g.wi + ix) * g.cr + sub * 8);
        const int tp = ky * 3 + kx;   // kw == 3 (dispatch guarantees it): compile-time register index
#pragma unroll
        for (int j = 0; j < 8; ++j) acc = fmaf(xv.v[j], w[tp][j], acc);
      }
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    acc += __shfl_xor_sync(0xffffffffu, acc, 4);
    if (sub == 0) {
      if (bias) acc += bias[0];
      out[pix] = from_f32<TO>(acc);
    }
  }
}

// expand1: out[p][c] = sum_taps in[p (+) tap] * W[tap][c]   (Conv2d 1->C forward, Conv2d C->1 dgrad).
// A thread owns 8 output channels for its whole life (its 9x8 weights stay in registers) and walks
// pixels with a grid stride: 9 scalar loads (L1-resident single-channel image) per 16 B stored.
template <typename TI, typename TO, bool SCATTER>
__global__ void __launch_bounds__(256) conv_expand1_kernel(const TI* __restrict__ in, const TI* __restrict__ W,
                                                           const float* __restrict__ bias, const float* __restrict__ colscale,
                                                           ConvGeom g, TO* __restrict__ out) {
  vg::pdl_entry();
  const unsigned cog = (unsigned)g.co / 8;
  const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned nthr = gridDim.x * blockDim.x;          // multiple of cog (host guarantees)
  const int cg = (int)(tid % cog);
  float w[9][8], b[8];
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    Vec8<TI> wv;
    wv.load(W + (long long)t * g.co + cg * 8);            // W is [tap][1][co]
#pragma unroll
    for (int j = 0; j < 8; ++j) w[t][j] = wv.v[j];
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) b[j] = bias ? bias[cg * 8 + j] : 0.f;
  const unsigned npix = (unsigned)g.n * g.ho * g.wo;
  for (unsigned pix = tid / cog; pix < npix; pix += nthr / cog) {
    const int ox = (int)(pix % (unsigned)g.wo);
    const unsigned t0 = pix / (unsigned)g.wo;
    const int oy = (int)(t0 % (unsigned)g.ho);
    const int n = (int)(t0 / (unsigned)g.ho);
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = b[j];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      int iy;
      if (SCATTER) { int ty = oy + g.pad - ky; if (ty < 0 || ty % g.stride != 0) continue; iy = ty / g.stride; }
      else iy = oy * g.stride - g.pad + ky;
      if (iy < 0 || iy >= g.hi) continue;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        int ix;
        if (SCATTER) { int tx = ox + g.pad - kx; if (tx < 0 || tx % g.stride != 0) continue; ix = tx / g.stride; }
        else ix = ox * g.stride - g.pad + kx;
        if (ix < 0 || ix >= g.wi) continue;
        const float xs = to_f32(in[((long long)n * g.hi + iy) * g.wi + ix]);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = fmaf(xs, w[ky * 3 + kx][j], acc[j]);
      }
    }
    if (colscale) {
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] *= colscale[(long long)n * g.co + cg * 8 + j];
    }
    Vec8<TO> ov;
#pragma unroll
    for (int j = 0; j < 8; ++j) ov.v[j] = acc[j];
    ov.store(out + (long long)pix * g.co + cg * 8);
  }
}

// ---- strip variants (3x3, stride 1, pad 1, width % 8 == 0): a thread walks 8 consecutive pixels of a
// row and keeps the 3x10 window of the single-channel tensor in registers, so per pixel it issues the
// 72 FMAs it must plus ~10 other instructions (the per-pixel kernels above spend ~4x that on index math,
// bounds checks and reloading the window).
template <typename T>
__device__ __forceinline__ void load_window_3x10(const T* __restrict__ S, int n, int h, int w, int oy, int ox0, float (&win)[3][10]) {
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const int iy = oy - 1 + r;
    const bool rowok = iy >= 0 && iy < h;
    const T* rp = S + ((long long)n * h + (rowok ? iy : 0)) * w;
#pragma unroll
    for (int c = 0; c < 10; ++c) {
      const int ix = ox0 - 1 + c;
      win[r][c] = (rowok && ix >= 0 && ix < w) ? to_f32(rp[ix]) : 0.f;
    }
  }
}

template <typename TI, typename TO, bool FLIP>
__global__ void __launch_bounds__(256) conv_expand1_strip_kernel(const TI* __restrict__ in, const TI* __restrict__ W,
                                                                 const float* __restrict__ bias, const float* __restrict__ colscale,
                                                                 ConvGeom g, TO* __restrict__ out) {
  vg::pdl_entry();
  const unsigned cog = (unsigned)g.co / 8;
  const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned nthr = gridDim.x * blockDim.x;
  const int cg = (int)(tid % cog);
  float w[9][8], b[8];
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    Vec8<TI> wv;
    wv.load(W + (long long)(FLIP ? 8 - t : t) * g.co + cg * 8);
#pragma unroll
    for (int j = 0; j < 8; ++j) w[t][j] = wv.v[j];
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) b[j] = bias ? bias[cg * 8 + j] : 0.f;
  const unsigned spr = (unsigned)g.wo / 8;
  const unsigned nstrips = (unsigned)g.n * g.ho * spr;
  for (unsigned st = tid / cog; st < nstrips; st += nthr / cog) {
    const int sx = (int)(st % spr);
    const unsigned t0 = st / spr;
    const int oy = (int)(t0 % (unsigned)g.ho);
    const int n = (int)(t0 / (unsigned)g.ho);
    float win[3][10];
    load_window_3x10(in, n, g.hi, g.wi, oy, sx * 8, win);
    float cs[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) cs[j] = colscale ? colscale[(long long)n * g.co + cg * 8 + j] : 1.f;
    TO* op = out + (((long long)n * g.ho + oy) * g.wo + sx * 8) * g.co + cg * 8;
#pragma unroll
    for (int px = 0; px < 8; ++px) {
      Vec8<TO> ov;
#pragma unroll
      for (int j = 0; j < 8; ++j) ov.v[j] = b[j];
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float xs = win[r][px + c];
#pragma unroll
          for (int j = 0; j < 8; ++j) ov.v[j] = fmaf(xs, w[r * 3 + c][j], ov.v[j]);
        }
#pragma unroll
      for (int j = 0; j < 8; ++j) ov.v[j] *= cs[j];
      ov.store(op + (long long)px * g.co);
    }
  }
}

template <typename T, bool FLIP>
__global__ void __launch_bounds__(256) wgrad_degenerate_strip_kernel(const T* __restrict__ V, const T* __restrict__ S, int n, int h,
                                                                     int w, int c, unsigned strips_per_block, float* __restrict__ dw,
                                                                     float* __restrict__ partials) {
  vg::pdl_entry();
  // [9 * c]; deterministic mode (partials != nullptr): one such slot per warp, combined in warp order, and the block's
  // sums go to partials[block][c * 9] (added in block order by ordered_reduce_f32) instead of atomics on dw
  extern __shared__ float sacc[];
  const int nslot = partials ? (int)(blockDim.x >> 5) : 1;
  for (int i = threadIdx.x; i < nslot * 9 * c; i += blockDim.x) sacc[i] = 0.f;
  __syncthreads();
  const int groups = c / 8;
  const int lanes = blockDim.x / groups;
  const int grp = threadIdx.x % groups, lane = threadIdx.x / groups;
  const unsigned spr = (unsigned)w / 8;
  const unsigned nstrips = (unsigned)n * h * spr;
  const unsigned s0 = blockIdx.x * strips_per_block;
  const unsigned s1 = min(nstrips, s0 + strips_per_block);
  float acc[9][8];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[t][j] = 0.f;
  for (unsigned st = s0 + lane; st < s1; st += lanes) {
    const int sx = (int)(st % spr);
    const unsigned t0 = st / spr;
    const int oy = (int)(t0 % (unsigned)h);
    const int nn = (int)(t0 / (unsigned)h);
    float win[3][10];
    load_window_3x10(S, nn, h, w, oy, sx * 8, win);
    const T* vp = V + (((long long)nn * h + oy) * w + sx * 8) * c + grp * 8;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      Vec8<T> v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u].load(vp + (long long)(half * 4 + u) * c);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int px = half * 4 + u;
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
          for (int cc = 0; cc < 3; ++cc) {
            const float sv = win[r][px + cc];
            const int t = FLIP ? 8 - (r * 3 + cc) : (r * 3 + cc);
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[t][j] = fmaf(v[u].v[j], sv, acc[t][j]);
          }
      }
    }
  }
  const int lid = threadIdx.x & 31;
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float a = acc[t][j];
      for (int off = groups; off < 32; off <<= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
      acc[t][j] = a;
    }
  if (lid < groups || groups >= 32) {
    float* slot = sacc + (partials ? (threadIdx.x >> 5) * 9 * c : 0);
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (partials) slot[t * c + grp * 8 + j] = acc[t][j];       // one writer per (warp, tap, channel)
        else atomicAdd(&slot[t * c + grp * 8 + j], acc[t][j]);
      }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 9 * c; i += blockDim.x) {
    const int tap = i / c, ch = i % c;
    if (partials) {
      float t = sacc[i];
      for (int ws = 1; ws < nslot; ++ws) t += sacc[ws * 9 * c + i];
      partials[(size_t)blockIdx.x * 9 * c + (size_t)ch * 9 + tap] = t;
    } else {
      atomicAdd(&dw[(long long)ch * 9 + tap], sacc[i]);
    }
  }
}


// ---- streaming variant of the single-channel weight gradient (round 2) ----------------------------------------------
// The strip kernel above keeps 168 registers per thread -> one 256-thread block per SM, no loads in flight while it
// computes: ncu (profiles/r2_*) shows 12 % occupancy, IPC 0.24, 97 us for a 75 MB tensor (HBM time: 12 us).  Here a
// producer warp streams tiles of R image rows of V (+ the R + 2 rows of the single-channel tensor S) into a two-stage
// shared-memory ring with bulk copies (cp.async.bulk + mbarrier, as in bn_stream.cu); the 256 consumer threads turn the S
// rows into a zero-padded fp32 window array once per tile and then do nothing but shared-memory loads and FMAs into
// their 9 x 8 accumulators (thread = 8 channels x 8-pixel strips of the tile).
namespace degs {
constexpr int kConsumers = 256;
constexpr int kThreads = kConsumers + 32;
constexpr int kStages = 2;
struct Args {
  const void* V;
  const void* S;
  float* dw;
  int n, h, w, c;
  int R;                 // image rows per tile (divides h)
  int groups;            // c / 8 (divides 256)
  long long ntiles;
  int v_bytes, sraw_bytes, sf_bytes, stage_bytes;
};
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc), "r"(bytes), "r"((uint32_t)__cvta_generic_to_shared(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"((uint32_t)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const long long t0 = clock64();
  while (true) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                 : "=r"(ok) : "r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
    if (ok) return;
    if (clock64() - t0 > 4000000000LL) {
      printf("vaegan_b200: degenerate wgrad mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
}
}  // namespace degs

template <typename T, bool FLIP>
__global__ void __launch_bounds__(degs::kThreads, 1) wgrad_degenerate_stream_kernel(const __grid_constant__ degs::Args a) {
  vg::pdl_entry();
  using namespace degs;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = (uint32_t)__cvta_generic_to_shared(smem_raw);
  uint8_t* ring = smem_raw + ((128u - (raw_addr & 127u)) & 127u);
  float* sacc = reinterpret_cast<float*>(ring + (size_t)kStages * a.stage_bytes);     // [9 * c]
  uint64_t* full = reinterpret_cast<uint64_t*>(sacc + 9 * a.c);
  uint64_t* empty = full + kStages;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int s = 0; s < kStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kConsumers / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < 9 * a.c; i += blockDim.x) sacc[i] = 0.f;
  __syncthreads();
  const int tiles_per_img = a.h / a.R;
  const int w = a.w, c = a.c, R = a.R, wp = a.w + 8;
  const uint32_t row_v = (uint32_t)((size_t)w * c * sizeof(T)), row_s = (uint32_t)((size_t)w * sizeof(T));

  if (warp == kConsumers / 32) {
    // producer warp (one lane issues)
    int stage = 0;
    uint32_t phase = 0;
    for (long long t = blockIdx.x; t < a.ntiles; t += gridDim.x) {
      mbar_wait(&empty[stage], phase ^ 1u);
      if (lane == 0) {
        const int n = (int)(t / tiles_per_img), y0 = (int)(t % tiles_per_img) * R;
        int s_rows = 0;
        for (int r = 0; r < R + 2; ++r) { const int iy = y0 - 1 + r; s_rows += (iy >= 0 && iy < a.h) ? 1 : 0; }
        uint8_t* st = ring + (size_t)stage * a.stage_bytes;
        mbar_expect(&full[stage], (uint32_t)R * row_v + (uint32_t)s_rows * row_s);
        const uint8_t* vsrc = reinterpret_cast<const uint8_t*>(a.V) + ((size_t)n * a.h + y0) * row_v;
        for (int r = 0; r < R; ++r) bulk_load(st + (size_t)r * row_v, vsrc + (size_t)r * row_v, row_v, &full[stage]);
        for (int r = 0; r < R + 2; ++r) {
          const int iy = y0 - 1 + r;
          if (iy >= 0 && iy < a.h)
            bulk_load(st + a.v_bytes + (size_t)r * row_s, reinterpret_cast<const uint8_t*>(a.S) + ((size_t)n * a.h + iy) * row_s, row_s,
                      &full[stage]);
        }
      }
      __syncwarp();
      if (++stage == kStages) { stage = 0; phase ^= 1u; }
    }
    return;
  }

  const int groups = a.groups;
  const int grp = tid % groups;                 // fixed per thread: 256 % groups == 0
  const int spr = w / 8;
  const int items = R * spr * groups;
  float acc[9][8];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[t][j] = 0.f;
  int stage = 0;
  uint32_t phase = 0;
  for (long long t = blockIdx.x; t < a.ntiles; t += gridDim.x) {
    const int y0 = (int)(t % tiles_per_img) * R;
    mbar_wait(&full[stage], phase);
    uint8_t* st = ring + (size_t)stage * a.stage_bytes;
    const T* sraw = reinterpret_cast<const T*>(st + a.v_bytes);
    float* sf = reinterpret_cast<float*>(st + a.v_bytes + a.sraw_bytes);
    // the single-channel rows as zero-padded fp32: sf[r][x + 4], r = image row y0 - 1 + r
    for (int i = tid; i < (R + 2) * wp; i += kConsumers) {
      const int r = i / wp, xx = i - r * wp - 4;
      const int iy = y0 - 1 + r;
      sf[i] = (xx >= 0 && xx < w && iy >= 0 && iy < a.h) ? to_f32(sraw[r * w + xx]) : 0.f;
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    for (int item = tid; item < items; item += kConsumers) {
      const int t2 = item / groups;
      const int sx = t2 % spr, ly = t2 / spr;
      float win[3][10];
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int cc = 0; cc < 10; ++cc) win[r][cc] = sf[(ly + r) * wp + sx * 8 + 3 + cc];
      const T* vp = reinterpret_cast<const T*>(st) + ((size_t)(ly * w + sx * 8)) * c + grp * 8;
#pragma unroll
      for (int px = 0; px < 8; ++px) {
        Vec8<T> v;
        v.load(vp + (size_t)px * c);
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
          for (int cc = 0; cc < 3; ++cc) {
            const float sv = win[r][px + cc];
            const int tp = FLIP ? 8 - (r * 3 + cc) : (r * 3 + cc);
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[tp][j] = fmaf(v.v[j], sv, acc[tp][j]);
          }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[stage]);
    if (++stage == kStages) { stage = 0; phase ^= 1u; }
  }
  // lanes of a warp with the same channel group first, then shared-memory atomics, then one global atomic per value
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = acc[t][j];
      for (int off = groups; off < 32; off <<= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
      acc[t][j] = v;
    }
  if (lane < groups || groups >= 32) {
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int j = 0; j < 8; ++j) atomicAdd(&sacc[t * c + grp * 8 + j], acc[t][j]);
  }
  asm volatile("bar.sync 1, 256;" ::: "memory");
  for (int i = tid; i < 9 * c; i += kConsumers) {
    const int tap = i / c, ch = i % c;
    atomicAdd(&a.dw[(long long)ch * 9 + tap], sacc[i]);
  }
}

// returns true (and launches) when the streaming kernel can take the problem
template <typename T>
static int try_degenerate_stream(bool flip, const void* V, const void* S, int n, int h, int w, int c, float* dw, cudaStream_t s, bool* taken) {
  *taken = false;
  if (g_det.on) return VG_OK;      // deterministic mode: the strip kernel has the ordered reduction
  const int groups = c / 8;
  if (c % 8 != 0 || groups > 256 || 256 % groups != 0 || w % 8 != 0) return VG_OK;
  if (((size_t)w * sizeof(T)) % 16 != 0 || ((uintptr_t)V & 15) != 0 || ((uintptr_t)S & 15) != 0) return VG_OK;
  degs::Args a;
  memset(&a, 0, sizeof(a));
  int R = 0;
  for (int r : {8, 4, 2, 1}) {
    if (h % r != 0) continue;
    const size_t vb = (size_t)r * w * c * sizeof(T);
    const size_t sr = (((size_t)(r + 2) * w * sizeof(T)) + 15) / 16 * 16;
    const size_t sfb = (((size_t)(r + 2) * (w + 8) * 4) + 127) / 128 * 128;
    const size_t stage = (vb + sr + sfb + 127) / 128 * 128;
    if (degs::kStages * stage + (size_t)9 * c * 4 + 256 <= 220 * 1024) {
      R = r;
      a.v_bytes = (int)vb; a.sraw_bytes = (int)sr; a.sf_bytes = (int)sfb; a.stage_bytes = (int)stage;
      break;
    }
  }
  if (R == 0) return VG_OK;
  a.V = V; a.S = S; a.dw = dw; a.n = n; a.h = h; a.w = w; a.c = c; a.R = R; a.groups = groups;
  a.ntiles = (long long)n * (h / R);
  const size_t smem = (size_t)degs::kStages * a.stage_bytes + (size_t)9 * c * 4 + 2 * degs::kStages * 8 + 128 + 16;
  const int grid = (int)std::max<long long>(1, std::min<long long>(a.ntiles, num_sms()));
  cudaError_t e;
  if (flip) {
    e = cudaFuncSetAttribute(wgrad_degenerate_stream_kernel<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024);
    if (e != cudaSuccess) { cudaGetLastError(); return VG_OK; }
    vg::Launch(grid, degs::kThreads, smem, s)(wgrad_degenerate_stream_kernel<T, true>, a);
  } else {
    e = cudaFuncSetAttribute(wgrad_degenerate_stream_kernel<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024);
    if (e != cudaSuccess) { cudaGetLastError(); return VG_OK; }
    vg::Launch(grid, degs::kThreads, smem, s)(wgrad_degenerate_stream_kernel<T, false>, a);
  }
  VG_LAUNCHED();
  *taken = true;
  return VG_OK;
}

// wgrad with a single-channel side: dw[c*taps + tap] += sum_q V[q][c] * S[shift(q, tap)]
//   a_mode = true : V on the coarse/output grid (Conv2d 1->C: V = dy, S = x),   S index = q*stride - pad + k
//   a_mode = false: V on the input grid         (Conv2d C->1: V = x,  S = dy),  S index = (q + pad - k)/stride
template <typename T, int VEC>
__global__ void __launch_bounds__(256, 2) wgrad_degenerate_kernel(const T* __restrict__ V, const T* __restrict__ S, int n, int hv,
                                                               int wv, int c, int hs, int ws, int kh, int kw, int stride, int pad,
                                                               bool a_mode, unsigned pix_per_block, float* __restrict__ dw,
                                                               float* __restrict__ partials) {
  vg::pdl_entry();
  extern __shared__ float sacc[];   // [taps * c]; deterministic mode: one slot per warp (see wgrad_degenerate_strip_kernel)
  const int taps = kh * kw;
  const int nslot = partials ? (int)(blockDim.x >> 5) : 1;
  for (int i = threadIdx.x; i < nslot * taps * c; i += blockDim.x) sacc[i] = 0.f;
  __syncthreads();
  const int groups = c / VEC;                 // channel groups per pixel
  const int lanes = blockDim.x / groups;      // pixels processed concurrently
  const int grp = threadIdx.x % groups, lane = threadIdx.x / groups;
  const unsigned npix = (unsigned)n * hv * wv;
  const unsigned p0 = blockIdx.x * pix_per_block;
  const unsigned p1 = min(npix, p0 + pix_per_block);
  float acc[9][VEC];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[t][j] = 0.f;
  if (lane < lanes) {
    constexpr int U = 2;
    for (unsigned qb = p0 + lane; qb < p1; qb += U * lanes) {
      float v[U][VEC];
      // issue all the streaming loads of this batch first (memory-level parallelism)
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const unsigned q = qb + u * lanes;
        if (q < p1) {
          if (VEC == 8) {
            Vec8<T> vv;
            vv.load(V + (long long)q * c + grp * 8);
#pragma unroll
            for (int j = 0; j < VEC; ++j) v[u][j] = vv.v[j];
          } else {
            v[u][0] = to_f32(V[(long long)q * c + grp]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < VEC; ++j) v[u][j] = 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const unsigned q = qb + u * lanes;
        if (q >= p1) break;
        const int xq = (int)(q % (unsigned)wv);
        const unsigned t0 = q / (unsigned)wv;
        const int yq = (int)(t0 % (unsigned)hv);
        const int nn = (int)(t0 / (unsigned)hv);
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
          if (ky >= kh) break;
          int sy;
          if (a_mode) sy = yq * stride - pad + ky;
          else { int ty = yq + pad - ky; if (ty < 0 || ty % stride != 0) continue; sy = ty / stride; }
          if (sy < 0 || sy >= hs) continue;
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) {
            if (kx >= kw) break;
            int sx;
            if (a_mode) sx = xq * stride - pad + kx;
            else { int tx = xq + pad - kx; if (tx < 0 || tx % stride != 0) continue; sx = tx / stride; }
            if (sx < 0 || sx >= ws) continue;
            const float sv = to_f32(S[((long long)nn * hs + sy) * ws + sx]);
#pragma unroll
            for (int j = 0; j < VEC; ++j) acc[ky * 3 + kx][j] = fmaf(v[u][j], sv, acc[ky * 3 + kx][j]);
          }
        }
      }
    }
    // reduce across the threads of this warp that own the same channel group (register shuffles),
    // then ONE plain shared store per (warp, tap, channel): no contended shared atomics
    const int lid = threadIdx.x & 31;
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        float a = acc[t][j];
        for (int off = groups; off < 32; off <<= 1) a += __shfl_xor_sync(0xffffffffu, a, off);
        acc[t][j] = a;
      }
    if (lid < groups || groups >= 32) {
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          if (ky >= kh || kx >= kw) continue;
#pragma unroll
          for (int j = 0; j < VEC; ++j) {
            float* dst = &sacc[(partials ? (threadIdx.x >> 5) * taps * c : 0) + (ky * kw + kx) * c + grp * VEC + j];
            if (partials) *dst = acc[ky * 3 + kx][j];                     // one writer per (warp, tap, channel)
            else atomicAdd(dst, acc[ky * 3 + kx][j]);                     // <= 8 warps contend per address
          }
        }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < taps * c; i += blockDim.x) {
    const int tap = i / c, ch = i % c;
    if (partials) {
      float t = sacc[i];
      for (int ws = 1; ws < nslot; ++ws) t += sacc[ws * taps * c + i];
      partials[(size_t)blockIdx.x * taps * c + (size_t)ch * taps + tap] = t;
    } else {
      atomicAdd(&dw[(long long)ch * taps + tap], sacc[i]);
    }
  }
}

// ---- generic weight gradient -----------------------------------------------------------------
// dw[cu][cs][tap] += sum_q U[q][cu] * S[q*s - p + k][cs];  U lives on the coarse grid (hu x wu),
// S on the fine grid (hs x ws).  Block tile 32(cu) x 32(cs), 256 threads, 2x2 micro tile.
struct WgradGeom {
  int n, hu, wu, cu, hs, ws, cs, kh, kw, stride, pad;
  long long q_per_split;
};

template <typename T>
__global__ void __launch_bounds__(256) wgrad_simt_kernel(const T* __restrict__ U, const T* __restrict__ S, WgradGeom g,
                                                          float* __restrict__ dw, int* __restrict__ det_locks) {
  vg::pdl_entry();
  __shared__ float su[32][33];
  __shared__ float ss[32][33];
  const int tiles_s = (g.cs + 31) / 32;
  const int tile_u = blockIdx.x / tiles_s, tile_s = blockIdx.x % tiles_s;
  const int tap = blockIdx.y;
  const int ky = tap / g.kw, kx = tap % g.kw;
  const long long qtot = (long long)g.n * g.hu * g.wu;
  const long long q0 = (long long)blockIdx.z * g.q_per_split;
  const long long q1 = (q0 + g.q_per_split < qtot) ? q0 + g.q_per_split : qtot;
  const int tid = threadIdx.x;
  const int tu = tid / 16, ts = tid % 16;   // micro tile rows tu*2.., cols ts*2..
  float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
  const int lc = tid % 32, lq = tid / 32;   // loader: channel lc, pixel row lq (8 per pass)
  for (long long qb = q0; qb < q1; qb += 32) {
#pragma unroll
    for (int pass = 0; pass < 4; ++pass) {
      int qq = lq + pass * 8;
      long long q = qb + qq;
      float uv = 0.f, sv = 0.f;
      if (q < q1) {
        int xq = (int)(q % g.wu);
        long long t = q / g.wu;
        int yq = (int)(t % g.hu);
        int n = (int)(t / g.hu);
        int cu = tile_u * 32 + lc;
        if (cu < g.cu) uv = to_f32(U[q * g.cu + cu]);
        int sy = yq * g.stride - g.pad + ky, sx = xq * g.stride - g.pad + kx;
        int cs = tile_s * 32 + lc;
        if (cs < g.cs && sy >= 0 && sy < g.hs && sx >= 0 && sx < g.ws)
          sv = to_f32(S[(((long long)n * g.hs + sy) * g.ws + sx) * g.cs + cs]);
      }
      su[qq][lc] = uv;
      ss[qq][lc] = sv;
    }
    __syncthreads();
#pragma unroll 8
    for (int qq = 0; qq < 32; ++qq) {
      float u0 = su[qq][tu * 2], u1 = su[qq][tu * 2 + 1];
      float s0 = ss[qq][ts * 2], s1 = ss[qq][ts * 2 + 1];
      acc[0][0] = fmaf(u0, s0, acc[0][0]);
      acc[0][1] = fmaf(u0, s1, acc[0][1]);
      acc[1][0] = fmaf(u1, s0, acc[1][0]);
      acc[1][1] = fmaf(u1, s1, acc[1][1]);
    }
    __syncthreads();
  }
  const int taps = g.kh * g.kw;
  // deterministic mode: the pixel splits (blockIdx.z) of one (tile, tap) add in split order
  int* const det_lock = det_locks ? det_locks + (blockIdx.y * gridDim.x + blockIdx.x) : nullptr;
  if (det_lock) {
    if (tid == 0) det_wait_turn(det_lock, (int)blockIdx.z);
    __syncthreads();
  }
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      int cu = tile_u * 32 + tu * 2 + a, cs = tile_s * 32 + ts * 2 + b;
      if (cu < g.cu && cs < g.cs) atomicAdd(&dw[((long long)cu * g.cs + cs) * taps + tap], acc[a][b]);
    }
  if (det_lock) {
    __threadfence();
    __syncthreads();
    if (tid == 0) det_publish_turn(det_lock, blockIdx.z + 1 == gridDim.z ? 0 : (int)blockIdx.z + 1);
  }
}

// dbias[c] += sum over rows of dy[row][c]
template <typename T>
__global__ void colsum_kernel(const T* __restrict__ x, long long rows, int c, long long rows_per_block, float* __restrict__ out,
                              float* __restrict__ partials) {
  vg::pdl_entry();
  long long r0 = (long long)blockIdx.x * rows_per_block;
  long long r1 = (r0 + rows_per_block < rows) ? r0 + rows_per_block : rows;
  for (int ch = threadIdx.x; ch < c; ch += blockDim.x) {
    float s = 0.f;
    for (long long r = r0; r < r1; ++r) s += to_f32(x[r * c + ch]);
    if (partials) partials[(size_t)blockIdx.x * c + ch] = s;
    else atomicAdd(&out[ch], s);
  }
}

// ---- host-side launchers (called from conv_api.cu) -------------------------------------------
template <typename TI, typename TO>
static int launch_direct(bool scatter, const TI* in, const TI* W, const float* bias, const float* colscale, const float* sigma,
                         int sigma_group_n, const ConvGeom& g, TO* out, cudaStream_t s) {
  const bool v8 = (g.co % 8 == 0);
  const long long total = (long long)g.n * g.ho * g.wo * (v8 ? g.co / 8 : g.co);
  if (total == 0) return VG_OK;
  VG_CHECK_ARG(total < (1LL << 31) && (long long)g.n * g.hi * g.wi * g.cr < (1LL << 40), "tensor too large for the CUDA-core conv path");
  // the single-channel special kernels have no sigma epilogue: a spectral-normed degenerate layer takes the generic kernel
  if (sigma == nullptr && g.co == 1 && g.cr == 64 && g.kh == 3 && g.kw == 3 && colscale == nullptr) {
    const long long thr = (long long)g.n * g.ho * g.wo * 8;
    int grid1 = (int)std::min<long long>(cdiv(thr, 256), (long long)num_sms() * 16);
    if (scatter) vg::Launch(grid1, 256, 0, s)(conv_reduce1_kernel<TI, TO, true, 9>, in, W, bias, g, out);
    else         vg::Launch(grid1, 256, 0, s)(conv_reduce1_kernel<TI, TO, false, 9>, in, W, bias, g, out);
    VG_LAUNCHED();
    return VG_OK;
  }
  if (sigma == nullptr && g.cr == 1 && v8 && g.kh == 3 && g.kw == 3 && g.stride == 1 && g.pad == 1 && g.wo % 8 == 0 && g.ho == g.hi &&
      g.wo == g.wi && 256 % (g.co / 8) == 0) {
    const long long thr = (long long)g.n * g.ho * (g.wo / 8) * (g.co / 8);
    int grid1 = (int)std::min<long long>(cdiv(thr, 256), (long long)num_sms() * 8);
    if (scatter) vg::Launch(grid1, 256, 0, s)(conv_expand1_strip_kernel<TI, TO, true>, in, W, bias, colscale, g, out);
    else         vg::Launch(grid1, 256, 0, s)(conv_expand1_strip_kernel<TI, TO, false>, in, W, bias, colscale, g, out);
    VG_LAUNCHED();
    return VG_OK;
  }
  if (sigma == nullptr && g.cr == 1 && v8 && g.kh == 3 && g.kw == 3 && 256 % (g.co / 8) == 0) {
    int grid1 = (int)std::min<long long>(cdiv(total, 256 * 2), (long long)num_sms() * 16);
    if (scatter) vg::Launch(grid1, 256, 0, s)(conv_expand1_kernel<TI, TO, true>, in, W, bias, colscale, g, out);
    else         vg::Launch(grid1, 256, 0, s)(conv_expand1_kernel<TI, TO, false>, in, W, bias, colscale, g, out);
    VG_LAUNCHED();
    return VG_OK;
  }
  int grid = (int)std::min<long long>(cdiv(total, 256), (long long)num_sms() * 32);
  if (scatter) {
    if (v8) vg::Launch(grid, 256, 0, s)(conv_direct_kernel<TI, TO, true, 8>, in, W, bias, colscale, sigma, sigma_group_n, g, out);
    else    vg::Launch(grid, 256, 0, s)(conv_direct_kernel<TI, TO, true, 1>, in, W, bias, colscale, sigma, sigma_group_n, g, out);
  } else {
    if (v8) vg::Launch(grid, 256, 0, s)(conv_direct_kernel<TI, TO, false, 8>, in, W, bias, colscale, sigma, sigma_group_n, g, out);
    else    vg::Launch(grid, 256, 0, s)(conv_direct_kernel<TI, TO, false, 1>, in, W, bias, colscale, sigma, sigma_group_n, g, out);
  }
  VG_LAUNCHED();
  return VG_OK;
}

int simt_conv_forward(const VgConvDesc* d, const void* x, const void* pack_nk, const float* bias, const float* colscale,
                      const float* sigma, int sigma_group_n, void* y, cudaStream_t s) {
  ConvGeom g{d->n, d->h_in, d->w_in, d->c_in, d->h_out, d->w_out, d->c_out, d->kh, d->kw, d->stride, d->pad};
  const bool scatter = d->transposed != 0;
  if (d->act_dtype == VG_BF16) {
    if (d->out_dtype == VG_BF16)
      return launch_direct<__nv_bfloat16, __nv_bfloat16>(scatter, (const __nv_bfloat16*)x, (const __nv_bfloat16*)pack_nk, bias, colscale, sigma,
                                                         sigma_group_n, g, (__nv_bfloat16*)y, s);
    return launch_direct<__nv_bfloat16, float>(scatter, (const __nv_bfloat16*)x, (const __nv_bfloat16*)pack_nk, bias, colscale, sigma,
                                               sigma_group_n, g, (float*)y, s);
  }
  VG_CHECK_ARG(d->out_dtype == VG_F32, "fp32 activations require fp32 output");
  return launch_direct<float, float>(scatter, (const float*)x, (const float*)pack_nk, bias, colscale, sigma, sigma_group_n, g, (float*)y, s);
}

int simt_conv_dgrad(const VgConvDesc* d, const void* dy, const void* pack_kn, const float* sigma, int sigma_group_n, void* dx,
                    cudaStream_t s) {
  // reduce over c_out; output has c_in channels on the input grid
  ConvGeom g{d->n, d->h_out, d->w_out, d->c_out, d->h_in, d->w_in, d->c_in, d->kh, d->kw, d->stride, d->pad};
  const bool scatter = d->transposed == 0;   // Conv2d dgrad scatters, ConvTranspose2d dgrad gathers
  if (d->act_dtype == VG_BF16)
    return launch_direct<__nv_bfloat16, __nv_bfloat16>(scatter, (const __nv_bfloat16*)dy, (const __nv_bfloat16*)pack_kn, nullptr, nullptr, sigma,
                                                       sigma_group_n, g, (__nv_bfloat16*)dx, s);
  return launch_direct<float, float>(scatter, (const float*)dy, (const float*)pack_kn, nullptr, nullptr, sigma, sigma_group_n, g, (float*)dx, s);
}

int simt_conv_wgrad(const VgConvDesc* d, const void* x, const void* dy, float* dw, cudaStream_t s) {
  WgradGeom g;
  const void *U, *S;
  if (!d->transposed) {   // dw[co][ci][tap]: U = dy on the output grid, S = x
    g = WgradGeom{d->n, d->h_out, d->w_out, d->c_out, d->h_in, d->w_in, d->c_in, d->kh, d->kw, d->stride, d->pad, 0};
    U = dy; S = x;
  } else {                // dw[ci][co][tap]: U = x on the input grid, S = dy
    g = WgradGeom{d->n, d->h_in, d->w_in, d->c_in, d->h_out, d->w_out, d->c_out, d->kh, d->kw, d->stride, d->pad, 0};
    U = x; S = dy;
  }
  const long long qtot = (long long)g.n * g.hu * g.wu;
  if (qtot == 0) return VG_OK;
  const int dg_c = (d->c_in == 1) ? d->c_out : d->c_in;
  const int dg_groups = (dg_c % 8 == 0) ? dg_c / 8 : dg_c;
  if (!d->transposed && d->kh <= 3 && d->kw <= 3 && (d->c_in == 1 || d->c_out == 1) && dg_groups <= 256 &&
      (dg_groups & (dg_groups - 1)) == 0 &&
      (long long)d->n * d->h_in * d->w_in < (1LL << 31) && std::max(d->c_in, d->c_out) * d->kh * d->kw * 4 <= 40000) {
    // one side has a single channel: memory-bound streaming kernel
    const bool a_mode = (d->c_in == 1);           // V = dy on the output grid, S = x
    const void* V = a_mode ? dy : x;
    const void* Sx = a_mode ? x : dy;
    const int c = a_mode ? d->c_out : d->c_in;
    const int hv = a_mode ? d->h_out : d->h_in, wv = a_mode ? d->w_out : d->w_in;
    const int hs = a_mode ? d->h_in : d->h_out, ws = a_mode ? d->w_in : d->w_out;
    const long long npix = (long long)d->n * hv * wv;
    if (c % 8 == 0 && d->kh == 3 && d->kw == 3 && d->stride == 1 && d->pad == 1 && wv % 8 == 0 && hv == hs && wv == ws &&
        256 % (c / 8) == 0 && (size_t)9 * c * sizeof(float) <= 40000) {
      {
        bool taken = false;
        int rcs = (d->act_dtype == VG_BF16) ? try_degenerate_stream<__nv_bfloat16>(!a_mode, V, Sx, d->n, hv, wv, c, dw, s, &taken)
                                            : try_degenerate_stream<float>(!a_mode, V, Sx, d->n, hv, wv, c, dw, s, &taken);
        if (rcs) return rcs;
        if (taken) return VG_OK;
      }
      const long long nstrips = npix / 8;
      long long blocks = std::min<long long>(cdiv(nstrips, 64), (long long)num_sms() * 4);
      unsigned spb = (unsigned)cdiv(nstrips, blocks);
      blocks = cdiv(nstrips, spb);
      size_t sm2 = (size_t)9 * c * sizeof(float);
      float* part = nullptr;
      if (g_det.on) {
        sm2 *= 8;                                                    // one slot per warp
        if (sm2 > 48 * 1024) VG_DET_UNSUPPORTED("single-channel weight gradient with more than 170 channels");
        if (!(part = (float*)det_scratch((size_t)blocks * 9 * c * sizeof(float)))) return VG_EINVAL;
      }
      if (d->act_dtype == VG_BF16) {
        if (a_mode) vg::Launch((unsigned)blocks, 256, sm2, s)(wgrad_degenerate_strip_kernel<__nv_bfloat16, false>, (const __nv_bfloat16*)V, (const __nv_bfloat16*)Sx, d->n, hv, wv, c, spb, dw, part);
        else        vg::Launch((unsigned)blocks, 256, sm2, s)(wgrad_degenerate_strip_kernel<__nv_bfloat16, true>, (const __nv_bfloat16*)V, (const __nv_bfloat16*)Sx, d->n, hv, wv, c, spb, dw, part);
      } else {
        if (a_mode) vg::Launch((unsigned)blocks, 256, sm2, s)(wgrad_degenerate_strip_kernel<float, false>, (const float*)V, (const float*)Sx, d->n, hv, wv, c, spb, dw, part);
        else        vg::Launch((unsigned)blocks, 256, sm2, s)(wgrad_degenerate_strip_kernel<float, true>, (const float*)V, (const float*)Sx, d->n, hv, wv, c, spb, dw, part);
      }
      VG_LAUNCHED();
      if (part) return ordered_reduce_f32(part, (int)blocks, 9LL * c, dw, s);
      return VG_OK;
    }
    const int vec = (c % 8 == 0 && c / 8 <= 256) ? 8 : 1;
    VG_CHECK_ARG(c / vec <= 256, "degenerate wgrad supports up to 256 channel groups");
    long long blocks = std::min<long long>(cdiv(npix, 1024), (long long)num_sms() * 4);
    unsigned ppb = (unsigned)cdiv(npix, blocks);
    blocks = cdiv(npix, ppb);
    size_t sm = (size_t)d->kh * d->kw * c * sizeof(float);
    float* part = nullptr;
    if (g_det.on) {
      sm *= 8;
      if (sm > 48 * 1024) VG_DET_UNSUPPORTED("single-channel weight gradient with this many channels");
      if (!(part = (float*)det_scratch((size_t)blocks * d->kh * d->kw * c * sizeof(float)))) return VG_EINVAL;
    }
    if (d->act_dtype == VG_BF16) {
      if (vec == 8) vg::Launch((unsigned)blocks, 256, sm, s)(wgrad_degenerate_kernel<__nv_bfloat16, 8>, (const __nv_bfloat16*)V, (const __nv_bfloat16*)Sx, d->n, hv, wv, c, hs, ws, d->kh, d->kw, d->stride, d->pad, a_mode, ppb, dw, part);
      else          vg::Launch((unsigned)blocks, 256, sm, s)(wgrad_degenerate_kernel<__nv_bfloat16, 1>, (const __nv_bfloat16*)V, (const __nv_bfloat16*)Sx, d->n, hv, wv, c, hs, ws, d->kh, d->kw, d->stride, d->pad, a_mode, ppb, dw, part);
    } else {
      if (vec == 8) vg::Launch((unsigned)blocks, 256, sm, s)(wgrad_degenerate_kernel<float, 8>, (const float*)V, (const float*)Sx, d->n, hv, wv, c, hs, ws, d->kh, d->kw, d->stride, d->pad, a_mode, ppb, dw, part);
      else          vg::Launch((unsigned)blocks, 256, sm, s)(wgrad_degenerate_kernel<float, 1>, (const float*)V, (const float*)Sx, d->n, hv, wv, c, hs, ws, d->kh, d->kw, d->stride, d->pad, a_mode, ppb, dw, part);
    }
    VG_LAUNCHED();
    if (part) return ordered_reduce_f32(part, (int)blocks, (long long)d->kh * d->kw * c, dw, s);
    return VG_OK;
  }
  const int tiles = ((g.cu + 31) / 32) * ((g.cs + 31) / 32);
  const int taps = g.kh * g.kw;
  long long want = std::max<long long>(1, (long long)num_sms() * 4 / ((long long)tiles * taps));
  long long splits = std::min<long long>(want, cdiv(qtot, 256));
  splits = std::max<long long>(1, std::min<long long>(splits, 65535));
  g.q_per_split = cdiv(cdiv(qtot, splits), 32) * 32;
  splits = cdiv(qtot, g.q_per_split);
  dim3 grid(tiles, taps, (unsigned)splits);
  int* locks = nullptr;
  if (g_det.on && splits > 1 && !(locks = det_locks((long long)tiles * taps))) return VG_EINVAL;
  if (d->act_dtype == VG_BF16)
    vg::Launch(grid, 256, 0, s)(wgrad_simt_kernel<__nv_bfloat16>, (const __nv_bfloat16*)U, (const __nv_bfloat16*)S, g, dw, locks);
  else
    vg::Launch(grid, 256, 0, s)(wgrad_simt_kernel<float>, (const float*)U, (const float*)S, g, dw, locks);
  VG_LAUNCHED();
  return VG_OK;
}

int simt_colsum(const void* x, long long rows, int c, int dtype, float* out, cudaStream_t s) {
  if (rows == 0) return VG_OK;
  long long blocks = std::min<long long>(cdiv(rows, 64), (long long)num_sms() * 4);
  long long rpb = cdiv(rows, blocks);
  blocks = cdiv(rows, rpb);
  int threads = std::min(1024, ((c + 31) / 32) * 32);
  float* part = nullptr;
  if (g_det.on && !(part = (float*)det_scratch((size_t)blocks * c * sizeof(float)))) return VG_EINVAL;
  if (dtype == VG_BF16)
    vg::Launch((int)blocks, threads, 0, s)(colsum_kernel<__nv_bfloat16>, (const __nv_bfloat16*)x, rows, c, rpb, out, part);
  else
    vg::Launch((int)blocks, threads, 0, s)(colsum_kernel<float>, (const float*)x, rows, c, rpb, out, part);
  VG_LAUNCHED();
  if (part) return ordered_reduce_f32(part, (int)blocks, c, out, s);
  return VG_OK;
}

int simt_pack_weights(const VgConvDesc* d, const float* w, const float* sigma, void* pack_kn, void* pack_nk, cudaStream_t s) {
  const int taps = d->kh * d->kw;
  const long long total = (long long)taps * d->c_in * d->c_out;
  if (total == 0) return VG_OK;
  const int n0 = d->transposed ? d->c_in : d->c_out, n1 = d->transposed ? d->c_out : d->c_in;
  if (total >= 4096 && (taps == 1 || taps == 9 || taps == 16)) {
    const bool bf = d->act_dtype == VG_BF16;
    if (taps == 1) {
      // [r0][r1] -> same layout (rows r0) + transpose (rows r1); which of pack_kn / pack_nk is which depends on `transposed`
      void* same = d->transposed ? pack_nk : pack_kn;
      void* transp = d->transposed ? pack_kn : pack_nk;
      dim3 tg((unsigned)cdiv(n1, 32), (unsigned)cdiv(n0, 32));
      if (bf) vg::Launch(tg, 256, 0, s)(pack_weights_1x1_kernel<__nv_bfloat16>, w, sigma, n0, n1, (__nv_bfloat16*)same, (__nv_bfloat16*)transp);
      else vg::Launch(tg, 256, 0, s)(pack_weights_1x1_kernel<float>, w, sigma, n0, n1, (float*)same, (float*)transp);
    } else {
      dim3 tg((unsigned)cdiv(n1, kPackR1), (unsigned)cdiv(n0, kPackR0));
      if (taps == 9) {
        if (bf) vg::Launch(tg, 256, 0, s)(pack_weights_tiled_kernel<__nv_bfloat16, 9>, w, sigma, n0, n1, d->transposed, (__nv_bfloat16*)pack_kn, (__nv_bfloat16*)pack_nk);
        else vg::Launch(tg, 256, 0, s)(pack_weights_tiled_kernel<float, 9>, w, sigma, n0, n1, d->transposed, (float*)pack_kn, (float*)pack_nk);
      } else {
        if (bf) vg::Launch(tg, 256, 0, s)(pack_weights_tiled_kernel<__nv_bfloat16, 16>, w, sigma, n0, n1, d->transposed, (__nv_bfloat16*)pack_kn, (__nv_bfloat16*)pack_nk);
        else vg::Launch(tg, 256, 0, s)(pack_weights_tiled_kernel<float, 16>, w, sigma, n0, n1, d->transposed, (float*)pack_kn, (float*)pack_nk);
      }
    }
    VG_LAUNCHED();
    return VG_OK;
  }
  int grid = (int)std::min<long long>(cdiv(total, 256), (long long)num_sms() * 8);
  if (d->act_dtype == VG_BF16)
    vg::Launch(grid, 256, 0, s)(pack_weights_kernel<__nv_bfloat16>, w, sigma, d->c_out, d->c_in, taps, d->transposed, (__nv_bfloat16*)pack_kn,
                                                            (__nv_bfloat16*)pack_nk);
  else
    vg::Launch(grid, 256, 0, s)(pack_weights_kernel<float>, w, sigma, d->c_out, d->c_in, taps, d->transposed, (float*)pack_kn, (float*)pack_nk);
  VG_LAUNCHED();
  return VG_OK;
}

}  // namespace vg
