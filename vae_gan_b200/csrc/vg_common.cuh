// Shared helpers for libvaegan_sm100.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>

#include "../../include/vaegan_b200.h"

namespace vg {

// ---- host-side error plumbing -------------------------------------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<unsigned long long> g_launches;
extern int g_num_sms;
extern int g_force_simt;
// deterministic-reduction mode (vg_set_deterministic): caller-owned scratch for per-block partial sums and a zeroed
// int array of turn counters for the split-K epilogues
struct DetState {
  int on;
  unsigned char* scratch;
  size_t scratch_bytes;
  int* locks;
  int n_locks;
};
extern DetState g_det;
// out[i] += sum over b (in block order) of partials[b * nvals + i]; one writer per element
int ordered_reduce_f64(const double* partials, int nblocks, long long nvals, double* out, cudaStream_t s);
int ordered_reduce_f32(const float* partials, int nblocks, long long nvals, float* out, cudaStream_t s);
// scratch for `bytes` of partial sums, or nullptr (with the error set) when the caller's buffer is too small
void* det_scratch(size_t bytes);
int* det_locks(long long n);
extern int g_pdl;   // VG_PDL: 1 (default) = kernels are launched with programmatic stream serialization, 0 = plain launches

#define VG_CHECK_ARG(cond, ...)                  \
  do {                                           \
    if (!(cond)) {                               \
      vg::set_error(__VA_ARGS__);                \
      return VG_EINVAL;                          \
    }                                            \
  } while (0)

#define VG_CUDA(expr)                                                                    \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) {                                                             \
      vg::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return VG_ECUDA;                                                                   \
    }                                                                                    \
  } while (0)

// kernels whose reductions have no ordered variant refuse to run in deterministic mode (loudly, like every other
// unsupported configuration) instead of silently breaking the bit-reproducibility the caller asked for
#define VG_DET_UNSUPPORTED(what)                                                          \
  do {                                                                                    \
    if (vg::g_det.on) {                                                                   \
      vg::set_error("deterministic mode: no ordered reduction for %s", what);             \
      return VG_EUNSUPPORTED;                                                             \
    }                                                                                     \
  } while (0)

// call after every kernel launch
#define VG_LAUNCHED()                                                                    \
  do {                                                                                   \
    vg::g_launches.fetch_add(1, std::memory_order_relaxed);                              \
    cudaError_t _e = cudaPeekAtLastError();                                              \
    if (_e != cudaSuccess) {                                                             \
      cudaGetLastError();                                                                \
      vg::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return VG_ECUDA;                                                                   \
    }                                                                                    \
  } while (0)

static inline cudaStream_t as_stream(vg_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
static inline size_t dtype_size(int dt) { return dt == VG_BF16 ? 2 : 4; }
static inline int num_sms() { return g_num_sms > 0 ? g_num_sms : 148; }
static inline long long cdiv(long long a, long long b) { return (a + b - 1) / b; }

// ---- kernel launch with programmatic dependent launch (PDL) --------------------------------------
// Every kernel of the library is launched with cudaLaunchAttributeProgrammaticStreamSerialization and calls
// pdl_entry() before its first global-memory access: `griddepcontrol.wait` blocks until the grid it depends on has
// completed and its memory is visible (a no-op for a plain launch), so no load or store of a kernel can pass the
// previous kernel's - while the launch itself, the CTA rasterisation and whatever a kernel does BEFORE pdl_entry()
// (mbarrier init, TMEM allocation, tensor-map prefetch in the tcgen05 / bulk-copy kernels) overlap the previous
// kernel's tail.  Inside the captured iteration these become programmatic edges of the CUDA graph.
// Measured on B200 (profiles/r2_pdl_ab.txt): batch 32 10.88 -> 10.59 ms/step, batch 256 unchanged.  Kernels do not
// trigger their dependents early (measured slower, DESIGN.md 3.5): the next grid starts once this one's CTAs have exited.
__device__ __forceinline__ void pdl_entry() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

struct Launch {
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[1];
  Launch(dim3 grid, dim3 block, size_t smem, cudaStream_t s) {
    cfg = cudaLaunchConfig_t{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = g_pdl ? 1 : 0;
  }
  template <typename... KArgs, typename... Args>
  void operator()(void (*kernel)(KArgs...), Args&&... args) {
    cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);   // errors surface in VG_LAUNCHED()
  }
};

// ---- deterministic split-K: the splits of one output tile add their partial sums in split order --------------------
// `turn`-th contributor waits until the tile's counter equals `turn`, adds its values, then publishes turn + 1 (the
// last one resets the counter to 0 for the next launch).  Lower splits have lower block / work-item indices, so they
// are always scheduled first: no deadlock (the serial split-K of CUTLASS relies on the same ordering).
__device__ __forceinline__ void det_wait_turn(const int* lock, int turn) {
  int v;
  long long t0 = 0;
  do {
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(lock) : "memory");
    if (v != turn) {
      if (t0 == 0) t0 = clock64();
      else if (clock64() - t0 > 8000000000LL) {
        printf("vaegan_b200: deterministic split-K turn wait timed out (block %d,%d,%d turn %d saw %d)\n", blockIdx.x, blockIdx.y,
               blockIdx.z, turn, v);
        __trap();
      }
      __nanosleep(64);
    }
  } while (v != turn);
}
__device__ __forceinline__ void det_publish_turn(int* lock, int next) {
  __threadfence();
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(lock), "r"(next) : "memory");
}

// ---- device helpers -----------------------------------------------------------------------
__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// 8-element vector access (16 B for bf16, 32 B for f32)
template <typename T> struct Vec8;
template <> struct Vec8<float> {
  float v[8];
  __device__ __forceinline__ void load(const float* p) {
    float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
  __device__ __forceinline__ void store(float* p) const {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
  }
};
template <> struct Vec8<__nv_bfloat16> {
  float v[8];
  __device__ __forceinline__ void load(const __nv_bfloat16* p) {
    uint4 r = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  __device__ __forceinline__ void store(__nv_bfloat16* p) const {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
  }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- Philox4x32-10 (counter-based; restated on the CPU in oracle/vaegan_oracle.py) ---------
struct Philox {
  uint32_t k0, k1, c2, c3;
  __device__ __forceinline__ Philox(unsigned long long seed, unsigned long long offset)
      : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)), c2((uint32_t)offset), c3((uint32_t)(offset >> 32)) {}
  // 4 words for block index `blk` (= element index / 4)
  __device__ __forceinline__ uint4 block(unsigned long long blk) const {
    uint32_t c0 = (uint32_t)blk, c1 = (uint32_t)(blk >> 32), d2 = c2, d3 = c3, a = k0, b = k1;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
      uint32_t hi1 = __umulhi(0xCD9E8D57u, d2), lo1 = 0xCD9E8D57u * d2;
      uint32_t n0 = hi1 ^ c1 ^ a, n2 = hi0 ^ d3 ^ b;
      c0 = n0; c1 = lo1; d2 = n2; d3 = lo0;
      a += 0x9E3779B9u; b += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, d2, d3);
  }
  __device__ __forceinline__ uint32_t word(unsigned long long idx) const {
    uint4 r = block(idx >> 2);
    uint32_t l = (uint32_t)idx & 3u;
    return l == 0 ? r.x : (l == 1 ? r.y : (l == 2 ? r.z : r.w));
  }
};
__device__ __forceinline__ uint32_t drop_threshold(float p) {
  double t = (double)p * 4294967296.0;
  return t >= 4294967295.0 ? 0xffffffffu : (uint32_t)t;
}

}  // namespace vg
