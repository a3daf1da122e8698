// C-ABI entry points for the convolutions: validation + dispatch between the tcgen05 implicit
// GEMM kernels (conv_tc.cu) and the CUDA-core kernels (conv_simt.cu).  Both are this library's
// own sm_100a kernels; there is no library (cuDNN/cuBLAS) or CPU fallback.
#include "vg_common.cuh"

namespace vg {
int simt_conv_forward(const VgConvDesc*, const void*, const void*, const float*, const float*, const float* sigma, int sigma_group_n, void*,
                      cudaStream_t);
int simt_conv_dgrad(const VgConvDesc*, const void*, const void*, const float* sigma, int sigma_group_n, void*, cudaStream_t);
int simt_conv_wgrad(const VgConvDesc*, const void*, const void*, float*, cudaStream_t);
int simt_colsum(const void*, long long, int, int, float*, cudaStream_t);
int simt_pack_weights(const VgConvDesc*, const float*, const float*, void*, void*, cudaStream_t);
int simt_pack_weights_batched(const VgPackItem* items, int n_items, int dtype, cudaStream_t);
bool tc_conv_supported(const VgConvDesc*, bool dgrad);
bool tc_wgrad_supported(const VgConvDesc*);
int tc_conv_run(const VgConvDesc*, bool dgrad, const void* in, const void* wpack, const float* bias, const float* colscale,
                const float* sigma, int sigma_group_n, void* out, int out_dtype, cudaStream_t, const VgConvEpilogue* ep = nullptr);
int tc_wgrad_run(const VgConvDesc*, const void* x, const void* dy, float* dw, float* workspace, cudaStream_t, bool acc_only = false);
int sn_backward_run(const float* dw_hat, const float* w_orig, const float* u, const float* v, const float* sigma, int rows, int cols,
                    float* dw_orig, float* dot_ws, cudaStream_t s);
int sn_backward_packed_run(const float* acc, const float* w_orig, const float* u, const float* v, const float* sigma, int cu, int cs,
                           int taps, float* dw_orig, float* dot_ws, cudaStream_t s);
int simt_colsum(const void* x, long long rows, int c, int dtype, float* out, cudaStream_t s);
int tc_tune_set(const VgConvDesc*, int dgrad, int bn, int form);
void tc_tune_clear();
void tc_tune_record(int on);
int tc_tune_seen(int* keys, int max_keys);
}  // namespace vg

using namespace vg;

static int check_conv(const VgConvDesc* d) {
  VG_CHECK_ARG(d != nullptr, "VgConvDesc is null");
  VG_CHECK_ARG(d->n >= 0 && d->h_in > 0 && d->w_in > 0 && d->c_in > 0 && d->c_out > 0, "bad conv dims");
  VG_CHECK_ARG(d->kh > 0 && d->kw > 0 && d->stride > 0 && d->pad >= 0, "bad conv kernel geometry");
  VG_CHECK_ARG(d->act_dtype == VG_F32 || d->act_dtype == VG_BF16, "bad act_dtype");
  VG_CHECK_ARG(d->out_dtype == VG_F32 || d->out_dtype == VG_BF16, "bad out_dtype");
  int eh, ew;
  if (d->transposed) {
    eh = (d->h_in - 1) * d->stride - 2 * d->pad + d->kh;
    ew = (d->w_in - 1) * d->stride - 2 * d->pad + d->kw;
  } else {
    eh = (d->h_in + 2 * d->pad - d->kh) / d->stride + 1;
    ew = (d->w_in + 2 * d->pad - d->kw) / d->stride + 1;
  }
  VG_CHECK_ARG(eh == d->h_out && ew == d->w_out, "output dims %dx%d inconsistent with geometry (expected %dx%d)", d->h_out, d->w_out, eh, ew);
  return VG_OK;
}

extern "C" int vg_conv_pack_weights(const VgConvDesc* d, const float* w, const float* sigma, void* pack_kn, void* pack_nk,
                                    vg_stream_t stream) {
  int rc = check_conv(d);
  if (rc) return rc;
  VG_CHECK_ARG(w && (pack_kn || pack_nk), "null pointer");
  return simt_pack_weights(d, w, sigma, pack_kn, pack_nk, as_stream(stream));
}

extern "C" int vg_conv_pack_weights_batched(const VgPackItem* items, int n_items, int dtype, vg_stream_t stream) {
  VG_CHECK_ARG(items != nullptr && n_items >= 0, "bad args");
  VG_CHECK_ARG(dtype == VG_F32 || dtype == VG_BF16, "bad dtype %d", dtype);
  if (n_items == 0) return VG_OK;
  return simt_pack_weights_batched(items, n_items, dtype, as_stream(stream));
}

extern "C" int vg_conv_forward(const VgConvDesc* d, const void* x, const void* pack_kn, const void* pack_nk, const float* bias,
                               const float* colscale, void* y, double* stats, vg_stream_t stream) {
  return vg_conv_forward_scaled(d, x, pack_kn, pack_nk, bias, colscale, nullptr, 0, y, stats, stream);
}

extern "C" int vg_conv_forward_scaled(const VgConvDesc* d, const void* x, const void* pack_kn, const void* pack_nk, const float* bias,
                                      const float* colscale, const float* sigma, int sigma_group_n, void* y, double* stats,
                                      vg_stream_t stream) {
  VgConvEpilogue ep{};
  ep.bias = bias; ep.colscale = colscale; ep.sigma = sigma; ep.sigma_group_n = sigma_group_n;
  ep.act_slope = 1.0f; ep.post_slope = 1.0f;
  return vg_conv_forward_fused(d, x, pack_kn, pack_nk, &ep, y, stats, stream);
}

extern "C" int vg_conv_forward_fused(const VgConvDesc* d, const void* x, const void* pack_kn, const void* pack_nk, const VgConvEpilogue* ep,
                                     void* y, double* stats, vg_stream_t stream) {
  int rc = check_conv(d);
  if (rc) return rc;
  VG_CHECK_ARG(ep != nullptr, "VgConvEpilogue is null");
  if (d->n == 0) return VG_OK;   // empty batch: nothing to do (pointers of empty tensors may be null)
  VG_CHECK_ARG(x && y && pack_kn && pack_nk, "null pointer");
  VG_CHECK_ARG(ep->sigma_group_n >= 0, "sigma_group_n must be >= 0");
  VG_CHECK_ARG(ep->y2 == nullptr || (ep->post_scale && ep->post_shift), "the second output needs post_scale / post_shift");
  const float* bias = ep->bias; const float* colscale = ep->colscale; const float* sigma = ep->sigma;
  const int sigma_group_n = ep->sigma_group_n;
  const bool inference_ep = ep->act_slope != 1.0f || ep->residual != nullptr || ep->y2 != nullptr;
  cudaStream_t s = as_stream(stream);
  if (tc_conv_supported(d, false) && !(d->c_out == 1 && colscale != nullptr))
    rc = tc_conv_run(d, false, x, pack_kn, bias, colscale, sigma, sigma_group_n, y, d->out_dtype, s, ep);
  else if (inference_ep) {
    set_error("the activation / residual / second-output epilogue exists on the tensor-core path only (bf16, channels %% 64 == 0)");
    return VG_EUNSUPPORTED;
  } else
    rc = simt_conv_forward(d, x, pack_nk, bias, colscale, sigma, sigma_group_n, y, s);
  if (rc) return rc;
  // BatchNorm statistics of y come from the separate streaming statistics kernel.  Accumulating them in the tensor-core
  // epilogue was measured slower on B200 twice and removed: with per-chunk shared-memory transposes +35 % per launch (8
  // epilogue warps) / +60 % (4) against a 20 us statistics kernel; with a 31-shuffle column sum per 32 x 32 chunk in every
  // kernel form (scripts/sweep_conv.py, batch 64) 64->64 @96 74.9 -> 163 us, 128->128 @96 151 -> 217 us, 512->512 @24
  // 110 -> 125 us, whole step 63.7 -> 68.2 ms against a 17 us kernel: the epilogue warps bound the short-reduction layers
  // and ~350 extra instructions per chunk double their work.
  if (stats != nullptr) {
    VgBnDesc b{};
    b.rows = (long long)d->n * d->h_out * d->w_out;
    b.c = d->c_out;
    b.hw = d->h_out * d->w_out;
    b.dtype = d->out_dtype;
    b.slope = 1.f;
    rc = vg_bn_stats(y, &b, stats, stream);
  }
  return rc;
}

extern "C" int vg_conv_dgrad(const VgConvDesc* d, const void* dy, const void* pack_kn, const void* pack_nk, void* dx,
                             vg_stream_t stream) {
  return vg_conv_dgrad_scaled(d, dy, pack_kn, pack_nk, nullptr, 0, dx, stream);
}

extern "C" int vg_conv_dgrad_scaled(const VgConvDesc* d, const void* dy, const void* pack_kn, const void* pack_nk, const float* sigma,
                                    int sigma_group_n, void* dx, vg_stream_t stream) {
  int rc = check_conv(d);
  if (rc) return rc;
  if (d->n == 0) return VG_OK;
  VG_CHECK_ARG(dy && dx && pack_kn && pack_nk, "null pointer");
  VG_CHECK_ARG(sigma_group_n >= 0, "sigma_group_n must be >= 0");
  cudaStream_t s = as_stream(stream);
  if (tc_conv_supported(d, true))
    return tc_conv_run(d, true, dy, pack_nk, nullptr, nullptr, sigma, sigma_group_n, dx, d->act_dtype, s);
  return simt_conv_dgrad(d, dy, pack_kn, sigma, sigma_group_n, dx, s);
}

extern "C" int vg_conv_wgrad(const VgConvDesc* d, const void* x, const void* dy, float* dw, float* dbias, float* workspace,
                             vg_stream_t stream) {
  int rc = check_conv(d);
  if (rc) return rc;
  if (d->n == 0) return VG_OK;
  VG_CHECK_ARG(x && dy && dw, "null pointer");
  cudaStream_t s = as_stream(stream);
  if (tc_wgrad_supported(d))
    rc = tc_wgrad_run(d, x, dy, dw, workspace, s);
  else
    rc = simt_conv_wgrad(d, x, dy, dw, s);
  if (rc) return rc;
  if (dbias != nullptr) rc = simt_colsum(dy, (long long)d->n * d->h_out * d->w_out, d->c_out, d->act_dtype, dbias, s);
  return rc;
}

// ---- weight gradient of a spectral-normed convolution in one call ----------------------------------------------------------
extern "C" int vg_conv_wgrad_sn_supported(const VgConvDesc* d) { return (d != nullptr && vg::tc_wgrad_supported(d)) ? 1 : 0; }

extern "C" int vg_conv_wgrad_sn(const VgConvDesc* d, const void* x, const void* dy, const float* w_orig, const float* u,
                                const float* v, const float* sigma, float* dw_orig, float* dbias, float* workspace,
                                vg_stream_t stream) {
  int rc = check_conv(d);
  if (rc) return rc;
  if (d->n == 0) return VG_OK;
  VG_CHECK_ARG(x && dy && w_orig && u && v && sigma && dw_orig && workspace, "null pointer");
  if (!tc_wgrad_supported(d)) {
    set_error("vg_conv_wgrad_sn needs a tensor-core layer (bf16, channels %% 64 == 0): use vg_conv_wgrad + vg_spectral_norm_backward");
    return VG_EUNSUPPORTED;
  }
  cudaStream_t s = as_stream(stream);
  const int taps = d->kh * d->kw;
  const int cu = d->transposed ? d->c_in : d->c_out, cs = d->transposed ? d->c_out : d->c_in;
  const size_t welems = (size_t)taps * cu * cs;
  // ONE memset for the gradient accumulator and the dot-product cell behind it
  VG_CUDA(cudaMemsetAsync(workspace, 0, (welems + 4) * sizeof(float), s));
  if ((rc = tc_wgrad_run(d, x, dy, nullptr, workspace, s, /*acc_only=*/true))) return rc;
  // spectral norm: rows = dim 0 of the torch-layout weight (c_u), cols = the rest (c_s * taps)
  if (taps > 1) rc = sn_backward_packed_run(workspace, w_orig, u, v, sigma, cu, cs, taps, dw_orig, workspace + welems, s);
  else rc = sn_backward_run(workspace, w_orig, u, v, sigma, cu, cs, dw_orig, workspace + welems, s);
  if (rc) return rc;
  if (dbias) rc = simt_colsum(dy, (long long)d->n * d->h_out * d->w_out, d->c_out, d->act_dtype, dbias, s);
  return rc;
}

// ---- tile table (SURVEY.md section 8f N4) ------------------------------------------------------------------------------
extern "C" int vg_conv_tune_set(const VgConvDesc* d, int dgrad, int bn, int form) { return vg::tc_tune_set(d, dgrad, bn, form); }
extern "C" int vg_conv_tune_clear(void) {
  vg::tc_tune_clear();
  return VG_OK;
}
extern "C" int vg_conv_tune_record(int on) {
  vg::tc_tune_record(on);
  return VG_OK;
}
extern "C" int vg_conv_tune_seen(int* keys, int max_keys, int* count) {
  VG_CHECK_ARG(count != nullptr && max_keys >= 0 && (keys != nullptr || max_keys == 0), "bad args");
  *count = vg::tc_tune_seen(keys, max_keys);
  return VG_OK;
}
