// extern "C" boundary of libe2fgvi_b200.so (declared in include/e2fgvi_b200.h): argument validation, error
// strings, launch accounting.  No torch types, no allocation; the only process-wide state is per-device-ordinal caches
// of immutable facts (SM count, "function attributes already set on device d", cluster occupancy; launch.h DeviceOnce).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "e2fgvi_b200.h"
#include "launch.h"

namespace e2f {

static thread_local char g_err[512] = {0};
static std::atomic<long long> g_launches{0};

void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

int num_sms() {
  static std::atomic<int> cache[64];
  const int dev = current_device();
  int v = (dev >= 0 && dev < 64) ? cache[dev].load(std::memory_order_relaxed) : 0;
  if (!v) {
    v = 148;
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    if (dev >= 0 && dev < 64) cache[dev].store(v, std::memory_order_relaxed);
  }
  return v;
}

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static int finish(int status, const char* what) {
  if (status > 0) set_error("%s: CUDA error %d (%s)", what, status, cudaGetErrorString(static_cast<cudaError_t>(status)));
  return status;
}

static bool aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

}  // namespace e2f

using namespace e2f;

extern "C" {

const char* e2f_version(void) { return "e2fgvi_b200 0.1.0 sm_100a"; }

const char* e2f_last_error(void) { return g_err; }

int64_t e2f_launch_count(void) { return static_cast<int64_t>(g_launches.load(std::memory_order_relaxed)); }

int e2f_flow_warp(const void* x, const float* flow, void* out, int n, int h, int w, int c, int dtype, int pad_mode,
                  void* stream) {
  if (!x || !flow || !out) { set_error("e2f_flow_warp: null pointer"); return E2F_ERR_BAD_ARG; }
  if (n < 0 || h <= 0 || w <= 0 || c <= 0) { set_error("e2f_flow_warp: bad shape n=%d h=%d w=%d c=%d", n, h, w, c); return E2F_ERR_BAD_ARG; }
  if (dtype != E2F_F32 && dtype != E2F_F16) { set_error("e2f_flow_warp: dtype %d", dtype); return E2F_ERR_BAD_ARG; }
  if (pad_mode != E2F_PAD_ZEROS && pad_mode != E2F_PAD_BORDER) { set_error("e2f_flow_warp: pad_mode %d", pad_mode); return E2F_ERR_BAD_ARG; }
  const int vec = dtype == E2F_F16 ? 8 : 4;
  if (c % vec) { set_error("e2f_flow_warp: C=%d must be a multiple of %d for the NHWC kernel (use e2f_flow_warp_nchw)", c, vec); return E2F_ERR_UNSUPPORTED; }
  if (!aligned(x, 16) || !aligned(out, 16) || !aligned(flow, 8)) { set_error("e2f_flow_warp: x/out need 16-byte, flow 8-byte alignment"); return E2F_ERR_ALIGNMENT; }
  return finish(launch_flow_warp_nhwc(x, flow, out, n, h, w, c, dtype, pad_mode, static_cast<cudaStream_t>(stream)), "e2f_flow_warp");
}

int e2f_flow_warp_nchw(const float* x, const float* flow, float* out, int n, int c, int h, int w, int pad_mode,
                       void* stream) {
  if (!x || !flow || !out) { set_error("e2f_flow_warp_nchw: null pointer"); return E2F_ERR_BAD_ARG; }
  if (n < 0 || h <= 0 || w <= 0 || c <= 0) { set_error("e2f_flow_warp_nchw: bad shape"); return E2F_ERR_BAD_ARG; }
  if (pad_mode != E2F_PAD_ZEROS && pad_mode != E2F_PAD_BORDER) { set_error("e2f_flow_warp_nchw: pad_mode %d", pad_mode); return E2F_ERR_BAD_ARG; }
  if (!aligned(flow, 8)) { set_error("e2f_flow_warp_nchw: flow needs 8-byte alignment"); return E2F_ERR_ALIGNMENT; }
  return finish(launch_flow_warp_nchw(x, flow, out, n, c, h, w, pad_mode, static_cast<cudaStream_t>(stream)), "e2f_flow_warp_nchw");
}

int e2f_dcn_pack_weight(const float* w, void* w_packed_f16, int cout, int cin, int deform_groups, void* stream) {
  if (!w || !w_packed_f16) { set_error("e2f_dcn_pack_weight: null pointer"); return E2F_ERR_BAD_ARG; }
  if (cout <= 0 || cin <= 0 || deform_groups <= 0 || cin % deform_groups) { set_error("e2f_dcn_pack_weight: bad shape"); return E2F_ERR_BAD_ARG; }
  return finish(launch_dcn_pack_weight(w, w_packed_f16, cout, cin, deform_groups, static_cast<cudaStream_t>(stream)), "e2f_dcn_pack_weight");
}

static int dcn_common_checks(const char* who, const void* x, const void* w_packed, const void* out, int n, int h, int w,
                             int out_dtype) {
  if (!x || !w_packed || !out) { set_error("%s: null pointer", who); return E2F_ERR_BAD_ARG; }
  if (n < 0 || h <= 0 || w <= 0) { set_error("%s: bad shape n=%d h=%d w=%d", who, n, h, w); return E2F_ERR_BAD_ARG; }
  if (out_dtype != E2F_F32 && out_dtype != E2F_F16) { set_error("%s: out_dtype %d", who, out_dtype); return E2F_ERR_BAD_ARG; }
  if (!aligned(x, 32) || !aligned(w_packed, 128) || !aligned(out, 16)) { set_error("%s: x needs 32-byte, w_packed 128-byte, out 16-byte alignment", who); return E2F_ERR_ALIGNMENT; }
  return 0;
}

int e2f_modulated_deform_conv2d(const void* x, const float* offset, const float* mask, const void* w_packed,
                                const float* bias, void* out, int n, int h, int w, int cin, int cout,
                                int deform_groups, int out_dtype, int x_layout, void* stream) {
  int st = dcn_common_checks("e2f_modulated_deform_conv2d", x, w_packed, out, n, h, w, out_dtype);
  if (st) return st;
  if (!offset || !mask) { set_error("e2f_modulated_deform_conv2d: null offset/mask"); return E2F_ERR_BAD_ARG; }
  if (!aligned(offset, 16) || !aligned(mask, 16)) { set_error("e2f_modulated_deform_conv2d: offset / mask need 16-byte alignment"); return E2F_ERR_ALIGNMENT; }
  if (x_layout != E2F_X_NHWC && x_layout != E2F_X_GROUPED) { set_error("e2f_modulated_deform_conv2d: x_layout %d", x_layout); return E2F_ERR_BAD_ARG; }
  return finish(launch_dcn(x, offset, mask, nullptr, nullptr, nullptr, w_packed, bias, out, n, h, w, cin, cout,
                           deform_groups, 0.f, out_dtype, x_layout, static_cast<cudaStream_t>(stream)),
                "e2f_modulated_deform_conv2d");
}

int e2f_deform_align_fused(const void* x, const float* head, const float* flow1, const float* flow2,
                           const void* w_packed, const float* bias, void* out, int n, int h, int w, int cin, int cout,
                           int deform_groups, float max_residue, int out_dtype, int x_layout, void* stream) {
  int st = dcn_common_checks("e2f_deform_align_fused", x, w_packed, out, n, h, w, out_dtype);
  if (st) return st;
  if (!head || !flow1 || !flow2) { set_error("e2f_deform_align_fused: null head/flow"); return E2F_ERR_BAD_ARG; }
  if (!aligned(head, 16) || !aligned(flow1, 8) || !aligned(flow2, 8)) { set_error("e2f_deform_align_fused: head needs 16-byte, flow 8-byte alignment"); return E2F_ERR_ALIGNMENT; }
  if (x_layout != E2F_X_NHWC && x_layout != E2F_X_GROUPED) { set_error("e2f_deform_align_fused: x_layout %d", x_layout); return E2F_ERR_BAD_ARG; }
  return finish(launch_dcn(x, nullptr, nullptr, head, flow1, flow2, w_packed, bias, out, n, h, w, cin, cout,
                           deform_groups, max_residue, out_dtype, x_layout, static_cast<cudaStream_t>(stream)),
                "e2f_deform_align_fused");
}

int e2f_deform_align_fused_split(const void* x, const float* head, const float* flow1, const float* flow2,
                                 const void* w_packed, const float* bias, float* out, void* out_hi, void* out_lo, int n,
                                 int h, int w, int cin, int cout, int deform_groups, float max_residue, int x_layout,
                                 void* stream) {
  const char* who = "e2f_deform_align_fused_split";
  int st = dcn_common_checks(who, x, w_packed, out, n, h, w, E2F_F32);
  if (st) return st;
  if (!head || !flow1 || !flow2 || !out_hi || !out_lo) { set_error("%s: null pointer", who); return E2F_ERR_BAD_ARG; }
  if (!aligned(head, 16) || !aligned(flow1, 8) || !aligned(flow2, 8) || !aligned(out_hi, 16) || !aligned(out_lo, 16)) { set_error("%s: head / out_hi / out_lo need 16-byte, flow 8-byte alignment", who); return E2F_ERR_ALIGNMENT; }
  if (x_layout != E2F_X_NHWC && x_layout != E2F_X_GROUPED) { set_error("%s: x_layout %d", who, x_layout); return E2F_ERR_BAD_ARG; }
  return finish(launch_dcn(x, nullptr, nullptr, head, flow1, flow2, w_packed, bias, out, n, h, w, cin, cout,
                           deform_groups, max_residue, E2F_F32, x_layout, static_cast<cudaStream_t>(stream), out_hi, out_lo), who);
}

int e2f_focal_window_attention(const void* qkv, const void* qkv_pooled, void* out, int b, int t, int h, int w,
                               int heads, int head_dim, int wh, int ww, int eh, int ew, int fh, int fw,
                               int use_pooled, float scale, int out_dtype, void* stream) {
  if (!qkv || !out || (use_pooled && !qkv_pooled)) { set_error("e2f_focal_window_attention: null pointer"); return E2F_ERR_BAD_ARG; }
  if (b < 0 || t <= 0 || h <= 0 || w <= 0 || heads <= 0 || wh <= 0 || ww <= 0 || eh < 0 || ew < 0) { set_error("e2f_focal_window_attention: bad shape"); return E2F_ERR_BAD_ARG; }
  if (h % wh || w % ww) { set_error("e2f_focal_window_attention: token grid %dx%d is not a multiple of the window %dx%d", h, w, wh, ww); return E2F_ERR_BAD_ARG; }
  if (use_pooled && (fh <= 0 || fw <= 0 || !(fh & 1) || !(fw & 1))) { set_error("e2f_focal_window_attention: pooled neighbourhood %dx%d must be odd", fh, fw); return E2F_ERR_BAD_ARG; }
  if (out_dtype != E2F_F32 && out_dtype != E2F_F16 && out_dtype != E2F_SPLIT_BF16) { set_error("e2f_focal_window_attention: out_dtype %d", out_dtype); return E2F_ERR_BAD_ARG; }
  if (head_dim != 128) { set_error("e2f_focal_window_attention: head_dim %d unsupported (128 only)", head_dim); return E2F_ERR_UNSUPPORTED; }
  if (!aligned(qkv, 16) || !aligned(out, 16) || (use_pooled && !aligned(qkv_pooled, 16))) { set_error("e2f_focal_window_attention: 16-byte alignment required"); return E2F_ERR_ALIGNMENT; }
  return finish(launch_focal_attention(qkv, qkv_pooled, out, b, t, h, w, heads, head_dim, wh, ww, eh, ew, fh, fw,
                                       use_pooled, scale, out_dtype, static_cast<cudaStream_t>(stream)),
                "e2f_focal_window_attention");
}

int e2f_dcn_pack_input(const float* a, const float* b, void* xg, int n, int h, int w, int ca, int cb, void* stream) {
  if (!a || !b || !xg) { set_error("e2f_dcn_pack_input: null pointer"); return E2F_ERR_BAD_ARG; }
  if (n < 0 || h <= 0 || w <= 0 || ca <= 0 || cb <= 0 || ca % 16 || cb % 16) { set_error("e2f_dcn_pack_input: bad shape (channels must be multiples of 16)"); return E2F_ERR_BAD_ARG; }
  if (!aligned(a, 16) || !aligned(b, 16) || !aligned(xg, 16)) { set_error("e2f_dcn_pack_input: 16-byte alignment required"); return E2F_ERR_ALIGNMENT; }
  return finish(launch_dcn_pack_input(a, b, xg, n, h, w, ca, cb, static_cast<cudaStream_t>(stream)), "e2f_dcn_pack_input");
}

static int t2t_checks(const char* who, const void* a, const void* b, int bt, int c, int h, int w, int k, int s, int p) {
  if (!a || !b) { set_error("%s: null pointer", who); return E2F_ERR_BAD_ARG; }
  if (bt < 0 || c <= 0 || h <= 0 || w <= 0 || k <= 0 || s <= 0 || p < 0 || h + 2 * p < k || w + 2 * p < k) { set_error("%s: bad shape", who); return E2F_ERR_BAD_ARG; }
  if ((c * k * k) % 4) { set_error("%s: C*k*k=%d must be a multiple of 4", who, c * k * k); return E2F_ERR_UNSUPPORTED; }
  if (!aligned(a, 16) || !aligned(b, 16)) { set_error("%s: 16-byte alignment required", who); return E2F_ERR_ALIGNMENT; }
  return 0;
}

int e2f_t2t_unfold(const float* img, float* tokens, void* tokens_hi, void* tokens_lo, int bt, int c, int h, int w, int k,
                   int stride, int pad, int gelu, void* stream) {
  if ((!tokens && !tokens_hi) || (!tokens_hi) != (!tokens_lo)) { set_error("e2f_t2t_unfold: need tokens and/or both of tokens_hi/tokens_lo"); return E2F_ERR_BAD_ARG; }
  int st = t2t_checks("e2f_t2t_unfold", img, tokens ? static_cast<const void*>(tokens) : tokens_hi, bt, c, h, w, k, stride, pad);
  if (st) return st;
  if (tokens_hi && (!aligned(tokens_hi, 16) || !aligned(tokens_lo, 16))) { set_error("e2f_t2t_unfold: 16-byte alignment required"); return E2F_ERR_ALIGNMENT; }
  return finish(launch_t2t_unfold(img, tokens, tokens_hi, tokens_lo, bt, c, h, w, k, stride, pad, gelu, 0, static_cast<cudaStream_t>(stream)), "e2f_t2t_unfold");
}

int e2f_t2t_unfold_nhwc(const float* img_nhwc, float* tokens, void* tokens_hi, void* tokens_lo, int bt, int c, int h, int w,
                        int k, int stride, int pad, int gelu, void* stream) {
  if ((!tokens && !tokens_hi) || (!tokens_hi) != (!tokens_lo)) { set_error("e2f_t2t_unfold_nhwc: need tokens and/or both of tokens_hi/tokens_lo"); return E2F_ERR_BAD_ARG; }
  int st = t2t_checks("e2f_t2t_unfold_nhwc", img_nhwc, tokens ? static_cast<const void*>(tokens) : tokens_hi, bt, c, h, w, k, stride, pad);
  if (st) return st;
  if (tokens_hi && (!aligned(tokens_hi, 16) || !aligned(tokens_lo, 16))) { set_error("e2f_t2t_unfold_nhwc: 16-byte alignment required"); return E2F_ERR_ALIGNMENT; }
  st = launch_t2t_unfold(img_nhwc, tokens, tokens_hi, tokens_lo, bt, c, h, w, k, stride, pad, gelu, 1, static_cast<cudaStream_t>(stream));
  if (st == E2F_ERR_UNSUPPORTED) { set_error("e2f_t2t_unfold_nhwc: channels_last input needs k=7 stride=3 pad=3 and C %% 8 == 0 (k=%d s=%d p=%d c=%d)", k, stride, pad, c); return st; }
  return finish(st, "e2f_t2t_unfold_nhwc");
}

int e2f_t2t_fold_unfold(const float* tokens_in, float* tokens, void* tokens_hi, void* tokens_lo, int bt, int c, int h,
                        int w, int k, int stride, int pad, int gelu, int out_pitch, void* stream) {
  if ((!tokens && !tokens_hi) || (!tokens_hi) != (!tokens_lo)) { set_error("e2f_t2t_fold_unfold: need tokens and/or both of tokens_hi/tokens_lo"); return E2F_ERR_BAD_ARG; }
  int st = t2t_checks("e2f_t2t_fold_unfold", tokens_in, tokens ? static_cast<const void*>(tokens) : tokens_hi, bt, c, h, w, k, stride, pad);
  if (st) return st;
  if (tokens_hi && (!aligned(tokens_hi, 16) || !aligned(tokens_lo, 16))) { set_error("e2f_t2t_fold_unfold: 16-byte alignment required"); return E2F_ERR_ALIGNMENT; }
  if (out_pitch == 0) out_pitch = c * k * k;
  if (out_pitch < c * k * k || out_pitch % 4) { set_error("e2f_t2t_fold_unfold: out_pitch=%d must be 0 or a multiple of 4 >= C*k*k=%d", out_pitch, c * k * k); return E2F_ERR_BAD_ARG; }
  st = launch_t2t_fold_unfold(tokens_in, tokens, tokens_hi, tokens_lo, bt, c, h, w, k, stride, pad, gelu, out_pitch, static_cast<cudaStream_t>(stream));
  if (st == E2F_ERR_UNSUPPORTED) { set_error("e2f_t2t_fold_unfold: only k=7 stride=3 pad=3, C %% 4 == 0, bt <= 65535 and W <= 1800 are fused (k=%d s=%d p=%d c=%d w=%d); compose e2f_t2t_fold + e2f_t2t_unfold", k, stride, pad, c, w); return st; }
  return finish(st, "e2f_t2t_fold_unfold");
}

int e2f_layernorm_pool_split(const float* x, const float* gamma, const float* beta, const float* pool_w,
                             const float* pool_b, void* out_hi, void* out_lo, int bt, int h, int w, int c, int wh, int ww,
                             float eps, void* stream) {
  const char* who = "e2f_layernorm_pool_split";
  if (!x || !gamma || !beta || !pool_w || !out_hi || !out_lo) { set_error("%s: null pointer", who); return E2F_ERR_BAD_ARG; }
  if (bt < 0 || h <= 0 || w <= 0 || c <= 0 || wh <= 0 || ww <= 0 || h % wh || w % ww) { set_error("%s: bad shape bt=%d h=%d w=%d c=%d window=%dx%d", who, bt, h, w, c, wh, ww); return E2F_ERR_BAD_ARG; }
  if (!aligned(x, 16) || !aligned(out_hi, 16) || !aligned(out_lo, 16) || !aligned(gamma, 4) || !aligned(beta, 4)) { set_error("%s: 16-byte alignment required", who); return E2F_ERR_ALIGNMENT; }
  return finish(launch_layernorm_pool_split(x, gamma, beta, pool_w, pool_b, out_hi, out_lo, bt, h, w, c, wh, ww, eps, static_cast<cudaStream_t>(stream)), who);
}

int e2f_window_pool(const void* x_hi, const void* x_lo, const float* weight, const float* bias, float* out, void* out_hi,
                    void* out_lo, int bt, int h, int w, int c, int wh, int ww, void* stream) {
  if (!x_hi || !x_lo || !weight) { set_error("e2f_window_pool: null pointer"); return E2F_ERR_BAD_ARG; }
  if ((!out && !out_hi) || (!out_hi) != (!out_lo)) { set_error("e2f_window_pool: need out and/or both of out_hi/out_lo"); return E2F_ERR_BAD_ARG; }
  if (bt < 0 || h <= 0 || w <= 0 || c <= 0 || wh <= 0 || ww <= 0) { set_error("e2f_window_pool: bad shape"); return E2F_ERR_BAD_ARG; }
  if (h % wh || w % ww) { set_error("e2f_window_pool: token grid %dx%d is not a multiple of the window %dx%d", h, w, wh, ww); return E2F_ERR_BAD_ARG; }
  if (c % 8 || wh > 8 || static_cast<size_t>(wh) * c * 4 > 48 * 1024 || bt > 65535) { set_error("e2f_window_pool: needs C %% 8 == 0, wh <= 8, wh*C <= 12288, bt <= 65535 (c=%d wh=%d bt=%d)", c, wh, bt); return E2F_ERR_UNSUPPORTED; }
  if (!aligned(x_hi, 16) || !aligned(x_lo, 16) || (out && !aligned(out, 16)) || (out_hi && (!aligned(out_hi, 16) || !aligned(out_lo, 16)))) { set_error("e2f_window_pool: 16-byte alignment required"); return E2F_ERR_ALIGNMENT; }
  return finish(launch_window_pool(x_hi, x_lo, weight, bias, out, out_hi, out_lo, bt, h, w, c, wh, ww, static_cast<cudaStream_t>(stream)), "e2f_window_pool");
}

int e2f_upsample2x_split(const float* x, void* out_hi, void* out_lo, int n, int h, int w, int c, void* stream) {
  if (!x || !out_hi || !out_lo) { set_error("e2f_upsample2x_split: null pointer"); return E2F_ERR_BAD_ARG; }
  if (n < 0 || h <= 0 || w <= 0 || c <= 0) { set_error("e2f_upsample2x_split: bad shape"); return E2F_ERR_BAD_ARG; }
  if (c % 8) { set_error("e2f_upsample2x_split: C=%d must be a multiple of 8", c); return E2F_ERR_UNSUPPORTED; }
  if (!aligned(x, 32) || !aligned(out_hi, 16) || !aligned(out_lo, 16)) { set_error("e2f_upsample2x_split: x needs 32-byte, out_hi / out_lo 16-byte alignment"); return E2F_ERR_ALIGNMENT; }
  return finish(launch_upsample2x_split(x, out_hi, out_lo, n, h, w, c, static_cast<cudaStream_t>(stream)), "e2f_upsample2x_split");
}

int e2f_layernorm_split(const float* x, const float* gamma, const float* beta, float* out, void* out_hi, void* out_lo,
                        int64_t rows, int c, float eps, void* stream) {
  if (!x || !gamma || !beta) { set_error("e2f_layernorm_split: null pointer"); return E2F_ERR_BAD_ARG; }
  if ((!out && !out_hi) || (!out_hi) != (!out_lo)) { set_error("e2f_layernorm_split: need out and/or both of out_hi/out_lo"); return E2F_ERR_BAD_ARG; }
  if (rows < 0 || c <= 0) { set_error("e2f_layernorm_split: bad shape"); return E2F_ERR_BAD_ARG; }
  if (!aligned(x, 16) || (out && !aligned(out, 16)) || (out_hi && (!aligned(out_hi, 16) || !aligned(out_lo, 16)))) { set_error("e2f_layernorm_split: 16-byte alignment required"); return E2F_ERR_ALIGNMENT; }
  return finish(launch_layernorm_split(x, gamma, beta, out, out_hi, out_lo, rows, c, eps, static_cast<cudaStream_t>(stream)), "e2f_layernorm_split");
}

int e2f_t2t_fold(const float* tokens, const float* bias, float* img, int bt, int c, int h, int w, int k, int stride,
                 int pad, int normalize, void* stream) {
  int st = t2t_checks("e2f_t2t_fold", tokens, img, bt, c, h, w, k, stride, pad);
  if (st) return st;
  return finish(launch_t2t_fold(tokens, bias, img, bt, c, h, w, k, stride, pad, normalize, static_cast<cudaStream_t>(stream)), "e2f_t2t_fold");
}

int e2f_t2t_fold_nhwc(const float* tokens, const float* bias, const float* residual_nhwc, float* img_nhwc, int bt, int c,
                      int h, int w, int k, int stride, int pad, int normalize, void* stream) {
  int st = t2t_checks("e2f_t2t_fold_nhwc", tokens, img_nhwc, bt, c, h, w, k, stride, pad);
  if (st) return st;
  if (residual_nhwc && !aligned(residual_nhwc, 16)) { set_error("e2f_t2t_fold_nhwc: 16-byte alignment required"); return E2F_ERR_ALIGNMENT; }
  st = launch_t2t_fold_nhwc(tokens, bias, residual_nhwc, img_nhwc, bt, c, h, w, k, stride, pad, normalize, static_cast<cudaStream_t>(stream));
  if (st == E2F_ERR_UNSUPPORTED) { set_error("e2f_t2t_fold_nhwc: needs k=7 stride=3 pad=3, C %% 8 == 0, bt <= 65535 (k=%d s=%d p=%d c=%d)", k, stride, pad, c); return st; }
  return finish(st, "e2f_t2t_fold_nhwc");
}

int e2f_split_bf16(const float* x, void* hi_bf16, void* lo_bf16, int64_t n, void* stream) {
  if (!x || !hi_bf16 || !lo_bf16) { set_error("e2f_split_bf16: null pointer"); return E2F_ERR_BAD_ARG; }
  if (n < 0 || n % 8) { set_error("e2f_split_bf16: n=%lld must be a non-negative multiple of 8", static_cast<long long>(n)); return E2F_ERR_BAD_ARG; }
  if (!aligned(x, 16) || !aligned(hi_bf16, 16) || !aligned(lo_bf16, 16)) { set_error("e2f_split_bf16: 16-byte alignment required"); return E2F_ERR_ALIGNMENT; }
  return finish(launch_split_bf16(x, hi_bf16, lo_bf16, n, static_cast<cudaStream_t>(stream)), "e2f_split_bf16");
}

int e2f_linear_bf16x3(const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo, const float* bias,
                      const float* residual, void* out, int m, int n, int k, int out_dtype, int tile_hint,
                      void* stream) {
  if (!a_hi || !a_lo || !w_hi || !w_lo || !out) { set_error("e2f_linear_bf16x3: null pointer"); return E2F_ERR_BAD_ARG; }
  if (m < 0 || n <= 0 || k <= 0) { set_error("e2f_linear_bf16x3: bad shape m=%d n=%d k=%d", m, n, k); return E2F_ERR_BAD_ARG; }
  if (out_dtype != E2F_F32 && out_dtype != E2F_F16) { set_error("e2f_linear_bf16x3: out_dtype %d", out_dtype); return E2F_ERR_BAD_ARG; }
  if (tile_hint != 0 && tile_hint != 128 && tile_hint != 256) { set_error("e2f_linear_bf16x3: tile_hint %d", tile_hint); return E2F_ERR_BAD_ARG; }
  if (k % 8 || n % (out_dtype == E2F_F16 ? 8 : 4)) { set_error("e2f_linear_bf16x3: K %% 8 and N %% %d must be 0 (k=%d n=%d)", out_dtype == E2F_F16 ? 8 : 4, k, n); return E2F_ERR_UNSUPPORTED; }
  if (!aligned(a_hi, 16) || !aligned(a_lo, 16) || !aligned(w_hi, 16) || !aligned(w_lo, 16) || !aligned(out, 16) || (residual && !aligned(residual, 16))) { set_error("e2f_linear_bf16x3: 16-byte alignment required"); return E2F_ERR_ALIGNMENT; }
  int bn = tile_hint;
  if (bn == 0) {
    // 256-wide tiles re-read A half as often; 128-wide ones only when they save more than ~15% of padded columns
    const int t128 = (n + 127) / 128, t256 = (n + 255) / 256;
    bn = (n < 512 || t128 * 115 < t256 * 200) ? 128 : 256;
  }
  return finish(launch_linear_bf16x3(a_hi, a_lo, w_hi, w_lo, bias, residual, out, m, n, k, out_dtype, bn, static_cast<cudaStream_t>(stream)), "e2f_linear_bf16x3");
}

int e2f_conv2d_rows_bf16x3(int nsrc, const void* const* src_hi, const void* const* src_lo, const int* src_channels,
                           int in_rows, const void* w_hi, const void* w_lo, const float* bias, const float* residual,
                           float* out, void* out_hi, void* out_lo, int out_lead, int n, int h, int w, int cout, int groups,
                           float leaky_slope, int ksize, int stride, int pad, void* stream) {
  const char* who = "e2f_conv2d_bf16x3";
  if (!src_hi || !src_lo || !src_channels || !w_hi || !w_lo) { set_error("%s: null pointer", who); return E2F_ERR_BAD_ARG; }
  if ((!out && !out_hi) || (!out_hi) != (!out_lo)) { set_error("%s: need out and/or both of out_hi/out_lo", who); return E2F_ERR_BAD_ARG; }
  if (out_hi && cout % 8) { set_error("%s: split output needs Cout %% 8 == 0", who); return E2F_ERR_UNSUPPORTED; }
  if (nsrc < 1 || nsrc > 4) { set_error("%s: nsrc=%d (1..4 supported)", who, nsrc); return E2F_ERR_UNSUPPORTED; }
  if (n < 0 || h <= 0 || w <= 0 || cout <= 0 || groups <= 0 || cout % groups) { set_error("%s: bad shape n=%d h=%d w=%d cout=%d groups=%d", who, n, h, w, cout, groups); return E2F_ERR_BAD_ARG; }
  if (ksize < 1 || ksize > 7 || (stride != 1 && stride != 2) || pad < 0 || h + 2 * pad < ksize || w + 2 * pad < ksize) { set_error("%s: unsupported geometry k=%d stride=%d pad=%d", who, ksize, stride, pad); return E2F_ERR_UNSUPPORTED; }
  if (out_lead < 0 || out_lead > 8 || (out_lead && !out_hi)) { set_error("%s: out_lead=%d needs a split output and 0..8", who, out_lead); return E2F_ERR_BAD_ARG; }
  if (out_lead && groups != 1) { set_error("%s: row-gapped output needs groups == 1", who); return E2F_ERR_UNSUPPORTED; }
  if (in_rows) {
    const int cin = src_channels[0];
    const bool pow2 = cin == 4 || cin == 8 || cin == 16 || cin == 32;
    if (nsrc != 1 || groups != 1 || !pow2 || (stride * cin * 2) % 16 || (ksize > 64 / cin && (64 / cin) % stride)) {
      set_error("%s: window-packed input needs one source, groups == 1, cin in {4,8,16,32} with stride*cin*2 %% 16 == 0 (nsrc=%d groups=%d cin=%d stride=%d)", who, nsrc, groups, cin, stride);
      return E2F_ERR_UNSUPPORTED;
    }
  }
  for (int i = 0; i < nsrc; ++i) {
    if (!src_hi[i] || !src_lo[i]) { set_error("%s: null source %d", who, i); return E2F_ERR_BAD_ARG; }
    if (!in_rows && (src_channels[i] <= 0 || src_channels[i] % 8 || src_channels[i] % groups)) { set_error("%s: source %d has %d channels (needs a multiple of 8 and of groups)", who, i, src_channels[i]); return E2F_ERR_UNSUPPORTED; }
    if (!aligned(src_hi[i], 16) || !aligned(src_lo[i], 16)) { set_error("%s: 16-byte alignment required", who); return E2F_ERR_ALIGNMENT; }
  }
  if (!aligned(w_hi, 16) || !aligned(w_lo, 16) || (out && !aligned(out, 16)) || (out_hi && (!aligned(out_hi, 16) || !aligned(out_lo, 16))) || (residual && !aligned(residual, 16))) { set_error("%s: 16-byte alignment required", who); return E2F_ERR_ALIGNMENT; }
  if (n == 0) return 0;
  return finish(launch_conv3x3(nsrc, src_hi, src_lo, src_channels, w_hi, w_lo, bias, residual, out, out_hi, out_lo, n, h, w, cout, groups, leaky_slope, ksize, stride, pad, in_rows ? 1 : 0, out_lead, static_cast<cudaStream_t>(stream)), who);
}

int e2f_conv_gather_bf16x3(int nsrc, const void* const* src_hi, const void* const* src_lo, const int* src_channels,
                           const void* w_hi, const void* w_lo, const float* bias, const float* bias_map,
                           const float* residual, float* out, void* out_hi, void* out_lo, int n, int h_in, int w_in,
                           int cout, float leaky_slope, int stride, int grid_h, int grid_w, int tile_w, int tile_h,
                           int ntaps, const int8_t* tap_dy, const int8_t* tap_dx, int nphase, const uint8_t* ph_tap0,
                           const uint8_t* ph_oy, const uint8_t* ph_ox, int ostep, int out_h, int out_w,
                           const int64_t* src_nstride, int64_t out_nstride, void* stream) {
  const char* who = "e2f_conv_gather_bf16x3";
  if (out_nstride < 0) { set_error("%s: negative out_nstride", who); return E2F_ERR_BAD_ARG; }
  if (!src_hi || !src_lo || !src_channels || !w_hi || !w_lo || !tap_dy || !tap_dx || !ph_tap0 || !ph_oy || !ph_ox) { set_error("%s: null pointer", who); return E2F_ERR_BAD_ARG; }
  if ((!out && !out_hi) || (!out_hi) != (!out_lo)) { set_error("%s: need out and/or both of out_hi/out_lo", who); return E2F_ERR_BAD_ARG; }
  if (out_hi && cout % 8) { set_error("%s: split output needs Cout %% 8 == 0", who); return E2F_ERR_UNSUPPORTED; }
  if (nsrc < 1 || nsrc > 4) { set_error("%s: nsrc=%d (1..4 supported)", who, nsrc); return E2F_ERR_UNSUPPORTED; }
  if (n < 0 || h_in <= 0 || w_in <= 0 || cout <= 0 || grid_h <= 0 || grid_w <= 0 || out_h <= 0 || out_w <= 0) { set_error("%s: bad shape", who); return E2F_ERR_BAD_ARG; }
  if (stride < 1 || stride > 8 || ntaps < 1 || ntaps > 64 || nphase < 1 || nphase > 9 || ostep < 1 || ostep > 8 || tile_w < 1 || tile_h < 1 || tile_w * tile_h > 128) { set_error("%s: unsupported geometry stride=%d taps=%d phases=%d ostep=%d tile=%dx%d", who, stride, ntaps, nphase, ostep, tile_w, tile_h); return E2F_ERR_UNSUPPORTED; }
  if (ph_tap0[0] != 0 || ph_tap0[nphase] != ntaps) { set_error("%s: ph_tap0 must start at 0 and end at ntaps", who); return E2F_ERR_BAD_ARG; }
  for (int i = 0; i < nphase; ++i) {
    if (ph_tap0[i] >= ph_tap0[i + 1] || ph_oy[i] >= ostep || ph_ox[i] >= ostep) { set_error("%s: phase %d is empty or its offset exceeds ostep", who, i); return E2F_ERR_BAD_ARG; }
  }
  for (int i = 0; i < nsrc; ++i) {
    if (!src_hi[i] || !src_lo[i]) { set_error("%s: null source %d", who, i); return E2F_ERR_BAD_ARG; }
    if (src_channels[i] <= 0 || src_channels[i] % 8) { set_error("%s: source %d has %d channels (needs a multiple of 8)", who, i, src_channels[i]); return E2F_ERR_UNSUPPORTED; }
    if (!aligned(src_hi[i], 16) || !aligned(src_lo[i], 16)) { set_error("%s: 16-byte alignment required", who); return E2F_ERR_ALIGNMENT; }
  }
  if (!aligned(w_hi, 16) || !aligned(w_lo, 16) || (out && !aligned(out, 16)) || (out_hi && (!aligned(out_hi, 16) || !aligned(out_lo, 16))) || (residual && !aligned(residual, 16)) || (bias_map && !aligned(bias_map, 16))) { set_error("%s: 16-byte alignment required", who); return E2F_ERR_ALIGNMENT; }
  if (n == 0) return 0;
  ConvGeom g;
  g.grid_h = grid_h; g.grid_w = grid_w; g.out_h = out_h; g.out_w = out_w; g.tile_w = tile_w; g.tile_h = tile_h;
  g.ntaps = ntaps; g.nphase = nphase; g.ostep = ostep; g.tap_dy = tap_dy; g.tap_dx = tap_dx; g.ph_tap0 = ph_tap0;
  g.ph_oy = ph_oy; g.ph_ox = ph_ox; g.bias_map = bias_map;
  long long sn[4] = {0, 0, 0, 0};
  for (int i = 0; src_nstride && i < nsrc; ++i) sn[i] = static_cast<long long>(src_nstride[i]);
  g.src_nstride = src_nstride ? sn : nullptr;
  g.out_nstride = static_cast<long long>(out_nstride);
  return finish(launch_conv3x3(nsrc, src_hi, src_lo, src_channels, w_hi, w_lo, bias, residual, out, out_hi, out_lo, n, h_in, w_in, cout, 1, leaky_slope, 0, stride, 0, 0, 0, static_cast<cudaStream_t>(stream), &g), who);
}

int e2f_conv3x3_tanh_nchw(const void* src_hi, const void* src_lo, int cin, const void* w_hi, const void* w_lo,
                          const float* bias, float* out, int n, int h, int w, int cout, void* stream) {
  const char* who = "e2f_conv3x3_tanh_nchw";
  if (!src_hi || !src_lo || !w_hi || !w_lo || !out) { set_error("%s: null pointer", who); return E2F_ERR_BAD_ARG; }
  if (n < 0 || h <= 0 || w <= 0 || cin <= 0 || cin % 8 || cout <= 0 || cout > 32 || (cout & 3) == 0) { set_error("%s: bad shape n=%d h=%d w=%d cin=%d cout=%d (cin %% 8 == 0, cout <= 32 and not a multiple of 4)", who, n, h, w, cin, cout); return E2F_ERR_UNSUPPORTED; }
  if (!aligned(src_hi, 16) || !aligned(src_lo, 16) || !aligned(w_hi, 16) || !aligned(w_lo, 16) || !aligned(out, 4)) { set_error("%s: alignment", who); return E2F_ERR_ALIGNMENT; }
  if (n == 0) return 0;
  const void* hi[1] = {src_hi};
  const void* lo[1] = {src_lo};
  const int ch[1] = {cin};
  return finish(launch_conv3x3(1, hi, lo, ch, w_hi, w_lo, bias, nullptr, out, nullptr, nullptr, n, h, w, cout, 1, 1.0f, 3, 1, 1, 0, 0, static_cast<cudaStream_t>(stream), nullptr, 3), who);
}

int e2f_conv_kxn_bf16x3(int nsrc, const void* const* src_hi, const void* const* src_lo, const int* src_channels,
                        const void* w_hi, const void* w_lo, const float* bias, const float* residual, float* out, void* out_hi,
                        void* out_lo, int n, int h, int w, int cout, int groups, int co_pad, int ksize, float leaky_slope,
                        int flags, void* stream) {
  const char* who = "e2f_conv_kxn_bf16x3";
  if (!src_hi || !src_lo || !src_channels || !w_hi || !w_lo) { set_error("%s: null pointer", who); return E2F_ERR_BAD_ARG; }
  if ((!out && !out_hi) || (!out_hi) != (!out_lo)) { set_error("%s: need out and/or both of out_hi/out_lo", who); return E2F_ERR_BAD_ARG; }
  if (nsrc < 1 || nsrc > 2) { set_error("%s: nsrc=%d (1..2 supported)", who, nsrc); return E2F_ERR_UNSUPPORTED; }
  if (n < 0 || h <= 0 || w <= 0 || cout <= 0 || groups <= 0) { set_error("%s: bad shape", who); return E2F_ERR_BAD_ARG; }
  if (flags & ~3) { set_error("%s: flags %d", who, flags); return E2F_ERR_BAD_ARG; }
  if ((flags & 2) && (!out || out_hi)) { set_error("%s: the NCHW store goes with an fp32-only output", who); return E2F_ERR_BAD_ARG; }
  for (int i = 0; i < nsrc; ++i) {
    if (!src_hi[i] || !src_lo[i]) { set_error("%s: null source %d", who, i); return E2F_ERR_BAD_ARG; }
    if (!aligned(src_hi[i], 16) || !aligned(src_lo[i], 16)) { set_error("%s: alignment", who); return E2F_ERR_ALIGNMENT; }
  }
  if (!aligned(w_hi, 16) || !aligned(w_lo, 16) || (out && !aligned(out, 16)) ||
      (out_hi && (!aligned(out_hi, 16) || !aligned(out_lo, 16))) || (residual && !aligned(residual, 8))) { set_error("%s: alignment", who); return E2F_ERR_ALIGNMENT; }
  if (n == 0) return 0;
  return finish(launch_conv_kxn(nsrc, src_hi, src_lo, src_channels, w_hi, w_lo, bias, residual, out, out_hi, out_lo, n, h, w, cout,
                                groups, co_pad, ksize, leaky_slope, flags, static_cast<cudaStream_t>(stream)), who);
}

int e2f_conv2d_bf16x3(int nsrc, const void* const* src_hi, const void* const* src_lo, const int* src_channels,
                      const void* w_hi, const void* w_lo, const float* bias, const float* residual, float* out,
                      void* out_hi, void* out_lo, int n, int h, int w, int cout, int groups, float leaky_slope, int ksize,
                      int stride, int pad, void* stream) {
  return e2f_conv2d_rows_bf16x3(nsrc, src_hi, src_lo, src_channels, 0, w_hi, w_lo, bias, residual, out, out_hi, out_lo, 0, n,
                                h, w, cout, groups, leaky_slope, ksize, stride, pad, stream);
}

int e2f_conv_rows_pitch(int w, int lead, int channels) { return (w <= 0 || lead < 0 || channels <= 0) ? E2F_ERR_BAD_ARG : conv_rows_pitch(w, lead, channels); }

int e2f_conv_rows_tail(int lead, int channels) { return (lead < 0 || channels <= 0) ? E2F_ERR_BAD_ARG : conv_rows_tail(lead, channels); }

int e2f_pack_rows_bf16(const float* x, void* out_hi, void* out_lo, int n, int c, int h, int w, int cin, int lead,
                       void* stream) {
  if (!x || !out_hi || !out_lo) { set_error("e2f_pack_rows_bf16: null pointer"); return E2F_ERR_BAD_ARG; }
  if (n < 0 || c <= 0 || h <= 0 || w <= 0 || lead < 0 || lead > 8) { set_error("e2f_pack_rows_bf16: bad shape"); return E2F_ERR_BAD_ARG; }
  if ((cin != 4 && cin != 8 && cin != 16 && cin != 32) || c > cin) { set_error("e2f_pack_rows_bf16: cin=%d must be 4, 8, 16 or 32 and >= C=%d", cin, c); return E2F_ERR_UNSUPPORTED; }
  if (!aligned(x, 4) || !aligned(out_hi, 16) || !aligned(out_lo, 16)) { set_error("e2f_pack_rows_bf16: alignment"); return E2F_ERR_ALIGNMENT; }
  return finish(launch_pack_rows(x, out_hi, out_lo, n, c, h, w, cin, lead, static_cast<cudaStream_t>(stream)), "e2f_pack_rows_bf16");
}

int e2f_conv3x3_bf16x3(int nsrc, const void* const* src_hi, const void* const* src_lo, const int* src_channels,
                       const void* w_hi, const void* w_lo, const float* bias, const float* residual, float* out,
                       void* out_hi, void* out_lo, int n, int h, int w, int cout, int groups, float leaky_slope,
                       void* stream) {
  return e2f_conv2d_bf16x3(nsrc, src_hi, src_lo, src_channels, w_hi, w_lo, bias, residual, out, out_hi, out_lo, n, h, w,
                           cout, groups, leaky_slope, 3, 1, 1, stream);
}

int e2f_prop_prologue(const float* prop, const float* feat_n2, const float* flow_n1, int64_t flow_n1_bstride,
                      const float* flow_prev, int64_t flow_prev_bstride, void* cond1_hi, void* cond1_lo, void* cond2_hi,
                      void* cond2_lo, float* flow1_out, float* flow2_out, void* flows_hi, void* flows_lo, void* x_grouped,
                      int n, int h, int w, int c, void* stream) {
  if (!prop || !flow_n1 || !cond1_hi || !cond1_lo || !cond2_hi || !cond2_lo || !flow1_out || !flow2_out || !flows_hi ||
      !flows_lo || !x_grouped) { set_error("e2f_prop_prologue: null pointer"); return E2F_ERR_BAD_ARG; }
  if ((feat_n2 == nullptr) != (flow_prev == nullptr)) { set_error("e2f_prop_prologue: feat_n2 and flow_prev must both be given or both be NULL"); return E2F_ERR_BAD_ARG; }
  if (n < 0 || h <= 0 || w <= 0 || c <= 0 || c % 16) { set_error("e2f_prop_prologue: bad shape n=%d h=%d w=%d c=%d (C must be a multiple of 16)", n, h, w, c); return E2F_ERR_BAD_ARG; }
  if (!aligned(prop, 16) || (feat_n2 && !aligned(feat_n2, 16)) || !aligned(cond1_hi, 8) || !aligned(cond1_lo, 8) || !aligned(cond2_hi, 8) ||
      !aligned(cond2_lo, 8) || !aligned(flow1_out, 8) || !aligned(flow2_out, 8) || !aligned(flows_hi, 16) || !aligned(flows_lo, 16) ||
      !aligned(x_grouped, 16)) { set_error("e2f_prop_prologue: alignment"); return E2F_ERR_ALIGNMENT; }
  return finish(launch_prop_prologue(prop, feat_n2, flow_n1, static_cast<long long>(flow_n1_bstride), flow_prev,
                                     static_cast<long long>(flow_prev_bstride), cond1_hi, cond1_lo, cond2_hi, cond2_lo, flow1_out,
                                     flow2_out, flows_hi, flows_lo, x_grouped, n, h, w, c, static_cast<cudaStream_t>(stream)),
                "e2f_prop_prologue");
}

int e2f_spynet_pyramid(const float* frames, float* pyramid, int b, int t, int l_t, int H, int W, int h, int w, int h_up,
                       int w_up, const float* mean3, const float* std3, void* stream) {
  const char* who = "e2f_spynet_pyramid";
  if (!frames || !pyramid || !mean3 || !std3) { set_error("%s: null pointer", who); return E2F_ERR_BAD_ARG; }
  if (b < 0 || t <= 0 || l_t <= 0 || l_t > t || H <= 0 || W <= 0 || h <= 1 || w <= 1 || h > H || w > W) { set_error("%s: bad shape b=%d t=%d l_t=%d %dx%d -> %dx%d", who, b, t, l_t, H, W, h, w); return E2F_ERR_BAD_ARG; }
  if (h_up < h || w_up < w || h_up % 32 || w_up % 32) { set_error("%s: the working size %dx%d must be multiples of 32 >= %dx%d", who, h_up, w_up, h, w); return E2F_ERR_BAD_ARG; }
  return finish(launch_spynet_pyramid(frames, pyramid, b, t, l_t, H, W, h, w, h_up, w_up, mean3, std3, static_cast<cudaStream_t>(stream)), who);
}

int e2f_spynet_level_input(const float* level_img, const float* prev_flow, void* rows_hi, void* rows_lo, float* flow_up,
                           int b, int l_t, int hk, int wk, int lead, void* stream) {
  const char* who = "e2f_spynet_level_input";
  if (!level_img || !rows_hi || !rows_lo || !flow_up) { set_error("%s: null pointer", who); return E2F_ERR_BAD_ARG; }
  if (b < 0 || l_t < 2 || hk <= 0 || wk <= 0 || lead < 0 || lead > 8 || (prev_flow && ((hk | wk) & 1))) { set_error("%s: bad shape b=%d l_t=%d %dx%d lead=%d", who, b, l_t, hk, wk, lead); return E2F_ERR_BAD_ARG; }
  if (!aligned(rows_hi, 16) || !aligned(rows_lo, 16) || !aligned(flow_up, 8) || (prev_flow && !aligned(prev_flow, 8))) { set_error("%s: alignment", who); return E2F_ERR_ALIGNMENT; }
  return finish(launch_spynet_level_input(level_img, prev_flow, rows_hi, rows_lo, flow_up, b, l_t, hk, wk, lead, static_cast<cudaStream_t>(stream)), who);
}

int e2f_spynet_final(const float* flow, float* flows_forward, float* flows_backward, int b, int l_t, int h, int w, int h_up,
                     int w_up, void* stream) {
  const char* who = "e2f_spynet_final";
  if (!flow || !flows_forward || !flows_backward) { set_error("%s: null pointer", who); return E2F_ERR_BAD_ARG; }
  if (b < 0 || l_t < 2 || h <= 0 || w <= 0 || h_up < h || w_up < w) { set_error("%s: bad shape", who); return E2F_ERR_BAD_ARG; }
  if (!aligned(flow, 8)) { set_error("%s: flow needs 8-byte alignment", who); return E2F_ERR_ALIGNMENT; }
  return finish(launch_spynet_final(flow, flows_forward, flows_backward, b, l_t, h, w, h_up, w_up, static_cast<cudaStream_t>(stream)), who);
}

int e2f_video_prepare_clip(const uint8_t* frames, const uint8_t* masks, const int* ids, float* out, int t, int h, int w,
                           int hp, int wp, void* stream) {
  if (!frames || !masks || !ids || !out) { set_error("e2f_video_prepare_clip: null pointer"); return E2F_ERR_BAD_ARG; }
  if (t < 0 || h <= 0 || w <= 0 || hp < h || wp < w || hp > 2 * h || wp > 2 * w) {
    set_error("e2f_video_prepare_clip: bad shape t=%d h=%d w=%d hp=%d wp=%d (mirror padding needs h <= hp <= 2h, w <= wp <= 2w)", t, h, w, hp, wp);
    return E2F_ERR_BAD_ARG;
  }
  return finish(launch_video_prepare_clip(frames, masks, ids, out, t, h, w, hp, wp, static_cast<cudaStream_t>(stream)), "e2f_video_prepare_clip");
}

int e2f_video_compose(const float* pred, const uint8_t* frames, const uint8_t* masks, const int* ids, uint8_t* img,
                      int n_local, int h, int w, int hp, int wp, void* stream) {
  if (!pred || !frames || !masks || !ids || !img) { set_error("e2f_video_compose: null pointer"); return E2F_ERR_BAD_ARG; }
  if (n_local < 0 || h <= 0 || w <= 0 || hp < h || wp < w) { set_error("e2f_video_compose: bad shape n_local=%d h=%d w=%d hp=%d wp=%d", n_local, h, w, hp, wp); return E2F_ERR_BAD_ARG; }
  return finish(launch_video_compose(pred, frames, masks, ids, img, n_local, h, w, hp, wp, static_cast<cudaStream_t>(stream)), "e2f_video_compose");
}

int e2f_video_blend(const uint8_t* img, const int* ids, const int* first, float* comp, int n_local, int64_t frame_elems,
                    void* stream) {
  if (!img || !ids || !first || !comp) { set_error("e2f_video_blend: null pointer"); return E2F_ERR_BAD_ARG; }
  if (n_local < 0 || frame_elems <= 0) { set_error("e2f_video_blend: bad shape"); return E2F_ERR_BAD_ARG; }
  return finish(launch_video_blend(img, ids, first, comp, n_local, static_cast<long long>(frame_elems), static_cast<cudaStream_t>(stream)), "e2f_video_blend");
}

int e2f_video_finalize(const float* comp, uint8_t* out, int64_t count, void* stream) {
  if (!comp || !out) { set_error("e2f_video_finalize: null pointer"); return E2F_ERR_BAD_ARG; }
  if (count < 0) { set_error("e2f_video_finalize: bad count"); return E2F_ERR_BAD_ARG; }
  return finish(launch_video_finalize(comp, out, static_cast<long long>(count), static_cast<cudaStream_t>(stream)), "e2f_video_finalize");
}

static int psnr_ssim_shape_checks(const char* who, int n, int h, int w, int win_size) {
  if (n <= 0 || h <= 0 || w <= 0) { set_error("%s: bad shape n=%d h=%d w=%d", who, n, h, w); return E2F_ERR_BAD_ARG; }
  if (win_size < 3 || !(win_size & 1)) { set_error("%s: win_size %d must be odd and >= 3", who, win_size); return E2F_ERR_BAD_ARG; }
  if (win_size > h || win_size > w) { set_error("%s: win_size %d exceeds the image side (h=%d w=%d)", who, win_size, h, w); return E2F_ERR_BAD_ARG; }
  if (win_size > psnr_ssim_max_win()) { set_error("%s: win_size %d > %d unsupported", who, win_size, psnr_ssim_max_win()); return E2F_ERR_UNSUPPORTED; }
  return 0;
}

size_t e2f_psnr_ssim_workspace_bytes(int n, int h, int w, int win_size) {
  if (psnr_ssim_shape_checks("e2f_psnr_ssim_workspace_bytes", n, h, w, win_size)) return 0;
  return psnr_ssim_workspace_bytes(n, h, w, win_size);
}

int e2f_psnr_ssim(const uint8_t* ref, const float* test, double* psnr, double* ssim, int n, int h, int w, int win_size,
                  double data_range, void* workspace, void* stream) {
  const char* who = "e2f_psnr_ssim";
  if (!ref || !test || !psnr || !ssim || !workspace) { set_error("%s: null pointer", who); return E2F_ERR_BAD_ARG; }
  const int st = psnr_ssim_shape_checks(who, n, h, w, win_size);
  if (st) return st;
  if (!(data_range > 0.0)) { set_error("%s: data_range must be positive", who); return E2F_ERR_BAD_ARG; }
  if (!aligned(test, 4) || !aligned(psnr, 8) || !aligned(ssim, 8) || !aligned(workspace, 8)) { set_error("%s: test needs 4-byte, psnr / ssim / workspace 8-byte alignment", who); return E2F_ERR_ALIGNMENT; }
  return finish(launch_psnr_ssim(ref, test, psnr, ssim, n, h, w, win_size, data_range, workspace, static_cast<cudaStream_t>(stream)), who);
}

}  // extern "C"
