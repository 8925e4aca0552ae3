// Internal host-side launcher declarations shared by api.cu and the kernel translation units.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdint>

namespace e2f {

// Function attributes (opt-in dynamic shared memory), SM counts and cluster occupancy are PER DEVICE: a process that
// drives several GPUs (model moved to cuda:1, one thread per device) must configure each of them.  One bit per device
// ordinal; devices >= 64 are simply configured on every call.  Setting an attribute twice is idempotent, so two threads
// racing on the same bit are harmless.
struct DeviceOnce {
  std::atomic<unsigned long long> done{0};
};
inline int current_device() {
  int d = 0;
  cudaGetDevice(&d);
  return d;
}
inline bool device_done(const DeviceOnce& o, int dev) {
  return dev >= 0 && dev < 64 && ((o.done.load(std::memory_order_acquire) >> dev) & 1ull);
}
inline void device_mark(DeviceOnce& o, int dev) {
  if (dev >= 0 && dev < 64) o.done.fetch_or(1ull << dev, std::memory_order_release);
}
int num_sms();                             // api.cu: SM count of the CURRENT device (cached per device ordinal)

void count_launch();                       // api.cu: atomic launch counter behind e2f_launch_count()
void set_error(const char* fmt, ...);      // api.cu: thread-local message behind e2f_last_error()

int launch_flow_warp_nhwc(const void* x, const float* flow, void* out, int n, int h, int w, int c, int dtype,
                          int pad_mode, cudaStream_t stream);
int launch_flow_warp_nchw(const float* x, const float* flow, float* out, int n, int c, int h, int w, int pad_mode,
                          cudaStream_t stream);

int launch_prop_prologue(const float* prop, const float* feat2, const float* flow1, long long f1_bs, const float* flowp,
                         long long fp_bs, void* c1h, void* c1l, void* c2h, void* c2l, float* f1_out, float* f2_out,
                         void* flh, void* fll, void* xg, int n, int h, int w, int c, cudaStream_t stream);

int launch_dcn_pack_weight(const float* w, void* w_packed, int cout, int cin, int dg, cudaStream_t stream);
// head != nullptr selects the fused (tanh / flow / sigmoid) prologue; otherwise offset+mask are final values.
int launch_dcn(const void* x, const float* offset, const float* mask, const float* head, const float* flow1,
               const float* flow2, const void* w_packed, const float* bias, void* out, int n, int h, int w, int cin,
               int cout, int dg, float max_residue, int out_dtype, int x_grouped, cudaStream_t stream,
               void* out_hi = nullptr, void* out_lo = nullptr);   // optional bf16 split of the fp32 result
int launch_dcn_pack_input(const float* a, const float* b, void* xg, int n, int h, int w, int ca, int cb,
                          cudaStream_t stream);

int launch_focal_attention(const void* qkv, const void* qkv_pooled, void* out, int b, int t, int h, int w, int heads,
                           int head_dim, int wh, int ww, int eh, int ew, int fh, int fw, int use_pooled, float scale,
                           int out_dtype, cudaStream_t stream);

int launch_t2t_unfold(const float* img, float* tok, void* tok_hi, void* tok_lo, int bt, int c, int h, int w, int k,
                      int s, int p, int gelu, int nhwc, cudaStream_t stream);
int launch_upsample2x_split(const float* x, void* hi, void* lo, int n, int h, int w, int c, cudaStream_t stream);
int launch_layernorm_split(const float* x, const float* gamma, const float* beta, float* out, void* hi, void* lo,
                           long long rows, int c, float eps, cudaStream_t stream);
int launch_layernorm_pool_split(const float* x, const float* gamma, const float* beta, const float* pool_w,
                                const float* pool_b, void* hi, void* lo, int bt, int h, int w, int c, int wh, int ww,
                                float eps, cudaStream_t stream);
int launch_window_pool(const void* xh, const void* xl, const float* weight, const float* bias, float* out, void* out_hi,
                       void* out_lo, int bt, int h, int w, int c, int wh, int ww, cudaStream_t stream);
int launch_t2t_fold_unfold(const float* tin, float* tok, void* tok_hi, void* tok_lo, int bt, int c, int h, int w, int k,
                           int s, int p, int gelu, int out_pitch, cudaStream_t stream);
int launch_t2t_fold_nhwc(const float* tok, const float* bias, const float* residual, float* img, int bt, int c, int h,
                         int w, int k, int s, int p, int normalize, cudaStream_t stream);
int launch_t2t_fold(const float* tok, const float* bias, float* img, int bt, int c, int h, int w, int k, int s,
                    int p, int normalize, cudaStream_t stream);

int launch_split_bf16(const float* x, void* hi, void* lo, long long n, cudaStream_t stream);
int launch_linear_bf16x3(const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo, const float* bias,
                         const float* residual, void* out, int m, int n, int k, int out_dtype, int block_n,
                         cudaStream_t stream);

// Optional generalised geometry of the implicit-GEMM conv ("gather conv", see conv.cu Params): explicit tap offsets,
// output phases and tile shape.  nullptr = the plain k x k / stride / pad conv.
struct ConvGeom {
  int grid_h, grid_w;            // GEMM grid (per phase): one accumulator row per grid pixel
  int out_h, out_w;              // output image; grid pixel (y, x) of phase ph -> (y*ostep + ph_oy[ph], x*ostep + ph_ox[ph])
  int tile_w, tile_h;            // grid pixels per tile, tile_w * tile_h <= 128
  int ntaps, nphase, ostep;
  const int8_t* tap_dy;          // [ntaps] input offset of tap i relative to (y*stride, x*stride)
  const int8_t* tap_dx;
  const uint8_t* ph_tap0;        // [nphase + 1]
  const uint8_t* ph_oy;          // [nphase]
  const uint8_t* ph_ox;
  const float* bias_map;         // fp32 [out_h][out_w][cout] or null
  const long long* src_nstride;  // [nsrc] pixels between consecutive images of each source (0 / null = dense)
  long long out_nstride;         // pixels between consecutive images of every output and of the residual (0 = dense)
};
int launch_conv3x3(int nsrc, const void* const* src_hi, const void* const* src_lo, const int* src_channels,
                   const void* w_hi, const void* w_lo, const float* bias, const float* residual, float* out,
                   void* out_hi, void* out_lo, int n, int h_in, int w_in, int cout, int groups, float slope, int ks,
                   int stride, int pad, int in_rows, int out_lead, cudaStream_t stream, const ConvGeom* geom = nullptr,
                   int epi_flags = 0);     // 1: tanh, 2: NCHW fp32 output (3-channel output conv only)
int launch_conv_kxn(int nsrc, const void* const* src_hi, const void* const* src_lo, const int* src_c, const void* w_hi,
                    const void* w_lo, const float* bias, const float* residual, float* out, void* out_hi, void* out_lo, int n,
                    int h, int w, int cout, int groups, int co_pad, int ks, float slope, int flags, cudaStream_t stream);
int conv_rows_tail(int lead, int channels);
int conv_rows_pitch(int w, int lead, int channels);
int launch_pack_rows(const float* x, void* hi, void* lo, int n, int c, int h, int w, int cin, int lead,
                     cudaStream_t stream);

int launch_spynet_pyramid(const float* frames, float* pyr, int b, int t, int lt, int H, int W, int h, int w, int hu, int wu,
                          const float* mean3, const float* std3, cudaStream_t stream);
int launch_spynet_level_input(const float* img, const float* prev, void* hi, void* lo, float* flow_up, int b, int lt, int hk,
                              int wk, int lead, cudaStream_t stream);
int launch_spynet_final(const float* flow, float* out_fwd, float* out_bwd, int b, int lt, int h, int w, int hu, int wu,
                        cudaStream_t stream);

int launch_video_prepare_clip(const uint8_t* frames, const uint8_t* masks, const int* ids, float* out, int t, int h,
                              int w, int hp, int wp, cudaStream_t stream);
int launch_video_compose(const float* pred, const uint8_t* frames, const uint8_t* masks, const int* ids, uint8_t* img,
                         int n_local, int h, int w, int hp, int wp, cudaStream_t stream);
int launch_video_blend(const uint8_t* img, const int* ids, const int* first, float* comp, int n_local,
                       long long frame_elems, cudaStream_t stream);
int launch_video_finalize(const float* comp, uint8_t* out, long long count, cudaStream_t stream);

size_t psnr_ssim_workspace_bytes(int n, int h, int w, int win);
int psnr_ssim_max_win();
int launch_psnr_ssim(const uint8_t* ref, const float* test, double* psnr, double* ssim, int n, int h, int w, int win,
                     double data_range, void* workspace, cudaStream_t stream);

}  // namespace e2f
