// Frame-quality metrics of the reference's evaluate.py (core/metrics.py:20-53): per-frame PSNR and SSIM of an fp32
// canvas against the uint8 original, as scikit-image 0.16's compare_ssim(data_range, multichannel=True, win_size)
// computes it with scipy's uniform_filter, in fp64 throughout.
//
// Only outputs whose whole window lies inside the image survive skimage's final crop by win_size/2, so no boundary
// handling is needed.  One CTA owns one frame, a strip of up to kRows output rows and the output columns whose windows
// fit in kCols input columns; it walks its input rows top to bottom:
//
//   A  stage the entering row i and the leaving row i - win (uint8 and fp32 -> float in shared memory, coalesced);
//      score the output row finished in the previous step; add the squared differences of the rows this CTA owns
//      for PSNR.
//   B  warp (q, c) — q in {x, y, x^2, y^2, xy}, c the channel — adds entering minus leaving values to its column sums
//      (registers, kK columns per lane), and writes the inclusive prefix over the strip's columns to shared memory,
//      so every window sum is one difference P[j + win] - P[j].
//
// For the inputs evaluation produces (uint8 originals, canvases that are multiples of 2^-d with d the blend depth)
// every product, sum and difference above is an exact fp64 value (all magnitudes stay below 2^40), so the only
// roundings are the final S formula and the mean; arbitrary fp32 inputs lose at most a few ulp of the sums.
//
// Each CTA writes (sum of S, sum of squared differences) to its own workspace slot; a second kernel sums a frame's
// slots in a fixed order.  No atomics: a frame's result depends only on its own pixels, not on the batch or the run.
#include <algorithm>
#include <cstdint>
#include "launch.h"

namespace e2f {
namespace metrics {

constexpr int kK = 8;                   // input columns per lane
constexpr int kCols = 32 * kK;          // input columns per CTA (the output strip is kCols - win + 1 wide)
constexpr int kRows = 16;               // output rows per CTA
constexpr int kWarps = 15;              // 5 quantities x 3 channels
constexpr int kThreads = 32 * kWarps;

struct Geometry {
  int pad, out_h, out_w, strip_w, strips_x, strips_y;
};

inline Geometry geometry(int h, int w, int win) {
  Geometry g;
  g.pad = win / 2;
  g.out_h = h - win + 1;
  g.out_w = w - win + 1;
  g.strip_w = kCols - (win - 1);
  g.strips_x = (g.out_w + g.strip_w - 1) / g.strip_w;
  g.strips_y = (g.out_h + kRows - 1) / kRows;
  return g;
}

// column ic of a staged row lives at (ic % kK) * 32 + ic / kK: lane l reads its kK columns without bank conflicts
__device__ __forceinline__ int swz(int ic) { return (ic % kK) * 32 + ic / kK; }

__device__ __forceinline__ double quantity(int q, double a, double b) {
  switch (q) {
    case 0: return a;
    case 1: return b;
    case 2: return __dmul_rn(a, a);
    case 3: return __dmul_rn(b, b);
    default: return __dmul_rn(a, b);
  }
}

__global__ void __launch_bounds__(kThreads) psnr_ssim_kernel(const uint8_t* __restrict__ ref,
                                                             const float* __restrict__ test,
                                                             double* __restrict__ partial, int h, int w, int win,
                                                             Geometry g, double c1, double c2) {
  __shared__ float sa[2][3][kCols];     // [enter, leave][channel][swizzled column]: original
  __shared__ float sb[2][3][kCols];     // canvas
  __shared__ double P[kWarps][kCols + 1];
  __shared__ double red[2][kWarps];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int q = warp / 3, qc = warp % 3;
  const int frame = blockIdx.y;
  const int sx = blockIdx.x % g.strips_x, sy = blockIdx.x / g.strips_x;
  const int ox0 = g.pad + sx * g.strip_w, ox1 = min(ox0 + g.strip_w, w - g.pad);
  const int oy0 = g.pad + sy * kRows, oy1 = min(oy0 + kRows, h - g.pad);
  const int tw = ox1 - ox0, ncols = tw + win - 1, ix0 = ox0 - g.pad;
  const int i_begin = oy0 - g.pad, i_end = oy1 + g.pad;
  // pixels whose squared difference this CTA adds for PSNR: a partition of the frame over the CTAs
  const int own_y0 = sy == 0 ? 0 : oy0, own_y1 = sy == g.strips_y - 1 ? h : oy1;
  const int own_x0 = sx == 0 ? 0 : ox0, own_x1 = sx == g.strips_x - 1 ? w : ox1;
  const double np = static_cast<double>(win) * win;
  const double cov_norm = __ddiv_rn(np, np - 1.0);
  const size_t frame_base = static_cast<size_t>(frame) * h * w * 3;

  if (tid < kWarps) P[tid][0] = 0.0;
  double colsum[kK];
#pragma unroll
  for (int k = 0; k < kK; ++k) colsum[k] = 0.0;
  double s_acc = 0.0, sq_acc = 0.0;

  // S for every output column of one finished row, from the prefix sums in P (skimage's formula and operand order)
  auto score_row = [&]() {
    for (int o = tid; o < tw * 3; o += kThreads) {
      const int j = o / 3, c = o - 3 * j;
      double m[5];
#pragma unroll
      for (int k = 0; k < 5; ++k) m[k] = __ddiv_rn(__dsub_rn(P[k * 3 + c][j + win], P[k * 3 + c][j]), np);
      const double ux = m[0], uy = m[1];
      const double vx = __dmul_rn(cov_norm, __dsub_rn(m[2], __dmul_rn(ux, ux)));
      const double vy = __dmul_rn(cov_norm, __dsub_rn(m[3], __dmul_rn(uy, uy)));
      const double vxy = __dmul_rn(cov_norm, __dsub_rn(m[4], __dmul_rn(ux, uy)));
      const double a1 = __dadd_rn(__dmul_rn(__dmul_rn(2.0, ux), uy), c1);
      const double a2 = __dadd_rn(__dmul_rn(2.0, vxy), c2);
      const double b1 = __dadd_rn(__dadd_rn(__dmul_rn(ux, ux), __dmul_rn(uy, uy)), c1);
      const double b2 = __dadd_rn(__dadd_rn(vx, vy), c2);
      s_acc = __dadd_rn(s_acc, __ddiv_rn(__dmul_rn(a1, a2), __dmul_rn(b1, b2)));
    }
  };

  for (int i = i_begin; i < i_end; ++i) {
    // ---- A
    if (i > i_begin + win - 1) score_row();                  // row i - 1 - pad was completed by the last step B
    const bool leave = i - win >= i_begin;
    for (int e = tid; e < 2 * kCols * 3; e += kThreads) {
      const int r = e / (kCols * 3), rest = e - r * kCols * 3, ic = rest / 3, c = rest - 3 * ic;
      float a = 0.f, b = 0.f;
      if (ic < ncols && (r == 0 || leave)) {
        const int row = r == 0 ? i : i - win;
        const size_t idx = frame_base + (static_cast<size_t>(row) * w + ix0 + ic) * 3 + c;
        a = static_cast<float>(__ldg(ref + idx));
        b = __ldg(test + idx);
        const int x = ix0 + ic;
        if (r == 0 && row >= own_y0 && row < own_y1 && x >= own_x0 && x < own_x1) {
          const double d = __dsub_rn(static_cast<double>(a), static_cast<double>(b));
          sq_acc = __dadd_rn(sq_acc, __dmul_rn(d, d));
        }
      }
      sa[r][c][swz(ic)] = a;
      sb[r][c][swz(ic)] = b;
    }
    __syncthreads();
    // ---- B
    double run = 0.0, pre[kK];
#pragma unroll
    for (int k = 0; k < kK; ++k) {
      const int s = k * 32 + lane;
      const double in = quantity(q, sa[0][qc][s], sb[0][qc][s]);
      const double out = quantity(q, sa[1][qc][s], sb[1][qc][s]);
      colsum[k] = __dsub_rn(__dadd_rn(colsum[k], in), out);
      run = __dadd_rn(run, colsum[k]);
      pre[k] = run;
    }
    double offset = run;                                      // inclusive scan of the lane totals
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const double v = __shfl_up_sync(0xffffffffu, offset, d);
      if (lane >= d) offset = __dadd_rn(offset, v);
    }
    offset = __shfl_up_sync(0xffffffffu, offset, 1);          // exclusive
    if (lane == 0) offset = 0.0;
#pragma unroll
    for (int k = 0; k < kK; ++k) P[warp][1 + lane * kK + k] = __dadd_rn(offset, pre[k]);
    __syncthreads();
  }
  score_row();

  // fixed-order CTA reduction
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    s_acc = __dadd_rn(s_acc, __shfl_down_sync(0xffffffffu, s_acc, d));
    sq_acc = __dadd_rn(sq_acc, __shfl_down_sync(0xffffffffu, sq_acc, d));
  }
  if (lane == 0) {
    red[0][warp] = s_acc;
    red[1][warp] = sq_acc;
  }
  __syncthreads();
  if (tid == 0) {
    double s = 0.0, sq = 0.0;
    for (int k = 0; k < kWarps; ++k) {
      s = __dadd_rn(s, red[0][k]);
      sq = __dadd_rn(sq, red[1][k]);
    }
    double* slot = partial + (static_cast<size_t>(frame) * gridDim.x + blockIdx.x) * 2;
    slot[0] = s;
    slot[1] = sq;
  }
}

__global__ void __launch_bounds__(128) psnr_ssim_finish_kernel(const double* __restrict__ partial,
                                                               double* __restrict__ psnr, double* __restrict__ ssim,
                                                               int n, int strips, double ssim_count, double px_count,
                                                               double data_range) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  double s = 0.0, sq = 0.0;
  for (int k = 0; k < strips; ++k) {
    s = __dadd_rn(s, partial[(static_cast<size_t>(f) * strips + k) * 2]);
    sq = __dadd_rn(sq, partial[(static_cast<size_t>(f) * strips + k) * 2 + 1]);
  }
  ssim[f] = __ddiv_rn(s, ssim_count);
  const double mse = __ddiv_rn(sq, px_count);
  psnr[f] = mse == 0.0 ? __longlong_as_double(0x7ff0000000000000ll) : 20.0 * log10(data_range / sqrt(mse));
}

}  // namespace metrics

size_t psnr_ssim_workspace_bytes(int n, int h, int w, int win) {
  const metrics::Geometry g = metrics::geometry(h, w, win);
  return static_cast<size_t>(n) * g.strips_x * g.strips_y * 2 * sizeof(double);
}

int psnr_ssim_max_win() { return metrics::kCols - 1; }

int launch_psnr_ssim(const uint8_t* ref, const float* test, double* psnr, double* ssim, int n, int h, int w, int win,
                     double data_range, void* workspace, cudaStream_t stream) {
  const metrics::Geometry g = metrics::geometry(h, w, win);
  const int strips = g.strips_x * g.strips_y;
  double* partial = static_cast<double*>(workspace);
  const double c1 = (0.01 * data_range) * (0.01 * data_range), c2 = (0.03 * data_range) * (0.03 * data_range);
  const size_t frame_elems = static_cast<size_t>(h) * w * 3;
  for (int f0 = 0; f0 < n; f0 += 65535) {              // grid.y limit; frames are independent
    const int nf = std::min(n - f0, 65535);
    metrics::psnr_ssim_kernel<<<dim3(strips, nf), metrics::kThreads, 0, stream>>>(
        ref + f0 * frame_elems, test + f0 * frame_elems, partial + static_cast<size_t>(f0) * strips * 2, h, w, win, g,
        c1, c2);
    count_launch();
    const int st = static_cast<int>(cudaGetLastError());
    if (st) return st;
  }
  metrics::psnr_ssim_finish_kernel<<<(n + 127) / 128, 128, 0, stream>>>(
      partial, psnr, ssim, n, strips, 3.0 * g.out_h * g.out_w, 3.0 * h * w, data_range);
  count_launch();
  return static_cast<int>(cudaGetLastError());
}

}  // namespace e2f
