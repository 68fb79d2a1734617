// Per-frame quality of a rollout against a target (gnca_rollout_metrics): the per-cell terms every kernel family adds
// up.  The premultiplied values and their differences are rounded one operation at a time (no FMA contraction), as
// torch forms them in utils/metrics.py, so the |diff| < eps and alpha > thr tests count the same cells as the
// metrics computed on the recorded frames.
#pragma once
#include "gnca_common.cuh"

namespace gnca {

// One part (a CTA's cells, or a block of a streaming sample) of one frame and sample: sum of the premultiplied-RGBA
// squared error, sum of the clipped-RGB squared error, pixel-perfect cells, alive cells.  The squares are exact in
// double; the counts are small integers.
struct MetAcc {
  double se, sr;
  int pp, al;
};

__device__ __forceinline__ void met_cell(MetAcc& m, float r, float g, float bl, float al,
                                         const float* __restrict__ tgt /* [4][HW] */, int cell, int HW, float eps,
                                         float thr) {
  const float p[4] = {__fmul_rn(r, al), __fmul_rn(g, al), __fmul_rn(bl, al), al};
  bool perfect = true;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float tc = __ldg(tgt + (size_t)c * HW + cell);
    const float d = __fsub_rn(p[c], tc);
    m.se += (double)d * (double)d;
    perfect = perfect && fabsf(d) < eps;
    if (c < 3) {
      const float e = __fsub_rn(fminf(fmaxf(p[c], 0.f), 1.f), fminf(fmaxf(tc, 0.f), 1.f));
      m.sr += (double)e * (double)e;
    }
  }
  m.pp += perfect ? 1 : 0;
  m.al += al > thr ? 1 : 0;
}

// butterfly over the warp: every lane ends with the same sums, in an order fixed by the lane indices
__device__ __forceinline__ void met_warp_sum(MetAcc& m) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    m.se += __shfl_xor_sync(0xffffffffu, m.se, o);
    m.sr += __shfl_xor_sync(0xffffffffu, m.sr, o);
    m.pp += __shfl_xor_sync(0xffffffffu, m.pp, o);
    m.al += __shfl_xor_sync(0xffffffffu, m.al, o);
  }
}

__device__ __forceinline__ void met_put(double* dst, const MetAcc& m) {
  dst[0] = m.se; dst[1] = m.sr; dst[2] = (double)m.pp; dst[3] = (double)m.al;
}

// SSIM of a frame (gnca_rollout_metrics_ssim, gnca_ssim_rgb): skimage's structural_similarity(pred, tgt,
// channel_axis=-1, data_range=1) with pred = clip(premultiplied RGB, 0, 1) and tgt = clip(target RGB, 0, 1).  A 7x7
// uniform window, cov_norm = 49/48, C1 = 0.01^2, C2 = 0.03^2, averaged over the (H-6)(W-6) interior cells only (a
// window never leaves the grid, so no padding mode enters).  Every family sums ssim_cell over its interior cells.
constexpr int kSsimWin = 7, kSsimR = 3;

__device__ __forceinline__ bool ssim_interior(int y, int x, int H, int W) {
  return y >= kSsimR && y < H - kSsimR && x >= kSsimR && x < W - kSsimR;
}

// S_R + S_G + S_B of the interior cell (y, x).  state(yy, xx) returns the raw (r, g, b, gated alpha) of a cell; the taps
// are visited in the same row-major order by every family, and the window moments are accumulated in double (every
// product of two fp32 values is exact there), so E[x^2] - ux^2 does not cancel in near-flat windows and every family
// gets the same bits for the same cell.
template <class State>
__device__ __forceinline__ double ssim_cell(const State& state, const float* __restrict__ tgt /* [4][HW] */, int y,
                                            int x, int W, int HW) {
  double sp[3] = {0.0, 0.0, 0.0}, sq[3] = {0.0, 0.0, 0.0}, spp[3] = {0.0, 0.0, 0.0}, sqq[3] = {0.0, 0.0, 0.0},
         spq[3] = {0.0, 0.0, 0.0};
#pragma unroll 1
  for (int i = -kSsimR; i <= kSsimR; ++i) {
#pragma unroll
    for (int j = -kSsimR; j <= kSsimR; ++j) {
      const int cell = (y + i) * W + (x + j);
      const float4 v = state(y + i, x + j);
      const float rgb[3] = {v.x, v.y, v.z};
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const double p = (double)fminf(fmaxf(__fmul_rn(rgb[c], v.w), 0.f), 1.f);
        const double q = (double)fminf(fmaxf(__ldg(tgt + (size_t)c * HW + cell), 0.f), 1.f);
        sp[c] += p; sq[c] += q; spp[c] += p * p; sqq[c] += q * q; spq[c] += p * q;
      }
    }
  }
  constexpr double inv_np = 1.0 / 49.0, cov_norm = 49.0 / 48.0, C1 = 0.01 * 0.01, C2 = 0.03 * 0.03;
  double s = 0.0;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const double ux = sp[c] * inv_np, uy = sq[c] * inv_np;
    const double vx = cov_norm * (spp[c] * inv_np - ux * ux), vy = cov_norm * (sqq[c] * inv_np - uy * uy);
    const double vxy = cov_norm * (spq[c] * inv_np - ux * uy);
    s += ((2.0 * ux * uy + C1) * (2.0 * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2));
  }
  return s;
}

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// dst[j] = sum over w in [w0, w1) of src[w * stride + j], in w order
__device__ __forceinline__ void met_sum_parts(double* dst, const double* src, int w0, int w1, int stride) {
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  for (int w = w0; w < w1; ++w) {
    s0 += src[w * stride]; s1 += src[w * stride + 1]; s2 += src[w * stride + 2]; s3 += src[w * stride + 3];
  }
  dst[0] = s0; dst[1] = s1; dst[2] = s2; dst[3] = s3;
}

}  // namespace gnca
