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

// dst[j] = sum over w in [w0, w1) of src[w * stride + j], in w order
__device__ __forceinline__ void met_sum_parts(double* dst, const double* src, int w0, int w1, int stride) {
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  for (int w = w0; w < w1; ++w) {
    s0 += src[w * stride]; s1 += src[w * stride + 1]; s2 += src[w * stride + 2]; s3 += src[w * stride + 3];
  }
  dst[0] = s0; dst[1] = s1; dst[2] = s2; dst[3] = s3;
}

}  // namespace gnca
