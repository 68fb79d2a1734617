// Stand-alone operators and training glue: perception fwd/bwd, alive mask, premultiplied-RGBA loss (+grad),
// per-tensor gradient normalisation + Adam, multiplicative damage masks.
#include "gnca_common.cuh"

namespace gnca {

// perception.py:21-26 ---------------------------------------------------------------------------------
__global__ void k_perception_fwd(int B, int C, int H, int W, const float* __restrict__ x, float* __restrict__ out) {
  const int HW = H * W;
  const size_t n = (size_t)B * C * HW;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int cell = (int)(i % HW);
    const int c = (int)((i / HW) % C);
    const int b = (int)(i / ((size_t)HW * C));
    const int y = cell / W, xx = cell - y * W;
    const float* p = x + i;
    const bool up = y > 0, dn = y < H - 1, lf = xx > 0, rt = xx < W - 1;
    float a00 = (up && lf) ? p[-W - 1] : 0.f, a01 = up ? p[-W] : 0.f, a02 = (up && rt) ? p[-W + 1] : 0.f;
    float a10 = lf ? p[-1] : 0.f, a11 = p[0], a12 = rt ? p[1] : 0.f;
    float a20 = (dn && lf) ? p[W - 1] : 0.f, a21 = dn ? p[W] : 0.f, a22 = (dn && rt) ? p[W + 1] : 0.f;
    float* o = out + ((size_t)b * 3 * C) * HW + cell;
    o[(size_t)c * HW] = a11;
    o[(size_t)(C + c) * HW] = (a00 - a02) + 2.f * (a10 - a12) + (a20 - a22);
    o[(size_t)(2 * C + c) * HW] = (a00 + 2.f * a01 + a02) - (a20 + 2.f * a21 + a22);
  }
}

// transpose of the above: gx[y,x] = gid[y,x] + sum_{i,j} kx[i][j]*gsx[y-i,x-j] + ky[i][j]*gsy[y-i,x-j], zero halo
__global__ void k_perception_bwd(int B, int C, int H, int W, const float* __restrict__ gy, float* __restrict__ gx) {
  const int HW = H * W;
  const size_t n = (size_t)B * C * HW;
  const float kx[3][3] = {{1.f, 0.f, -1.f}, {2.f, 0.f, -2.f}, {1.f, 0.f, -1.f}};
  const float ky[3][3] = {{1.f, 2.f, 1.f}, {0.f, 0.f, 0.f}, {-1.f, -2.f, -1.f}};
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int cell = (int)(i % HW);
    const int c = (int)((i / HW) % C);
    const int b = (int)(i / ((size_t)HW * C));
    const int y = cell / W, xx = cell - y * W;
    const float* g0 = gy + ((size_t)b * 3 * C) * HW;
    const float* gsx = g0 + (size_t)(C + c) * HW;
    const float* gsy = g0 + (size_t)(2 * C + c) * HW;
    float acc = g0[(size_t)c * HW + cell];
#pragma unroll
    for (int di = -1; di <= 1; ++di) {
#pragma unroll
      for (int dj = -1; dj <= 1; ++dj) {
        const int yy = y - di, xq = xx - dj;   // output position whose stencil tap (di,dj) reads (y,x)
        if (yy < 0 || yy >= H || xq < 0 || xq >= W) continue;
        acc = fmaf(kx[di + 1][dj + 1], gsx[yy * W + xq], acc);
        acc = fmaf(ky[di + 1][dj + 1], gsy[yy * W + xq], acc);
      }
    }
    gx[i] = acc;
  }
}

__global__ void k_alive_mask(int B, int C, int H, int W, const float* __restrict__ x, float thr, float* __restrict__ m) {
  const int HW = H * W;
  const size_t n = (size_t)B * HW;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int cell = (int)(i % HW);
    const int b = (int)(i / HW);
    const int y = cell / W, xx = cell - y * W;
    m[i] = alive_at(x + ((size_t)b * C + 3) * HW, y, xx, H, W, thr) ? 1.f : 0.f;
  }
}

// train_graph_augmented_nca.py:52-61 -- one block per sample, deterministic
// MT (gnca_loss_premult_rgba_targets): tgt is [B / per][4][H][W] and sample b reads target b / per; per is unused
// otherwise.  A compile-time flag with a trailing parameter, so the single-target kernel keeps its code.
template <bool MT>
__global__ void k_loss_premult(int B, int C, int H, int W, const float* __restrict__ x, const float* __restrict__ tgt,
                               float* __restrict__ per_sample, float* __restrict__ gx, float scale, int per) {
  const int b = blockIdx.x, HW = H * W;
  if constexpr (MT) tgt += (size_t)(b / per) * 4 * HW;
  const float* xb = x + (size_t)b * C * HW;
  const float inv = 1.0f / (4.0f * (float)HW);
  double acc = 0.0;
  for (int cell = threadIdx.x; cell < HW; cell += blockDim.x) {
    const float r = xb[cell], g = xb[HW + cell], bl = xb[2 * HW + cell], al = xb[3 * HW + cell];
    const float d0 = r * al - tgt[cell], d1 = g * al - tgt[HW + cell], d2 = bl * al - tgt[2 * HW + cell],
                d3 = al - tgt[3 * HW + cell];
    acc += (double)(d0 * d0) + (double)(d1 * d1) + (double)(d2 * d2) + (double)(d3 * d3);
    if (gx) {
      float* gb = gx + (size_t)b * C * HW;
      const float s = 2.0f * inv * scale;
      gb[cell] = s * d0 * al;
      gb[HW + cell] = s * d1 * al;
      gb[2 * HW + cell] = s * d2 * al;
      gb[3 * HW + cell] = s * (d3 + d0 * r + d1 * g + d2 * bl);
      for (int c = 4; c < C; ++c) gb[(size_t)c * HW + cell] = 0.f;
    }
  }
  __shared__ double sred[32];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sred[w];
    per_sample[b] = (float)(t * (double)inv);
  }
}

// train_graph_augmented_nca.py:370-375 + torch.optim.Adam (coupled L2): one block per parameter tensor
struct Segments {
  int64_t off[33];
  int32_t has_grad[32];
  int n;
};

__global__ void k_normalize_adam(Segments S, float* __restrict__ p, float* __restrict__ g, float* __restrict__ m,
                                 float* __restrict__ v, int normalize, float lr, float b1, float b2, float eps, float wd,
                                 float bc1, float bc2_sqrt) {
  const int s = blockIdx.x;
  if (!S.has_grad[s]) return;
  const int64_t lo = S.off[s], hi = S.off[s + 1];
  __shared__ double sred[32];
  __shared__ float s_scale;
  float scale = 1.f;
  if (normalize) {
    double acc = 0.0;
    for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) acc += (double)g[i] * (double)g[i];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sred[w];
      s_scale = 1.0f / ((float)sqrt(t) + 1e-8f);
    }
    __syncthreads();
    scale = s_scale;
  }
  for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
    float gi = g[i] * scale;
    g[i] = gi;                                   // the reference normalises p.grad in place
    const float pi = p[i];
    if (wd != 0.f) gi = fmaf(wd, pi, gi);
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = pi - (lr / bc1) * (mi / denom);
  }
}

__global__ void k_apply_mask(int64_t n, float* __restrict__ x, const float* __restrict__ mask) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    x[i] *= mask[i];
}

inline int grid_for(size_t n, int threads = 256) {
  size_t g = (n + threads - 1) / threads;
  return (int)(g < 1 ? 1 : (g > 148 * 16 ? 148 * 16 : g));
}


// ------------------------------------------------------------------------------------------------
// damage descriptor -> per-cell plane (utils/damage.py:16-98 in closed form; one thread per cell)
// ------------------------------------------------------------------------------------------------
__global__ void k_damage_plane(gnca_damage d, int B, int C, int H, int W, const float* __restrict__ state,
                               float* __restrict__ plane) {
  const int HW = H * W;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)B * HW) return;
  const int b = (int)(i / HW), cell = (int)(i - (size_t)b * HW), y = cell / W, x = cell - y * W;
  float v = 1.f;
  switch (d.kind) {
    case GNCA_DK_SQUARE: {                       // state[b, :, y0:y0+size, x0:x0+size] = 0       damage.py:16-24
      const long long y0 = d.pos[2 * b], x0 = d.pos[2 * b + 1];
      if (y >= y0 && y < y0 + d.size && x >= x0 && x < x0 + d.size) v = 0.f;
    } break;
    case GNCA_DK_CIRCLE: {                       // (yy-cy)^2 + (xx-cx)^2 <= r^2 -> 0              damage.py:27-37
      const long long dy = y - d.pos[2 * b], dx = x - d.pos[2 * b + 1];
      if (dy * dy + dx * dx <= (long long)d.size * d.size) v = 0.f;
    } break;
    case GNCA_DK_STRIPE_H: { const long long s0 = d.pos[0]; if (y >= s0 && y < s0 + d.size) v = 0.f; } break;   // :40-51
    case GNCA_DK_STRIPE_V: { const long long s0 = d.pos[0]; if (x >= s0 && x < s0 + d.size) v = 0.f; } break;
    case GNCA_DK_GAUSSIAN: {                     // clamp(1 - exp(-r2 / (2 (R*soft)^2)), 0, 1)      damage.py:87-98
      const long long dy = y - d.pos[2 * b], dx = x - d.pos[2 * b + 1];
      const float r2 = (float)(dy * dy + dx * dx);
      const float sg = (float)d.size * fmaxf(1e-6f, d.softness);
      const float m = expf(-(r2 / (2.0f * sg * sg)));
      v = fminf(fmaxf(1.0f - m, 0.f), 1.f);
    } break;
    case GNCA_DK_ALPHA_DROP:                     // (rand < p) * (alpha > thr) -> 0, all channels   damage.py:54-66
      if (d.rand[i] < d.p && state[((size_t)b * C + 3) * HW + cell] > d.alpha_thr) v = 0.f;
      break;
    case GNCA_DK_SALTPEPPER:                     // rand < p -> alpha 0                             damage.py:69-73
      if (d.rand[i] < d.p) v = 0.f;
      break;
  }
  plane[i] = v;
}

__global__ void k_apply_plane(int B, int C, int HW, float* __restrict__ x, const float* __restrict__ plane, int alpha_only) {
  const size_t n = (size_t)B * C * HW;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t bc = i / HW;
    const int c = (int)(bc % C);
    if (alpha_only && c != 3) continue;
    x[i] *= plane[(bc / C) * HW + (i - bc * HW)];
  }
}
}  // namespace gnca

using namespace gnca;

extern "C" {

int gnca_perception_fwd(int B, int C, int H, int W, const float* x_dev, float* y_dev, void* stream) {
  if (!x_dev || !y_dev || B <= 0 || C <= 0 || H <= 0 || W <= 0) return GNCA_ERR_ARG;
  k_perception_fwd<<<grid_for((size_t)B * C * H * W), 256, 0, (cudaStream_t)stream>>>(B, C, H, W, x_dev, y_dev);
  GNCA_LAUNCH_CHECK();
  return 0;
}

int gnca_perception_bwd(int B, int C, int H, int W, const float* gy_dev, float* gx_dev, void* stream) {
  if (!gy_dev || !gx_dev || B <= 0 || C <= 0 || H <= 0 || W <= 0) return GNCA_ERR_ARG;
  k_perception_bwd<<<grid_for((size_t)B * C * H * W), 256, 0, (cudaStream_t)stream>>>(B, C, H, W, gy_dev, gx_dev);
  GNCA_LAUNCH_CHECK();
  return 0;
}

int gnca_alive_mask(int B, int C, int H, int W, const float* x_dev, float thr, float* mask_dev, void* stream) {
  if (!x_dev || !mask_dev || B <= 0 || C < 4 || H <= 0 || W <= 0) return GNCA_ERR_ARG;
  k_alive_mask<<<grid_for((size_t)B * H * W), 256, 0, (cudaStream_t)stream>>>(B, C, H, W, x_dev, thr, mask_dev);
  GNCA_LAUNCH_CHECK();
  return 0;
}

int gnca_loss_premult_rgba(int B, int C, int H, int W, const float* x_dev, const float* target_dev,
                           float* per_sample_dev, float* gx_dev, float scale, void* stream) {
  if (!x_dev || !target_dev || !per_sample_dev || B <= 0 || C < 4 || H <= 0 || W <= 0) return GNCA_ERR_ARG;
  k_loss_premult<false><<<B, 256, 0, (cudaStream_t)stream>>>(B, C, H, W, x_dev, target_dev, per_sample_dev, gx_dev,
                                                              scale, 0);
  GNCA_LAUNCH_CHECK();
  return 0;
}

int gnca_loss_premult_rgba_targets(int B, int C, int H, int W, const float* x_dev, const float* targets_dev,
                                   int n_targets, float* per_sample_dev, float* gx_dev, float scale, void* stream) {
  if (!x_dev || !targets_dev || !per_sample_dev || B <= 0 || C < 4 || H <= 0 || W <= 0) return GNCA_ERR_ARG;
  if (n_targets < 1 || B % n_targets != 0) return GNCA_ERR_ARG;
  k_loss_premult<true><<<B, 256, 0, (cudaStream_t)stream>>>(B, C, H, W, x_dev, targets_dev, per_sample_dev, gx_dev,
                                                             scale, B / n_targets);
  GNCA_LAUNCH_CHECK();
  return 0;
}

int gnca_normalize_adam(float* params_dev, float* grads_dev, float* exp_avg_dev, float* exp_avg_sq_dev,
                        const int64_t* seg_off_host, const int32_t* seg_has_grad_host, int n_seg, int normalize,
                        float lr, float beta1, float beta2, float eps, float weight_decay, int64_t step, void* stream) {
  if (!params_dev || !grads_dev || !exp_avg_dev || !exp_avg_sq_dev || !seg_off_host) return GNCA_ERR_ARG;
  if (n_seg <= 0 || n_seg > 32 || step < 1) return GNCA_ERR_ARG;
  Segments S;
  S.n = n_seg;
  for (int i = 0; i <= n_seg; ++i) S.off[i] = seg_off_host[i];
  for (int i = 0; i < n_seg; ++i) S.has_grad[i] = seg_has_grad_host ? seg_has_grad_host[i] : 1;
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  k_normalize_adam<<<n_seg, 256, 0, (cudaStream_t)stream>>>(S, params_dev, grads_dev, exp_avg_dev, exp_avg_sq_dev,
                                                            normalize, lr, beta1, beta2, eps, weight_decay, (float)bc1,
                                                            (float)sqrt(bc2));
  GNCA_LAUNCH_CHECK();
  return 0;
}

int gnca_apply_mask(int64_t n, float* x_dev, const float* mask_dev, void* stream) {
  if (!x_dev || !mask_dev || n <= 0) return GNCA_ERR_ARG;
  k_apply_mask<<<grid_for((size_t)n), 256, 0, (cudaStream_t)stream>>>(n, x_dev, mask_dev);
  GNCA_LAUNCH_CHECK();
  return 0;
}

int gnca_damage_plane(const gnca_damage* d, int B, int C, int H, int W, const float* state_dev, float* plane_dev,
                      int32_t* layout_out, void* stream) {
  if (!d || !plane_dev || B <= 0 || C <= 0 || H <= 0 || W <= 0) return GNCA_ERR_ARG;
  if (d->kind < GNCA_DK_SQUARE || d->kind > GNCA_DK_SALTPEPPER) return GNCA_ERR_UNSUPPORTED;
  const bool needs_pos = d->kind <= GNCA_DK_GAUSSIAN, needs_rand = d->kind >= GNCA_DK_ALPHA_DROP;
  if ((needs_pos && !d->pos) || (needs_rand && !d->rand)) return GNCA_ERR_ARG;
  if (d->kind == GNCA_DK_ALPHA_DROP && (!state_dev || C < 4)) return GNCA_ERR_ARG;
  const size_t n = (size_t)B * H * W;
  k_damage_plane<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(*d, B, C, H, W, state_dev, plane_dev);
  GNCA_LAUNCH_CHECK();
  if (layout_out) *layout_out = d->kind == GNCA_DK_SALTPEPPER ? GNCA_DMG_PLANE_ALPHA : GNCA_DMG_PLANE;
  return 0;
}

int gnca_apply_plane(int B, int C, int H, int W, float* state_dev, const float* plane_dev, int32_t layout, void* stream) {
  if (!state_dev || !plane_dev || B <= 0 || C <= 0 || H <= 0 || W <= 0) return GNCA_ERR_ARG;
  if (layout != GNCA_DMG_PLANE && layout != GNCA_DMG_PLANE_ALPHA) return GNCA_ERR_ARG;
  if (layout == GNCA_DMG_PLANE_ALPHA && C < 4) return GNCA_ERR_ARG;
  k_apply_plane<<<grid_for((size_t)B * C * H * W), 256, 0, (cudaStream_t)stream>>>(B, C, H * W, state_dev, plane_dev,
                                                                                 layout == GNCA_DMG_PLANE_ALPHA);
  GNCA_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
