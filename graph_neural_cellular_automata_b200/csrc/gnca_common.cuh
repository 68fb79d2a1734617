// Shared device helpers for the graph-NCA kernels (sm_100a).
// Semantics follow the reference step (SURVEY 0.1 / 0.2); citations are to /root/reference/src/modules.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <atomic>
#include "../../include/gnca.h"

#define GNCA_CHECK_CUDA(expr)                      \
  do {                                             \
    cudaError_t _e = (expr);                       \
    if (_e != cudaSuccess) return (int)_e;         \
  } while (0)

// every kernel launch in the library is followed by this macro: it also counts launches (gnca_launch_count)
#define GNCA_LAUNCH_CHECK()                        \
  do {                                             \
    ::gnca::g_launches.fetch_add(1, std::memory_order_relaxed); \
    cudaError_t _e = cudaGetLastError();           \
    if (_e != cudaSuccess) return (int)_e;         \
  } while (0)

namespace gnca {

extern std::atomic<unsigned long long> g_launches;   // defined in gnca_fwd.cu

// optional per-kernel timing with CUDA events on the launching stream (gnca_profile_enable / gnca_profile_read)
enum ProfId { PROF_UPDATE = 0, PROF_APPLY = 1, PROF_RESIDENT_FWD = 2, PROF_BWD_MLP = 3, PROF_BWD_NORM = 4,
              PROF_BWD_GATHER = 5, PROF_RESIDENT_BWD = 6, PROF_COUNT = 8 };
void prof_begin(int id, cudaStream_t st);
void prof_end(int id, cudaStream_t st);

// ------------------------------------------------------------------------------------------------
// Packed (kernel-side) weight buffer.  All offsets are multiples of 4 floats (float4 loads).
// ------------------------------------------------------------------------------------------------
struct Packed {
  int w1t;    // [3C][hid]   transposed update_net.0.weight  (forward MLP: broadcast LDS.128 over 4 hidden units)
  int b1;     // [hid]
  int w2t;    // [hid][C]    transposed update_net.2.weight
  int w1;     // [hid][3C]   original orientation (backward)
  int w2;     // [C][hid]
  int gamma;  // [C]
  int beta;   // [C]
  int wm;     // [C][C]      msg_proj weight  (out, in)
  int wmt;    // [C][C]      transposed       (in, out)
  int bm;     // [C]
  int wq, bq, wk, bk, scaling;  // [d][C],[d],[d][C],[d],[1]
  int w1c;    // [2][hid x 3C]  update_net.0.weight split into tf32 (hi, lo), canonical no-swizzle K-major UMMA layout
  int w2c;    // [2][C x hid]   update_net.2.weight, same (gnca_tc.cuh); filled when C % 8 == 0 and hid % 8 == 0
  int total;
};

__host__ __device__ inline int pad4(int n) { return (n + 3) & ~3; }

__host__ __device__ inline Packed make_packed(int C, int hid, int d, bool graph) {
  Packed p;
  int o = 0;
  p.w1t = o; o += 3 * C * hid;
  p.b1 = o; o += pad4(hid);
  p.w2t = o; o += hid * C;
  p.w1 = o; o += hid * 3 * C;
  p.w2 = o; o += C * hid;
  p.gamma = o; o += pad4(C);
  p.beta = o; o += pad4(C);
  if (graph) {
    p.wm = o; o += pad4(C * C);
    p.wmt = o; o += pad4(C * C);
    p.bm = o; o += pad4(C);
    p.wq = o; o += pad4(d * C);
    p.bq = o; o += pad4(d);
    p.wk = o; o += pad4(d * C);
    p.bk = o; o += pad4(d);
    p.scaling = o; o += 4;
  } else {
    p.wm = p.wmt = p.bm = p.wq = p.bq = p.wk = p.bk = p.scaling = -1;
  }
  p.w1c = o; o += 2 * hid * 3 * C;
  p.w2c = o; o += 2 * C * hid;
  p.total = o;
  return p;
}

inline gnca_layout make_layout(const gnca_model& m) {
  gnca_layout L;
  const bool graph = (m.flags & GNCA_F_GRAPH) != 0;
  int64_t o = 0;
  L.w1 = o; o += (int64_t)m.hidden * 3 * m.C;
  L.b1 = o; o += m.hidden;
  L.w2 = o; o += (int64_t)m.C * m.hidden;
  L.gamma = o; o += m.C;
  L.beta = o; o += m.C;
  if (graph) {
    L.wm = o; o += (int64_t)m.C * m.C;
    L.bm = o; o += m.C;
    L.wq = o; o += (int64_t)m.d_model * m.C;
    L.bq = o; o += m.d_model;
    L.wk = o; o += (int64_t)m.d_model * m.C;
    L.bk = o; o += m.d_model;
    L.scaling = o; o += 1;
  } else {
    L.wm = L.bm = L.wq = L.bq = L.wk = L.bk = L.scaling = -1;
  }
  L.total = o;
  L.packed_total = make_packed(m.C, m.hidden, m.d_model, graph).total;
  return L;
}

inline bool model_supported(const gnca_model& m) {
  if (!(m.C == 4 || m.C == 8 || m.C == 16 || m.C == 32)) return false;
  if (m.hidden < 4 || m.hidden > 256 || (m.hidden & 3)) return false;
  if ((m.flags & GNCA_F_GRAPH) && (m.d_model < 1 || m.d_model > 64)) return false;
  return true;
}

// ------------------------------------------------------------------------------------------------
// Per-launch description of one step (by value in kernel params).
// ------------------------------------------------------------------------------------------------
struct Offsets {
  int8_t dy[GNCA_MAX_K];
  int8_t dx[GNCA_MAX_K];
};

struct StepArgs {
  int B, H, W, t, k;
  uint32_t flags;
  float update_gain, alpha_thr, graph_alpha_thr, gn_eps;
  float fire_rate, message_gain;      // host scalars (used when the *_dev pointers are null)
  const float* fire_rate_dev;         // [T]
  const float* message_gain_dev;      // [T]
  const int8_t* offsets_dev;          // [T][k][2]
  const int32_t* steps;               // [B] or null
  const float* fire_u;                // [B][H][W] of THIS step, or null
  uint64_t philox_seed, philox_offset;
  const float* attn_w;                // [B][k] per-sample softmax weights (zero-pad mode) or null (uniform 1/k)
  const float* x_in;
  float* x_out;
  float* u;                           // [B][C][H][W]
  float* stats;                       // [B][2]  (mean, rstd)
  double* partials;                   // [B][nchunks][2]
  int nchunks, chunk;                 // k_update work split: cells per block and blocks per sample
  int npart;                          // GroupNorm partial slots per sample in `partials` (nchunks, or 3*nchunks: k_update_tc)
  const uint32_t* actbits;            // [B][ceil(HW/32)] active (alive & fire) bits of this step written by k_compact, or null
  const uint32_t* alivebits;          // same layout: sender-alive bits (3x3 alpha max > graph_alpha_thr) of x_in, or null
  Offsets off;                        // host-supplied offsets (single step)
};

__device__ __forceinline__ float step_fire_rate(const StepArgs& a) {
  return a.fire_rate_dev ? a.fire_rate_dev[a.t] : a.fire_rate;
}
__device__ __forceinline__ float step_message_gain(const StepArgs& a) {
  return a.message_gain_dev ? a.message_gain_dev[a.t] : a.message_gain;
}
__device__ __forceinline__ void step_offset(const StepArgs& a, int i, int& dy, int& dx) {
  if (a.offsets_dev) {
    const int8_t* o = a.offsets_dev + ((size_t)a.t * a.k + i) * 2;
    dy = o[0]; dx = o[1];
  } else {
    dy = a.off.dy[i]; dx = a.off.dx[i];
  }
}
__device__ __forceinline__ bool sample_active(const StepArgs& a, int b) {
  return a.steps == nullptr || a.steps[b] > a.t;
}

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (counter based) for in-kernel fire uniforms.  Own stream layout, NOT torch's.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0; key.y += W1;
  }
  return ctr;
}

// uniform in [0,1) for (step t, sample b, cell) -- one Philox block serves 4 consecutive cells
__device__ __forceinline__ float philox_uniform(uint64_t seed, uint64_t offset, int t, int b, int B, int cell, int HW) {
  uint64_t idx = ((uint64_t)t * B + b) * (uint64_t)HW + (uint64_t)cell;
  uint64_t blk = (idx >> 2) + offset;
  uint4 r = philox4x32_10(make_uint4((uint32_t)blk, (uint32_t)(blk >> 32), 0u, 0u),
                          make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  uint32_t v = (idx & 3) == 0 ? r.x : (idx & 3) == 1 ? r.y : (idx & 3) == 2 ? r.z : r.w;
  return (float)(v >> 8) * (1.0f / 16777216.0f);
}

// ------------------------------------------------------------------------------------------------
// alive: maxpool3x3(alpha) > thr with a -inf halo   (nca.py:55-62, ncagraph.py:85-92)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float alive_max(const float* __restrict__ alpha, int y, int x, int H, int W) {
  float m = -INFINITY;
#pragma unroll
  for (int i = -1; i <= 1; ++i) {
    int yy = y + i;
    if (yy < 0 || yy >= H) continue;
#pragma unroll
    for (int j = -1; j <= 1; ++j) {
      int xx = x + j;
      if (xx < 0 || xx >= W) continue;
      m = fmaxf(m, __ldg(alpha + yy * W + xx));
    }
  }
  return m;
}
__device__ __forceinline__ bool alive_at(const float* __restrict__ alpha, int y, int x, int H, int W, float thr) {
  return alive_max(alpha, y, x, H, W) > thr;
}

// pre-gate updated alpha x~_3 = x_3 + gain * tanh(gn(u_3)) (ncagraph.py:153-155) with EXPLICIT roundings: the streaming
// backward recomputes it for the post-alive mask (ncagraph.py:158) and must land on the forward's bits -- a contracted
// FMA on one side flips the mask of a cell within an ulp of the threshold (seen as a 2e-3 error of dL/dx0 of one sample
// in the 64-step gradient fixture).  idle3 = __fmul_rn(tanhf(bi3), gain).
__device__ __forceinline__ float updated_alpha(float alpha, bool act, float u3, float sc3, float bi3, float idle3, float gain) {
  return __fadd_rn(alpha, act ? __fmul_rn(tanhf(fmaf(u3, sc3, bi3)), gain) : idle3);
}

// fire decision of (b, cell) at this step: (u <= fire_rate), skipped entirely when fire_rate >= 1 (ncagraph.py:144)
__device__ __forceinline__ bool fires(const StepArgs& a, float fire_rate, int b, int cell) {
  if (fire_rate >= 1.0f) return true;
  const int HW = a.H * a.W;
  float u = a.fire_u ? __ldg(a.fire_u + (size_t)b * HW + cell)
                     : philox_uniform(a.philox_seed, a.philox_offset, a.t, b, a.B, cell, HW);
  return u <= fire_rate;
}

// ------------------------------------------------------------------------------------------------
// perception of one cell from a global NCHW sample (zero halo, cross-correlation)  perception.py:9-26
//   y[0..C) identity, y[C..2C) sobel_x = sum_i w_i (in[y+i,x-1] - in[y+i,x+1]), y[2C..3C) sobel_y
// ------------------------------------------------------------------------------------------------
template <int C>
__device__ __forceinline__ void perceive(const float* __restrict__ xs /* sample base [C][H][W] */, int y, int x,
                                         int H, int W, float (&out)[3 * C]) {
  const int HW = H * W;
  const bool up = y > 0, dn = y < H - 1, lf = x > 0, rt = x < W - 1;
  const int c0 = y * W + x;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const float* p = xs + c * HW + c0;
    float a00 = (up && lf) ? __ldg(p - W - 1) : 0.f, a01 = up ? __ldg(p - W) : 0.f, a02 = (up && rt) ? __ldg(p - W + 1) : 0.f;
    float a10 = lf ? __ldg(p - 1) : 0.f, a11 = __ldg(p), a12 = rt ? __ldg(p + 1) : 0.f;
    float a20 = (dn && lf) ? __ldg(p + W - 1) : 0.f, a21 = dn ? __ldg(p + W) : 0.f, a22 = (dn && rt) ? __ldg(p + W + 1) : 0.f;
    out[c] = a11;
    out[C + c] = (a00 - a02) + 2.f * (a10 - a12) + (a20 - a22);
    out[2 * C + c] = (a00 + 2.f * a01 + a02) - (a20 + 2.f * a21 + a22);
  }
}

// ------------------------------------------------------------------------------------------------
// update MLP forward for P cells per thread: dx = W2 relu(W1 y + b1)   (ncagraph.py:60-65,131)
// weights are read from shared memory with warp-uniform (broadcast) float4 loads.
// ------------------------------------------------------------------------------------------------
template <int C, int P, int JU = 4>
__device__ __forceinline__ void mlp_forward(const float (&y)[P][3 * C], float (&dx)[P][C], const float* __restrict__ sW1T,
                                            const float* __restrict__ sb1, const float* __restrict__ sW2T, int hid) {
  static_assert(JU % 4 == 0, "hidden units per pass: multiples of 4 (float4 weight rows)");
#pragma unroll
  for (int p = 0; p < P; ++p)
#pragma unroll
    for (int c = 0; c < C; ++c) dx[p][c] = 0.f;
#pragma unroll 1
  for (int j = 0; j < hid; j += JU) {        // hid % JU == 0 is checked by the launcher
    float h[P][JU];
#pragma unroll
    for (int q = 0; q < JU / 4; ++q) {
      const float4 bb = *reinterpret_cast<const float4*>(sb1 + j + 4 * q);
#pragma unroll
      for (int p = 0; p < P; ++p) { h[p][4 * q] = bb.x; h[p][4 * q + 1] = bb.y; h[p][4 * q + 2] = bb.z; h[p][4 * q + 3] = bb.w; }
    }
#pragma unroll
    for (int k = 0; k < 3 * C; ++k) {
#pragma unroll
      for (int q = 0; q < JU / 4; ++q) {
        const float4 w = *reinterpret_cast<const float4*>(sW1T + k * hid + j + 4 * q);
#pragma unroll
        for (int p = 0; p < P; ++p) {
          h[p][4 * q + 0] = fmaf(w.x, y[p][k], h[p][4 * q + 0]);
          h[p][4 * q + 1] = fmaf(w.y, y[p][k], h[p][4 * q + 1]);
          h[p][4 * q + 2] = fmaf(w.z, y[p][k], h[p][4 * q + 2]);
          h[p][4 * q + 3] = fmaf(w.w, y[p][k], h[p][4 * q + 3]);
        }
      }
    }
#pragma unroll
    for (int jj = 0; jj < JU; ++jj) {
#pragma unroll
      for (int p = 0; p < P; ++p) h[p][jj] = fmaxf(h[p][jj], 0.f);
#pragma unroll
      for (int c4 = 0; c4 < C / 4; ++c4) {
        const float4 w2 = *reinterpret_cast<const float4*>(sW2T + (j + jj) * C + c4 * 4);
#pragma unroll
        for (int p = 0; p < P; ++p) {
          dx[p][c4 * 4 + 0] = fmaf(w2.x, h[p][jj], dx[p][c4 * 4 + 0]);
          dx[p][c4 * 4 + 1] = fmaf(w2.y, h[p][jj], dx[p][c4 * 4 + 1]);
          dx[p][c4 * 4 + 2] = fmaf(w2.z, h[p][jj], dx[p][c4 * 4 + 2]);
          dx[p][c4 * 4 + 3] = fmaf(w2.w, h[p][jj], dx[p][c4 * 4 + 3]);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// graph message of one receiver cell, using linearity of the 1x1 msg_proj:
//   agg = sum_i w_i * shift_i(M * A_send) = Wm * xs + bm * as,
//   xs = sum_i w_i * A(q_i) * x(q_i),  as = sum_i w_i * A(q_i),  q_i = sender of offset i
// (graph_augmentation.py:109-111,116-133,156-158; shift(M)*shift(A) == shift(M*A)).
// torus: q = ((y-dy) mod H, (x-dx) mod W)  (:94-97);  zero-pad: q = (y-dy, x) if in range (:85-92, dx is a no-op)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool sender_of(int y, int x, int dy, int dx, int H, int W, bool torus, int& qy, int& qx) {
  if (torus) {
    qy = y - dy; qx = x - dx;
    qy = qy < 0 ? qy + H : (qy >= H ? qy - H : qy);
    qx = qx < 0 ? qx + W : (qx >= W ? qx - W : qx);
    // offsets larger than the grid (tiny grids): full modulo
    if (qy < 0 || qy >= H) qy = ((qy % H) + H) % H;
    if (qx < 0 || qx >= W) qx = ((qx % W) + W) % W;
    return true;
  }
  qy = y - dy; qx = x;
  return qy >= 0 && qy < H;
}

template <int C>
__device__ __forceinline__ void gather_senders(const StepArgs& a, const float* __restrict__ xs_base /* sample [C][H][W] */,
                                               int b, int y, int x, float (&xs)[C], float& as) {
  const int H = a.H, W = a.W, HW = H * W;
  const bool torus = (a.flags & GNCA_F_TORUS) != 0;
  const bool a2a = (a.flags & GNCA_F_ALIVE_TO_ALIVE) != 0;
#pragma unroll
  for (int c = 0; c < C; ++c) xs[c] = 0.f;
  as = 0.f;
  const float wuni = a.k > 0 ? 1.0f / (float)a.k : 0.f;
  for (int i = 0; i < a.k; ++i) {
    int dy, dx, qy, qx;
    step_offset(a, i, dy, dx);
    if (!sender_of(y, x, dy, dx, H, W, torus, qy, qx)) continue;
    if (a2a && !alive_at(xs_base + 3 * HW, qy, qx, H, W, a.graph_alpha_thr)) continue;
    const float w = a.attn_w ? __ldg(a.attn_w + (size_t)b * a.k + i) : wuni;
    const float* q = xs_base + qy * W + qx;
#pragma unroll
    for (int c = 0; c < C; ++c) xs[c] = fmaf(w, __ldg(q + c * HW), xs[c]);
    as += w;
  }
}

// agg[c] = bm[c]*as + sum_c' WmT[c'][c] * xs[c']   (all C channels)
template <int C>
__device__ __forceinline__ void msg_project(const float (&xs)[C], float as, const float* __restrict__ sWmT,
                                            const float* __restrict__ sbm, float (&agg)[C]) {
#pragma unroll
  for (int c = 0; c < C; ++c) agg[c] = sbm[c] * as;
#pragma unroll
  for (int ci = 0; ci < C; ++ci) {
#pragma unroll
    for (int c4 = 0; c4 < C / 4; ++c4) {
      const float4 w = *reinterpret_cast<const float4*>(sWmT + ci * C + c4 * 4);
      agg[c4 * 4 + 0] = fmaf(w.x, xs[ci], agg[c4 * 4 + 0]);
      agg[c4 * 4 + 1] = fmaf(w.y, xs[ci], agg[c4 * 4 + 1]);
      agg[c4 * 4 + 2] = fmaf(w.z, xs[ci], agg[c4 * 4 + 2]);
      agg[c4 * 4 + 3] = fmaf(w.w, xs[ci], agg[c4 * 4 + 3]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// damage mask of a rollout (gnca_schedule.damage / damage_layout): dense [B][C][HW], or a per-cell plane [B][HW] applied
// to every channel or to the alpha channel only
// ------------------------------------------------------------------------------------------------
struct DamageView {
  const float* p;      // null: no damage
  int layout;
  __device__ __forceinline__ float at(int b, int ch, int cell, int C, int HW) const {
    if (layout == GNCA_DMG_DENSE) return p[((size_t)b * C + ch) * HW + cell];
    if (layout == GNCA_DMG_PLANE_ALPHA && ch != 3) return 1.f;
    return p[(size_t)b * HW + cell];
  }
};

// ------------------------------------------------------------------------------------------------
// reductions
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// copy n floats (n % 4 == 0, 16B aligned) global -> shared with the whole block
__device__ __forceinline__ void block_copy(float* __restrict__ dst, const float* __restrict__ src, int n) {
  const float4* s = reinterpret_cast<const float4*>(src);
  float4* d = reinterpret_cast<float4*>(dst);
  for (int i = threadIdx.x; i < (n >> 2); i += blockDim.x) d[i] = __ldg(s + i);
}

}  // namespace gnca
