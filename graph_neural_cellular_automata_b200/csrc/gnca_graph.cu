// GraphAugmentation.forward as a stand-alone operator (graph_augmentation.py:104-169) with its backward, and the
// backward of the zero-padded-shift attention weights (softmax over pooled Q.K logits), shared with the step.
//
// The k shifted copies of K / M / A_send the reference materialises are never built: the message uses the
// linearity of the 1x1 msg_proj (agg = Wm * sum_i w_i A x(q_i) + bm * sum_i w_i A(q_i)) and reads the senders in
// place; pooled logits come from per-row sums of x (Q_pooled = Wq mean(x) + bq, mean(shift_dy K) is a row-range sum).
#include "gnca_common.cuh"
#include "gnca_internal.h"

namespace gnca {

constexpr int kGCells = 256;   // cells per block of the stand-alone graph kernels

// ------------------------------------------------------------------------------------------------
// forward: m[b,c,p] for every cell and channel
// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(kGCells) k_graph_fwd(StepArgs a, Packed P, const float* __restrict__ packed,
                                                        float* __restrict__ msg) {
  __shared__ __align__(16) float sWmT[C * C];
  __shared__ __align__(16) float sbm[C];
  for (int i = threadIdx.x; i < C * C; i += blockDim.x) sWmT[i] = packed[P.wmt + i];
  if (threadIdx.x < C) sbm[threadIdx.x] = packed[P.bm + threadIdx.x];
  __syncthreads();
  const int b = blockIdx.y, H = a.H, W = a.W, HW = H * W;
  const int cell = blockIdx.x * blockDim.x + threadIdx.x;
  if (cell >= HW) return;
  const int y = cell / W, x = cell - y * W;
  const float* xs_base = a.x_in + (size_t)b * C * HW;
  float xs[C], agg[C], as;
  gather_senders<C>(a, xs_base, b, y, x, xs, as);
  msg_project<C>(xs, as, sWmT, sbm, agg);
#pragma unroll
  for (int c = 0; c < C; ++c) msg[((size_t)b * C + c) * HW + cell] = (a.k > 0) ? agg[c] : 0.f;
}

// ------------------------------------------------------------------------------------------------
// backward, cell phase: g_xs = Wm^T gm -> global; dWm, dbm partials per block; dL/dw_i partials (zero-pad)
// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(kGCells) k_graph_bwd_cells(StepArgs a, Packed P, const float* __restrict__ packed,
                                                              const float* __restrict__ gmsg, float* __restrict__ gxs,
                                                              float* __restrict__ wpart /*[B*nblk][C*C+C]*/,
                                                              float* __restrict__ gw_part /*[B][nblk][MAX_K] or null*/) {
  constexpr int NP = kGCells + 4;
  extern __shared__ __align__(16) float sm[];
  float* GAt = sm;                 // [C][NP]  gm of the block's cells
  float* XSt = GAt + C * NP;       // [C][NP]  gathered sender state
  float* GXt = XSt + C * NP;       // [C][NP]  Wm^T gm
  float* AS = GXt + C * NP;        // [NP]
  float* GB = AS + NP;             // [NP]     bm . gm
  float* sWm = GB + NP;            // [C][C]
  float* sbm = sWm + C * C;        // [C]
  for (int i = threadIdx.x; i < C * C; i += blockDim.x) sWm[i] = packed[P.wm + i];
  if (threadIdx.x < C) sbm[threadIdx.x] = packed[P.bm + threadIdx.x];
  const int b = blockIdx.y, H = a.H, W = a.W, HW = H * W;
  const int cell = blockIdx.x * blockDim.x + threadIdx.x;
  const int cl = threadIdx.x;
  const bool valid = cell < HW;
  const int y = valid ? cell / W : 0, x = valid ? cell - y * W : 0;
  const float* xs_base = a.x_in + (size_t)b * C * HW;
  __syncthreads();
  {
    float xs[C], as = 0.f, gm[C];
#pragma unroll
    for (int c = 0; c < C; ++c) { xs[c] = 0.f; gm[c] = 0.f; }
    if (valid) {
      gather_senders<C>(a, xs_base, b, y, x, xs, as);
#pragma unroll
      for (int c = 0; c < C; ++c) gm[c] = gmsg[((size_t)b * C + c) * HW + cell];
    }
    float gb = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) { GAt[c * NP + cl] = gm[c]; XSt[c * NP + cl] = xs[c]; gb = fmaf(sbm[c], gm[c], gb); }
    AS[cl] = as; GB[cl] = gb;
#pragma unroll
    for (int ci = 0; ci < C; ++ci) {
      float v = 0.f;
#pragma unroll
      for (int co = 0; co < C; ++co) v = fmaf(sWm[co * C + ci], gm[co], v);
      GXt[ci * NP + cl] = v;
      if (valid) gxs[((size_t)b * C + ci) * HW + cell] = v;
    }
  }
  __syncthreads();
  const int nb = min(kGCells, HW - blockIdx.x * kGCells);
  float* wp = wpart + ((size_t)b * gridDim.x + blockIdx.x) * (C * C + C);
  for (int idx = threadIdx.x; idx < C * C + C; idx += blockDim.x) {
    float acc = 0.f;
    if (idx < C * C) {
      const int co = idx / C, ci = idx % C;
      for (int i = 0; i < nb; ++i) acc = fmaf(GAt[co * NP + i], XSt[ci * NP + i], acc);
    } else {
      const int c = idx - C * C;
      for (int i = 0; i < nb; ++i) acc = fmaf(GAt[c * NP + i], AS[i], acc);
    }
    wp[idx] = acc;
  }
  if (gw_part) {   // dL/dw_i = sum_p [ g_xs(p) . A x(q_i(p)) + (bm . gm(p)) A(q_i(p)) ]
    const bool torus = (a.flags & GNCA_F_TORUS) != 0, a2a = (a.flags & GNCA_F_ALIVE_TO_ALIVE) != 0;
    for (int oi = threadIdx.x; oi < a.k; oi += blockDim.x) {
      int dy, dx;
      step_offset(a, oi, dy, dx);
      float acc = 0.f;
      for (int i = 0; i < nb; ++i) {
        const int pc = blockIdx.x * kGCells + i, py = pc / W, px = pc - py * W;
        int qy, qx;
        if (!sender_of(py, px, dy, dx, H, W, torus, qy, qx)) continue;
        if (a2a && !alive_at(xs_base + 3 * HW, qy, qx, H, W, a.graph_alpha_thr)) continue;
        float v = GB[i];
        for (int c = 0; c < C; ++c) v = fmaf(GXt[c * NP + i], __ldg(xs_base + (size_t)c * HW + qy * W + qx), v);
        acc += v;
      }
      gw_part[((size_t)b * gridDim.x + blockIdx.x) * GNCA_MAX_K + oi] = acc;
    }
  }
}

// backward, gather phase: gx(q) = A(q) * sum_i w_i g_xs(receiver of q at offset i) + grow[b][c][row]
template <int C>
__global__ void __launch_bounds__(256) k_graph_bwd_gather(StepArgs a, const float* __restrict__ gxs,
                                                           const float* __restrict__ grow, float* __restrict__ gx) {
  const int b = blockIdx.y, H = a.H, W = a.W, HW = H * W;
  const int cell = blockIdx.x * blockDim.x + threadIdx.x;
  if (cell >= HW) return;
  const int y = cell / W, x = cell - y * W;
  const bool torus = (a.flags & GNCA_F_TORUS) != 0;
  const float* xs_base = a.x_in + (size_t)b * C * HW;
  float g[C];
#pragma unroll
  for (int c = 0; c < C; ++c) g[c] = 0.f;
  if (a.k > 0 && (!(a.flags & GNCA_F_ALIVE_TO_ALIVE) || alive_at(xs_base + 3 * HW, y, x, H, W, a.graph_alpha_thr))) {
    const float wuni = 1.0f / (float)a.k;
    for (int i = 0; i < a.k; ++i) {
      int dy, dx, py, px;
      step_offset(a, i, dy, dx);
      if (torus) {
        py = ((y + dy) % H + H) % H; px = ((x + dx) % W + W) % W;
      } else {
        py = y + dy; px = x;
        if (py < 0 || py >= H) continue;
      }
      const float w = a.attn_w ? a.attn_w[(size_t)b * a.k + i] : wuni;
      const float* gp = gxs + (size_t)b * C * HW + py * W + px;
#pragma unroll
      for (int c = 0; c < C; ++c) g[c] = fmaf(w, gp[(size_t)c * HW], g[c]);
    }
  }
#pragma unroll
  for (int c = 0; c < C; ++c) {
    float v = g[c];
    if (grow) v += grow[((size_t)b * C + c) * H + y];
    gx[((size_t)b * C + c) * HW + cell] = v;
  }
}

// ------------------------------------------------------------------------------------------------
// attention backward (zero-padded shift), one block per sample
// ------------------------------------------------------------------------------------------------
__global__ void k_attn_bwd(StepArgs a, Packed P, int C, int d, const float* __restrict__ packed,
                           const float* __restrict__ rowsum, const float* __restrict__ gw_part, int nparts,
                           float* __restrict__ grow, float* __restrict__ pw, int stage, int accumulate) {
  extern __shared__ float sm[];
  const int b = blockIdx.x, H = a.H, W = a.W, k = a.k;
  float* xbar = sm;              // [C]
  float* qp = xbar + C;          // [d]
  float* gqp = qp + d;           // [d]
  float* wkq = gqp + d;          // [C]   sum_j Wk[j][c] qp[j]
  float* gxb = wkq + C;          // [C]   Wq^T gqp
  float* S = gxb + C;            // [k][C] row-range sums
  float* KP = S + k * C;         // [k][d]
  float* lg = KP + k * d;        // [k] logits -> then a_i
  float* wv = lg + k;            // [k] softmax weights
  float* gL = wv + k;            // [k]
  int* rlo = reinterpret_cast<int*>(gL + k);   // [k]
  int* rhi = rlo + k;                           // [k]
  float* swq = reinterpret_cast<float*>(rhi + k);   // [d][C] weights / biases staged like the row sums (see k_attn_weights)
  float* swk = swq + d * C;
  float* sbq = swk + d * C;
  float* sbk = sbq + d;
  float* rss = sbk + d;                             // [C][H] when staged
  __shared__ float s_gtau;
  const float* rs = rowsum + (size_t)b * C * H;
  const float invHW = 1.0f / (float)(H * W);
  const bool torus = (a.flags & GNCA_F_TORUS) != 0;
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int i = tid; i < d * C; i += nt) { swq[i] = packed[P.wq + i]; swk[i] = packed[P.wk + i]; }
  for (int i = tid; i < d; i += nt) { sbq[i] = packed[P.bq + i]; sbk[i] = packed[P.bk + i]; }
  if (stage) {
    for (int i = tid; i < C * H; i += nt) rss[i] = rs[i];
    rs = rss;
  }
  for (int i = tid; i < k; i += nt) {
    int dy, dx;
    step_offset(a, i, dy, dx);
    int lo = 0, hi = H;
    if (!torus) { lo = max(0, -dy); hi = min(H, H - dy); }
    rlo[i] = lo; rhi[i] = max(lo, hi);
    float gw = 0.f;               // dL/dw_i: the partials of the cell kernels, in order (one thread per offset)
    for (int pidx = 0; pidx < nparts; ++pidx) gw += gw_part[((size_t)b * nparts + pidx) * GNCA_MAX_K + i];
    gL[i] = gw;
  }
  __syncthreads();
  for (int c = tid; c < C; c += nt) {
    float s = 0.f;
    for (int y = 0; y < H; ++y) s += rs[c * H + y];
    xbar[c] = s * invHW;
  }
  __syncthreads();
  for (int j = tid; j < d; j += nt) {
    float s = 0.f;
    for (int c = 0; c < C; ++c) s = fmaf(swq[j * C + c], xbar[c], s);
    qp[j] = s + sbq[j];
  }
  for (int idx = tid; idx < k * C; idx += nt) {
    const int i = idx / C, c = idx % C;
    float s = 0.f;
    for (int y = rlo[i]; y < rhi[i]; ++y) s += rs[c * H + y];
    S[idx] = s;
  }
  __syncthreads();
  for (int idx = tid; idx < k * d; idx += nt) {
    const int i = idx / d, j = idx % d;
    float s = 0.f;
    for (int c = 0; c < C; ++c) s = fmaf(swk[j * C + c], S[i * C + c], s);
    KP[idx] = (s + (float)(rhi[i] - rlo[i]) * (float)W * sbk[j]) * invHW;
  }
  for (int c = tid; c < C; c += nt) {
    float s = 0.f;
    for (int j = 0; j < d; ++j) s = fmaf(swk[j * C + c], qp[j], s);
    wkq[c] = s;
  }
  __syncthreads();
  for (int i = tid; i < k; i += nt) {
    float s = 0.f;
    for (int j = 0; j < d; ++j) s = fmaf(qp[j], KP[i * d + j], s);
    lg[i] = s;
  }
  __syncthreads();
  if (tid == 0) {
    float mx = -INFINITY;
    for (int i = 0; i < k; ++i) mx = fmaxf(mx, lg[i]);
    const float sc = packed[P.scaling];
    const float tau = fabsf(sc) + 1e-6f;
    float se = 0.f;
    for (int i = 0; i < k; ++i) { lg[i] = (lg[i] - mx) / tau; wv[i] = expf(lg[i]); se += wv[i]; }
    float dot = 0.f;
    for (int i = 0; i < k; ++i) {
      wv[i] /= se;
      dot = fmaf(wv[i], gL[i], dot);          // gL holds dL/dw_i for now
    }
    float gtau = 0.f;
    for (int i = 0; i < k; ++i) {
      const float ga = wv[i] * (gL[i] - dot);
      gtau -= ga * lg[i] / tau;
      gL[i] = ga / tau;           // dL/dlogit_i
    }
    s_gtau = gtau * (sc >= 0.f ? 1.f : -1.f);
  }
  __syncthreads();
  for (int j = tid; j < d; j += nt) {
    float s = 0.f;
    for (int i = 0; i < k; ++i) s = fmaf(gL[i], KP[i * d + j], s);
    gqp[j] = s;
  }
  __syncthreads();
  for (int c = tid; c < C; c += nt) {
    float s = 0.f;
    for (int j = 0; j < d; ++j) s = fmaf(swq[j * C + c], gqp[j], s);
    gxb[c] = s;
  }
  // per-sample parameter gradients: [wq d*C][bq d][wk d*C][bk d][scaling]; `accumulate`: added to the slot (a BPTT sums the
  // steps here and reduces over the samples once at the end) instead of overwriting it
  float* pwb = pw + (size_t)b * (2 * d * C + 2 * d + 1);
  auto put = [&](int i, float v) { pwb[i] = accumulate ? pwb[i] + v : v; };
  for (int idx = tid; idx < d * C; idx += nt) {
    const int j = idx / C, c = idx % C;
    put(idx, gqp[j] * xbar[c]);
    float s = 0.f;
    for (int i = 0; i < k; ++i) s = fmaf(gL[i], S[i * C + c], s);
    put(d * C + d + idx, qp[j] * s * invHW);
  }
  for (int j = tid; j < d; j += nt) {
    put(d * C + j, gqp[j]);
    float s = 0.f;
    for (int i = 0; i < k; ++i) s += gL[i] * (float)(rhi[i] - rlo[i]);
    put(2 * d * C + d + j, qp[j] * s * (float)W * invHW);
  }
  if (tid == 0) put(2 * d * C + 2 * d, s_gtau);
  __syncthreads();
  // additive row term of dL/dx: (Wq^T gqp)[c]/HW + wkq[c]/HW * sum_{i: y in rows_i} gL_i
  for (int idx = tid; idx < C * H; idx += nt) {
    const int c = idx / H, y = idx % H;
    float s = 0.f;
    for (int i = 0; i < k; ++i) if (y >= rlo[i] && y < rhi[i]) s += gL[i];
    grow[((size_t)b * C + c) * H + y] = (gxb[c] + wkq[c] * s) * invHW;
  }
}

// MS: blockIdx.y = model of a stack: B is its sample count, its rows of pw and its gparams row
template <bool MS>
__global__ void k_attn_param_reduce(int B, int C, int d, gnca_layout L, const float* __restrict__ pw,
                                    float* __restrict__ gparams) {
  const int n = 2 * d * C + 2 * d + 1;
  if constexpr (MS) {
    pw += (size_t)blockIdx.y * B * n;
    gparams += (size_t)blockIdx.y * L.total;
  }
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int b0 = 0; b0 < B; b0 += 8) {          // 8 loads in flight, added in sample order
      float v[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) v[q] = b0 + q < B ? pw[(size_t)(b0 + q) * n + idx] : 0.f;
#pragma unroll
      for (int q = 0; q < 8; ++q) if (b0 + q < B) s += v[q];
    }
    int64_t dst;
    if (idx < d * C) dst = L.wq + idx;
    else if (idx < d * C + d) dst = L.bq + (idx - d * C);
    else if (idx < 2 * d * C + d) dst = L.wk + (idx - d * C - d);
    else if (idx < 2 * d * C + 2 * d) dst = L.bk + (idx - 2 * d * C - d);
    else dst = L.scaling;
    gparams[dst] += s;
  }
}

__global__ void k_graph_wpart_reduce(int nparts, int C, gnca_layout L, const float* __restrict__ wpart,
                                     float* __restrict__ gparams) {
  const int n = C * C + C;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int p = 0; p < nparts; ++p) s += wpart[(size_t)p * n + idx];
    gparams[(idx < C * C) ? L.wm + idx : L.bm + (idx - C * C)] += s;
  }
}

// ------------------------------------------------------------------------------------------------
static inline size_t al256(size_t v) { return (v + 255) / 256 * 256; }

AttnBwdScratch carve_attn_bwd(void* base, const gnca_model& m, int B, int H, int nparts) {
  AttnBwdScratch s;
  char* p = reinterpret_cast<char*>(base);
  size_t o = 0;
  s.gw_part = reinterpret_cast<float*>(p + o); o = al256(o + (size_t)B * nparts * GNCA_MAX_K * 4);
  s.grow = reinterpret_cast<float*>(p + o); o = al256(o + (size_t)B * m.C * H * 4);
  s.pw = reinterpret_cast<float*>(p + o); o = al256(o + (size_t)B * (2 * m.d_model * m.C + 2 * m.d_model + 1) * 4);
  return s;
}

size_t attn_bwd_scratch_bytes(const gnca_model& m, int B, int H, int nparts) {
  return al256((size_t)B * nparts * GNCA_MAX_K * 4) + al256((size_t)B * m.C * H * 4) +
         al256((size_t)B * (2 * m.d_model * m.C + 2 * m.d_model + 1) * 4);
}

// defer_reduce: the per-sample parameter gradients are ACCUMULATED in sc.pw (zeroed by the caller before the first step)
// and run_attn_param_reduce adds them to gparams once, after the last step of a BPTT
int run_attn_bwd(const gnca_model& m, const Packed& P, const float* packed, const StepArgs& a, const float* rowsum,
                 const AttnBwdScratch& sc, int nparts, float* gparams, cudaStream_t st, bool defer_reduce) {
  const int C = m.C, d = m.d_model, k = a.k;
  const int stage = (size_t)C * a.H * 4 <= 32 * 1024;
  const size_t smem = (size_t)(4 * C + 2 * d + k * C + k * d + 3 * k) * 4 + 2 * k * 4 + (size_t)2 * d * (C + 1) * 4 + (stage ? (size_t)C * a.H * 4 : 0) + 64;
  if (smem > 48 * 1024)
    GNCA_CHECK_CUDA(cudaFuncSetAttribute(k_attn_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_attn_bwd<<<a.B, 128, smem, st>>>(a, P, C, d, packed, rowsum, sc.gw_part, nparts, sc.grow, sc.pw, stage, defer_reduce ? 1 : 0);
  GNCA_LAUNCH_CHECK();
  if (!defer_reduce) return run_attn_param_reduce(m, a.B, sc, gparams, st);
  return 0;
}

int run_attn_param_reduce(const gnca_model& m, int B, const AttnBwdScratch& sc, float* gparams, cudaStream_t st,
                          int n_models) {
  const auto kern = n_models > 1 ? k_attn_param_reduce<true> : k_attn_param_reduce<false>;
  kern<<<dim3(4, n_models), 256, 0, st>>>(B / n_models, m.C, m.d_model, make_layout(m), sc.pw, gparams);
  GNCA_LAUNCH_CHECK();
  return 0;
}

size_t graph_workspace_bytes(const gnca_model& m, int B, int H, int W) {
  const int nblk = (H * W + kGCells - 1) / kGCells;
  return al256((size_t)B * m.C * H * W * 4) + al256((size_t)B * nblk * (m.C * m.C + m.C) * 4) + attn_bwd_scratch_bytes(m, B, H, nblk);
}

template <int C>
static int launch_graph_fwd(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a, const FwdWorkspace& ws,
                            float* msg, float* attn, cudaStream_t st) {
  if (!(m.flags & GNCA_F_TORUS) && a.k > 0) {
    int rc = run_attn_prepass(m, P, packed, a, ws, st);
    if (rc) return rc;
  }
  dim3 g((a.H * a.W + kGCells - 1) / kGCells, a.B);
  k_graph_fwd<C><<<g, kGCells, 0, st>>>(a, P, packed, msg);
  GNCA_LAUNCH_CHECK();
  if (attn) return run_attn_map(m, P, packed, a, ws, attn, st);
  return 0;
}

template <int C>
static int launch_graph_bwd(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a, const FwdWorkspace& ws,
                            char* scratch, const float* gmsg, float* gx, float* gparams, cudaStream_t st) {
  const bool zp = !(m.flags & GNCA_F_TORUS) && a.k > 0;
  if (zp) {
    int rc = run_attn_prepass(m, P, packed, a, ws, st);
    if (rc) return rc;
  }
  const int HW = a.H * a.W, nblk = (HW + kGCells - 1) / kGCells;
  float* gxs = reinterpret_cast<float*>(scratch);
  size_t o = al256((size_t)a.B * C * HW * 4);
  float* wpart = reinterpret_cast<float*>(scratch + o);
  o += al256((size_t)a.B * nblk * (C * C + C) * 4);
  AttnBwdScratch sc = carve_attn_bwd(scratch + o, m, a.B, a.H, nblk);
  const size_t smem = (size_t)((3 * C + 2) * (kGCells + 4) + C * C + C) * 4;
  GNCA_CHECK_CUDA(cudaFuncSetAttribute(k_graph_bwd_cells<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 g(nblk, a.B);
  k_graph_bwd_cells<C><<<g, kGCells, smem, st>>>(a, P, packed, gmsg, gxs, wpart, zp ? sc.gw_part : nullptr);
  GNCA_LAUNCH_CHECK();
  k_graph_wpart_reduce<<<2, 256, 0, st>>>(a.B * nblk, C, make_layout(m), wpart, gparams);
  GNCA_LAUNCH_CHECK();
  if (zp) {
    int rc = run_attn_bwd(m, P, packed, a, ws.rowsum, sc, nblk, gparams, st, false);
    if (rc) return rc;
  }
  dim3 g2((HW + 255) / 256, a.B);
  k_graph_bwd_gather<C><<<g2, 256, 0, st>>>(a, gxs, zp ? sc.grow : nullptr, gx);
  GNCA_LAUNCH_CHECK();
  return 0;
}

}  // namespace gnca

using namespace gnca;

extern "C" {

int gnca_graph_fwd(const gnca_model* m, const float* packed_dev, int B, int H, int W, const float* x_dev,
                   const int32_t* offsets_host, int k, float* msg_dev, float* attn_dev, void* workspace_dev,
                   size_t workspace_bytes, void* stream) {
  if (!m || !packed_dev || !x_dev || !msg_dev || !workspace_dev || B <= 0 || H <= 0 || W <= 0) return GNCA_ERR_ARG;
  if (!model_supported(*m) || !(m->flags & GNCA_F_GRAPH)) return GNCA_ERR_UNSUPPORTED;
  FwdWorkspace ws = carve_fwd_workspace(workspace_dev, *m, B, H, W);
  if (ws.bytes > workspace_bytes) return GNCA_ERR_WORKSPACE;
  StepArgs a;
  fill_step_args(a, *m, B, H, W);
  int rc = set_host_offsets(a, offsets_host, k);
  if (rc) return rc;
  a.x_in = x_dev;
  const Packed P = make_packed(m->C, m->hidden, m->d_model, true);
  cudaStream_t st = (cudaStream_t)stream;
  switch (m->C) {
    case 4: return launch_graph_fwd<4>(*m, P, packed_dev, a, ws, msg_dev, attn_dev, st);
    case 8: return launch_graph_fwd<8>(*m, P, packed_dev, a, ws, msg_dev, attn_dev, st);
    case 16: return launch_graph_fwd<16>(*m, P, packed_dev, a, ws, msg_dev, attn_dev, st);
    case 32: return launch_graph_fwd<32>(*m, P, packed_dev, a, ws, msg_dev, attn_dev, st);
  }
  return GNCA_ERR_UNSUPPORTED;
}

int gnca_graph_bwd(const gnca_model* m, const float* packed_dev, int B, int H, int W, const float* x_dev,
                   const int32_t* offsets_host, int k, const float* gmsg_dev, float* gx_dev, float* gparams_dev,
                   void* workspace_dev, size_t workspace_bytes, void* stream) {
  if (!m || !packed_dev || !x_dev || !gmsg_dev || !gx_dev || !gparams_dev || !workspace_dev) return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0) return GNCA_ERR_ARG;
  if (!model_supported(*m) || !(m->flags & GNCA_F_GRAPH)) return GNCA_ERR_UNSUPPORTED;
  FwdWorkspace ws = carve_fwd_workspace(workspace_dev, *m, B, H, W);
  if (ws.bytes + graph_workspace_bytes(*m, B, H, W) > workspace_bytes) return GNCA_ERR_WORKSPACE;
  StepArgs a;
  fill_step_args(a, *m, B, H, W);
  int rc = set_host_offsets(a, offsets_host, k);
  if (rc) return rc;
  a.x_in = x_dev;
  const Packed P = make_packed(m->C, m->hidden, m->d_model, true);
  cudaStream_t st = (cudaStream_t)stream;
  char* scratch = reinterpret_cast<char*>(workspace_dev) + ws.bytes;
  switch (m->C) {
    case 4: return launch_graph_bwd<4>(*m, P, packed_dev, a, ws, scratch, gmsg_dev, gx_dev, gparams_dev, st);
    case 8: return launch_graph_bwd<8>(*m, P, packed_dev, a, ws, scratch, gmsg_dev, gx_dev, gparams_dev, st);
    case 16: return launch_graph_bwd<16>(*m, P, packed_dev, a, ws, scratch, gmsg_dev, gx_dev, gparams_dev, st);
    case 32: return launch_graph_bwd<32>(*m, P, packed_dev, a, ws, scratch, gmsg_dev, gx_dev, gparams_dev, st);
  }
  return GNCA_ERR_UNSUPPORTED;
}

}  // extern "C"
