// Cluster-resident forward rollout: ONE launch runs all T steps of a batch, state in shared memory.
//
// A sample is owned by a thread-block cluster of NC CTAs (NC in {8,4,2,1}: largest that keeps the batch
// co-resident and divides H into bands of at least HALO rows).  CTA r holds, in shared memory and for the whole
// rollout, the band of rows [r*own, (r+1)*own) of every channel plus HALO = radius+1 rows of each neighbouring
// band (torus-wrapped, so the mid-range message reads its senders in place).  HBM is touched at the rollout
// boundaries (x_0 in, x_T out) and, only when BPTT history is requested, by one store of x_t per step.
//
// Per step (reference semantics: ncagraph.py:106-168):
//   P1  alive & fire test on own cells, deterministic compaction of the active cells
//   P2  perception + MLP (+ graph message) on active cells in staged batches (FFMA register tiles, weights in smem)
//   --  per-sample GroupNorm statistics: block partial -> DSMEM all-gather           [cluster barrier 1]
//   P3  bounded update in place; idle update of the halo copies; pre-gate alpha rows pushed to the neighbours
//                                                                                    [cluster barrier 2]
//   P4  post-alive gate; gated alpha rows and the active cells' channels pushed into the neighbours' halos
//                                                                                    [cluster barrier 3]
#include <cooperative_groups.h>
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include "gnca_common.cuh"
#include "gnca_internal.h"
#include "gnca_metrics.cuh"
#include "gnca_ptx.cuh"

namespace cg = cooperative_groups;

namespace gnca {

constexpr int kRThreads = 512;
constexpr int kRWarps = kRThreads / 32;

struct ResidentArgs {
  StepArgs s;                 // model scalars + schedule pointers (t / fire_u are set per step in-kernel)
  int T, NC, own_rows, halo, MB, plane_stride;
  double inv_n;               // 1 / (C*H*W)
  const float* fire_u_base;   // [T][B][H][W] or null
  const float* x0;
  float* xT;
  float* hist;                // [T/hist_every+1][B][C][HW] or null: x_t of the steps t % hist_every == 0, in slot t/hist_every
  int hist_every;
  float* stats_hist;          // [T][B][2] or null
  float* u_hist;              // [T][B][C][HW] or null: masked pre-norm update of the active cells (for the backward)
  DamageView damage;          // schedule.damage (dense or plane) or null
  int damage_step;
  unsigned long long* dbg;    // optional phase-cycle counters (GNCA_PHASE_TIMING=<cta index>), else null
  int dbg_cta;
};

// phase counters accumulate in shared memory (a global RMW per mark would sit on the critical path)
#ifdef GNCA_PHASE_COUNTERS          /* build with -DGNCA_PHASE_COUNTERS for the per-phase cycle counters */
#define GNCA_PHASE_MARK(idx)                                                        \
  do {                                                                              \
    if (R.dbg && tid == 0) {                                                        \
      const long long _n = clock64();                                               \
      s_dbg[idx] += (unsigned long long)(_n - t_prev);                              \
      t_prev = _n;                                                                  \
    }                                                                               \
  } while (0)
#else
#define GNCA_PHASE_MARK(idx) do { } while (0)
#endif

// Out-of-line helpers: the per-step code of the resident kernel has to stay small enough for the instruction
// caches (every phase is executed once per step by few warps, so cold-code fetch latency is on the critical path).
__device__ __noinline__ float tanh_ool(float v) { return tanhf(v); }

__device__ __noinline__ double warp_sum_ool(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// alive(maxpool3x3 > thr) around local row lr / column x of an alpha-like plane with row stride W; rows outside
// the image (by GLOBAL row gy of the centre) count as -inf exactly like F.max_pool2d (nca.py:61).
__device__ __noinline__ bool alive_local_ool(const float* plane, int lr, int x, int gy, int H, int W, float thr) {
  float m = -INFINITY;
#pragma unroll
  for (int i = -1; i <= 1; ++i) {
    const int gyy = gy + i;
    if (gyy < 0 || gyy >= H) continue;
#pragma unroll
    for (int j = -1; j <= 1; ++j) {
      const int xx = x + j;
      if (xx < 0 || xx >= W) continue;
      m = fmaxf(m, plane[(lr + i) * W + xx]);
    }
  }
  return m > thr;
}

// MET (gnca_rollout_metrics): at every step t % M.every == 0 each CTA reduces its own rows (the cells store_own writes)
// against M.target and writes one partial per (frame, sample, rank); M is unused otherwise.
// MS (a stack of models, gnca_rollout_*_models): sample b stages its weights from packed + (b / S.per_model) * S.stride;
// S is unused otherwise.  A compile-time flag: a runtime field moves the register allocation of the plain kernels.
// MET with MS: sample b measures against M.target + (b / S.per_model) * target_stride (0: one target for the stack), a
// trailing parameter as ssim_part is; unused otherwise.
// SS (with MET, gnca_rollout_metrics_ssim): at the same steps each CTA also sums the SSIM of the interior cells of its
// own rows into ssim_part[frame][b][rank], reading the window rows it does not own from their owners over DSMEM between
// two cluster barriers; ssim_part is unused otherwise.
template <int C, bool MET, bool MS, bool SS>
__global__ void __launch_bounds__(kRThreads, 1) k_resident_fwd(ResidentArgs R, Packed P, int hid,
                                                               const float* __restrict__ packed, FrameMetrics M,
                                                               ModelStack S, double* ssim_part, int target_stride) {
  static_assert(MET || !SS, "SSIM rides on the metrics steps");
  cg::cluster_group cluster = cg::this_cluster();
  constexpr int C3 = 3 * C;
  constexpr int CQ = C / 4;                                     // channel quads (power of two)
  constexpr int LCQ = (CQ == 1) ? 0 : (CQ == 2) ? 1 : (CQ == 4) ? 2 : 3;
  StepArgs a = R.s;
  const int NC = R.NC;
  const int rank = (int)cluster.block_rank();
  const int b = blockIdx.x / NC;
  const int H = a.H, W = a.W, HW = H * W;
  const bool graph = (a.flags & GNCA_F_GRAPH) != 0;
  const bool gn = (a.flags & GNCA_F_GROUPNORM) != 0;
  const bool a2a = (a.flags & GNCA_F_ALIVE_TO_ALIVE) != 0;
  const int c_lo = ((a.flags & GNCA_F_HIDDEN_ONLY) && C >= 4) ? 4 : 0;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int own = R.own_rows, HALO = R.halo, RS = own + 2 * HALO;
  const int r0 = rank * own;                 // first global row of the band
  const int nown = own * W;                  // own cells
  const int PL = R.plane_stride;             // padded plane stride (== 1 mod 32: bank-conflict free across channels)
  const int MB = R.MB, MBP = MB + 4;
  const int kk = a.k > 0 ? a.k : 1;

  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* sW1T = reinterpret_cast<float*>(smem_raw);     // [3C][hid], hidden index permuted (see below)
  float* sb1 = sW1T + C3 * hid;                         // [hid] same permutation
  float* sW2T = sb1 + hid;                              // [hid][C]
  float* sWmT = sW2T + hid * C;
  float* sbm = sWmT + (graph ? C * C : 0);
  float* sX = sbm + (graph ? C : 0);                    // [C][RS][W]   resident state: band + halos
  float* sAt = sX + pad4(C * PL);                       // [own+2][W]   pre-gate updated alpha (1-row halo)
  float* Yt = sAt + pad4((own + 2) * W);                // [3C][MBP]
  float* XSt = Yt + C3 * MBP;                           // [C][MBP]
  float* AS = XSt + C * MBP;                            // [MBP]
  float* MSGt = AS + MBP;                               // [C][MBP]
  float* Ht = MSGt + C * MBP;                           // [hid][MBP]
  float* Ut = Ht + hid * MBP;                           // [C][nown] masked pre-norm update of active cells
  int* s_q = reinterpret_cast<int*>(Ut + (size_t)C * nown);   // [MB][k] sender (lr*W+x) or -1
  int* s_actlist = s_q + MB * kk;                       // [nown] own-cell index of active cells (compacted)
  int* s_slot = s_actlist + nown;                       // [nown] slot in the active list or -1
  unsigned char* s_oy = reinterpret_cast<unsigned char*>(s_slot + nown);   // [nown] own row of an own cell
  unsigned char* s_ox = s_oy + ((nown + 15) & ~15);                         // [nown] column
  float* s_fr = reinterpret_cast<float*>(s_ox + ((nown + 15) & ~15));      // [T] fire rate per step (16B aligned)
  float* s_gain = s_fr + R.T;                                               // [T] message gain per step
  signed char* s_off = reinterpret_cast<signed char*>(s_gain + R.T);        // [T][k][2] offsets
  __shared__ float s_partsf[8][2];           // (sum u, sum u^2) of every CTA of the cluster, pushed by its owner
  __shared__ float s_wredf[kRWarps][2];
  __shared__ float s_sc[C], s_bi[C], s_idle[C], s_gam[C], s_bet[C];
  __shared__ int s_wcount[kRWarps], s_wbase[kRWarps + 1];
  __shared__ unsigned long long s_dbg[16];
  if (tid < 16) s_dbg[tid] = 0;

  // ---- weights -> smem.  Hidden units are permuted so that lane l of a warp owns units {g*128 + l + 32*jj}:
  //      its 4 weights of one input k are one float4, and the warp's stores of h are bank-conflict free.
  //      These are the only reads of `packed`.
  if constexpr (MS) packed += (size_t)(b / S.per_model) * S.stride;
#pragma unroll 1
  for (int i = tid; i < C3 * hid; i += kRThreads) {
    const int k = i / hid, jp = i - k * hid;                   // jp = g*128 + l*4 + jj
    const int g = jp >> 7, l = (jp & 127) >> 2, jj = jp & 3;
    sW1T[i] = packed[P.w1t + k * hid + (g * 128 + l + 32 * jj)];
  }
#pragma unroll 1
  for (int jp = tid; jp < hid; jp += kRThreads) {
    const int g = jp >> 7, l = (jp & 127) >> 2, jj = jp & 3;
    sb1[jp] = packed[P.b1 + g * 128 + l + 32 * jj];
  }
  block_copy(sW2T, packed + P.w2t, hid * C);
  if (graph) { block_copy(sWmT, packed + P.wmt, C * C); block_copy(sbm, packed + P.bm, C); }
  if (tid < C) { s_gam[tid] = packed[P.gamma + tid]; s_bet[tid] = packed[P.beta + tid]; }
  // the whole schedule comes on chip once: no global-memory latency inside the step loop
#pragma unroll 1
  for (int i = tid; i < R.T; i += kRThreads) {
    s_fr[i] = a.fire_rate_dev[i];
    s_gain[i] = graph ? a.message_gain_dev[i] : 0.f;
  }
#pragma unroll 1
  for (int i = tid; i < R.T * a.k * 2; i += kRThreads) s_off[i] = a.offsets_dev[i];
#pragma unroll 1
  for (int oc = tid; oc < nown; oc += kRThreads) {
    const int orow = oc / W;
    s_oy[oc] = (unsigned char)orow;
    s_ox[oc] = (unsigned char)(oc - orow * W);
  }

  const size_t sample_off = (size_t)b * C * HW;
  auto wrap_row = [&](int lr) { int gr = (r0 - HALO + lr) % H; return gr < 0 ? gr + H : gr; };
  // ---- x_0 -> smem (band + wrapped halos) ---------------------------------------------------------------
#pragma unroll 1
  for (int row = warp; row < C * RS; row += kRWarps) {
    const int c = row / RS, lr = row - c * RS;
    const float* src = R.x0 + sample_off + (size_t)c * HW + wrap_row(lr) * W;
#pragma unroll 1
    for (int x = lane; x < W; x += 32) sX[(size_t)c * PL + lr * W + x] = src[x];
  }
  float* sA = sX + (size_t)3 * PL;                      // alpha plane
  // neighbour CTAs (torus order) and their views of our pushes
  const int prev = (rank + NC - 1) % NC, next = (rank + 1) % NC;
  float* pX = cluster.map_shared_rank(sX, prev);
  float* nX = cluster.map_shared_rank(sX, next);
  float* pAt = cluster.map_shared_rank(sAt, prev);
  float* nAt = cluster.map_shared_rank(sAt, next);
  __syncthreads();
  cluster_sync_no_acquire();

  const int my_steps = a.steps ? min(a.steps[b], R.T) : R.T;
  long long t_prev = clock64();

  auto store_own = [&](float* dst) {   // own rows of every channel -> global [C][H][W] slice of this sample
#pragma unroll 1
    for (int c = 0; c < C; ++c)
#pragma unroll 1
      for (int oc = tid; oc < nown; oc += kRThreads)
        dst[(size_t)c * HW + r0 * W + oc] = sX[(size_t)c * PL + HALO * W + oc];
  };
  auto store_hist = [&](int t) {        // x_t into its history slot when step t is kept
    if (R.hist && t % R.hist_every == 0) store_own(R.hist + (size_t)(t / R.hist_every) * a.B * C * HW + sample_off);
  };
  // frame metrics of x_t over the own rows; the warps' partials go through the head of the hidden-layer staging
  // buffer Ht, which is free outside P2
  // sample b's target, formed at each use from %ctaid.x and the parameters: the volatile read keeps the compiler from
  // hoisting the rebased pointer out of the step loop, where it would cost two registers (at C = 32 with SSIM, spills)
  auto met_target = [&]() -> const float* {
    if constexpr (MS) {
      unsigned cta;
      asm volatile("mov.u32 %0, %%ctaid.x;" : "=r"(cta));
      return M.target + (size_t)((int)cta / NC / S.per_model) * target_stride;
    }
    return M.target;
  };
  auto met_frame = [&](int t) {
    const float* tgt = met_target();
    MetAcc acc{0.0, 0.0, 0, 0};
#pragma unroll 1
    for (int oc = tid; oc < nown; oc += kRThreads) {
      const float* px = sX + HALO * W + oc;
      met_cell(acc, px[0], px[PL], px[2 * (size_t)PL], px[3 * (size_t)PL], tgt, r0 * W + oc, HW, M.eps,
               a.alpha_thr);
    }
    met_warp_sum(acc);
    double* s_met = reinterpret_cast<double*>(Ht);
    if (lane == 0) met_put(s_met + warp * 4, acc);
    __syncthreads();
    if (tid == 0) met_sum_parts(M.part + (((size_t)(t / M.every) * a.B + b) * NC + rank) * 4, s_met, 0, kRWarps, 4);
    __syncthreads();
  };
  // SSIM of x_t over the interior cells of the own rows.  A window reaches 3 rows beyond the band, more than the halo
  // may hold, so every row is read from the CTA that owns it; the first barrier makes every CTA's x_t (after this step's
  // damage) visible, the second keeps the rows unchanged until every peer has read them.
  auto ssim_frame = [&](int t) {
    cluster.sync();
    const float* tgt = met_target();
    auto state = [&](int yy, int xx) {
      const int q = yy / own;
      const float* p = cluster.map_shared_rank(sX, q) + (size_t)(HALO + yy - q * own) * W + xx;
      return make_float4(p[0], p[PL], p[2 * (size_t)PL], p[3 * (size_t)PL]);
    };
    double s = 0.0;
#pragma unroll 1
    for (int oc = tid; oc < nown; oc += kRThreads) {
      const int y = r0 + oc / W, x = oc % W;
      if (ssim_interior(y, x, H, W)) s += ssim_cell(state, tgt, y, x, W, HW);
    }
    s = warp_sum_f64(s);
    double* s_ss = reinterpret_cast<double*>(Ht);
    if (lane == 0) s_ss[warp] = s;
    __syncthreads();
    if (tid == 0) {
      double v = 0.0;
      for (int w = 0; w < kRWarps; ++w) v += s_ss[w];
      ssim_part[((size_t)(t / M.every) * a.B + b) * NC + rank] = v;
    }
    cluster.sync();
  };
  auto alive_local = [&](const float* plane, int lr, int x, int gy, float thr) {
    return alive_local_ool(plane, lr, x, gy, H, W, thr);
  };

  for (int t = 0; t < R.T; ++t) {
    if (R.damage.p && t == R.damage_step) {    // multiplicative damage on every copy we hold (own + halos)
#pragma unroll 1
      for (int row = warp; row < C * RS; row += kRWarps) {
        const int c = row / RS, lr = row - c * RS;
        const int cell0 = wrap_row(lr) * W;
#pragma unroll 1
        for (int x = lane; x < W; x += 32) sX[(size_t)c * PL + lr * W + x] *= R.damage.at(b, c, cell0 + x, C, HW);
      }
      __syncthreads();
    }
    store_hist(t);
    if constexpr (MET) if (t % M.every == 0) met_frame(t);
    if constexpr (SS) if (t % M.every == 0) ssim_frame(t);
    if (t >= my_steps) continue;               // frozen sample (whole cluster agrees): state passes through
    a.t = t;
    a.fire_u = R.fire_u_base ? R.fire_u_base + (size_t)t * a.B * HW : nullptr;
    const float fr = s_fr[t];
    const float gain_m = s_gain[t];
    const bool msg_on = graph && gain_m != 0.f && a.k > 0;

    // ---- P1: alive & fire on own cells, deterministic compaction ------------------------------------------
    int cnt = 0;
    const int per = ((nown + kRThreads - 1) / kRThreads) * 32;     // own cells per warp (multiple of 32)
    const int lo = warp * per;
    for (int base = lo; base < lo + per; base += 32) {
      const int oc = base + lane;
      bool act = false;
      if (oc < nown) {
        const int orow = s_oy[oc], x = s_ox[oc];
        act = alive_local(sA, HALO + orow, x, r0 + orow, a.alpha_thr) && fires(a, fr, b, (r0 + orow) * W + x);
        s_slot[oc] = act ? 1 : -1;
      }
      cnt += __popc(__ballot_sync(0xffffffffu, act));
    }
    if (lane == 0) s_wcount[warp] = cnt;
    __syncthreads();
    if (warp == 0) {                        // exclusive scan of the per-warp counts
      const int v = lane < kRWarps ? s_wcount[lane] : 0;
      int incl = v;
#pragma unroll
      for (int o = 1; o < kRWarps; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
      }
      if (lane < kRWarps) s_wbase[lane] = incl - v;
      if (lane == kRWarps - 1) s_wbase[kRWarps] = incl;
    }
    __syncthreads();
    int pos = s_wbase[warp];
    for (int base = lo; base < lo + per; base += 32) {
      const int oc = base + lane;
      const bool act = oc < nown && s_slot[oc] > 0;
      const unsigned bal = __ballot_sync(0xffffffffu, act);
      if (act) {
        const int slot = pos + __popc(bal & ((1u << lane) - 1u));
        s_actlist[slot] = oc;
        s_slot[oc] = slot;
      }
      pos += __popc(bal);
    }
    __syncthreads();
    const int nact = s_wbase[kRWarps];
    GNCA_PHASE_MARK(0);
    if (R.dbg && tid == 0) s_dbg[8] += nact;

    // ---- P2: perception + MLP + message on the active cells, in batches of MB ----------------------------
    float ps1 = 0.f, ps2 = 0.f;
    for (int base = 0; base < nact; base += MB) {
      const int nb = min(MB, nact - base);
      const int G = nb > 32 ? 8 : 4;                    // cells per warp tile (layer 1 + layer 2 stay inside one warp)
      const int nbp = ((nb + G - 1) / G) * G;           // staged cells (zero padded to the tile)
      // 2a: sender table, one lane per (cell, offset): local index of the (alive) sender or -1
      if (msg_on) {
        for (int i = tid; i < nb * a.k; i += kRThreads) {
          const int cl = i / a.k, oi = i - cl * a.k;
          const int oc = s_actlist[base + cl];
          const int orow = s_oy[oc], x = s_ox[oc], gy = r0 + orow;
          const int dy = s_off[(t * a.k + oi) * 2], dx = s_off[(t * a.k + oi) * 2 + 1];
          int gq = (gy - dy) % H; gq = gq < 0 ? gq + H : gq;       // sender's global row (torus)
          int qx = (x - dx) % W; qx = qx < 0 ? qx + W : qx;
          const int lq = HALO + orow - dy;                          // its local row (halo holds the wrap)
          int q = lq * W + qx;
          if (a2a && !alive_local(sA, lq, qx, gq, a.graph_alpha_thr)) q = -1;
          s_q[cl * kk + oi] = q;
        }
        __syncthreads();
      }
      // 2b: one half-warp per cell, lane = channel: perception (9 independent loads) and the gathered sender
      //     state xs = sum_i w x(q_i) with the k loads issued back to back (invalid senders get weight 0)
      const int hw = tid >> 4, l16 = tid & 15;
      const float wuni = a.k > 0 ? 1.0f / (float)a.k : 0.f;
      for (int cl = hw; cl < nbp; cl += kRThreads / 16) {
        const bool valid = cl < nb;
        int orow = 0, x = 0;
        if (valid) { const int oc = s_actlist[base + cl]; orow = s_oy[oc]; x = s_ox[oc]; }
        const int gy = r0 + orow;
        const bool up = gy > 0, dn = gy < H - 1, lf = x > 0, rt = x < W - 1;
        int nvalid = 0;
        for (int c = l16; c < C; c += 16) {
          float vid = 0.f, vsx = 0.f, vsy = 0.f, xs = 0.f;
          if (valid) {
            const float* pc = sX + (size_t)c * PL;
            const float* p = pc + (HALO + orow) * W + x;
            const float a00 = (up && lf) ? p[-W - 1] : 0.f, a01 = up ? p[-W] : 0.f, a02 = (up && rt) ? p[-W + 1] : 0.f;
            const float a10 = lf ? p[-1] : 0.f, a12 = rt ? p[1] : 0.f;
            const float a20 = (dn && lf) ? p[W - 1] : 0.f, a21 = dn ? p[W] : 0.f, a22 = (dn && rt) ? p[W + 1] : 0.f;
            vid = p[0];
            vsx = (a00 - a02) + 2.f * (a10 - a12) + (a20 - a22);
            vsy = (a00 + 2.f * a01 + a02) - (a20 + 2.f * a21 + a22);
            if (msg_on) {
              nvalid = 0;
              const int* qrow = s_q + cl * kk;
              for (int o4 = 0; o4 < a.k; o4 += 4) {
                int q0, q1, q2, q3;
                if ((kk & 3) == 0) {
                  const int4 qq = *reinterpret_cast<const int4*>(qrow + o4);
                  q0 = qq.x; q1 = qq.y; q2 = qq.z; q3 = qq.w;
                } else {
                  q0 = qrow[o4];
                  q1 = (o4 + 1 < a.k) ? qrow[o4 + 1] : -1;
                  q2 = (o4 + 2 < a.k) ? qrow[o4 + 2] : -1;
                  q3 = (o4 + 3 < a.k) ? qrow[o4 + 3] : -1;
                }
                const float v0 = pc[max(q0, 0)], v1 = pc[max(q1, 0)], v2 = pc[max(q2, 0)], v3 = pc[max(q3, 0)];
                xs = fmaf(q0 >= 0 ? wuni : 0.f, v0, xs);
                xs = fmaf(q1 >= 0 ? wuni : 0.f, v1, xs);
                xs = fmaf(q2 >= 0 ? wuni : 0.f, v2, xs);
                xs = fmaf(q3 >= 0 ? wuni : 0.f, v3, xs);
                nvalid += (q0 >= 0) + (q1 >= 0) + (q2 >= 0) + (q3 >= 0);
              }
            }
          }
          Yt[c * MBP + cl] = vid;
          Yt[(C + c) * MBP + cl] = vsx;
          Yt[(2 * C + c) * MBP + cl] = vsy;
          XSt[c * MBP + cl] = xs;
        }
        if (l16 == 0) {
          float as = 0.f;
          for (int n = 0; n < nvalid; ++n) as += wuni;     // same summation as the streaming path
          AS[cl] = as;
        }
        __syncwarp();     // nbp is even: both half-warps of a warp run this loop the same number of times
        // message projection by the first CQ lanes of the half-warp:
        //   MSGt[c][cl] = gain * tanh(bm[c]*as + sum_ci Wm[c][ci] xs[ci]) on the gated channels, else 0
        if (l16 < CQ) {
          const int cq = l16;
          float agg[4] = {0.f, 0.f, 0.f, 0.f};
          if (msg_on && valid && 4 * cq + 3 >= c_lo) {
            const float as = AS[cl];
            const float4 bmv = *reinterpret_cast<const float4*>(sbm + 4 * cq);
            agg[0] = bmv.x * as; agg[1] = bmv.y * as; agg[2] = bmv.z * as; agg[3] = bmv.w * as;
#pragma unroll 4
            for (int ci = 0; ci < C; ++ci) {
              const float xv = XSt[ci * MBP + cl];
              const float4 w = *reinterpret_cast<const float4*>(sWmT + ci * C + 4 * cq);
              agg[0] = fmaf(w.x, xv, agg[0]); agg[1] = fmaf(w.y, xv, agg[1]);
              agg[2] = fmaf(w.z, xv, agg[2]); agg[3] = fmaf(w.w, xv, agg[3]);
            }
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) agg[cc] = (4 * cq + cc >= c_lo) ? tanhf(agg[cc]) * gain_m : 0.f;
          }
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) MSGt[(4 * cq + cc) * MBP + cl] = agg[cc];
        }
      }
      __syncthreads();
      GNCA_PHASE_MARK(10);
      // 2c: layer 1 + layer 2 inside ONE warp per tile of G cells (no block barrier in between): lane = 4 permuted
      //     hidden units for layer 1; for layer 2 the warp re-reads its own h columns with the hidden dimension
      //     split over 4 lane groups (j = 4*jj + kq) and reduces with two shuffle levels.
      auto mlp_tile = [&](auto gtag) {
        constexpr int GG = decltype(gtag)::value;
        const int ngroups = nbp / GG;
        for (int cgp = warp; cgp < ngroups; cgp += kRWarps) {
          const int jp = lane * 4;                      // permuted index of this lane's 4 hidden units
          {
            float acc[GG][4];
            const float4 bb = *reinterpret_cast<const float4*>(sb1 + jp);
#pragma unroll
            for (int m = 0; m < GG; ++m) { acc[m][0] = bb.x; acc[m][1] = bb.y; acc[m][2] = bb.z; acc[m][3] = bb.w; }
#pragma unroll 4
            for (int k = 0; k < C3; ++k) {
              const float4 w = *reinterpret_cast<const float4*>(sW1T + k * hid + jp);
              float ym[GG];
#pragma unroll
              for (int m4 = 0; m4 < GG / 4; ++m4) {
                const float4 yv = *reinterpret_cast<const float4*>(Yt + k * MBP + GG * cgp + 4 * m4);
                ym[4 * m4] = yv.x; ym[4 * m4 + 1] = yv.y; ym[4 * m4 + 2] = yv.z; ym[4 * m4 + 3] = yv.w;
              }
#pragma unroll
              for (int m = 0; m < GG; ++m) {
                acc[m][0] = fmaf(ym[m], w.x, acc[m][0]); acc[m][1] = fmaf(ym[m], w.y, acc[m][1]);
                acc[m][2] = fmaf(ym[m], w.z, acc[m][2]); acc[m][3] = fmaf(ym[m], w.w, acc[m][3]);
              }
            }
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
              const int j = lane + 32 * jj;             // true hidden index (row of Ht / W2T)
#pragma unroll
              for (int m4 = 0; m4 < GG / 4; ++m4) {
                float4 hv;
                hv.x = fmaxf(acc[4 * m4][jj], 0.f); hv.y = fmaxf(acc[4 * m4 + 1][jj], 0.f);
                hv.z = fmaxf(acc[4 * m4 + 2][jj], 0.f); hv.w = fmaxf(acc[4 * m4 + 3][jj], 0.f);
                *reinterpret_cast<float4*>(Ht + j * MBP + GG * cgp + 4 * m4) = hv;
              }
            }
          }
          __syncwarp();
          const int kq = lane >> 3, tl = lane & 7;
          constexpr int NSUB = (GG / 2) * CQ;           // sub-tiles of 2 cells x 4 channels
#pragma unroll 1
          for (int st0 = 0; st0 < NSUB; st0 += 8) {
            const int st = st0 + tl;
            const bool on = st < NSUB;
            const int cp = on ? st % (GG / 2) : 0, cq = on ? st / (GG / 2) : 0;
            float o2[2][4];
#pragma unroll
            for (int m = 0; m < 2; ++m)
#pragma unroll
              for (int cc = 0; cc < 4; ++cc) o2[m][cc] = 0.f;
#pragma unroll 4
            for (int jj = 0; jj < 32; ++jj) {
              const int j = 4 * jj + kq;
              const float2 hv = *reinterpret_cast<const float2*>(Ht + j * MBP + GG * cgp + 2 * cp);
              const float4 w = *reinterpret_cast<const float4*>(sW2T + j * C + 4 * cq);
              o2[0][0] = fmaf(hv.x, w.x, o2[0][0]); o2[0][1] = fmaf(hv.x, w.y, o2[0][1]);
              o2[0][2] = fmaf(hv.x, w.z, o2[0][2]); o2[0][3] = fmaf(hv.x, w.w, o2[0][3]);
              o2[1][0] = fmaf(hv.y, w.x, o2[1][0]); o2[1][1] = fmaf(hv.y, w.y, o2[1][1]);
              o2[1][2] = fmaf(hv.y, w.z, o2[1][2]); o2[1][3] = fmaf(hv.y, w.w, o2[1][3]);
            }
#pragma unroll
            for (int m = 0; m < 2; ++m)
#pragma unroll
              for (int cc = 0; cc < 4; ++cc) {
                float v = o2[m][cc];
                v += __shfl_xor_sync(0xffffffffu, v, 8);
                v += __shfl_xor_sync(0xffffffffu, v, 16);
                o2[m][cc] = v;
              }
            if (on && kq == 0) {
#pragma unroll
              for (int m = 0; m < 2; ++m) {
                const int cl = GG * cgp + 2 * cp + m;
                if (cl < nb) {
#pragma unroll
                  for (int cc = 0; cc < 4; ++cc) {
                    const int c = 4 * cq + cc;
                    const float v = o2[m][cc] + MSGt[c * MBP + cl];
                    Ut[(size_t)c * nown + base + cl] = v;
                    if (R.u_hist)
                      R.u_hist[(((size_t)t * a.B + b) * C + c) * HW + r0 * W + s_actlist[base + cl]] = v;
                    ps1 += v;
                    ps2 = fmaf(v, v, ps2);
                  }
                }
              }
            }
          }
          __syncwarp();
        }
      };
      if (G == 8) mlp_tile(std::integral_constant<int, 8>{}); else mlp_tile(std::integral_constant<int, 4>{});
      __syncthreads();     // staging buffers are reused by the next batch
    }
    GNCA_PHASE_MARK(1);

    // ---- GroupNorm(1,C) statistics over the whole sample: block partial -> DSMEM all-gather ----------------
    float mu = 0.f, rstd = 1.f;
    if (gn) {
      // fp32 tree (warp shuffles -> 16 warps -> NC CTAs); every CTA reduces the same values in the same order
      const float f1 = warp_sum(ps1), f2 = warp_sum(ps2);
      if (lane == 0) { s_wredf[warp][0] = f1; s_wredf[warp][1] = f2; }
      __syncthreads();
      if (warp == 0) {
        float t1 = lane < kRWarps ? s_wredf[lane][0] : 0.f, t2 = lane < kRWarps ? s_wredf[lane][1] : 0.f;
        t1 = warp_sum(t1); t2 = warp_sum(t2);
        if (lane < NC) {                       // push our partial into slot `rank` of every CTA (incl. ourselves)
          float* dst = cluster.map_shared_rank(&s_partsf[0][0], lane);
          dst[rank * 2] = t1; dst[rank * 2 + 1] = t2;
        }
      }
      GNCA_PHASE_MARK(2);
      cluster_sync_no_acquire();                                              // barrier 1
      GNCA_PHASE_MARK(3);
      if (warp == 0) {
        float t1 = 0.f, t2 = 0.f;
        if (lane < NC) { t1 = s_partsf[lane][0]; t2 = s_partsf[lane][1]; }
        const float a1 = warp_sum(t1), a2 = warp_sum(t2);
        const float invn = (float)R.inv_n;
        const float m_ = a1 * invn;
        const float var = fmaxf(fmaf(a2, invn, -m_ * m_), 0.f);
        const float r_ = 1.0f / sqrtf(var + a.gn_eps);
        if (lane == 0 && rank == 0 && R.stats_hist) {
          R.stats_hist[((size_t)t * a.B + b) * 2] = m_;
          R.stats_hist[((size_t)t * a.B + b) * 2 + 1] = r_;
        }
        if (lane < C) {                       // C <= 32: the same warp finishes the per-channel affine
          const float sc = r_ * s_gam[lane];
          const float bi = s_bet[lane] - m_ * sc;
          s_sc[lane] = sc; s_bi[lane] = bi;
          s_idle[lane] = tanhf(bi) * a.update_gain;
        }
      }
    } else if (tid < C) {
      s_sc[tid] = 1.f; s_bi[tid] = 0.f; s_idle[tid] = 0.f;
    }
    __syncthreads();
    (void)mu; (void)rstd;
    GNCA_PHASE_MARK(4);

    // ---- P3: bounded update in place (own cells); idle update of the halo copies; pre-gate alpha rows -------
    // inactive own cells: x += idle_c (their masked pre-norm update is 0); lanes <-> consecutive cells
    for (int item = warp; item < ((nown + 31) >> 5) * CQ; item += kRWarps) {
      const int cq = item & (CQ - 1), oc = (item >> LCQ) * 32 + lane;
      if (oc >= nown || s_slot[oc] >= 0) continue;
      float* px = sX + (size_t)(4 * cq) * PL + HALO * W + oc;
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        const int c = 4 * cq + cc;
        const float v = px[(size_t)cc * PL] + s_idle[c];
        if (c == 3) {
          sAt[W + oc] = v;                                   // rows 1..own of sAt
          const int orow = s_oy[oc];
          if (orow == 0) pAt[(own + 1) * W + oc] = v;        // our top row = prev's bottom halo row
          if (orow == own - 1) nAt[oc - (own - 1) * W] = v;  // our bottom row = next's top halo row
        } else {
          px[(size_t)cc * PL] = v;
        }
      }
    }
    // active cells: x += gain * tanh(gn(u)); one lane per (slot, channel), lanes <-> consecutive slots
    for (int item = warp; item < ((nact + 31) >> 5) * C; item += kRWarps) {
      const int c = item & (C - 1), sl = (item / C) * 32 + lane;
      if (sl >= nact) continue;
      const int oc = s_actlist[sl];
      const float d = tanhf(fmaf(Ut[(size_t)c * nown + sl], s_sc[c], s_bi[c])) * a.update_gain;
      float* px = sX + (size_t)c * PL + HALO * W + oc;
      const float v = *px + d;
      if (c == 3) {
        sAt[W + oc] = v;
        const int orow = s_oy[oc];
        if (orow == 0) pAt[(own + 1) * W + oc] = v;
        if (orow == own - 1) nAt[oc - (own - 1) * W] = v;
      } else {
        *px = v;
      }
    }
    for (int item = warp; item < ((2 * HALO * W + 31) >> 5) * CQ; item += kRWarps) {   // halo cells, channels != 3
      const int cq = item & (CQ - 1), hc = (item >> LCQ) * 32 + lane;
      if (hc >= 2 * HALO * W) continue;
      const int off = hc < HALO * W ? hc : own * W + hc;                    // top halo | bottom halo
      float* px = sX + (size_t)(4 * cq) * PL + off;
#pragma unroll
      for (int cc = 0; cc < 4; ++cc)
        if (4 * cq + cc != 3) px[(size_t)cc * PL] += s_idle[4 * cq + cc];
    }
    __syncthreads();
    GNCA_PHASE_MARK(5);
    cluster_sync_no_acquire();                                                // barrier 2
    GNCA_PHASE_MARK(6);
    // ---- P4: post-alive gate on own cells; push gated alpha rows + active cells' channels to the halos -------
    for (int oc = tid; oc < nown; oc += kRThreads) {
      const int orow = s_oy[oc], x = s_ox[oc];
      const bool post = alive_local(sAt, 1 + orow, x, r0 + orow, a.alpha_thr);
      const float v = post ? sAt[W + oc] : 0.f;
      sA[HALO * W + oc] = v;
      if (orow < HALO) pX[(size_t)3 * PL + (HALO + own) * W + oc] = v;                 // prev's bottom halo
      if (orow >= own - HALO) nX[(size_t)3 * PL + oc - (own - HALO) * W] = v;           // next's top halo
    }
    for (int item = warp; item < ((nact + 31) >> 5) * CQ; item += kRWarps) {
      const int cq = item & (CQ - 1), sl = (item >> LCQ) * 32 + lane;
      if (sl >= nact) continue;
      const int oc = s_actlist[sl];
      const int orow = s_oy[oc];
      const bool to_prev = orow < HALO, to_next = orow >= own - HALO;
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        const int c = 4 * cq + cc;
        if (c == 3) continue;
        const float v = sX[(size_t)c * PL + HALO * W + oc];
        if (to_prev) pX[(size_t)c * PL + (HALO + own) * W + oc] = v;
        if (to_next) nX[(size_t)c * PL + oc - (own - HALO) * W] = v;
      }
    }
    __syncthreads();
    GNCA_PHASE_MARK(7);
    cluster_sync_no_acquire();                                                // barrier 3
    GNCA_PHASE_MARK(9);
  }

  store_hist(R.T);
  if constexpr (MET) if (R.T % M.every == 0) met_frame(R.T);
  if constexpr (SS) if (R.T % M.every == 0) ssim_frame(R.T);
  store_own(R.xT + sample_off);
  if (R.dbg && blockIdx.x == R.dbg_cta && tid < 16) R.dbg[tid] = s_dbg[tid];
  cluster_sync_no_acquire();     // nobody exits while a neighbour may still address its shared memory
}

// ------------------------------------------------------------------------------------------------
static int plane_stride_of(int own, int halo, int W) {
  const int pl = (own + 2 * halo) * W;
  return pl + ((33 - pl % 32) % 32);        // == 1 (mod 32)
}

static size_t resident_smem_bytes(int C, int hid, bool graph, int own, int halo, int W, int MB, int k, int T) {
  const int MBP = MB + 4;
  size_t f = (size_t)3 * C * hid + hid + (size_t)hid * C;
  if (graph) f += C * C + C;
  f += (size_t)pad4(C * plane_stride_of(own, halo, W));
  f += (size_t)pad4((own + 2) * W);
  f += (size_t)3 * C * MBP + (size_t)C * MBP + MBP + (size_t)C * MBP + (size_t)hid * MBP;
  f += (size_t)C * own * W;
  size_t bytes = f * sizeof(float);
  bytes += (size_t)MB * (k > 0 ? k : 1) * sizeof(int) + 2 * (size_t)own * W * sizeof(int) + 2 * (size_t)((own * W + 15) & ~15);
  bytes += 16 + (size_t)T * 8 + (size_t)T * k * 2;        // schedule: fire rate, gain, offsets
  return bytes + 64;
}

template <int C>
static int launch_resident(const gnca_model& m, const Packed& P, const float* packed, ResidentArgs& R, int B, int radius,
                           cudaStream_t st, const FrameMetrics* met, ModelStack S, const SsimFrames* ss,
                           int target_stride) {
  const bool graph = (m.flags & GNCA_F_GRAPH) != 0;
  const int H = R.s.H, W = R.s.W;
  if (m.hidden != 128 || C < 4 || W > 255) return GNCA_ERR_UNSUPPORTED;   // layer 1 + 2 of a tile live in one warp: 32 lanes x 4 units
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int halo = (graph && R.s.k > 0 ? radius : 0) + 1;
  const char* env_nc = getenv("GNCA_RESIDENT_NC");      // development override of the cluster size
  const bool debug = getenv("GNCA_DEBUG") != nullptr;
  // Cluster size: the largest NC in {8,4,2,1} whose bands are at least `halo` rows, that fits shared memory and
  // keeps ALL B clusters co-resident (B <= cudaOccupancyMaxActiveClusters); if the batch is too large for that,
  // the smallest NC that fits (most clusters per wave) and the launch runs in waves.
  // the metrics (and SSIM) instantiations have the plain one's shared memory and register cap: the same launch
  // configuration
  const bool stack = S.stride != 0, ssim = met && ss;
  auto kfn = stack ? (ssim ? k_resident_fwd<C, true, true, true>
                           : met ? k_resident_fwd<C, true, true, false> : k_resident_fwd<C, false, true, false>)
                   : (ssim ? k_resident_fwd<C, true, false, true>
                           : met ? k_resident_fwd<C, true, false, false> : k_resident_fwd<C, false, false, false>);
  // the dynamic carve shares the opt-in limit with the kernel's static shared memory (about 1.1 KB at C = 32)
  const size_t cap = dynamic_smem_cap((const void*)kfn);
  const int cands[4] = {8, 4, 2, 1};
  int pick = -1, pick_MB = 0, pick_nclusters = 0;
  size_t pick_smem = 0;
  for (int pass = 0; pass < 2 && pick < 0; ++pass) {
    for (int ci = (pass == 0 ? 0 : 3); ci >= 0 && ci < 4; ci += (pass == 0 ? 1 : -1)) {
      const int NC = cands[ci];
      if (env_nc && atoi(env_nc) != NC) continue;
      if (H % NC != 0 || H / NC < halo || H / NC > 255) continue;
      const int own = H / NC;
      int MB = 64;
      size_t smem = resident_smem_bytes(C, m.hidden, graph, own, halo, W, MB, R.s.k, R.T);
      if (smem > cap) { MB = 32; smem = resident_smem_bytes(C, m.hidden, graph, own, halo, W, MB, R.s.k, R.T); }
      if (smem > cap) { MB = 16; smem = resident_smem_bytes(C, m.hidden, graph, own, halo, W, MB, R.s.k, R.T); }   // 40x40x32
      if (smem > cap) continue;
      GNCA_CHECK_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      cudaLaunchConfig_t q{};
      q.gridDim = dim3(B * NC); q.blockDim = dim3(kRThreads); q.dynamicSmemBytes = smem; q.stream = st;
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = NC; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
      q.attrs = qa; q.numAttrs = 1;
      int nclusters = 0;
      if (cudaOccupancyMaxActiveClusters(&nclusters, kfn, &q) != cudaSuccess || nclusters < 1) {
        cudaGetLastError();
        continue;
      }
      if (pass == 0 && B > nclusters && !env_nc) continue;      // would need a second wave: try a smaller cluster
      pick = NC; pick_MB = MB; pick_smem = smem; pick_nclusters = nclusters;
      break;
    }
  }
  if (pick < 0) return GNCA_ERR_UNSUPPORTED;
  {
    const int NC = pick, own = H / NC, MB = pick_MB;
    const size_t smem = pick_smem;
    GNCA_CHECK_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(B * NC);
    cfg.blockDim = dim3(kRThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = NC; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    const int nclusters = pick_nclusters;
    if (debug)
      fprintf(stderr, "[gnca] resident fwd: B=%d NC=%d own_rows=%d halo=%d MB=%d smem=%zu maxActiveClusters=%d\n", B, NC,
              own, halo, MB, smem, nclusters);
    R.NC = NC; R.own_rows = own; R.halo = halo; R.MB = MB; R.plane_stride = plane_stride_of(own, halo, W);
    R.inv_n = 1.0 / ((double)C * (double)H * (double)W);
    static unsigned long long* dbg_buf = nullptr;
    if (getenv("GNCA_PHASE_TIMING")) {
      if (!dbg_buf) cudaMalloc(&dbg_buf, 16 * sizeof(unsigned long long));
      cudaMemsetAsync(dbg_buf, 0, 16 * sizeof(unsigned long long), st);
      R.dbg = dbg_buf;
      R.dbg_cta = atoi(getenv("GNCA_PHASE_TIMING"));
    }
    prof_begin(PROF_RESIDENT_FWD, st);
    cudaError_t e = cudaLaunchKernelEx(&cfg, kfn, R, P, m.hidden, packed, met ? *met : FrameMetrics{}, S,
                                       ssim ? ss->part : nullptr, target_stride);
    prof_end(PROF_RESIDENT_FWD, st);
    if (e != cudaSuccess) return (int)e;
    GNCA_LAUNCH_CHECK();
    if (met) {
      const int rc = run_metrics_reduce((R.T / met->every + 1) * B, NC, met->part, met->sums, met->counts, st);
      if (rc) return rc;
    }
    if (ssim) {
      const int rc = run_ssim_reduce((R.T / met->every + 1) * B, NC, ss->part, ss->ssim, H, W, st);
      if (rc) return rc;
    }
    if (R.dbg) {   // development only: synchronous read-back of the phase counters of CTA 0
      unsigned long long h[16];
      cudaStreamSynchronize(st);
      cudaMemcpy(h, dbg_buf, sizeof(h), cudaMemcpyDeviceToHost);
      const char* names[16] = {"P1 alive+compact", "P2 tail(reduce)", "stats reduce", "barrier1", "stats finish",
                               "P3 update", "barrier2", "P4 gate+push", "(sum nact)", "barrier3", "P2 stage",
                               "P2 msg+layer1", "P2 layer2", "st:dsmem-ld", "st:warpsum", "st:math"};
      fprintf(stderr, "[gnca phase cycles, CTA%d, T=%d]", R.dbg_cta, R.T);
      for (int i = 0; i < 16; ++i) fprintf(stderr, " %s=%llu", names[i], h[i]);
      fprintf(stderr, "\n");
    }
    return 0;
  }
}

// entry used by gnca_rollout_fwd (impl 2 / auto)
int run_resident_fwd(const gnca_model& m, const Packed& P, const float* packed, int B, int H, int W,
                     const gnca_schedule& sched, const float* x0, float* xT, float* hist, float* stats_hist,
                     float* u_hist, float* ping, float* pong, float* alpha_tmp, cudaStream_t st, int hist_every,
                     const FrameMetrics* met, ModelStack ms, const SsimFrames* ss, int target_stride) {
  (void)ping; (void)pong; (void)alpha_tmp;
  const bool graph = (m.flags & GNCA_F_GRAPH) != 0;
  if (graph && !(m.flags & GNCA_F_TORUS) && sched.k > 0) return GNCA_ERR_UNSUPPORTED;   // zero-pad: streaming path
  if (graph && sched.k > 0 && sched.max_offset <= 0) return GNCA_ERR_UNSUPPORTED;       // halo depth unknown
  ResidentArgs R{};
  fill_step_args(R.s, m, B, H, W);
  R.s.k = graph ? sched.k : 0;
  R.s.fire_rate_dev = sched.fire_rate;
  R.s.message_gain_dev = sched.message_gain;
  R.s.offsets_dev = sched.offsets;
  R.s.steps = sched.steps;
  R.s.philox_seed = sched.philox_seed;
  R.s.philox_offset = sched.philox_offset;
  R.fire_u_base = sched.fire_u;
  R.T = sched.T;
  R.x0 = x0; R.xT = xT; R.hist = hist; R.hist_every = hist_every; R.stats_hist = stats_hist; R.u_hist = u_hist;
  R.damage = DamageView{sched.damage, sched.damage_layout}; R.damage_step = sched.damage_step;
  const int radius = sched.max_offset;       // largest |dy| / |dx| in the schedule: sets the halo depth
  switch (m.C) {
    case 4: return launch_resident<4>(m, P, packed, R, B, radius, st, met, ms, ss, target_stride);
    case 8: return launch_resident<8>(m, P, packed, R, B, radius, st, met, ms, ss, target_stride);
    case 16: return launch_resident<16>(m, P, packed, R, B, radius, st, met, ms, ss, target_stride);
    case 32: return launch_resident<32>(m, P, packed, R, B, radius, st, met, ms, ss, target_stride);
  }
  return GNCA_ERR_UNSUPPORTED;
}

}  // namespace gnca
