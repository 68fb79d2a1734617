// Replicated-state cluster rollout (forward): ONE launch runs all T steps, state in shared memory.
//
// A sample is owned by a thread-block cluster of NC CTAs (8/4/2/1).  EVERY CTA keeps the WHOLE sample in shared
// memory for the whole rollout, cell-major ([cell][C], alpha in two dense planes), so
//   * the active cells of a step (fire & pre-alive, reference ncagraph.py:144-150) are split EVENLY over the
//     cluster whatever their position (a band split leaves the edge bands idle while the centre bands work);
//   * perception (3x3, zero halo) and the mid-range torus senders are read in place with no halo logic;
//   * the masks are linear cell bitmaps: max-pool > thr is a 3x3 dilation of (alpha > thr) done with funnel
//     shifts, compaction is popcount prefix sums, and pre_alive(t+1) == post_alive(t) is reused, not recomputed.
// Per step (reference semantics: ncagraph.py:106-168):
//   S2  warp-autonomous tiles of 2/4/8 cells over MY share of the active list: sender table, perception, message,
//       layer 1 in registers, layer 2 as a shuffle reduce-scatter -- no block barrier, no hidden layer in smem.
//       Warps without a tile generate the next step's Philox fire bits meanwhile; the BPTT history / records of the
//       step are stored before the hand-over below.
//   --  GroupNorm partials: warp -> block -> every CTA of the cluster with st.async, counted (8 bytes per peer) on the
//       peer's mbarrier A.  A peer's partial arriving also says "that peer has finished reading x_t".
//   S3  warp 0 finishes the statistics; my active cells get x + gain*tanh(gn(u)) and are pushed as 64-byte lines into
//       ALL NC replicas with st.async (transaction bytes counted on the destination's mbarrier B); while those
//       travel every CTA runs its local idle update x += idle_c of all inactive cells.
//   S4  (after mbarrier B) post-alive gate from the bitmap of the updated alpha, fused with the active bitmap /
//       balanced list of the next step.
// No cluster barrier and no MEMBAR.GPU inside the step loop (a barrier-based exchange remains as GNCA_REP_SYNC=barrier).
// HBM is touched at x_0 / x_T and by the optional BPTT history (x_t, u_t of the active cells, statistics).
#include <cooperative_groups.h>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <mutex>
#include <utility>
#include <type_traits>
#include "gnca_common.cuh"
#include "gnca_internal.h"
#include "gnca_metrics.cuh"
#include "gnca_ptx.cuh"
#include "gnca_rep.h"

namespace cg = cooperative_groups;

namespace gnca {

constexpr int kPT = 512;          // threads per CTA
constexpr int kPW = kPT / 32;     // warps
constexpr int kW2S = 20;          // padded row stride of W2^T (floats): conflict-free per-lane LDS.128 rows
constexpr int kMaxRows = 64;      // H, W <= 64
constexpr int kMaxWords = kMaxRows * kMaxRows / 32;   // words of a linear cell bitmap

struct RepArgs {
  StepArgs s;
  int T, NC, ucap, KP, listcap, HWp, zd;
  float inv_n;
  const float* fire_u_base;   // [T][B][H][W] or null
  const float* x0;
  float* xT;
  float* hist;                // [T/hist_every+1][B][C][HW] or null: x_t of the steps t % hist_every == 0, in slot t/hist_every
  int hist_every;
  float* stats_hist;          // [T][B][2] or null
  float* u_hist;              // [T][B][C][HW] or null (dense layout, active cells only)
  float* rec;                 // [T][B][HW][kRecStride] or null: per-active-cell records for the resident backward
  uint32_t* masks;            // [T][B][3][kMaskWords] or null: sender-alive, active, post-alive bitmaps of every step
  float* u_over;              // [B*NC][over_cap][C] overflow of the in-smem u buffer
  int over_cap;
  DamageView damage;          // schedule.damage (dense or plane) or null
  int damage_step;
  unsigned long long* dbg;
  int dbg_cta;
  int use_async;              // 1: st.async + mbarrier transaction counts between the CTAs, 0: two cluster barriers per step
  // absolute step of the launch's local step 0 (a checkpoint segment starts at t0 = j * every).  The caller hands
  // run_rep_fwd a schedule already rebased to the launch (arrays, fire_u, Philox counter, damage_step: segment_schedule
  // in gnca_rollout.cu); the kernel needs t0 only for the per-sample step counts steps[b], which stay absolute
  int t0;
  // a stack of models (ModelStack): sample b stages its weights from packed + (b / model_per) * model_stride;
  // model_stride = 0: every sample runs the model at `packed`
  int model_stride, model_per;
  // MET with per-model targets (run_rep_fwd's target_stride): sample b measures against M.target + (b / model_per) *
  // target_stride; 0 = one target.  It fills the struct's tail padding, so the parameters of the plain instantiations
  // keep their offsets.
  int target_stride;
};

#ifdef GNCA_PHASE_COUNTERS          /* build with -DGNCA_PHASE_COUNTERS for the per-phase cycle counters */
#define REP_MARK(idx)                                                               \
  do {                                                                              \
    if (R.dbg && tid == 0) {                                                        \
      const long long _n = clock64();                                               \
      s_dbg[idx] += (unsigned long long)(_n - t_prev);                              \
      t_prev = _n;                                                                  \
    }                                                                               \
  } while (0)
#else
#define REP_MARK(idx) do { } while (0)
#endif

__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, int rank) {
  uint32_t o;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(o) : "r"(addr), "r"(rank));
  return o;
}
__device__ __forceinline__ void st_cluster_f32(uint32_t addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
// remote store that signals `bytes written` on an mbarrier of the destination CTA: the consumer waits for the
// expected byte count instead of a cluster-wide barrier (and no MEMBAR on the producer side)
__device__ __forceinline__ void st_async_f32(uint32_t raddr, float v, uint32_t rmbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.f32 [%0], %1, [%2];" ::"r"(raddr), "f"(v), "r"(rmbar)
               : "memory");
}
// eight consecutive lanes each hold a nibble (4 cells): OR them into the 32-bit word of those 32 cells
__device__ __forceinline__ uint32_t pack_nibbles(uint32_t nib, int lane) {
  uint32_t w = nib << (4 * (lane & 7));
  w |= __shfl_xor_sync(0xffffffffu, w, 1);
  w |= __shfl_xor_sync(0xffffffffu, w, 2);
  w |= __shfl_xor_sync(0xffffffffu, w, 4);
  return w;
}

// Frame metrics of x_t (cell-major sX, alpha plane sAg) over cells [lo, hi), spread over warps [w0, kPW): each warp
// leaves its partial as 4 doubles at the head of its own perception tile in sY, which is free from the end of its tiles
// to the next step's tiles.  rep_met_flush (one thread, after a barrier) adds them in warp order.
__device__ __forceinline__ void rep_met_cells(const FrameMetrics& M, const float* tgt, const float* sX, const float* sAg,
                                              float* sY, int lo, int hi, int HW, float thr, int w0) {
  constexpr int C = 16, kTile = 3 * C * 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  MetAcc acc{0.0, 0.0, 0, 0};
#pragma unroll 1
  for (int cell = lo + (warp - w0) * 32 + lane; cell < hi; cell += (kPW - w0) * 32) {
    const float4 v = *reinterpret_cast<const float4*>(sX + (size_t)cell * C);
    met_cell(acc, v.x, v.y, v.z, sAg[cell], tgt, cell, HW, M.eps, thr);
  }
  met_warp_sum(acc);
  if (lane == 0) met_put(reinterpret_cast<double*>(sY + warp * kTile), acc);
}
__device__ __forceinline__ void rep_met_flush(const float* sY, int w0, double* dst) {
  met_sum_parts(dst, reinterpret_cast<const double*>(sY), w0, kPW, 3 * 16 * 8 / 2);
}

// SSIM of x_t over the interior cells among [lo, hi), spread over warps [w0, kPW) like rep_met_cells: the 7x7 windows are
// read from the replica (sX, sAg), which holds all of x_t.  Each warp leaves its sum as the fifth double of its tile head.
__device__ __forceinline__ void rep_ssim_cells(const float* sX, const float* sAg, float* sY, const float* tgt, int lo,
                                               int hi, int H, int W, int w0) {
  constexpr int C = 16, kTile = 3 * C * 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  auto state = [&](int yy, int xx) {
    const int cell = yy * W + xx;
    float4 v = *reinterpret_cast<const float4*>(sX + (size_t)cell * C);
    v.w = sAg[cell];
    return v;
  };
  double s = 0.0;
#pragma unroll 1
  for (int cell = lo + (warp - w0) * 32 + lane; cell < hi; cell += (kPW - w0) * 32) {
    const int y = cell / W, x = cell - y * W;
    if (ssim_interior(y, x, H, W)) s += ssim_cell(state, tgt, y, x, W, H * W);
  }
  s = warp_sum_f64(s);
  if (lane == 0) reinterpret_cast<double*>(sY + warp * kTile)[4] = s;
}
__device__ __forceinline__ void rep_ssim_flush(const float* sY, int w0, double* dst) {
  double s = 0.0;
  for (int w = w0; w < kPW; ++w) s += reinterpret_cast<const double*>(sY + w * 3 * 16 * 8)[4];
  *dst = s;
}

// the target sample b is measured against: M.target, or its model's with per-model targets (R.target_stride)
__device__ __forceinline__ const float* rep_met_target(const RepArgs& R, const FrameMetrics& M, int b) {
  return R.target_stride ? M.target + (size_t)(b / R.model_per) * R.target_stride : M.target;
}

// a whole frame's metrics (SS: and SSIM, into *ss_dst) by all warps, outside the tile phase of a step
template <bool SS>
__device__ __forceinline__ void rep_met_frame(const FrameMetrics& M, const float* tgt, const float* sX, const float* sAg,
                                              float* sY, int lo, int hi, int HW, float thr, double* dst, double* ss_dst,
                                              int H, int W) {
  rep_met_cells(M, tgt, sX, sAg, sY, lo, hi, HW, thr, 0);
  if constexpr (SS) rep_ssim_cells(sX, sAg, sY, tgt, lo, hi, H, W, 0);
  __syncthreads();
  if (threadIdx.x == 0) {
    rep_met_flush(sY, 0, dst);
    if constexpr (SS) rep_ssim_flush(sY, 0, ss_dst);
  }
  __syncthreads();
}

// ZP: zero-padded graph shift (the module default, graph_augmentation.py:85-92): senders (y - dy, x) -- the reference's
// _shift2d_pad slices the x padding away again, so dx is a no-op -- and per-sample softmax weights over the k offsets
// (graph_augmentation.py:114,136-154), recomputed from the resident state at the top of every step.  A separate
// instantiation: the torus kernel (trainer, bench) is compiled exactly as before.
// Z (ZP with records only, else unused): the softmax weights and row sums of every message step, for k_rep_bwd.
// MET (gnca_rollout_metrics): at every step t % M.every == 0 each CTA reduces the cells it stores for the history,
// [my_lo, my_hi), against M.target and writes one partial per (frame, sample, rank); M is unused otherwise.  With
// R.target_stride (a stack with per-model targets) each reduction reads sample b's model's target (rep_met_target).
// SS (with MET, gnca_rollout_metrics_ssim): at the same steps each CTA also sums the SSIM of its interior cells among
// [my_lo, my_hi) into ssim_part[frame][b][rank]; ssim_part is unused otherwise.
template <int C, bool ZP, bool MET, bool SS>
__global__ void __launch_bounds__(kPT, 1) k_rep_fwd(RepArgs R, Packed P, const float* __restrict__ packed, ZpRec Z,
                                                     FrameMetrics M, double* ssim_part) {
  static_assert(MET || !SS, "SSIM rides on the metrics steps");
  static_assert(C == 16, "lane mapping: 2 cells x 16 channels per warp row");
  constexpr int C3 = 3 * C, HID = 128;
  constexpr int CPL = 32 / C;                    // cells per lane row (2)
  cg::cluster_group cluster = cg::this_cluster();
  const StepArgs& a = R.s;
  const int NC = R.NC;
  const int rank = (int)cluster.block_rank();
  const int b = blockIdx.x / NC;
  const int H = a.H, W = a.W, HW = H * W, HWp = R.HWp;
  const int NQ = HW >> 2;                        // quads of 4 consecutive cells (W % 4 == 0: a quad never straddles rows)
  const int NW = (HW + 31) >> 5;                 // 32-bit words of a linear cell bitmap
  const bool graph = (a.flags & GNCA_F_GRAPH) != 0;
  const bool gn = (a.flags & GNCA_F_GROUPNORM) != 0;
  const bool a2a = (a.flags & GNCA_F_ALIVE_TO_ALIVE) != 0;
  const int c_lo = ((a.flags & GNCA_F_HIDDEN_ONLY) && C >= 4) ? 4 : 0;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int hwi = lane / C, c = lane % C;
  const int k = a.k, KP = R.KP, lkp = (R.KP == 16) ? 4 : 3;
  const int lnc = NC == 8 ? 3 : NC == 4 ? 2 : NC == 2 ? 1 : 0;
  const float thr = a.alpha_thr, gthr = a.graph_alpha_thr;
  const bool fast_alive = (thr >= 0.f) && (gthr == thr);
  // From step 1 on, a cell that is not post-alive has alpha == 0 exactly (the gate), an inactive cell moves by at most
  // update_gain, and only alive cells are active: with update_gain <= alpha_thr a cell outside dilate(alive(t)) cannot be
  // alive at t+1, so its fire bit is never read and its Philox draw can be skipped.
  const bool sparse_fire = fast_alive && a.update_gain <= thr && a.update_gain >= 0.f;

  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* sW1T = reinterpret_cast<float*>(smem_raw);           // [3C][HID] hidden index permuted: lane l owns 4l..4l+3
  float* sb1 = sW1T + C3 * HID;                               // [HID] same permutation
  float* sW2P = sb1 + HID;                                    // [HID][kW2S] W2^T rows (true hidden index), padded
  float* sX = sW2P + HID * kW2S;                              // [HW][C] state, cell-major (slot 3 unused: alpha planes)
  float* sAg = sX + (size_t)HW * C;                           // [HWp] alpha of x_t (gated)
  float* sAt = sAg + HWp;                                     // [HWp] updated alpha before the post-alive gate
  float* sY = sAt + HWp;                                      // [kPW][3C][8] per-warp perception tile
  float* sU = sY + kPW * C3 * 8;                              // [ucap][C] masked pre-norm update of MY active cells
  short* sq = reinterpret_cast<short*>(sU + (size_t)R.ucap * C);            // [kPW][8][16] sender cell or -1
  unsigned short* s_list = reinterpret_cast<unsigned short*>(sq + kPW * 8 * 16);   // [listcap] (y<<8|x) of my cells

  // linear cell bitmaps (bit = cell index); bits >= HW are always 0
  __shared__ uint32_t s_bAlive[kMaxWords], s_bAliveS2[kMaxWords], s_bAct[kMaxWords], s_bRaw[kMaxWords], s_bRawB[kMaxWords],
      s_bRaw2B[kMaxWords];
  __shared__ uint32_t s_bFire[2][kMaxWords];
  __shared__ __align__(16) int s_wtot[kPW];
  __shared__ int s_ctr;
  __shared__ __align__(8) unsigned long long s_mbar[2];      // A: statistics of the peers, B: updated cells of the peers
  __shared__ float s_parts[2][8][2];
  __shared__ float s_wred[kPW][2];
  __shared__ __align__(16) float s_aff[3][C];                 // per-channel scale, bias, idle update of the step
  __shared__ float s_astab[17];                               // n * (1/k) summed sequentially (same as the streaming path)
  __shared__ float s_fr[2], s_gain[2];
  __shared__ signed char s_off[2][2 * 16];
  __shared__ unsigned long long s_dbg[24];
  if (tid < 24) s_dbg[tid] = 0;

  // ---- weights -> smem (the only reads of `packed`) -------------------------------------------------------------
  if (R.model_stride) packed += (size_t)(b / R.model_per) * R.model_stride;
#pragma unroll 1
  for (int i = tid; i < C3 * HID; i += kPT) {
    const int kk = i / HID, jp = i - kk * HID;                 // jp = l*4 + jj  <->  true unit l + 32*jj
    const int l = jp >> 2, jj = jp & 3;
    sW1T[i] = packed[P.w1t + kk * HID + (l + 32 * jj)];
  }
  if (tid < HID) { const int l = tid >> 2, jj = tid & 3; sb1[tid] = packed[P.b1 + l + 32 * jj]; }
#pragma unroll 1
  for (int i = tid; i < HID * C; i += kPT) { const int j = i / C, cc = i - j * C; sW2P[j * kW2S + cc] = packed[P.w2t + i]; }
  __shared__ __align__(16) float s_wm[C][C + 4];                // Wm rows (registers are the scarce resource of this kernel)
  __shared__ float s_gbb[3][C];                                  // gamma, beta, bm (registers are scarce)
#pragma unroll
  for (int ci = 0; ci < C; ++ci) if (tid < C) s_wm[tid][ci] = graph ? packed[P.wm + tid * C + ci] : 0.f;
  if (tid < C) { s_gbb[0][tid] = packed[P.gamma + tid]; s_gbb[1][tid] = packed[P.beta + tid]; s_gbb[2][tid] = graph ? packed[P.bm + tid] : 0.f; }
  const float wuni = k > 0 ? 1.0f / (float)k : 0.f;
  if (tid == 0) { float as = 0.f; for (int n = 0; n <= 16; ++n) { s_astab[n] = as; as += wuni; } }
  // zero-padded shift: row sums of the state, pooled query / keys, softmax weights of the step
  constexpr int kZD = ZP ? 32 : 1;                              // d_model <= 32
  __shared__ float s_rowsum[ZP ? C : 1][ZP ? kMaxRows : 1];
  __shared__ float s_zq[2][kZD][ZP ? C : 1];                    // Wq, Wk
  __shared__ float s_zb[3][kZD];                                // bq, bk, (pooled query)
  __shared__ float s_w[16];                                     // attention weight of offset i at this step
  __shared__ float s_zscale;
  const int zd = ZP ? R.zd : 0;
  if constexpr (ZP) {
    for (int i = tid; i < zd * C; i += kPT) { s_zq[0][i / C][i % C] = packed[P.wq + i]; s_zq[1][i / C][i % C] = packed[P.wk + i]; }
    if (tid < zd) { s_zb[0][tid] = packed[P.bq + tid]; s_zb[1][tid] = packed[P.bk + tid]; }
    if (tid == 0) s_zscale = fabsf(packed[P.scaling]) + 1e-6f;
  }
  const size_t sample_off = (size_t)b * C * HW;
  // global [C][HW] <-> smem [cell][C]; lanes = 8 cells x 4 channels (32 B global sectors, 4-way smem conflict)
  auto store_item = [&](float* dst, int lo, int hi, int i) {
    const int ci = i & 7, c4 = (i >> 3) & 3, rest = i >> 5;
    const int cq = rest & 3, cgp = rest >> 2;
    const int cell = lo + cgp * 8 + ci, ch = cq * 4 + c4;
    if (cell < hi) dst[(size_t)ch * HW + cell] = (ch == 3) ? sAg[cell] : sX[cell * C + ch];
  };
  auto store_state = [&](float* dst, int lo, int hi) {       // cells [lo, hi) of x_t -> global [C][HW]
    const int n = (hi - lo + 7) & ~7;
#pragma unroll 1
    for (int i = tid; i < n * C; i += kPT) store_item(dst, lo, hi, i);
  };
  auto hist_at = [&](int t) -> float* {                       // history slot of x_t, or null when step t is not kept
    if (!R.hist || t % R.hist_every != 0) return nullptr;
    return R.hist + (size_t)(t / R.hist_every) * a.B * C * HW + sample_off;
  };
  {
    const int n8 = (HW + 7) & ~7;
#pragma unroll 1
    for (int i = tid; i < n8 * C; i += kPT) {
      const int ci = i & 7, c4 = (i >> 3) & 3, rest = i >> 5;
      const int cq = rest & 3, cgp = rest >> 2;
      const int cell = cgp * 8 + ci, ch = cq * 4 + c4;
      if (cell < HW) {
        const float v = R.x0[sample_off + (size_t)ch * HW + cell];
        if (ch == 3) sAg[cell] = v; else sX[cell * C + ch] = v;
      }
    }
  }
  const int my_lo = (HW * rank) >> lnc, my_hi = (HW * (rank + 1)) >> lnc;
  const int hist_items = ((my_hi - my_lo + 7) & ~7) * C;
  const int n_fire_tasks = (NQ + 31) >> 5, n_hist_tasks = R.hist ? (hist_items + 255) >> 8 : 0;
  // frame metrics: the partial of this CTA's cells of frame t goes to part[frame][b][rank]
  double* met_dst = MET ? M.part + ((size_t)b * NC + rank) * 4 : nullptr;
  const size_t met_frame_stride = MET ? (size_t)a.B * NC * 4 : 0;
  // ---- schedule: registers hold step t+2 while step t runs; smem buffers hold t and t+1 ---------------------
  float nx_fr = 0.f, nx_gain = 0.f;
  signed char nx_off = 0;
  auto sched_fetch = [&](int tn) {
    if (tn < R.T) {
      if (tid == 0) { nx_fr = a.fire_rate_dev[tn]; nx_gain = graph ? a.message_gain_dev[tn] : 0.f; }
      if (tid >= 32 && tid < 32 + 2 * k) nx_off = a.offsets_dev[(size_t)tn * k * 2 + (tid - 32)];
    }
  };
  auto sched_commit = [&](int buf) {
    if (tid == 0) { s_fr[buf] = nx_fr; s_gain[buf] = nx_gain; }
    if (tid >= 32 && tid < 32 + 2 * k) s_off[buf][tid - 32] = nx_off;
  };
  // fire bits of 32 consecutive quads of step tn (fire_rate in s_fr[buf]) -> s_bFire[buf]  (ncagraph.py:144-146: u <= fr)
  // `sparse`: the caller guarantees that a cell outside the 3x3 dilation of the CURRENT alive bitmap cannot be alive at
  // step tn (see sparse_fire below); a task none of whose cells is near an alive cell just writes zero words.
  auto fire_task = [&](int task, int tn, int buf, bool sparse) {
    if (sparse) {
      const int c0 = task * 128 - W - 1, c1 = task * 128 + 127 + W + 1;          // cells whose alive bit can matter
      const int w0 = max(c0, 0) >> 5, w1 = min(c1, HW - 1) >> 5;
      uint32_t any = 0;
      for (int w = w0 + lane; w <= w1; w += 32) any |= s_bAlive[w];
      if (!__any_sync(0xffffffffu, any != 0)) {
        const int q = task * 32 + lane;
        if ((lane & 7) == 0) s_bFire[buf][q >> 3] = 0u;
        return;
      }
    }
    const float frn = s_fr[buf];
    const int q = task * 32 + lane, qq = min(q, NQ - 1);     // every lane computes (clamped): no divergence before the shuffles
    uint32_t nib;
    if (frn >= 1.0f) {
      nib = 15u;
    } else if (R.fire_u_base) {
      const float4 u = __ldg(reinterpret_cast<const float4*>(R.fire_u_base + ((size_t)tn * a.B + b) * HW) + qq);
      nib = (u.x <= frn ? 1u : 0u) | (u.y <= frn ? 2u : 0u) | (u.z <= frn ? 4u : 0u) | (u.w <= frn ? 8u : 0u);
    } else {
      const uint64_t blk = ((((uint64_t)tn * a.B + b) * (uint64_t)HW) >> 2) + qq + a.philox_offset;
      const uint4 r = philox4x32_10(make_uint4((uint32_t)blk, (uint32_t)(blk >> 32), 0u, 0u),
                                    make_uint2((uint32_t)a.philox_seed, (uint32_t)(a.philox_seed >> 32)));
      const float s24 = 1.0f / 16777216.0f;
      nib = ((float)(r.x >> 8) * s24 <= frn ? 1u : 0u) | ((float)(r.y >> 8) * s24 <= frn ? 2u : 0u) |
            ((float)(r.z >> 8) * s24 <= frn ? 4u : 0u) | ((float)(r.w >> 8) * s24 <= frn ? 8u : 0u);
    }
    nib = (q < NQ) ? nib : 0u;
    const uint32_t w = pack_nibbles(nib, lane);
    if ((lane & 7) == 0) s_bFire[buf][q >> 3] = w;
  };
  // ---- masks: one quad of 4 consecutive cells per thread (static), linear bitmaps in smem --------------------------
  const int q = tid, qcell = 4 * tid;
  const bool qv = q < NQ;
  const int qy = qcell / W, qx0 = qcell - qy * W;
  const bool firstcol = qx0 == 0, lastcol = qx0 + 4 == W;
  const int qsh = 4 * (lane & 7), qword = q >> 3;
  // Lanes without a quad must not branch differently from their warp in front of the packing shuffles (a diverged
  // __shfl_sync takes the BRA.DIV slow path: ~2k cycles per step for the half-valid warp).  They LOAD quad ql and
  // STORE to a scratch quad behind the planes (the planes are padded), and their bits are masked with vmask.
  const int QP = (NQ + 31) & ~31;
  const int ql = min(q, QP - 1), qs = qv ? q : QP, qwordc = min(qword, NW - 1);
  const uint32_t vmask = qv ? 15u : 0u;
  uint32_t* s_bAliveS = fast_alive ? s_bAlive : s_bAliveS2;
  auto nib_gt = [&](const float4& v, float th) -> uint32_t {
    return (v.x > th ? 1u : 0u) | (v.y > th ? 2u : 0u) | (v.z > th ? 4u : 0u) | (v.w > th ? 8u : 0u);
  };
  auto pack_store = [&](uint32_t* arr, uint32_t nib) -> uint32_t {      // returns the packed word of my 8-lane group
    const uint32_t w = pack_nibbles(nib, lane);
    if ((lane & 7) == 0) arr[qword] = w;            // qword < kMaxWords always; words >= NW are never read
    return w;
  };
  // bits [start, start+6) of a bitmap (zero outside the grid); branch-free (start >= -1)
  auto field6 = [&](const uint32_t* bm, int start) -> uint32_t {
    const int s0 = max(start, 0), w = s0 >> 5;
    const uint32_t lo = bm[w], hi = bm[min(w + 1, NW - 1)];
    uint32_t f = __funnelshift_r(lo, (w + 1 < NW) ? hi : 0u, s0 & 31);
    f = (start < 0) ? (f << 1) : f;
    return f & 63u;
  };
  // 3x3 dilation of a thresholded plane == (max_pool2d(alpha,3,1,1) > thr) (nca.py:55-62; out-of-grid = -inf): my 4 cells
  const int qcc = qv ? qcell : 0;              // lanes without a quad compute on cell 0 and discard (no divergence)
  const int st_up = (qv && qy > 0) ? qcc - W - 1 : 0, st_dn = (qv && qy < H - 1) ? qcc + W - 1 : 0;
  const uint32_t m_up = (qv && qy > 0) ? 63u : 0u, m_dn = (qv && qy < H - 1) ? 63u : 0u;
  const uint32_t m_mid = qv ? (63u & ~(firstcol ? 1u : 0u) & ~(lastcol ? 32u : 0u)) : 0u;
  auto dil = [&](const uint32_t* bm) -> uint32_t {
    uint32_t f = field6(bm, qcc - 1) | (field6(bm, st_up) & m_up) | (field6(bm, st_dn) & m_dn);
    f &= m_mid;
    return ((f | (f >> 1) | (f << 1)) >> 1) & 15u;
  };
  // active = alive & fire of my quad; packed words + counts: in-warp exclusive prefix of my word, warp total -> smem
  uint32_t r_actnib = 0, r_actword = 0;
  int r_pre = 0;
  auto act_count = [&](uint32_t alive_nib, int firebuf) {
    const uint32_t fw = s_bFire[firebuf][qwordc];
    const uint32_t fire_nib = (fw >> qsh) & vmask;
    r_actnib = alive_nib & fire_nib;
    r_actword = pack_store(s_bAct, r_actnib);
    const int cnt = __popc(r_actword);
    const int c0 = __shfl_sync(0xffffffffu, cnt, 0), c1 = __shfl_sync(0xffffffffu, cnt, 8),
              c2 = __shfl_sync(0xffffffffu, cnt, 16), c3 = __shfl_sync(0xffffffffu, cnt, 24);
    const int g = lane >> 3;
    r_pre = (g > 0 ? c0 : 0) + (g > 1 ? c1 : 0) + (g > 2 ? c2 : 0);
    if (lane == 0) s_wtot[warp] = c0 + c1 + c2 + c3;
  };
  // balanced list of MY share of the active cells (slot order = cell order, deterministic)
  int n_my = 0, nact = 0, lo_my = 0;
  auto list_pass = [&]() {
    int base = 0, tot = 0;
#pragma unroll
    for (int w4 = 0; w4 < kPW / 4; ++w4) {
      const int4 v = *reinterpret_cast<const int4*>(&s_wtot[4 * w4]);
      const int vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) { base += (4 * w4 + j < warp) ? vv[j] : 0; tot += vv[j]; }
    }
    nact = tot;
    const int lo = (tot * rank) >> lnc, hi = (tot * (rank + 1)) >> lnc;
    n_my = hi - lo;
    lo_my = lo;
    if (r_actnib) {
      int slot = base + r_pre + __popc(r_actword & ((1u << qsh) - 1u));
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (r_actnib & (1u << j)) {
          if (slot >= lo && slot < hi) s_list[slot - lo] = (unsigned short)((qy << 8) | (qx0 + j));
          ++slot;
        }
      }
    }
    if (tid == 0) s_ctr = 0;
  };
  // alive / sender-alive / active bitmaps and my list from thresholded bitmaps of the gated alpha   [2 barriers]
  auto alive_from_raw = [&](const uint32_t* raw1, const uint32_t* raw2, int firebuf) {
    const uint32_t al = dil(raw1);
    pack_store(s_bAlive, al);
    if (!fast_alive) pack_store(s_bAliveS2, dil(raw2));
    act_count(al, firebuf);
    __syncthreads();
    list_pass();
    __syncthreads();
  };
  // everything step tn needs from the CURRENT state (alpha in sAg)   [3 barriers]
  auto prepare_from_state = [&](int tn) {
    const float4 v = reinterpret_cast<const float4*>(sAg)[ql];
    pack_store(s_bRawB, nib_gt(v, thr) & vmask);
    if (!fast_alive) pack_store(s_bRaw2B, nib_gt(v, gthr) & vmask);
    __syncthreads();
    alive_from_raw(s_bRawB, s_bRaw2B, tn & 1);
  };

  sched_fetch(0);
  sched_commit(0);
  sched_fetch(1);
  sched_commit(1);
  sched_fetch(2);
  __syncthreads();
  if (R.T > 0) for (int task = warp; task < n_fire_tasks; task += kPW) fire_task(task, 0, 0, false);
  __syncthreads();
  prepare_from_state(0);

  const uint32_t mbarA = smem_u32(&s_mbar[0]), mbarB = smem_u32(&s_mbar[1]);
  const bool use_async = R.use_async != 0 && NC > 1;
  if (tid == 0) {
    mbar_init(mbarA, 1);
    mbar_init(mbarB, 1);
    mbar_init_fence();
  }
  cluster_arrive(); cluster_wait();              // every replica initialised before any remote store

  const int my_steps = a.steps ? min(a.steps[b] - R.t0, R.T) : R.T;
  long long t_prev = clock64();
  float* myY = sY + warp * (C3 * 8);
  short* myq = sq + warp * (8 * 16);

  for (int t = 0; t < R.T; ++t) {
    const int cur = t & 1;
    if (R.damage.p && t == R.damage_step) {      // multiplicative damage on every replica (utils/damage.py masks)
      const int n8 = (HW + 7) & ~7;
#pragma unroll 1
      for (int i = tid; i < n8 * C; i += kPT) {
        const int ci = i & 7, c4 = (i >> 3) & 3, rest = i >> 5;
        const int cq = rest & 3, cgp = rest >> 2;
        const int cell = cgp * 8 + ci, ch = cq * 4 + c4;
        if (cell < HW) {
          const float d = R.damage.at(b, ch, cell, C, HW);
          if (ch == 3) sAg[cell] *= d; else sX[cell * C + ch] *= d;
        }
      }
      __syncthreads();
      prepare_from_state(t);
    }
    if (t >= my_steps) {                         // frozen sample (whole cluster agrees): state passes through
      if (float* h = hist_at(t)) store_state(h, my_lo, my_hi);
      if constexpr (MET)
        if (t % M.every == 0)
          rep_met_frame<SS>(M, rep_met_target(R, M, b), sX, sAg, sY, my_lo, my_hi, HW, a.alpha_thr,
                            met_dst + (t / M.every) * met_frame_stride,
                            ssim_part + ((size_t)(t / M.every) * a.B + b) * NC + rank, H, W);
      continue;
    }
    const float gain_m = s_gain[cur];
    const bool msg_on = graph && gain_m != 0.f && k > 0;
    if constexpr (ZP) {
      if (msg_on) {
        // per-(channel, row) sums of x_t from my replica (every CTA computes all of them: 25.6 k adds, no exchange)
        for (int row = warp; row < H; row += kPW) {               // warp per row, lane = (cell parity, channel): 128-byte loads
          const int c = lane & 15, hw = lane >> 4;
          const float* p = (c == 3) ? (sAg + row * W) : (sX + (size_t)row * W * C + c);
          const int st = (c == 3) ? 1 : C;
          float s0 = 0.f, s1 = 0.f;                              // W % 4 == 0: cells hw, hw+2, hw+4, ... in two chains
          for (int x = hw; x < W; x += 4) { s0 += p[x * st]; s1 += p[(x + 2) * st]; }
          float sv = s0 + s1;
          sv += __shfl_xor_sync(0xffffffffu, sv, 16);
          if (lane < C) s_rowsum[c][row] = sv;
        }
        __syncthreads();
        // one warp per offset (k <= 16 = the warps of the CTA): lanes c < C sum the kept rows, lane j forms its component
        // of the pooled query (recomputed by every warp: 16 FMAs) and of the mean shifted key, one shuffle tree per offset
        if (warp < k) {
          const float invHW = 1.0f / (float)HW;
          float xs_all = 0.f, ss = 0.f;
          const int dy = (int)s_off[cur][2 * warp];
          const int lo = max(0, -dy), hi = min(H, H - dy), nrows = max(0, hi - lo);
          if (lane < C) {
            for (int y = 0; y < H; ++y) xs_all += s_rowsum[lane][y];                 // pooled query (:114)
            for (int y = lo; y < hi; ++y) ss += s_rowsum[lane][y];                   // dy-shifted, zero-filled K (:126,136-138)
          }
          float qp = 0.f, kp = 0.f;
#pragma unroll
          for (int c = 0; c < C; ++c) {
            const float xm = __shfl_sync(0xffffffffu, xs_all, c) * invHW, sc = __shfl_sync(0xffffffffu, ss, c);
            if (lane < zd) { qp = fmaf(s_zq[0][lane][c], xm, qp); kp = fmaf(s_zq[1][lane][c], sc, kp); }
          }
          float li = 0.f;
          if (lane < zd) {
            qp += s_zb[0][lane];
            kp = (kp + (float)nrows * (float)W * s_zb[1][lane]) * invHW;
            li = qp * kp;
          }
          li = warp_sum(li);
          if (lane == 0) s_w[warp] = li;                         // logit of offset `warp`
        }
        __syncthreads();
        if (warp == 0) {                                         // softmax over the k offsets (:150-154)
          const float logit = lane < k ? s_w[lane] : -INFINITY;
          float mx = logit;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
          const float e = lane < k ? expf((logit - mx) / s_zscale) : 0.f;
          const float se = warp_sum(e);
          __syncwarp();
          if (lane < 16) s_w[lane] = lane < k ? e / se : 0.f;
        }
        __syncthreads();
        if (Z.w && rank == 0) {                                  // what the attention backward of this step reads
          if (tid < 16) Z.w[((size_t)t * a.B + b) * 16 + tid] = s_w[tid];
          float* zr = Z.rowsum + ((size_t)t * a.B + b) * C * H;
          for (int i = tid; i < C * H; i += kPT) zr[i] = s_rowsum[i / H][i - (i / H) * H];
        }
      }
    }
    REP_MARK(0);
    if (R.dbg && tid == 0) s_dbg[8] += n_my;
    if (R.masks && rank == 0 && tid < NW) {
      uint32_t* mk = R.masks + ((size_t)t * a.B + b) * 3 * kMaskWords;
      mk[tid] = s_bAliveS[tid];
      mk[kMaskWords + tid] = s_bAct[tid];
    }

    // ---- S2: warp-autonomous tiles of G cells; then the side jobs of the step (fire bits of step t+1, BPTT
    //      history of x_t) handed out in chunks by a shared counter, so the warps without a tile take them ----------
    float ps1 = 0.f, ps2 = 0.f;
    auto run_tile = [&](auto gtag, const int slot0, const int lim) {      // cells [slot0, min(slot0 + G, lim)) of my list
      constexpr int G = decltype(gtag)::value;
      constexpr int MPL = G / CPL;                         // cells per lane
      {
        // 2a: sender table of the tile: (cell, offset) -> sender cell index or -1   (graph_augmentation.py:94-97,116-133)
        if (msg_on) {
          for (int p = lane; p < G * KP; p += 32) {
            const int m = p >> lkp, i = p & (KP - 1);
            short q = -1;
            if (i < k) {
              const unsigned ent = s_list[min(slot0 + m, lim - 1)];
              int qy = (int)(ent >> 8) - (int)s_off[cur][2 * i], qx = (int)(ent & 255u) - (int)s_off[cur][2 * i + 1];
              bool inside = true;
              if constexpr (ZP) {
                qx = (int)(ent & 255u);                          // dx is a no-op in the reference's zero-padded shift
                inside = qy >= 0 && qy < H;
                qy = inside ? qy : 0;
              } else {
                qy += qy < 0 ? H : 0; qy -= qy >= H ? H : 0;
                qx += qx < 0 ? W : 0; qx -= qx >= W ? W : 0;
              }
              const int qc = qy * W + qx;
              if (inside && (!a2a || ((s_bAliveS[qc >> 5] >> (qc & 31)) & 1u))) q = (short)qc;
            }
            myq[m * KP + i] = q;
          }
          __syncwarp();
        }
        REP_MARK(13);
        // 2b: perception (perception.py:9-26, zero halo) + gathered sender state, lane = (cell hwi+2r, channel c)
        float xs[MPL], asv[MPL], msg[MPL];
        const bool isA = (c == 3);
        const float* pb = isA ? sAg : (sX + c);
        const int st = isA ? 1 : C;
#pragma unroll
        for (int r = 0; r < MPL; ++r) {
          const int m = hwi + CPL * r;
          const unsigned ent = s_list[min(slot0 + m, lim - 1)];
          const int y = (int)(ent >> 8), x = (int)(ent & 255u);
          const float* p = pb + (y * W + x) * st;
          const bool up = y > 0, dn = y < H - 1, lf = x > 0, rt = x < W - 1;
          const float a00 = (up && lf) ? p[(-W - 1) * st] : 0.f, a01 = up ? p[-W * st] : 0.f,
                      a02 = (up && rt) ? p[(-W + 1) * st] : 0.f;
          const float a10 = lf ? p[-st] : 0.f, a12 = rt ? p[st] : 0.f;
          const float a20 = (dn && lf) ? p[(W - 1) * st] : 0.f, a21 = dn ? p[W * st] : 0.f,
                      a22 = (dn && rt) ? p[(W + 1) * st] : 0.f;
          const float v_id = p[0];
          myY[c * G + m] = v_id;
          myY[(C + c) * G + m] = (a00 - a02) + 2.f * (a10 - a12) + (a20 - a22);
          myY[(2 * C + c) * G + m] = (a00 + 2.f * a01 + a02) - (a20 + 2.f * a21 + a22);
          float xsv = 0.f, as = 0.f;
          if (msg_on) {
            int nv = 0;
            const short* qrow = myq + m * KP;
            for (int o8 = 0; o8 < KP; o8 += 8) {
              const int4 qq = *reinterpret_cast<const int4*>(qrow + o8);
              const int qs[8] = {(short)(qq.x & 0xffff), qq.x >> 16, (short)(qq.y & 0xffff), qq.y >> 16,
                                 (short)(qq.z & 0xffff), qq.z >> 16, (short)(qq.w & 0xffff), qq.w >> 16};
              float vq[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) vq[j] = pb[max(qs[j], 0) * st];
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                if constexpr (ZP) {
                  const float wj = qs[j] >= 0 ? s_w[o8 + j] : 0.f;
                  xsv = fmaf(wj, vq[j], xsv);
                  as += wj;
                } else {
                  xsv = fmaf(qs[j] >= 0 ? wuni : 0.f, vq[j], xsv);
                  nv += qs[j] >= 0;
                }
              }
            }
            if constexpr (!ZP) as = s_astab[nv];
          }
          xs[r] = xsv; asv[r] = as;
          if (R.rec && slot0 + m < lim) {          // forward half of the record (gnca_rep.h): y | u | xs | tanh(agg) | as
            float* rc = R.rec + (((size_t)t * a.B + b) * HW + (size_t)(lo_my + slot0 + m)) * kRecStride;
            rc[c] = v_id; rc[C + c] = myY[(C + c) * G + m]; rc[2 * C + c] = myY[(2 * C + c) * G + m];
            rc[kRecXs + c] = xsv;
            if (c == 0) rc[kRecAs] = as;
          }
        }
        REP_MARK(14);
        // 2c: message projection + channel policy (ncagraph.py:94-104,141): lane's row of Wm in registers
#pragma unroll
        for (int r = 0; r < MPL; ++r) {
          float mval = 0.f;
          if (msg_on) {
            float agg = s_gbb[2][c] * asv[r];
#pragma unroll
            for (int c4 = 0; c4 < C / 4; ++c4) {
              const float4 w4 = *reinterpret_cast<const float4*>(&s_wm[c][4 * c4]);
              agg = fmaf(w4.x, __shfl_sync(0xffffffffu, xs[r], (lane & 16) | (4 * c4)), agg);
              agg = fmaf(w4.y, __shfl_sync(0xffffffffu, xs[r], (lane & 16) | (4 * c4 + 1)), agg);
              agg = fmaf(w4.z, __shfl_sync(0xffffffffu, xs[r], (lane & 16) | (4 * c4 + 2)), agg);
              agg = fmaf(w4.w, __shfl_sync(0xffffffffu, xs[r], (lane & 16) | (4 * c4 + 3)), agg);
            }
            const float th = tanhf(agg);
            if (c >= c_lo) mval = th * gain_m;
            if (R.rec && slot0 + hwi + CPL * r < lim)
              R.rec[(((size_t)t * a.B + b) * HW + (size_t)(lo_my + slot0 + hwi + CPL * r)) * kRecStride + kRecTh + c] = th;
          }
          msg[r] = mval;
        }
        __syncwarp();
        REP_MARK(15);
        // 2d: layer 1, lane = 4 hidden units (permuted), G cells: broadcast y, per-lane w
        float acc[G][4];
        {
          const float4 bb = *reinterpret_cast<const float4*>(sb1 + 4 * lane);
#pragma unroll
          for (int m = 0; m < G; ++m) { acc[m][0] = bb.x; acc[m][1] = bb.y; acc[m][2] = bb.z; acc[m][3] = bb.w; }
#pragma unroll 8
          for (int kk = 0; kk < C3; ++kk) {
            const float4 w = *reinterpret_cast<const float4*>(sW1T + kk * HID + 4 * lane);
            float ym[G];
            if constexpr (G == 2) {
              const float2 yv = *reinterpret_cast<const float2*>(myY + kk * G);
              ym[0] = yv.x; ym[1] = yv.y;
            } else {
#pragma unroll
              for (int m4 = 0; m4 < G / 4; ++m4) {
                const float4 yv = *reinterpret_cast<const float4*>(myY + kk * G + 4 * m4);
                ym[4 * m4] = yv.x; ym[4 * m4 + 1] = yv.y; ym[4 * m4 + 2] = yv.z; ym[4 * m4 + 3] = yv.w;
              }
            }
#pragma unroll
            for (int m = 0; m < G; ++m) {
              acc[m][0] = fmaf(ym[m], w.x, acc[m][0]); acc[m][1] = fmaf(ym[m], w.y, acc[m][1]);
              acc[m][2] = fmaf(ym[m], w.z, acc[m][2]); acc[m][3] = fmaf(ym[m], w.w, acc[m][3]);
            }
          }
        }
        REP_MARK(16);
        // 2e: layer 2: per-lane partial over its 4 hidden units, then a shuffle reduce-scatter that leaves
        //     (cell hwi+2e of the half, channel c) in this lane -- the same ownership as the message.
        constexpr int GB = G < 4 ? G : 4;                  // cells per reduce-scatter block
        constexpr int NPV = GB * C;                          // partial sums per lane and block
#pragma unroll
        for (int blk = 0; blk < G / GB; ++blk) {
          float pv[NPV];
#pragma unroll
          for (int i = 0; i < NPV; ++i) pv[i] = 0.f;
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const float* w2row = sW2P + (lane + 32 * jj) * kW2S;
            float hm[GB];
#pragma unroll
            for (int m = 0; m < GB; ++m) hm[m] = fmaxf(acc[GB * blk + m][jj], 0.f);
#pragma unroll
            for (int c4 = 0; c4 < C / 4; ++c4) {
              const float4 w = *reinterpret_cast<const float4*>(w2row + 4 * c4);
              const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
              for (int m = 0; m < GB; ++m)
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                  const int idx = (m & 1) * (NPV / 2) + (4 * c4 + cc) * (GB / 2) + (m >> 1);
                  pv[idx] = fmaf(hm[m], wv[cc], pv[idx]);
                }
            }
          }
#define REP_RS_STAGE(N2, SH)                                                          \
          {                                                                           \
            const bool upper = (lane & SH) != 0;                                      \
            _Pragma("unroll") for (int i = 0; i < (N2); ++i) {                        \
              const float send = upper ? pv[i] : pv[i + (N2)];                        \
              const float keep = upper ? pv[i + (N2)] : pv[i];                        \
              pv[i] = keep + __shfl_xor_sync(0xffffffffu, send, SH);                  \
            }                                                                         \
          }
          REP_RS_STAGE(NPV / 2, 16) REP_RS_STAGE(NPV / 4, 8) REP_RS_STAGE(NPV / 8, 4) REP_RS_STAGE(NPV / 16, 2)
          REP_RS_STAGE(NPV / 32, 1)
#undef REP_RS_STAGE
#pragma unroll
          for (int e = 0; e < GB / 2; ++e) {
            const int r = (GB / 2) * blk + e, m = hwi + CPL * r;
            const int slot = slot0 + m;
            if (slot < lim) {
              const float u = pv[e] + msg[r];
              if (R.rec) R.rec[(((size_t)t * a.B + b) * HW + (size_t)(lo_my + slot)) * kRecStride + kRecU + c] = u;
              float* dst = slot < R.ucap ? sU + slot * C + c
                                         : R.u_over + ((size_t)blockIdx.x * R.over_cap + (slot - R.ucap)) * C + c;
              *dst = u;
              if (R.u_hist) {
                const unsigned ent = s_list[slot];
                R.u_hist[(((size_t)t * a.B + b) * C + c) * HW + (ent >> 8) * W + (ent & 255u)] = u;
              }
              ps1 += u;
              ps2 = fmaf(u, u, ps2);
            }
          }
        }
        __syncwarp();
        REP_MARK(17);
      }
    };
    // tile size: as many warps as possible get a tile (latency), larger tiles amortise the weight reads (throughput)
    // Tile schedule.  Few cells (<= 64): tiles of 2 (<= 32 cells) or 4 handed out round-robin -- the phase is bound by
    // shared-memory weight reads + instruction issue, fewer/larger tiles cost fewer instructions, and the warps without a
    // tile do the side jobs meanwhile.  Many cells: every warp takes a contiguous, equally sized range and covers it with
    // tiles of 8 / 4 / 2 cells, so all warps finish together (17 round-robin tiles of 8 would mean two full rounds).
    static_assert(kPW == 16, "per-warp ranges");
    if (n_my <= 64) {
      if (n_my <= 32) {
#pragma unroll 1
        for (int s0 = 2 * warp; s0 < n_my; s0 += 2 * kPW) run_tile(std::integral_constant<int, 2>{}, s0, n_my);
      } else {
#pragma unroll 1
        for (int s0 = 4 * warp; s0 < n_my; s0 += 4 * kPW) run_tile(std::integral_constant<int, 4>{}, s0, n_my);
      }
    } else {
      const int w_lo = (n_my * warp) >> 4, w_hi = (n_my * (warp + 1)) >> 4;
#pragma unroll 1
      for (int s0 = w_lo; s0 < w_hi;) {
        const int rem = w_hi - s0;
        if (rem > 4) { run_tile(std::integral_constant<int, 8>{}, s0, w_hi); s0 += 8; }
        else if (rem > 2) { run_tile(std::integral_constant<int, 4>{}, s0, w_hi); s0 += 4; }
        else { run_tile(std::integral_constant<int, 2>{}, s0, w_hi); s0 += 2; }
      }
    }
    REP_MARK(9);
    // Side jobs of the step, statically spread over warps 1..15 (warp 0 runs the GroupNorm exchange).  The BPTT history
    // of x_t must be stored BEFORE my partial goes out (that message tells the peers they may overwrite x_t here); the
    // fire bits of step t+1 touch no state, so a warp that had a tile generates them in the shadow of the exchange.
    // the sparse-fire invariant (non-alive => alpha == 0) does not hold for the state a damage mask just produced: a cell
    // kept alive by a neighbour the mask killed still carries its alpha and can cross the threshold by the idle drift
    const bool dmg_now = R.damage.p && t == R.damage_step;
    auto side_jobs = [&](const bool fire, const bool hist) {
      const int nf = (t + 1 < R.T) ? n_fire_tasks : 0;
      float* hdst = hist_at(t);
      if (fire) {
#pragma unroll 1
        for (int task = kPW - 1 - warp; task < nf; task += kPW - 1) fire_task(task, t + 1, cur ^ 1, sparse_fire && t >= 1 && !dmg_now);
      }
      if (hist && hdst) {
#pragma unroll 1
        for (int task = warp - 1; task < n_hist_tasks; task += kPW - 1) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int i = task * 256 + j * 32 + lane;
            if (i < hist_items) store_item(hdst, my_lo, my_hi, i);
          }
        }
      }
      if constexpr (MET)
        if (hist && t % M.every == 0)
          rep_met_cells(M, rep_met_target(R, M, b), sX, sAg, sY, my_lo, my_hi, HW, a.alpha_thr, 1);
      if constexpr (SS)
        if (hist && t % M.every == 0) rep_ssim_cells(sX, sAg, sY, rep_met_target(R, M, b), my_lo, my_hi, H, W, 1);
    };
    const bool had_tile = n_my <= 32 ? (2 * warp < n_my) : n_my <= 64 ? (4 * warp < n_my) : (((n_my * warp) >> 4) < ((n_my * (warp + 1)) >> 4));
    const bool fire_early = !use_async || !had_tile;
    if (warp > 0) side_jobs(fire_early, true);
    REP_MARK(1);

    // ---- GroupNorm(1,C) partials (ncagraph.py:153): warp -> block -> every CTA of the cluster -------------------
    if (gn) {
      const float f1 = warp_sum(ps1), f2 = warp_sum(ps2);
      if (lane == 0) { s_wred[warp][0] = f1; s_wred[warp][1] = f2; }
    }
    __syncthreads();
    if constexpr (MET)
      if (tid == 32 && t % M.every == 0) {
        rep_met_flush(sY, 1, met_dst + (t / M.every) * met_frame_stride);
        if constexpr (SS) rep_ssim_flush(sY, 1, ssim_part + ((size_t)(t / M.every) * a.B + b) * NC + rank);
      }
    if (!use_async) {
      if (gn && warp == 0) {
        float t1 = lane < kPW ? s_wred[lane][0] : 0.f, t2 = lane < kPW ? s_wred[lane][1] : 0.f;
        t1 = warp_sum(t1); t2 = warp_sum(t2);
        if (lane < NC) {
          float* dst = cluster.map_shared_rank(&s_parts[cur][0][0], lane);
          dst[rank * 2] = t1; dst[rank * 2 + 1] = t2;
        }
      }
      REP_MARK(2);
      cluster_arrive();                                                       // ---- cluster barrier 1
      sched_commit(cur);                  // step t+2 -> the buffer step t no longer needs (visible after later barriers)
      sched_fetch(t + 3);
      cluster_wait();
    } else {
      // my partial -> every peer (8 bytes each, counted on the peer's mbarrier A); a peer's partial arriving here also
      // says that peer has finished reading x_t, so its cells may be overwritten once all of them are in
      if (warp == 0) {
        float t1 = lane < kPW ? s_wred[lane][0] : 0.f, t2 = lane < kPW ? s_wred[lane][1] : 0.f;
        t1 = warp_sum(t1); t2 = warp_sum(t2);
        if (lane == 0) mbar_expect_tx(mbarA, (uint32_t)(NC - 1) * 8u);
        if (lane == 0) { s_parts[cur][rank][0] = t1; s_parts[cur][rank][1] = t2; }
#pragma unroll
        for (int pr = 0; pr < 7; ++pr) {
          if (lane == pr + 1 && pr + 1 < NC) {
            const int peer = (rank + pr + 1) & (NC - 1);
            const uint32_t la = mapa_u32(smem_u32(&s_parts[cur][rank][0]), peer), lm = mapa_u32(mbarA, peer);
            st_async_f32(la, t1, lm);
            st_async_f32(la + 4, t2, lm);
          }
        }
      }
      REP_MARK(2);
      sched_commit(cur);
      sched_fetch(t + 3);
      if (warp > 0 && !fire_early) side_jobs(true, false);
      if (warp == 0) mbar_wait(mbarA, (uint32_t)(t & 1));
    }
    REP_MARK(3);

    // ---- S3: statistics (warp 0), idle update of all inactive cells (local), my active cells -> all replicas ------
    if (warp == 0 && lane < C) {
      float sc = 1.f, bi = 0.f, idle = 0.f;
      if (gn) {
        float t1 = 0.f, t2 = 0.f;
        for (int r = 0; r < NC; ++r) { t1 += s_parts[cur][r][0]; t2 += s_parts[cur][r][1]; }
        const float m_ = t1 * R.inv_n;
        const float var = fmaxf(fmaf(t2, R.inv_n, -m_ * m_), 0.f);
        const float r_ = 1.0f / sqrtf(var + a.gn_eps);
        sc = r_ * s_gbb[0][lane];             // lane == c for lanes < C
        bi = s_gbb[1][lane] - m_ * sc;
        idle = tanhf(bi) * a.update_gain;
        if (lane == 0 && rank == 0 && R.stats_hist) {
          R.stats_hist[((size_t)t * a.B + b) * 2] = m_;
          R.stats_hist[((size_t)t * a.B + b) * 2 + 1] = r_;
        }
      }
      s_aff[0][lane] = sc; s_aff[1][lane] = bi; s_aff[2][lane] = idle;
    }
    if (use_async && tid == 32) mbar_expect_tx(mbarB, (uint32_t)(nact - n_my) * (uint32_t)(C * 4));
    __syncthreads();
    REP_MARK(10);
    // (my active cells first: the pushes travel to the peers while everybody runs its local idle pass)
    {
      // my active cells: x + gain * tanh(gn(u)); written into every replica (alpha: pre-gate plane)
      const float sc = s_aff[0][c], bi = s_aff[1][c];
#pragma unroll 1
      for (int slot = warp * CPL + hwi; slot < n_my; slot += kPW * CPL) {
        {
          const unsigned ent = s_list[slot];
          const int cell = (int)(ent >> 8) * W + (int)(ent & 255u);
          const float u = slot < R.ucap ? sU[slot * C + c] : R.u_over[((size_t)blockIdx.x * R.over_cap + (slot - R.ucap)) * C + c];
          const float d = tanhf(fmaf(u, sc, bi)) * a.update_gain;
          float* loc = (c == 3) ? (sAt + cell) : (sX + cell * C + c);
          const float v = ((c == 3) ? sAg[cell] : *loc) + d;
          *loc = v;
          const uint32_t la = smem_u32(loc);
          if (use_async) {
#pragma unroll
            for (int pr = 0; pr < 7; ++pr)
              if (pr + 1 < NC) st_async_f32(mapa_u32(la, (rank + pr + 1) & (NC - 1)), v, mapa_u32(mbarB, (rank + pr + 1) & (NC - 1)));
          } else {
#pragma unroll
            for (int pr = 0; pr < 7; ++pr)
              if (pr + 1 < NC) st_cluster_f32(mapa_u32(la, (rank + pr + 1) & (NC - 1)), v);
          }
        }
      }
    }
    REP_MARK(12);
    {
      // inactive cells: x_c += idle_c (their masked pre-norm update is 0, ncagraph.py:149-155); float4 per (cell, quad)
      const float4 i4 = *reinterpret_cast<const float4*>(&s_aff[2][4 * (tid & 3)]);
      // item = tid + 512 j  <->  cell (tid>>2) + 128 j, channel quad tid&3: the active bit sits at a per-thread constant
      // position of word (tid>>7) + 4 j, and every address is a constant offset from a per-thread base
      float4* X4 = reinterpret_cast<float4*>(sX) + tid;
      const uint32_t* aw = s_bAct + (tid >> 7);
      const int abit = (tid >> 2) & 31;
      const int nfull = (HW * 4) / kPT;
#pragma unroll 4
      for (int j = 0; j < nfull; ++j) {
        if (!((aw[4 * j] >> abit) & 1u)) {
          float4 v = X4[j * kPT];
          v.x += i4.x; v.y += i4.y; v.z += i4.z; v.w += i4.w;
          X4[j * kPT] = v;
        }
      }
      if (nfull * kPT + tid < HW * 4 && !((aw[4 * nfull] >> abit) & 1u)) {
        float4 v = X4[nfull * kPT];
        v.x += i4.x; v.y += i4.y; v.z += i4.z; v.w += i4.w;
        X4[nfull * kPT] = v;
      }
      REP_MARK(11);
      // (the alpha of the inactive cells, alpha + idle_3, is formed in S4 where the plane is read anyway)
    }
    REP_MARK(4);
    if (use_async) {
      mbar_wait(mbarB, (uint32_t)(t & 1));                                    // every peer's cells have landed here
      __syncthreads();                                                        // ... and my own warps' writes are done
    } else {
      cluster_arrive(); cluster_wait();                                       // ---- cluster barrier 2
    }
    REP_MARK(5);

    // ---- S4 + S1 of the next step: post-alive gate (ncagraph.py:158-166) from bitmaps; pre_alive(t+1) ==
    //      post_alive(t) when both thresholds agree (a cell above thr is never gated), so one dilation serves both ----
    const uint32_t nib_now = r_actnib;        // active cells of my quad in THIS step (act_count below replaces it)
    const float idle3 = s_aff[2][3];
    {
      // updated alpha before the gate: active cells were written into sAt by their owners (locally or pushed), every
      // other cell moves by the idle update of the alpha channel
      float4 at = reinterpret_cast<const float4*>(sAt)[ql];
      {
        const float4 ag = reinterpret_cast<const float4*>(sAg)[ql];
        at.x = (nib_now & 1u) ? at.x : ag.x + idle3; at.y = (nib_now & 2u) ? at.y : ag.y + idle3;
        at.z = (nib_now & 4u) ? at.z : ag.z + idle3; at.w = (nib_now & 8u) ? at.w : ag.w + idle3;
      }
      pack_store(s_bRaw, nib_gt(at, thr) & vmask);
      __syncthreads();
      const uint32_t post = dil(s_bRaw);
      at.x = (post & 1u) ? at.x : 0.f; at.y = (post & 2u) ? at.y : 0.f;
      at.z = (post & 4u) ? at.z : 0.f; at.w = (post & 8u) ? at.w : 0.f;
      reinterpret_cast<float4*>(sAg)[qs] = at;
      if (R.masks) {
        const uint32_t pw = pack_nibbles(post, lane);
        if (rank == 0 && (lane & 7) == 0 && qword < NW) R.masks[(((size_t)t * a.B + b) * 3 + 2) * kMaskWords + qword] = pw;
      }
      if (fast_alive) {
        pack_store(s_bAlive, post);
        act_count(post, cur ^ 1);
        __syncthreads();
        list_pass();
        __syncthreads();
      } else {
        pack_store(s_bRawB, nib_gt(at, thr) & vmask);
        pack_store(s_bRaw2B, nib_gt(at, gthr) & vmask);
        __syncthreads();
        alive_from_raw(s_bRawB, s_bRaw2B, cur ^ 1);
      }
    }
    REP_MARK(6);
  }

  __syncthreads();
  if (float* h = hist_at(R.T)) store_state(h, my_lo, my_hi);
  if constexpr (MET)
    if (R.T % M.every == 0)
      rep_met_frame<SS>(M, rep_met_target(R, M, b), sX, sAg, sY, my_lo, my_hi, HW, a.alpha_thr,
                        met_dst + (R.T / M.every) * met_frame_stride,
                        ssim_part + ((size_t)(R.T / M.every) * a.B + b) * NC + rank, H, W);
  store_state(R.xT + sample_off, my_lo, my_hi);
  if (R.dbg && blockIdx.x == R.dbg_cta && tid < 24) R.dbg[tid] = s_dbg[tid];
  cluster_arrive(); cluster_wait();      // nobody exits while a peer may still address its shared memory
}

// ------------------------------------------------------------------------------------------------
size_t dynamic_smem_cap(const void* kfn) {
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> cache;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return 0; }
  std::lock_guard<std::mutex> lock(mu);
  const auto key = std::make_pair(kfn, dev);
  const auto it = cache.find(key);
  if (it != cache.end()) return it->second;
  cudaFuncAttributes fa{};
  int optin = 0;
  if (cudaFuncGetAttributes(&fa, kfn) != cudaSuccess ||
      cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  const size_t limit = (size_t)optin > fa.sharedSizeBytes ? (size_t)optin - fa.sharedSizeBytes : 0;
  const size_t cap = limit < (size_t)226 * 1024 ? limit : (size_t)226 * 1024;
  cache.emplace(key, cap);
  return cap;
}

static size_t rep_smem_bytes(int C, int HW, int ucap, int listcap) {
  const int HWp = 4 * (((HW >> 2) + 31) & ~31) + 16;
  size_t f = (size_t)3 * C * 128 + 128 + 128 * kW2S + (size_t)HW * C + 2 * (size_t)HWp + (size_t)kPW * 3 * C * 8 +
             (size_t)ucap * C;
  size_t bytes = f * sizeof(float);
  bytes += (size_t)kPW * 8 * 16 * sizeof(short) + (size_t)((listcap + 7) & ~7) * sizeof(unsigned short);
  return bytes + 32;
}

int run_rep_fwd(const gnca_model& m, const Packed& P, const float* packed, int B, int H, int W,
                const gnca_schedule& sched, const float* x0, float* xT, float* hist, float* stats_hist,
                float* u_hist, float* rec, uint32_t* masks, float* scratch /* >= B*C*H*W floats */, cudaStream_t st,
                int hist_every, int t0, const ZpRec* zpr, const FrameMetrics* met, ModelStack ms, const SsimFrames* ss,
                int target_stride) {
  const bool graph = (m.flags & GNCA_F_GRAPH) != 0;
  if (m.C != 16 || m.hidden != 128) return GNCA_ERR_UNSUPPORTED;
  if (H > kMaxRows || W > kMaxRows || H < 1 || W < 4 || (W & 3)) return GNCA_ERR_UNSUPPORTED;   // quads of 4 cells per row
  if (H * W > 4 * kPT) return GNCA_ERR_UNSUPPORTED;                                            // one quad per thread
  const int k = graph ? sched.k : 0;
  const bool zp = graph && k > 0 && !(m.flags & GNCA_F_TORUS);      // zero-padded shift: the ZP instantiation
  if (zp && m.d_model > 32) return GNCA_ERR_UNSUPPORTED;
  if (zp && (rec || masks) && !zpr) return GNCA_ERR_UNSUPPORTED;     // its records are useless without w and the row sums
  if (k > 16) return GNCA_ERR_UNSUPPORTED;
  if (sched.fire_u && ((uintptr_t)sched.fire_u & 15)) return GNCA_ERR_UNSUPPORTED;    // float4 loads of the uniforms
  if (k > 0 && (sched.max_offset <= 0 || sched.max_offset >= H || sched.max_offset >= W)) return GNCA_ERR_UNSUPPORTED;
  if (sched.T > 0 && (!sched.fire_rate || (graph && !sched.message_gain) || (k > 0 && !sched.offsets)))
    return GNCA_ERR_ARG;
  const int C = 16, HW = H * W;
  RepArgs R{};
  fill_step_args(R.s, m, B, H, W);
  R.s.k = k;
  R.s.fire_rate_dev = sched.fire_rate;
  R.s.message_gain_dev = sched.message_gain;
  R.s.offsets_dev = sched.offsets;
  R.s.steps = sched.steps;
  R.s.philox_seed = sched.philox_seed;
  R.s.philox_offset = sched.philox_offset;
  R.fire_u_base = sched.fire_u;
  R.T = sched.T;
  R.t0 = t0;
  R.x0 = x0; R.xT = xT; R.hist = hist; R.hist_every = hist_every; R.stats_hist = stats_hist; R.u_hist = u_hist;
  R.rec = rec; R.masks = masks;
  R.damage = DamageView{sched.damage, sched.damage_layout}; R.damage_step = sched.damage_step;
  R.KP = k > 8 ? 16 : 8;
  R.zd = zp ? m.d_model : 0;
  R.model_stride = ms.stride; R.model_per = ms.per_model; R.target_stride = target_stride;
  // the metrics (and SSIM) instantiations have the same shared memory and register cap as the plain ones: the same
  // launch configuration, so x_T is bit-equal to the rollout without metrics
  const bool ssim = met && ss;
  const void* kfn = zp ? (ssim ? (const void*)k_rep_fwd<16, true, true, true>
                               : met ? (const void*)k_rep_fwd<16, true, true, false> : (const void*)k_rep_fwd<16, true, false, false>)
                       : (ssim ? (const void*)k_rep_fwd<16, false, true, true>
                               : met ? (const void*)k_rep_fwd<16, false, true, false> : (const void*)k_rep_fwd<16, false, false, false>);
  R.HWp = 4 * (((HW >> 2) + 31) & ~31) + 16;      // planes padded to whole warps of quads + one scratch quad
  R.inv_n = (float)(1.0 / ((double)C * (double)H * (double)W));

  const char* env_nc = getenv("GNCA_RESIDENT_NC");
  const bool debug = getenv("GNCA_DEBUG") != nullptr;
  // the dynamic carve shares the opt-in limit with the kernel's static shared memory (6 KB, 15 KB for the ZP
  // instantiation): near 2048 cells the dynamic cap of 226 KB alone would ask for more than a block may have
  const size_t cap = dynamic_smem_cap(kfn);
  const int cands[4] = {8, 4, 2, 1};
  int pick = -1, pick_ucap = 0, pick_list = 0, pick_ncl = 0;
  size_t pick_smem = 0;
  for (int pass = 0; pass < 2 && pick < 0; ++pass) {
    for (int ci = (pass == 0 ? 0 : 3); ci >= 0 && ci < 4; ci += (pass == 0 ? 1 : -1)) {
      const int NC = cands[ci];
      if (env_nc && atoi(env_nc) != NC) continue;
      const int share = (HW + NC - 1) / NC + 1;
      int ucap = share < 384 ? share : 384;
      size_t smem = rep_smem_bytes(C, HW, ucap, share);
      while (smem > cap && ucap > 128) { ucap -= 64; smem = rep_smem_bytes(C, HW, ucap, share); }
      if (smem > cap) continue;
      if (ucap < share && !scratch) continue;
      GNCA_CHECK_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      cudaLaunchConfig_t q{};
      q.gridDim = dim3(B * NC); q.blockDim = dim3(kPT); q.dynamicSmemBytes = smem; q.stream = st;
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = NC; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
      q.attrs = qa; q.numAttrs = 1;
      int ncl = 0;
      if (cudaOccupancyMaxActiveClusters(&ncl, kfn, &q) != cudaSuccess || ncl < 1) {
        cudaGetLastError();
        continue;
      }
      if (pass == 0 && B > ncl && !env_nc) continue;     // would need a second wave: try a smaller cluster
      pick = NC; pick_ucap = ucap; pick_list = share; pick_smem = smem; pick_ncl = ncl;
      break;
    }
  }
  if (pick < 0) return GNCA_ERR_UNSUPPORTED;
  R.NC = pick; R.ucap = pick_ucap; R.listcap = (pick_list + 7) & ~7;
  R.u_over = scratch;
  R.over_cap = (HW + pick - 1) / pick + 1 > pick_ucap ? (HW + pick - 1) / pick + 1 - pick_ucap : 0;
  if ((size_t)pick * R.over_cap > (size_t)HW) return GNCA_ERR_UNSUPPORTED;   // scratch holds B*C*HW floats
  GNCA_CHECK_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pick_smem));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(B * pick);
  cfg.blockDim = dim3(kPT);
  cfg.dynamicSmemBytes = pick_smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = pick; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  { const char* e = getenv("GNCA_REP_SYNC"); R.use_async = !(e && e[0] == 'b'); }     // development: "barrier"
  if (debug)
    fprintf(stderr, "[gnca] replicated fwd: B=%d NC=%d ucap=%d over=%d smem=%zu maxActiveClusters=%d\n", B, pick,
            R.ucap, R.over_cap, pick_smem, pick_ncl);
  static unsigned long long* dbg_buf = nullptr;
  if (getenv("GNCA_PHASE_TIMING")) {
    if (!dbg_buf) cudaMalloc(&dbg_buf, 24 * sizeof(unsigned long long));
    cudaMemsetAsync(dbg_buf, 0, 24 * sizeof(unsigned long long), st);
    R.dbg = dbg_buf;
    R.dbg_cta = atoi(getenv("GNCA_PHASE_TIMING"));
  }
  prof_begin(PROF_RESIDENT_FWD, st);
  const ZpRec Z = (zp && zpr && rec) ? *zpr : ZpRec{nullptr, nullptr};
  const FrameMetrics M = met ? *met : FrameMetrics{};
  double* ssp = ssim ? ss->part : nullptr;
  cudaError_t e = zp ? (ssim ? cudaLaunchKernelEx(&cfg, k_rep_fwd<16, true, true, true>, R, P, packed, Z, M, ssp)
                        : met ? cudaLaunchKernelEx(&cfg, k_rep_fwd<16, true, true, false>, R, P, packed, Z, M, ssp)
                              : cudaLaunchKernelEx(&cfg, k_rep_fwd<16, true, false, false>, R, P, packed, Z, M, ssp))
                     : (ssim ? cudaLaunchKernelEx(&cfg, k_rep_fwd<16, false, true, true>, R, P, packed, Z, M, ssp)
                        : met ? cudaLaunchKernelEx(&cfg, k_rep_fwd<16, false, true, false>, R, P, packed, Z, M, ssp)
                              : cudaLaunchKernelEx(&cfg, k_rep_fwd<16, false, false, false>, R, P, packed, Z, M, ssp));
  prof_end(PROF_RESIDENT_FWD, st);
  if (e != cudaSuccess) return (int)e;
  GNCA_LAUNCH_CHECK();
  if (met) {
    const int rc = run_metrics_reduce((R.T / met->every + 1) * B, pick, met->part, met->sums, met->counts, st);
    if (rc) return rc;
  }
  if (ssim) {
    const int rc = run_ssim_reduce((R.T / met->every + 1) * B, pick, ss->part, ss->ssim, H, W, st);
    if (rc) return rc;
  }
  if (R.dbg) {
    unsigned long long h[24];
    cudaStreamSynchronize(st);
    cudaMemcpy(h, dbg_buf, sizeof(h), cudaMemcpyDeviceToHost);
    const char* names[18] = {"top", "S2 side jobs", "stats push", "wait A", "S3 idle alpha", "wait B",
                             "S4 gate + S1 list", "-", "(sum n_my)", "S2 tiles rest(warp0)", "S3 finalize+sync", "S3 idle x", "S3 active+push",
                             "tile: sender table", "tile: perception+gather", "tile: message", "tile: layer 1", "tile: layer 2 + RS"};
    fprintf(stderr, "[gnca rep phase cycles, CTA%d, T=%d]", R.dbg_cta, R.T);
    for (int i = 0; i < 18; ++i) fprintf(stderr, " %s=%llu", names[i], h[i]);
    fprintf(stderr, "\n");
  }
  return 0;
}

}  // namespace gnca
