// Cluster-resident BPTT for the replicated-state rollout (gnca_rep.cu) -- SURVEY Appendix A, restated for records.
//
// The forward kept, for every ACTIVE cell of every step, a record (gnca_rep.h): perception y, masked pre-norm update u,
// gathered sender state xs, tanh of the message pre-activation, `as`; plus three bitmaps and (mean, rstd) per step.
// Nothing else of the forward is needed: no x_t history, no gathers, no perception recompute.
//
//   k_rep_bwd   ONE launch walks t = T-1 .. 0.  A sample is owned by a cluster of NC CTAs.  The sequential part of BPTT
//               is only the propagation of g = dL/dx_t; per step:
//                 A0  inactive cells of my band: per-channel sums of the gated gradient (their tanh' is a per-channel
//                     constant) -> their share of the GroupNorm-backward sums S1, S2, dgamma, dbeta
//                 A   active cells of my band: gz = g * eta * tanh' -> L2 scratch (by slot)
//                 --  S1, S2 partials -> every CTA of the cluster (DSMEM)                        [cluster barrier 1]
//                 B   my SHARE of the active cells (balanced over the cluster like the forward), warp-autonomous tiles:
//                     gd = dL/du, hidden layer recomputed from y in registers, gh, gy = W1^T gh as
//                     three 16-channel shuffle reduce-scatters, message backward; gd / gm go back into the record, gy and
//                     g_xs of the cell into an L2-resident per-cell scratch                       [cluster barrier 2]
//                 C   my band of cells: g_t = gated g_{t+1} + perception transpose (gather from active neighbours) +
//                     message transpose (gather from active receivers at +offset), in place in shared memory
//               g itself never leaves shared memory (each CTA owns a band of it for the whole sweep); only gz of the
//               active cells and their gy / g_xs travel through L2 between the CTAs of the cluster.
//   k_rep_wgrad weight gradients have no sequential dependence: one fully parallel pass over ALL records of the rollout
//               (batches of 64 cells through the small GEMMs as FFMA register tiles, accumulators in registers for the
//               whole kernel, one partial per block, no atomics) -> k_rep_wreduce sums the partials in a fixed order.
#include <cooperative_groups.h>
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include "gnca_common.cuh"
#include "gnca_internal.h"
#include "gnca_ptx.cuh"
#include "gnca_rep.h"

namespace cg = cooperative_groups;

namespace gnca {

constexpr int kQT = 512;          // threads per CTA (k_rep_bwd)
constexpr int kQW = kQT / 32;
constexpr int kQW2S = 20;         // padded row stride of W2^T
constexpr int kQW1S = 132;        // padded row stride of W1^T (floats): rows c, c+8 share banks only pairwise (2-way)

struct RepBwdArgs {
  StepArgs s;
  int T, NC, gmax;            // gmax: largest tile (8, or 4 when the whole sample sits in one CTA and smem is short)
  float inv_n;
  float* rec;
  float* hgh;                 // [T][B][HW][kHghStride] h | gh of every record (written here, read by k_rep_wgrad)
  const uint32_t* masks;
  const float* stats;         // [T][B][2]
  const float* gT;            // [B][C][HW]
  float* g0;                  // [B][C][HW]
  float* GZ;                  // [B][HW][C] gz of the active cells of the current step, by slot (L2)
  float* RG;                  // [B][HW][64]   gy (48) | g_xs (16) of the active cells of the current step (L2)
  float* affpart;             // [B*NC][2C] dgamma | dbeta partials
  DamageView damage;
  int damage_step;
  // kFrames: add frame T / every to g_T when T % every == 0.  0 in a checkpoint segment, whose frame at T is the next
  // segment's first, added there already.  It sits in the padding before `dbg`, so the struct keeps its size and every
  // later kernel parameter its offset: the instantiations without frames compile to the same SASS as without the field
  int gT_frame;
  unsigned long long* dbg;    // optional phase-cycle counters (GNCA_PHASE_TIMING=<cta>)
  int dbg_cta;
  int t0;                     // absolute step of local step 0 (see RepArgs::t0): only steps[b] is absolute
};

#ifdef GNCA_PHASE_COUNTERS          /* build with -DGNCA_PHASE_COUNTERS for the per-phase cycle counters */
#define REPB_MARK(idx)                                                              \
  do {                                                                              \
    if (R.dbg && tid == 0) {                                                        \
      const long long _n = clock64();                                               \
      s_dbg[idx] += (unsigned long long)(_n - t_prev);                              \
      t_prev = _n;                                                                  \
    }                                                                               \
  } while (0)
#else
#define REPB_MARK(idx) do { } while (0)
#endif

// Bulk asynchronous stores shared -> global (async proxy, tracked per thread in bulk groups).  The 1 KB per record of
// h | gh that only k_rep_wgrad reads goes out this way: the cluster barriers' release fence then no longer waits for
// those stores to drain (they were ~70 % of the bytes a CTA writes per step), and the warp issues 2 instructions per
// cell instead of 16 STG.128.
__device__ __forceinline__ void bulk_store_512(float* gdst, const float* ssrc) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], 512;" ::"l"(__cvta_generic_to_global(gdst)),
               "r"((uint32_t)__cvta_generic_to_shared(ssrc)) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// kFrames: gframes ([F][B][C][HW]) holds dL/dframe_f of the state step f * every consumes; it is added to g_t at
// t = f * every (before that step's damage mask, since the frame is the post-damage state) and, with R.gT_frame, to g_T
// when T % every == 0.  The instantiation without it is the one every plain BPTT launches (its parameters go unused).
// ZP: zero-padded graph shift (k_rep_fwd<16, true>, buffers in Z; Z is unused otherwise).  Senders (y - dy_i, x) with
// the per-sample softmax weights w_i: the message transpose of phase C drops receivers outside the grid and weighs by
// w_i, and on message steps it also sums dL/dw_i (sender side: A(s) [g_xs(r) . x_t(s) + bm . gm(r)]).  The k partials
// are reduced over the cluster in a fixed order (third cluster barrier), then every CTA runs the softmax / pooled Q.K
// backward of k_attn_bwd and adds its row term `grow` to its band of g_t; rank 0 accumulates the Q/K/scaling
// gradients of the sample in Z.pw.
// MS (a stack of models, gnca_rollout_bwd_bptt_*_models): sample b reads its weights from packed + (b / S.per_model) *
// S.stride.  `packed` is rebased once at entry, so every later read (gamma / beta in the step loop, the attention
// parameters of ZP) goes through the rebased pointer.  A compile-time flag with a trailing parameter, not a RepBwdArgs
// field: the kernel runs at its register cap, and the instantiations without MS keep their SASS.
template <int C, bool kFrames, bool ZP, bool MS = false>
__global__ void __launch_bounds__(kQT, 1) k_rep_bwd(RepBwdArgs R, Packed P, const float* __restrict__ packed,
                                                   const float* __restrict__ gframes, int every, ZpBwd Z,
                                                   ModelStack S) {
  static_assert(C == 16, "lane mapping: 2 cells x 16 channels per warp row");
  constexpr int C3 = 3 * C, HID = 128, CPL = 32 / C;
  cg::cluster_group cluster = cg::this_cluster();
  const StepArgs& a = R.s;
  const int NC = R.NC;
  const int rank = (int)cluster.block_rank();
  const int b = blockIdx.x / NC;
  const int H = a.H, W = a.W, HW = H * W;
  const int NQ = HW >> 2, NW = (HW + 31) >> 5;
  const bool graph = (a.flags & GNCA_F_GRAPH) != 0;
  const bool gn = (a.flags & GNCA_F_GROUPNORM) != 0;
  const bool a2a = (a.flags & GNCA_F_ALIVE_TO_ALIVE) != 0;
  const int c_lo = ((a.flags & GNCA_F_HIDDEN_ONLY) && C >= 4) ? 4 : 0;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int hwi = lane / C, c = lane % C;
  const int k = a.k;
  const int lnc = NC == 8 ? 3 : NC == 4 ? 2 : NC == 2 ? 1 : 0;
  const float eta = a.update_gain;

  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* sW1T = reinterpret_cast<float*>(smem_raw);           // [3C][HID] permuted (lane l owns 4l..4l+3 <-> units l+32jj)
  float* sb1 = sW1T + C3 * kQW1S;
  float* sW2P = sb1 + HID;                                    // [HID][kQW2S]
  const int band_lo = (HW * rank) >> lnc, band_hi = (HW * (rank + 1)) >> lnc, nband = band_hi - band_lo;
  const int bandcap = ((HW + NC - 1) / NC) + 1;
  float* sG = sW2P + HID * kQW2S;                             // [bandcap][C] my band of g (cell-major)
  const int GM = R.gmax;
  float* sY = sG + (size_t)bandcap * C;                       // [kQW][3C][GM]
  float* sGD = sY + kQW * C3 * GM;                            // [kQW][C][GM]
  float* sGH = sGD + kQW * C * GM;                            // [kQW][GM][HID] gh of the tile (permuted unit order)
  unsigned short* s_list = reinterpret_cast<unsigned short*>(sGH + kQW * GM * HID);  // [bandcap] my SHARE of the active cells
  unsigned short* s_blist = s_list + ((bandcap + 7) & ~7);                          // [bandcap] active cells of my BAND
  // ZP: attention-backward scratch behind the band lists (kZpSmemFloats)
  float* const zrs = reinterpret_cast<float*>(s_blist + ((bandcap + 7) & ~7));      // [C][H] row sums of x_t
  float* const zw = zrs + 64 * 16;                                                  // [16] w_i
  float* const zgww = zw + 16;                                                      // [kQW][16] dL/dw_i per warp
  float* const zgwc = zgww + 16 * 16;                                               // [8][16] per CTA (pushed by the peers)
  float* const zgL = zgwc + 8 * 16;                                                 // [16] dL/dw_i, then dL/dlogit_i
  float* const zlg = zgL + 16;                                                      // [16] logits
  int* const zrlo = reinterpret_cast<int*>(zlg + 16);                               // [16] kept rows of offset i
  int* const zrhi = zrlo + 16;
  float* const zbm = reinterpret_cast<float*>(zrhi + 16);                           // [C] bm
  float* const zxbar = zbm + 16;                                                    // [C] mean of x_t
  float* const zwkq = zxbar + 16;                                                   // [C] Wk^T qp
  float* const zgxb = zwkq + 16;                                                    // [C] Wq^T gqp
  float* const zqp = zgxb + 16;                                                     // [32] pooled query
  float* const zgqp = zqp + 32;                                                     // [32] its gradient
  float* const zS = zgqp + 32;                                                      // [16][C] row-range sums
  float* const zKP = zS + 16 * 16;                                                  // [16][32] mean shifted keys
  float* const zsL = zKP + 16 * 32;                                                 // [64] sum of dL/dlogit_i over offsets keeping row y
  float* const zmisc = zsL + 64;                                                    // [0] dL/dscaling of the step

  __shared__ uint32_t s_bAS[kMaskWords], s_bAct[kMaskWords], s_bPost[kMaskWords];
  __shared__ __align__(16) int s_wtot[kQW];
  __shared__ float s_parts[8][2];
  __shared__ float s_wred[kQW][2];
  __shared__ float s_chs[kQW][2][C];       // per-warp per-channel sums (A0)
  __shared__ float s_aff[4][C];            // sc, bi, k_c = eta(1 - tanh(bi)^2), inactive gz factor ...
  __shared__ signed char s_off[2 * 16];
  __shared__ float s_gain;
  __shared__ int s_bandbase[2];            // slot of the first active cell at / after band_lo, band_hi
  __shared__ unsigned long long s_dbg[16];
  if (threadIdx.x < 16) s_dbg[threadIdx.x] = 0;
  long long t_prev = clock64();

  if constexpr (MS) packed += (size_t)(b / S.per_model) * S.stride;
#pragma unroll 1
  for (int i = tid; i < C3 * HID; i += kQT) {
    const int kk = i / HID, jp = i - kk * HID;
    const int l = jp >> 2, jj = jp & 3;
    sW1T[kk * kQW1S + jp] = packed[P.w1t + kk * HID + (l + 32 * jj)];
  }
  if (tid < HID) { const int l = tid >> 2, jj = tid & 3; sb1[tid] = packed[P.b1 + l + 32 * jj]; }
#pragma unroll 1
  for (int i = tid; i < HID * C; i += kQT) { const int j = i / C, cc = i - j * C; sW2P[j * kQW2S + cc] = packed[P.w2t + i]; }
  __shared__ __align__(16) float s_wmT[C][C + 4];               // s_wmT[c][cc] = Wm[cc][c] (kept out of the registers)
#pragma unroll
  for (int cc = 0; cc < C; ++cc) if (tid < C) s_wmT[tid][cc] = graph ? packed[P.wm + cc * C + tid] : 0.f;
  const float gam_c = gn ? packed[P.gamma + c] : 1.f;
  if constexpr (ZP) {
    if (tid < C) zbm[tid] = packed[P.bm + tid];
  }

  const size_t sample_off = (size_t)b * C * HW;
  float* GZs = R.GZ + (size_t)b * HW * C;
  float* RGs = R.RG + (size_t)b * HW * 64;

  // g_T (NCHW) -> my band in smem (g never leaves shared memory: the band owner gates it and gathers into it)
  {
    const int n8 = (nband + 7) & ~7;
#pragma unroll 1
    for (int i = tid; i < n8 * C; i += kQT) {
      const int ci = i & 7, c4 = (i >> 3) & 3, rest = i >> 5;
      const int cq = rest & 3, cgp = rest >> 2;
      const int cl = cgp * 8 + ci, ch = cq * 4 + c4;
      if (cl < nband) {
        float v = R.gT[sample_off + (size_t)ch * HW + band_lo + cl];
        if constexpr (kFrames)
          if (R.gT_frame && R.T % every == 0) v += __ldg(gframes + ((size_t)(R.T / every) * a.B * C + (size_t)b * C + ch) * HW + band_lo + cl);
        sG[cl * C + ch] = v;
      }
    }
  }
  __syncthreads();
  cluster_sync_acquire();

  const int my_steps = a.steps ? min(a.steps[b] - R.t0, R.T) : R.T;
  const int q = tid, qcell = 4 * tid;
  const bool qv = q < NQ;
  const int qsh = 4 * (lane & 7), qword = min(q >> 3, kMaskWords - 1);
  float* myY = sY + warp * (C3 * GM);
  float* myGD = sGD + warp * (C * GM);
  float* myGH = sGH + warp * (GM * HID);
  float dgam = 0.f, dbet = 0.f;              // this lane's channel c, summed over its cells / steps

  for (int t = R.T - 1; t >= 0; --t) {
    const bool dmg = R.damage.p && t == R.damage_step;
    // dL/dframe of step t (my sample), or null when step t keeps no frame
    const float* gfr = (kFrames && t % every == 0) ? gframes + ((size_t)(t / every) * a.B + b) * C * HW : nullptr;
    if (t >= my_steps) {                     // frozen: g passes through (the damage mask still multiplies x)
      if constexpr (kFrames) {
        if (dmg || gfr) {
#pragma unroll 1
          for (int i = tid; i < nband * C; i += kQT) {
            const int cl = i / C, ch = i - cl * C;
            float v = sG[i];
            if (gfr) v += __ldg(gfr + (size_t)ch * HW + band_lo + cl);
            if (dmg) v *= R.damage.at(b, ch, band_lo + cl, C, HW);
            sG[i] = v;
          }
          __syncthreads();
        }
        continue;
      }
      if (dmg) {
#pragma unroll 1
        for (int i = tid; i < nband * C; i += kQT) {
          const int cl = i / C, ch = i - cl * C;
          sG[i] *= R.damage.at(b, ch, band_lo + cl, C, HW);
        }
        __syncthreads();
      }
      continue;
    }
    REPB_MARK(0);
    // ---- masks, schedule, statistics of step t ----------------------------------------------------------------
    if (tid < NW) {
      const uint32_t* mk = R.masks + ((size_t)t * a.B + b) * 3 * kMaskWords;
      s_bAS[tid] = mk[tid]; s_bAct[tid] = mk[kMaskWords + tid]; s_bPost[tid] = mk[2 * kMaskWords + tid];
    }
    if (tid >= 64 && tid < 64 + 2 * k) s_off[tid - 64] = a.offsets_dev[(size_t)t * k * 2 + (tid - 64)];
    if (tid == 96) s_gain = graph ? a.message_gain_dev[t] : 0.f;
    if constexpr (ZP) {
      if (tid >= 160 && tid < 176) zw[tid - 160] = Z.w[((size_t)t * a.B + b) * 16 + (tid - 160)];
    }
    if (tid >= 128 && tid < 128 + C) {
      const int ch = tid - 128;
      float sc = 1.f, bi = 0.f;
      if (gn) {
        const float mu = R.stats[((size_t)t * a.B + b) * 2], rstd = R.stats[((size_t)t * a.B + b) * 2 + 1];
        sc = rstd * packed[P.gamma + ch];
        bi = packed[P.beta + ch] - mu * sc;
      }
      const float th = tanhf(bi);
      s_aff[0][ch] = sc; s_aff[1][ch] = bi; s_aff[2][ch] = eta * (1.f - th * th);
    }
    __syncthreads();
    const float gain_m = s_gain;
    const bool msg_on = graph && gain_m != 0.f && k > 0;
    const float mu = gn ? R.stats[((size_t)t * a.B + b) * 2] : 0.f, rstd = gn ? R.stats[((size_t)t * a.B + b) * 2 + 1] : 1.f;
    const float uh0 = -mu * rstd;            // normalised update of an inactive cell
    // ---- balanced list of my share of the active cells (same order as the forward: cell order) -------------------
    int n_my, lo_my, nact;
    {
      const uint32_t wd = s_bAct[qword];
      const uint32_t nib = qv ? (wd >> qsh) & 15u : 0u;
      const int cnt = ((lane & 7) == 0 && qv) ? __popc(wd) : 0;
      const int c0 = __shfl_sync(0xffffffffu, cnt, 0), c1 = __shfl_sync(0xffffffffu, cnt, 8),
                c2 = __shfl_sync(0xffffffffu, cnt, 16), c3 = __shfl_sync(0xffffffffu, cnt, 24);
      const int g = lane >> 3;
      const int pre = (g > 0 ? c0 : 0) + (g > 1 ? c1 : 0) + (g > 2 ? c2 : 0);
      if (lane == 0) s_wtot[warp] = c0 + c1 + c2 + c3;
      __syncthreads();
      int base = 0, tot = 0;
#pragma unroll
      for (int w4 = 0; w4 < kQW / 4; ++w4) {
        const int4 v = *reinterpret_cast<const int4*>(&s_wtot[4 * w4]);
        const int vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) { base += (4 * w4 + j < warp) ? vv[j] : 0; tot += vv[j]; }
      }
      nact = tot;
      const int lo = (tot * rank) >> lnc, hi = (tot * (rank + 1)) >> lnc;
      n_my = hi - lo; lo_my = lo;
      const int slot_q = base + pre + __popc(wd & ((1u << qsh) - 1u));      // slot of the first active cell of my quad
      if (qv && qcell == band_lo) s_bandbase[0] = slot_q;                   // band_lo, band_hi are multiples of 4
      if (qv && qcell == band_hi) s_bandbase[1] = slot_q;
      if (tid == 0 && band_hi == HW) s_bandbase[1] = tot;
      __syncthreads();
      if (nib) {
        int slot = slot_q;
        const int bb = s_bandbase[0];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (nib & (1u << j)) {
            if (slot >= lo && slot < hi) s_list[slot - lo] = (unsigned short)(qcell + j);
            if (qcell >= band_lo && qcell < band_hi) s_blist[slot - bb] = (unsigned short)(qcell + j);
            ++slot;
          }
        }
      }
    }
    const int bandbase = s_bandbase[0], n_band = s_bandbase[1] - s_bandbase[0];
    // u of my band's active cells (phase A) is requested NOW: one L2 round trip that phase A0 overlaps, instead of
    // n_band / 32 dependent ones at the top of phase A (the record loads were 5 % of the kernel's stall samples)
    constexpr int kAPre = 6;                 // 6 x 32 band cells up front; a longer band list falls back to the loop
    const size_t rec_base = ((size_t)t * a.B + b) * HW;
    float upre[kAPre];
#pragma unroll
    for (int i = 0; i < kAPre; ++i) {
      const int bi_ = warp * CPL + hwi + i * (kQW * CPL);
      upre[i] = bi_ < n_band ? __ldcg(R.rec + (rec_base + bandbase + bi_) * kRecStride + kRecU + c) : 0.f;
    }
    REPB_MARK(1);
    // ---- A0: inactive cells of my band: per-channel sums of the gated gradient --------------------------------------
    float s1 = 0.f, s2 = 0.f;
    {
      float acc0 = 0.f;                      // channel c (= tid & 15), cells (tid >> 4) + 32 j of the band
#pragma unroll 4
      for (int cl = tid >> 4; cl < nband; cl += kQT / C) {
        const int cell = band_lo + cl;
        const bool act = (s_bAct[cell >> 5] >> (cell & 31)) & 1u;
        float g = sG[cl * C + c];
        if (c == 3 && !((s_bPost[cell >> 5] >> (cell & 31)) & 1u)) g = 0.f;
        acc0 += act ? 0.f : g;
      }
      acc0 += __shfl_xor_sync(0xffffffffu, acc0, 16);
      if (lane < C) s_chs[warp][0][lane] = acc0;
    }
    __syncthreads();
    if (warp == 0 && lane < C) {
      float ac = 0.f;
      for (int w = 0; w < kQW; ++w) ac += s_chs[w][0][lane];
      const float gzs = ac * s_aff[2][lane];          // sum over the inactive cells of gz for this channel
      if (gn) {
        const float gu = gzs * gam_c;                 // lane == c here
        s1 = gu; s2 = gu * uh0;
        dgam += gzs * uh0; dbet += gzs;
      }
    }
    REPB_MARK(2);
    // ---- A: active cells of my BAND (g is resident here): gz = gated g * eta * (1 - tanh^2(gn(u)))  -> GZ[slot] in L2
    //         (ncagraph.py:153-166 backward); the heavy part (B) is done by whichever CTA the balanced split picks
    const float sc_c = s_aff[0][c], bi_c = s_aff[1][c];
    auto band_cell = [&](const int bi_, const float u) {
      const int cell = s_blist[bi_];
      float g = sG[(cell - band_lo) * C + c];
      if (c == 3 && !((s_bPost[cell >> 5] >> (cell & 31)) & 1u)) g = 0.f;
      const float th = tanhf(fmaf(u, sc_c, bi_c));
      const float gz = g * eta * (1.f - th * th);
      GZs[(size_t)(bandbase + bi_) * C + c] = gz;
      if (gn) {
        const float uh = (u - mu) * rstd, gu = gz * gam_c;
        s1 += gu; s2 = fmaf(gu, uh, s2);
        dgam = fmaf(gz, uh, dgam); dbet += gz;
      }
    };
#pragma unroll
    for (int i = 0; i < kAPre; ++i) {
      const int bi_ = warp * CPL + hwi + i * (kQW * CPL);
      if (bi_ < n_band) band_cell(bi_, upre[i]);
    }
#pragma unroll 2
    for (int bi_ = warp * CPL + hwi + kAPre * (kQW * CPL); bi_ < n_band; bi_ += kQW * CPL)
      band_cell(bi_, __ldcg(R.rec + (rec_base + bandbase + bi_) * kRecStride + kRecU + c));
    REPB_MARK(3);
    // ---- S1, S2: warp -> block -> every CTA of the cluster ---------------------------------------------------------
    {
      const float f1 = warp_sum(s1), f2 = warp_sum(s2);
      if (lane == 0) { s_wred[warp][0] = f1; s_wred[warp][1] = f2; }
    }
    __syncthreads();
    if (warp == 0) {
      float t1 = lane < kQW ? s_wred[lane][0] : 0.f, t2 = lane < kQW ? s_wred[lane][1] : 0.f;
      t1 = warp_sum(t1); t2 = warp_sum(t2);
      if (lane < NC) {
        float* dst = cluster.map_shared_rank(&s_parts[0][0], lane);
        dst[rank * 2] = t1; dst[rank * 2 + 1] = t2;
      }
    }
    REPB_MARK(4);
    cluster_sync_acquire();                                                   // ---- cluster barrier 1: S1/S2 partials, GZ visible
    REPB_MARK(5);
    float s1n = 0.f, s2n = 0.f;
    if (gn) {
      for (int r = 0; r < NC; ++r) { s1n += s_parts[r][0]; s2n += s_parts[r][1]; }
      s1n *= R.inv_n; s2n *= R.inv_n;
    }
    // ---- B: my share of the active cells; every warp covers an equal contiguous range with tiles of 8 / 4 / 2 cells ---
    auto bwd_tile = [&](auto gtag, const int slot0, const int lim) {
      constexpr int G = decltype(gtag)::value;
      constexpr int MPL = G / CPL;
      float gxs[MPL];
      int cellr[MPL];
      bool valid[MPL];
#pragma unroll
      for (int r = 0; r < MPL; ++r) {
        const int m = hwi + CPL * r, sl = slot0 + m;
        valid[r] = sl < lim;
        const int slc = min(sl, lim - 1);
        cellr[r] = s_list[slc];
        float* rc = R.rec + (rec_base + lo_my + slc) * kRecStride;
        myY[c * G + m] = __ldcg(rc + c);
        myY[(C + c) * G + m] = __ldcg(rc + C + c);
        myY[(2 * C + c) * G + m] = __ldcg(rc + 2 * C + c);
        const float gz = __ldcg(GZs + (size_t)(lo_my + slc) * C + c);
        float gd = gz;
        if (gn) {
          const float uh = (__ldcg(rc + kRecU + c) - mu) * rstd;
          gd = rstd * (gz * gam_c - s1n - uh * s2n);
        }
        gd = valid[r] ? gd : 0.f;
        myGD[c * G + m] = gd;
        float gm = 0.f;
        if (msg_on && c >= c_lo) {
          const float th = __ldcg(rc + kRecTh + c);
          gm = gd * gain_m * (1.f - th * th);
        }
        if (valid[r]) { rc[kRecU + c] = gd; rc[kRecTh + c] = gm; }           // record now holds gd | gm (weight gradients)
        if constexpr (ZP) {                                                  // bm . gm of the cell (dL/dw_i, phase C)
          if (msg_on) {
            float bg = zbm[c] * gm;
            bg += __shfl_xor_sync(0xffffffffu, bg, 8); bg += __shfl_xor_sync(0xffffffffu, bg, 4);
            bg += __shfl_xor_sync(0xffffffffu, bg, 2); bg += __shfl_xor_sync(0xffffffffu, bg, 1);
            if (c == 0 && valid[r]) Z.bg[(size_t)b * HW + cellr[r]] = bg;
          }
        }
        float acc = 0.f;                                                     // g_xs[c] = sum_cc Wm[cc][c] gm[cc]
        if (msg_on) {
#pragma unroll
          for (int c4 = 0; c4 < C / 4; ++c4) {
            const float4 w4 = *reinterpret_cast<const float4*>(&s_wmT[c][4 * c4]);
            acc = fmaf(w4.x, __shfl_sync(0xffffffffu, gm, (lane & 16) | (4 * c4)), acc);
            acc = fmaf(w4.y, __shfl_sync(0xffffffffu, gm, (lane & 16) | (4 * c4 + 1)), acc);
            acc = fmaf(w4.z, __shfl_sync(0xffffffffu, gm, (lane & 16) | (4 * c4 + 2)), acc);
            acc = fmaf(w4.w, __shfl_sync(0xffffffffu, gm, (lane & 16) | (4 * c4 + 3)), acc);
          }
        }
        gxs[r] = acc;
      }
      __syncwarp();
      // hidden pre-activations of my 4 units (recomputed): acc1[m][jj]
      float acc1[G][4];
      {
        const float4 bb = *reinterpret_cast<const float4*>(sb1 + 4 * lane);
#pragma unroll
        for (int m = 0; m < G; ++m) { acc1[m][0] = bb.x; acc1[m][1] = bb.y; acc1[m][2] = bb.z; acc1[m][3] = bb.w; }
#pragma unroll 8
        for (int kk = 0; kk < C3; ++kk) {
          const float4 w = *reinterpret_cast<const float4*>(sW1T + kk * kQW1S + 4 * lane);
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
            acc1[m][0] = fmaf(ym[m], w.x, acc1[m][0]); acc1[m][1] = fmaf(ym[m], w.y, acc1[m][1]);
            acc1[m][2] = fmaf(ym[m], w.z, acc1[m][2]); acc1[m][3] = fmaf(ym[m], w.w, acc1[m][3]);
          }
        }
      }
      // gh[m][jj] = [h > 0] * sum_c W2[c][j] gd[c][m]   (the ReLU mask as bits, the accumulators reuse acc1's registers)
      uint32_t hmask = 0;
      // h rows -> the warp's smem tile -> one 512-byte bulk store per cell (lane m issues cell m); the tile's previous
      // bulk reads (gh of the warp's last tile) must have finished before it is overwritten
      float* const hgh_row = R.hgh + (rec_base + lo_my + slot0 + min(lane, G - 1)) * kHghStride;
      const bool issuer = lane < G && slot0 + lane < lim;
      if (lane < G) bulk_wait_read_all();
      __syncwarp();
#pragma unroll
      for (int m = 0; m < G; ++m) {
        *reinterpret_cast<float4*>(myGH + m * HID + 4 * lane) =
            make_float4(fmaxf(acc1[m][0], 0.f), fmaxf(acc1[m][1], 0.f), fmaxf(acc1[m][2], 0.f), fmaxf(acc1[m][3], 0.f));
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) { hmask |= acc1[m][jj] > 0.f ? (1u << (4 * m + jj)) : 0u; acc1[m][jj] = 0.f; }
      }
      fence_proxy_async();
      __syncwarp();
      if (issuer) bulk_store_512(hgh_row, myGH + lane * HID);
      if (lane < G) bulk_commit();
#pragma unroll
      for (int c4 = 0; c4 < C / 4; ++c4) {
        float4 w2[4];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) w2[jj] = *reinterpret_cast<const float4*>(sW2P + (lane + 32 * jj) * kQW2S + 4 * c4);
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
          float gm4[G];
          if constexpr (G == 2) {
            const float2 gv = *reinterpret_cast<const float2*>(myGD + (4 * c4 + cc) * G);
            gm4[0] = gv.x; gm4[1] = gv.y;
          } else {
#pragma unroll
            for (int m4 = 0; m4 < G / 4; ++m4) {
              const float4 gv = *reinterpret_cast<const float4*>(myGD + (4 * c4 + cc) * G + 4 * m4);
              gm4[4 * m4] = gv.x; gm4[4 * m4 + 1] = gv.y; gm4[4 * m4 + 2] = gv.z; gm4[4 * m4 + 3] = gv.w;
            }
          }
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const float wv = cc == 0 ? w2[jj].x : cc == 1 ? w2[jj].y : cc == 2 ? w2[jj].z : w2[jj].w;
#pragma unroll
            for (int m = 0; m < G; ++m) acc1[m][jj] = fmaf(wv, gm4[m], acc1[m][jj]);
          }
        }
      }
      // gy[kk][m] = sum_j W1[j][kk] gh[j][m].  gh goes through the warp's shared-memory tile so that the lane that owns
      // (cell hwi+2e, channel c) can run the three 128-long dot products itself (rows c, 16+c, 32+c of W1^T = identity /
      // sobel_x / sobel_y parts): no cross-lane reduction.
      if (lane < G) bulk_wait_read_all();        // the h rows have left the tile (issued before the gh loop above)
      __syncwarp();
#pragma unroll
      for (int m = 0; m < G; ++m) {
        float4 v;
        v.x = (hmask >> (4 * m)) & 1u ? acc1[m][0] : 0.f; v.y = (hmask >> (4 * m + 1)) & 1u ? acc1[m][1] : 0.f;
        v.z = (hmask >> (4 * m + 2)) & 1u ? acc1[m][2] : 0.f; v.w = (hmask >> (4 * m + 3)) & 1u ? acc1[m][3] : 0.f;
        *reinterpret_cast<float4*>(myGH + m * HID + 4 * lane) = v;
      }
      fence_proxy_async();
      __syncwarp();
      if (issuer) bulk_store_512(hgh_row + HID, myGH + lane * HID);
      if (lane < G) bulk_commit();
      {
        float gy[3][MPL];
#pragma unroll
        for (int kb = 0; kb < 3; ++kb)
#pragma unroll
          for (int e = 0; e < MPL; ++e) gy[kb][e] = 0.f;
        const float* w0 = sW1T + c * kQW1S;
#pragma unroll 2
        for (int i = 0; i < HID / 4; ++i) {
          float4 gv[MPL];
#pragma unroll
          for (int e = 0; e < MPL; ++e) gv[e] = *reinterpret_cast<const float4*>(myGH + (hwi + CPL * e) * HID + 4 * i);
#pragma unroll
          for (int kb = 0; kb < 3; ++kb) {
            const float4 w = *reinterpret_cast<const float4*>(w0 + kb * C * kQW1S + 4 * i);
#pragma unroll
            for (int e = 0; e < MPL; ++e)
              gy[kb][e] = fmaf(w.x, gv[e].x, fmaf(w.y, gv[e].y, fmaf(w.z, gv[e].z, fmaf(w.w, gv[e].w, gy[kb][e]))));
          }
        }
#pragma unroll
        for (int kb = 0; kb < 3; ++kb)
#pragma unroll
          for (int e = 0; e < MPL; ++e)
            if (valid[e]) RGs[(size_t)cellr[e] * 64 + kb * C + c] = gy[kb][e];
      }
#pragma unroll
      for (int r = 0; r < MPL; ++r)
        if (valid[r]) RGs[(size_t)cellr[r] * 64 + 3 * C + c] = gxs[r];
      __syncwarp();
    };
    {
      const int w_lo = (n_my * warp) >> 4, w_hi = (n_my * (warp + 1)) >> 4;
#pragma unroll 1
      for (int s0 = w_lo; s0 < w_hi;) {
        const int rem = w_hi - s0;
        if (rem > 4 && R.gmax >= 8) { bwd_tile(std::integral_constant<int, 8>{}, s0, w_hi); s0 += 8; }
        else if (rem > 2) { bwd_tile(std::integral_constant<int, 4>{}, s0, w_hi); s0 += 4; }
        else { bwd_tile(std::integral_constant<int, 2>{}, s0, w_hi); s0 += 2; }
      }
    }
    REPB_MARK(6);
    cluster_sync_acquire();                                                   // ---- cluster barrier 2: RG visible
    REPB_MARK(7);
    // ---- C: my band: g_t = gated g_{t+1} + perception^T (gy of active neighbours) + message^T (g_xs of receivers) --
    float gwp[ZP ? 16 : 1];                  // ZP: this thread's share of dL/dw_i
#pragma unroll
    for (int i = 0; i < (ZP ? 16 : 1); ++i) gwp[i] = 0.f;
    {
      const float wuni = k > 0 ? 1.0f / (float)k : 0.f;
      auto actbit = [&](int cell) -> bool { return (s_bAct[cell >> 5] >> (cell & 31)) & 1u; };
#pragma unroll 1
      for (int it = tid; it < nband * 4; it += kQT) {
        const int cl = it >> 2, cq = it & 3;
        const int cell = band_lo + cl, py = cell / W, px = cell - py * W;
        float4 g = *reinterpret_cast<const float4*>(sG + cl * C + 4 * cq);
        if (cq == 0 && !((s_bPost[cell >> 5] >> (cell & 31)) & 1u)) g.w = 0.f;
        // active neighbours as a 9-bit mask, then ALL loads of the item are issued before the first use (predicated, no
        // branches between them): one L2 round trip per item instead of one per neighbour
        uint32_t nbm = 0;
#pragma unroll
        for (int ay = -1; ay <= 1; ++ay)
#pragma unroll
          for (int ax = -1; ax <= 1; ++ax) {
            const int yy = py + ay, xx = px + ax;
            const bool inb = yy >= 0 && yy < H && xx >= 0 && xx < W;
            const int ac = inb ? yy * W + xx : cell;
            nbm |= (inb && actbit(ac)) ? (1u << ((ay + 1) * 3 + (ax + 1))) : 0u;
          }
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        float4 vid = z4, vsx[6], vsy[6];
        if (nbm & (1u << 4)) vid = __ldcg(reinterpret_cast<const float4*>(RGs + (size_t)cell * 64 + 4 * cq));
        {
          int ix = 0, iy = 0;
#pragma unroll
          for (int ay = -1; ay <= 1; ++ay)
#pragma unroll
            for (int ax = -1; ax <= 1; ++ax) {
              const bool on = (nbm >> ((ay + 1) * 3 + (ax + 1))) & 1u;
              const float* rg = RGs + (size_t)(cell + ay * W + ax) * 64 + 4 * cq;
              if (ax != 0) { vsx[ix] = on ? __ldcg(reinterpret_cast<const float4*>(rg + C)) : z4; ++ix; }
              if (ay != 0) { vsy[iy] = on ? __ldcg(reinterpret_cast<const float4*>(rg + 2 * C)) : z4; ++iy; }
            }
        }
        uint32_t rm = 0;
        int rcell[16];
        const bool sender = msg_on && (!a2a || ((s_bAS[cell >> 5] >> (cell & 31)) & 1u));
        if (sender) {
          if constexpr (ZP) {
            // receiver (y + dy_i, x): dx is a no-op, a receiver outside the grid does not exist
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              rcell[i] = cell;
              if (i < k) {
                const int ry = py + (int)s_off[2 * i];
                const bool inside = ry >= 0 && ry < H;
                rcell[i] = inside ? ry * W + px : cell;
                rm |= (inside && actbit(rcell[i])) ? (1u << i) : 0u;
              }
            }
          } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            rcell[i] = cell;
            if (i < k) {
              int ry = py + (int)s_off[2 * i], rx = px + (int)s_off[2 * i + 1];
              ry += ry < 0 ? H : 0; ry -= ry >= H ? H : 0;
              rx += rx < 0 ? W : 0; rx -= rx >= W ? W : 0;
              rcell[i] = ry * W + rx;
              rm |= actbit(rcell[i]) ? (1u << i) : 0u;
            }
          }
          }
        }
        g.x += vid.x; g.y += vid.y; g.z += vid.z; g.w += vid.w;
        {
          int ix = 0, iy = 0;
#pragma unroll
          for (int ay = -1; ay <= 1; ++ay)
#pragma unroll
            for (int ax = -1; ax <= 1; ++ax) {
              if (ax != 0) {
                const float kx = (ax > 0 ? 1.f : -1.f) * (ay == 0 ? 2.f : 1.f);
                g.x = fmaf(kx, vsx[ix].x, g.x); g.y = fmaf(kx, vsx[ix].y, g.y);
                g.z = fmaf(kx, vsx[ix].z, g.z); g.w = fmaf(kx, vsx[ix].w, g.w);
                ++ix;
              }
              if (ay != 0) {
                const float ky = (ay > 0 ? 1.f : -1.f) * (ax == 0 ? 2.f : 1.f);
                g.x = fmaf(ky, vsy[iy].x, g.x); g.y = fmaf(ky, vsy[iy].y, g.y);
                g.z = fmaf(ky, vsy[iy].z, g.z); g.w = fmaf(ky, vsy[iy].w, g.w);
                ++iy;
              }
            }
        }
        if (rm) {
          float4 vr[16];
#pragma unroll
          for (int i = 0; i < 16; ++i)
            vr[i] = (rm >> i) & 1u ? __ldcg(reinterpret_cast<const float4*>(RGs + (size_t)rcell[i] * 64 + 3 * C + 4 * cq)) : z4;
          if constexpr (ZP) {
            // x_t of my 4 channels of the sender, and bm . gm of the receivers (counted once, by the quad-0 thread)
            const float* xs = Z.x + ((size_t)t * a.B + b) * C * HW + (size_t)(4 * cq) * HW + cell;
            const float x0 = __ldcg(xs), x1 = __ldcg(xs + HW), x2 = __ldcg(xs + 2 * HW), x3 = __ldcg(xs + 3 * HW);
            float bgr[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) bgr[i] = (cq == 0 && ((rm >> i) & 1u)) ? __ldcg(Z.bg + (size_t)b * HW + rcell[i]) : 0.f;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float wi = zw[i];
              g.x = fmaf(wi, vr[i].x, g.x); g.y = fmaf(wi, vr[i].y, g.y);
              g.z = fmaf(wi, vr[i].z, g.z); g.w = fmaf(wi, vr[i].w, g.w);
              gwp[i] += fmaf(vr[i].x, x0, fmaf(vr[i].y, x1, fmaf(vr[i].z, x2, fmaf(vr[i].w, x3, bgr[i]))));
            }
          } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            g.x = fmaf(wuni, vr[i].x, g.x); g.y = fmaf(wuni, vr[i].y, g.y);
            g.z = fmaf(wuni, vr[i].z, g.z); g.w = fmaf(wuni, vr[i].w, g.w);
          }
          }
        }
        if constexpr (kFrames) {
          if (gfr) {
            const float* gf = gfr + (size_t)(4 * cq) * HW + cell;
            g.x += __ldg(gf); g.y += __ldg(gf + HW); g.z += __ldg(gf + 2 * HW); g.w += __ldg(gf + 3 * HW);
          }
        }
        if (dmg) {
          g.x *= R.damage.at(b, 4 * cq, cell, C, HW); g.y *= R.damage.at(b, 4 * cq + 1, cell, C, HW);
          g.z *= R.damage.at(b, 4 * cq + 2, cell, C, HW); g.w *= R.damage.at(b, 4 * cq + 3, cell, C, HW);
        }
        *reinterpret_cast<float4*>(sG + cl * C + 4 * cq) = g;
      }
    }
    __syncthreads();
    REPB_MARK(8);
    if (R.dbg && tid == 0) s_dbg[9] += n_my;
    (void)nact;
    if constexpr (ZP) {
      if (msg_on) {
        // ---- dL/dw_i: lanes -> warps -> CTA -> every CTA of the cluster, each level in a fixed order ----------------
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float v = warp_sum(gwp[i]);
          if (lane == 0) zgww[warp * 16 + i] = v;
        }
        __syncthreads();
        if (tid < 16) {
          float v = 0.f;
          for (int w = 0; w < kQW; ++w) v += zgww[w * 16 + tid];
          for (int r = 0; r < NC; ++r) cluster.map_shared_rank(zgwc, r)[rank * 16 + tid] = v;
        }
        const float* rsg = Z.rowsum + ((size_t)t * a.B + b) * C * H;
        for (int i = tid; i < C * H; i += kQT) zrs[i] = __ldcg(rsg + i);
        cluster_sync_acquire();                                               // ---- cluster barrier 3: dL/dw_i partials
        // ---- softmax / pooled Q.K backward of the step (k_attn_bwd), redundantly on every CTA -----------------------
        const int d = Z.d;
        const float invHW = 1.0f / (float)HW;
        if (tid < k) {
          float gw = 0.f;
          for (int r = 0; r < NC; ++r) gw += zgwc[r * 16 + tid];
          zgL[tid] = gw;
          const int dy = (int)s_off[2 * tid];
          const int lo = max(0, -dy), hi = min(H, H - dy);
          zrlo[tid] = lo; zrhi[tid] = max(lo, hi);
        }
        __syncthreads();
        if (tid < C) {
          float sacc = 0.f;
          for (int y = 0; y < H; ++y) sacc += zrs[tid * H + y];
          zxbar[tid] = sacc * invHW;
        }
        for (int idx = tid; idx < k * C; idx += kQT) {
          const int i = idx / C, cc = idx % C;
          float sacc = 0.f;
          for (int y = zrlo[i]; y < zrhi[i]; ++y) sacc += zrs[cc * H + y];
          zS[idx] = sacc;
        }
        __syncthreads();
        if (tid < d) {
          float sacc = 0.f;
          for (int cc = 0; cc < C; ++cc) sacc = fmaf(__ldg(packed + P.wq + tid * C + cc), zxbar[cc], sacc);
          zqp[tid] = sacc + __ldg(packed + P.bq + tid);
        }
        for (int idx = tid; idx < k * d; idx += kQT) {
          const int i = idx / d, j = idx % d;
          float sacc = 0.f;
          for (int cc = 0; cc < C; ++cc) sacc = fmaf(__ldg(packed + P.wk + j * C + cc), zS[i * C + cc], sacc);
          zKP[i * 32 + j] = (sacc + (float)(zrhi[i] - zrlo[i]) * (float)W * __ldg(packed + P.bk + j)) * invHW;
        }
        __syncthreads();
        if (tid < C) {
          float sacc = 0.f;
          for (int j = 0; j < d; ++j) sacc = fmaf(__ldg(packed + P.wk + j * C + tid), zqp[j], sacc);
          zwkq[tid] = sacc;
        }
        if (tid >= 32 && tid < 32 + k) {
          const int i = tid - 32;
          float sacc = 0.f;
          for (int j = 0; j < d; ++j) sacc = fmaf(zqp[j], zKP[i * 32 + j], sacc);
          zlg[i] = sacc;
        }
        __syncthreads();
        if (tid == 0) {                      // the forward's weights; logits only for dL/dscaling
          float mx = -INFINITY;
          for (int i = 0; i < k; ++i) mx = fmaxf(mx, zlg[i]);
          const float sc = packed[P.scaling];
          const float tau = fabsf(sc) + 1e-6f;
          float dot = 0.f;
          for (int i = 0; i < k; ++i) dot = fmaf(zw[i], zgL[i], dot);
          float gtau = 0.f;
          for (int i = 0; i < k; ++i) {
            const float ga = zw[i] * (zgL[i] - dot);
            gtau -= ga * ((zlg[i] - mx) / tau) / tau;
            zgL[i] = ga / tau;               // dL/dlogit_i
          }
          zmisc[0] = gtau * (sc >= 0.f ? 1.f : -1.f);
        }
        __syncthreads();
        if (tid < d) {
          float sacc = 0.f;
          for (int i = 0; i < k; ++i) sacc = fmaf(zgL[i], zKP[i * 32 + tid], sacc);
          zgqp[tid] = sacc;
        }
        if (tid >= 64 && tid < 64 + H) {
          const int y = tid - 64;
          float sacc = 0.f;
          for (int i = 0; i < k; ++i) if (y >= zrlo[i] && y < zrhi[i]) sacc += zgL[i];
          zsL[y] = sacc;
        }
        __syncthreads();
        if (tid < C) {
          float sacc = 0.f;
          for (int j = 0; j < d; ++j) sacc = fmaf(__ldg(packed + P.wq + j * C + tid), zgqp[j], sacc);
          zgxb[tid] = sacc;
        }
        __syncthreads();
        // grow = dL/dx_t through the pooled Q / K, for every cell alive or not; part of dL/dx_t, so the damage mask of
        // step t multiplies it like the rest of g_t (phase C applied it to the rest)
#pragma unroll 1
        for (int i = tid; i < nband * C; i += kQT) {
          const int cl = i / C, ch = i - cl * C;
          const int cell = band_lo + cl;
          float v = (zgxb[ch] + zwkq[ch] * zsL[cell / W]) * invHW;
          if (dmg) v *= R.damage.at(b, ch, cell, C, HW);
          sG[i] += v;
        }
        if (rank == 0) {                     // per-sample Q/K/scaling gradients, summed over the steps
          float* pwb = Z.pw + (size_t)b * (2 * d * C + 2 * d + 1);
          for (int idx = tid; idx < d * C; idx += kQT) {
            const int j = idx / C, ch = idx % C;
            pwb[idx] += zgqp[j] * zxbar[ch];
            float sacc = 0.f;
            for (int i = 0; i < k; ++i) sacc = fmaf(zgL[i], zS[i * C + ch], sacc);
            pwb[d * C + d + idx] += zqp[j] * sacc * invHW;
          }
          for (int j = tid; j < d; j += kQT) {
            pwb[d * C + j] += zgqp[j];
            float sacc = 0.f;
            for (int i = 0; i < k; ++i) sacc += zgL[i] * (float)(zrhi[i] - zrlo[i]);
            pwb[2 * d * C + d + j] += zqp[j] * sacc * (float)W * invHW;
          }
          if (tid == 0) pwb[2 * d * C + 2 * d] += zmisc[0];
        }
        __syncthreads();
      }
    }
  }

  // dL/dx_0 (NCHW) from my band; per-CTA dgamma / dbeta partials
  __syncthreads();
  {
    const int n8 = (nband + 7) & ~7;
#pragma unroll 1
    for (int i = tid; i < n8 * C; i += kQT) {
      const int ci = i & 7, c4 = (i >> 3) & 3, rest = i >> 5;
      const int cq = rest & 3, cgp = rest >> 2;
      const int cl = cgp * 8 + ci, ch = cq * 4 + c4;
      if (cl < nband) R.g0[sample_off + (size_t)ch * HW + band_lo + cl] = sG[cl * C + ch];
    }
  }
  if (R.dbg && blockIdx.x == R.dbg_cta && tid < 16) R.dbg[tid] = s_dbg[tid];
  dgam += __shfl_xor_sync(0xffffffffu, dgam, 16);
  dbet += __shfl_xor_sync(0xffffffffu, dbet, 16);
  if (lane < C) { s_chs[warp][0][lane] = dgam; s_chs[warp][1][lane] = dbet; }
  __syncthreads();
  if (tid < 2 * C) {
    const int which = tid / C, ch = tid % C;
    float ac = 0.f;
    for (int w = 0; w < kQW; ++w) ac += s_chs[w][which][ch];
    R.affpart[(size_t)blockIdx.x * 2 * C + tid] = ac;
  }
  if (lane < 8) bulk_wait_all();               // every h | gh row has reached global memory before the kernel ends
  cluster_sync_acquire();
}

// ------------------------------------------------------------------------------------------------
// Weight gradients from the records, all steps at once.
// ------------------------------------------------------------------------------------------------
constexpr int kWT = 256;          // threads
constexpr int kWNB = 32;          // records per batch
constexpr int kWMaxSeg = 256;     // (t, b) segments per block and round

struct WgradArgs {
  const float* rec;
  const float* hgh;
  const uint32_t* masks;
  const int32_t* steps;       // [B] or null (absolute step counts)
  int T, B, HW, NW;
  int t0;                     // absolute step of record step 0
  uint32_t flags;
  float* wpart;               // [gridDim.x][wtotal]
  int64_t wtotal;
  gnca_layout L;
  // a stack of models: samples [i*per, (i+1)*per) run model i, and blocks [i*nbm, (i+1)*nbm) sum its records only.
  // (read by the MS instantiation only)
  int per, nbm;
};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// dW1 += gh (x) y, db1 += gh, dW2 += gd (x) h, dWm += gm (x) xs, dbm += gm * as over all records: operands are read
// record-major straight from the cp.async buffers (a thread's 4 hidden units are one float4 of the permuted h / gh rows).
template <int C, bool MS>
__global__ void __launch_bounds__(kWT, 2) k_rep_wgrad(WgradArgs A) {
  constexpr int C3 = 3 * C, HID = 128, NB = kWNB;
  constexpr int TK = 6, KG = C3 / TK;          // dW1 tile: 4 hidden units (one permuted float4) x 6 consecutive inputs
  constexpr int JQ = HID / 4;
  constexpr int RAWR = NB * kRecStride, RAWH = NB * kHghStride;
  static_assert(JQ * KG == kWT, "dW1 tiling");
  const bool graph = (A.flags & GNCA_F_GRAPH) != 0;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* RAW = reinterpret_cast<float*>(smem_raw);      // [2][NB][kRecStride]
  float* RH = RAW + 2 * RAWR;                           // [2][NB][kHghStride]
  __shared__ int s_cnt[kWMaxSeg];
  const int tid = threadIdx.x;

  float aW1[4][TK], ab1[4], aW2[4][2], aWm = 0.f, abm = 0.f;
#pragma unroll
  for (int jj = 0; jj < 4; ++jj) { ab1[jj] = 0.f; aW2[jj][0] = aW2[jj][1] = 0.f; for (int kk = 0; kk < TK; ++kk) aW1[jj][kk] = 0.f; }
  const int kg = tid % KG, jg = tid / KG;               // dW1: units jg + 32 jj (float4 at 4 jg), inputs 6 kg .. 6 kg + 5
  const int cp2 = tid % (C / 2), jg2 = tid / (C / 2);   // dW2: channels 2 cp2, 2 cp2 + 1, units jg2 + 32 jj
  const int mc = tid / C, mci = tid % C;                // dWm[mc][mci]

  // MS: my model's segments (t, b), b in [model*per, (model+1)*per), in the local order ls = t*per + (b - model*per); I
  // take ls = lb, lb + nbm, ...  With one model that is the partition of the plain instantiation (ls = t*B + b), which
  // keeps the single-model code without the mapping
  const unsigned nbm = MS ? (unsigned)A.nbm : gridDim.x;
  const int model = MS ? (int)blockIdx.x / A.nbm : 0;
  const int lb = MS ? (int)blockIdx.x - model * A.nbm : blockIdx.x;
  const int nseg = A.T * (MS ? A.per : A.B);
  auto gseg = [&](int ls) {
    if constexpr (MS) { const int t = ls / A.per; return t * A.B + model * A.per + (ls - t * A.per); }
    return ls;
  };
  for (int seg0 = lb; seg0 < nseg; seg0 += nbm * kWMaxSeg) {
    __syncthreads();
    for (int si = tid; si < kWMaxSeg; si += kWT) {        // record counts of my segments (popcount of the active bitmap)
      const int ls = seg0 + si * nbm;
      int cnt = 0;
      if (ls < nseg) {
        const int seg = gseg(ls);
        const int t = seg / A.B, b = seg - t * A.B;
        if (!(A.steps && A.steps[b] - A.t0 <= t)) {
          const uint32_t* mk = A.masks + ((size_t)seg * 3 + 1) * kMaskWords;
          for (int i = 0; i < A.NW; ++i) cnt += __popc(__ldg(mk + i));
        }
      }
      s_cnt[si] = cnt;
    }
    __syncthreads();
    int si = 0, base = 0;
    auto skip_empty = [&](int& s_, int& b_) { while (s_ < kWMaxSeg && b_ >= s_cnt[s_]) { ++s_; b_ = 0; } };
    auto issue = [&](int s_, int b_, int buf) {
      if (s_ < kWMaxSeg) {
        const int seg = gseg(seg0 + s_ * nbm);
        const int nb = min(NB, s_cnt[s_] - b_);
        const float* src = A.rec + ((size_t)seg * A.HW + b_) * kRecStride;
        const float* srch = A.hgh + ((size_t)seg * A.HW + b_) * kHghStride;
        float* dst = RAW + buf * RAWR;
        float* dsth = RH + buf * RAWH;
        for (int i = tid; i < nb * (kRecStride / 4); i += kWT) cp_async16(dst + 4 * i, src + 4 * i);
        for (int i = tid; i < nb * (kHghStride / 4); i += kWT) cp_async16(dsth + 4 * i, srch + 4 * i);
      }
      cp_async_commit();
    };
    skip_empty(si, base);
    issue(si, base, 0);
    int buf = 0;
    while (si < kWMaxSeg) {
      const int nb = min(NB, s_cnt[si] - base);
      int nsi = si, nbase = base + NB;
      skip_empty(nsi, nbase);
      issue(nsi, nbase, buf ^ 1);
      cp_async_wait<1>();
      __syncthreads();                                   // this batch has landed
      const float* raw = RAW + buf * RAWR;
      const float* rh = RH + buf * RAWH;
#pragma unroll 4
      for (int cl = 0; cl < nb; ++cl) {
        const float* rc = raw + cl * kRecStride;
        const float4 g = *reinterpret_cast<const float4*>(rh + cl * kHghStride + HID + 4 * jg);
        const float2 y01 = *reinterpret_cast<const float2*>(rc + TK * kg);
        const float2 y23 = *reinterpret_cast<const float2*>(rc + TK * kg + 2);
        const float2 y45 = *reinterpret_cast<const float2*>(rc + TK * kg + 4);
        const float gj[4] = {g.x, g.y, g.z, g.w};
        const float yk[TK] = {y01.x, y01.y, y23.x, y23.y, y45.x, y45.y};
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
#pragma unroll
          for (int kk = 0; kk < TK; ++kk) aW1[jj][kk] = fmaf(gj[jj], yk[kk], aW1[jj][kk]);
          if (kg == 0) ab1[jj] += gj[jj];
        }
        const float4 hv = *reinterpret_cast<const float4*>(rh + cl * kHghStride + 4 * jg2);
        const float2 gd2 = *reinterpret_cast<const float2*>(rc + kRecU + 2 * cp2);
        const float hj[4] = {hv.x, hv.y, hv.z, hv.w};
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          aW2[jj][0] = fmaf(gd2.x, hj[jj], aW2[jj][0]);
          aW2[jj][1] = fmaf(gd2.y, hj[jj], aW2[jj][1]);
        }
        if (graph) {
          const float gmv = rc[kRecTh + mc];
          aWm = fmaf(gmv, rc[kRecXs + mci], aWm);
          if (mci == 0) abm = fmaf(gmv, rc[kRecAs], abm);
        }
      }
      __syncthreads();                                   // everybody is done with this buffer before it is refilled
      si = nsi; base = nbase; buf ^= 1;
    }
    cp_async_wait<0>();
  }
  // one partial per block (canonical layout)
  float* wp = A.wpart + (size_t)blockIdx.x * A.wtotal;
#pragma unroll
  for (int jj = 0; jj < 4; ++jj) {
    const int j = jg + JQ * jj;
#pragma unroll
    for (int kk = 0; kk < TK; ++kk) wp[A.L.w1 + (int64_t)j * C3 + (TK * kg + kk)] = aW1[jj][kk];
    if (kg == 0) wp[A.L.b1 + j] = ab1[jj];
    wp[A.L.w2 + (int64_t)(2 * cp2) * HID + (jg2 + JQ * jj)] = aW2[jj][0];
    wp[A.L.w2 + (int64_t)(2 * cp2 + 1) * HID + (jg2 + JQ * jj)] = aW2[jj][1];
  }
  if (graph) {
    wp[A.L.wm + mc * C + mci] = aWm;
    if (mci == 0) wp[A.L.bm + mc] = abm;
  }
}

// gparams[i] += sum over blocks of wpart[blk][i] (fixed order); + dgamma / dbeta partials of the resident kernel.
// MS: blockIdx.y = model of a stack: its nblk partials, its naff affine partials (its samples' CTAs) and its gparams row
template <bool MS>
__global__ void k_rep_wreduce(int nblk, int64_t total, const float* __restrict__ wpart, int naff, int C,
                              const float* __restrict__ affpart, gnca_layout L, float* __restrict__ gparams) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  if constexpr (MS) {
    wpart += (size_t)blockIdx.y * nblk * total;
    affpart += (size_t)blockIdx.y * naff * 2 * C;
    gparams += (size_t)blockIdx.y * total;
  }
  float acc = 0.f;
  for (int bl = 0; bl < nblk; ++bl) acc += wpart[(size_t)bl * total + i];
  if (i >= L.gamma && i < L.gamma + C) for (int r = 0; r < naff; ++r) acc += affpart[(size_t)r * 2 * C + (i - L.gamma)];
  if (i >= L.beta && i < L.beta + C) for (int r = 0; r < naff; ++r) acc += affpart[(size_t)r * 2 * C + C + (i - L.beta)];
  gparams[i] += acc;
}

// ------------------------------------------------------------------------------------------------
static size_t rep_bwd_smem_bytes(int C, int HW, int NC, int gmax) {
  const int bandcap = ((HW + NC - 1) / NC) + 1;
  size_t f = (size_t)3 * C * kQW1S + 128 + 128 * kQW2S + (size_t)bandcap * C + (size_t)kQW * 3 * C * gmax + (size_t)kQW * C * gmax +
             (size_t)kQW * gmax * 128;
  return f * sizeof(float) + 2 * (size_t)((bandcap + 7) & ~7) * sizeof(unsigned short) + 32;
}

size_t rep_bptt_bytes(const gnca_model& m, int B, int H, int W, int T) {
  if (m.C != 16 || m.hidden != 128 || H > 64 || W > 64 || W < 4 || (W & 3) || H * W > 2048) return 0;
  const size_t HW = (size_t)H * W;
  size_t bytes = (size_t)T * B * HW * kRecStride * sizeof(float);
  bytes = (bytes + 255) & ~(size_t)255;
  bytes += (size_t)T * B * HW * kHghStride * sizeof(float);
  bytes += (size_t)T * B * 3 * kMaskWords * sizeof(uint32_t);
  bytes += (size_t)T * B * 2 * sizeof(float) + 256;
  return bytes;
}

void rep_bptt_carve(void* base, int B, int H, int W, int T, float** rec, uint32_t** masks, float** stats, float** hgh) {
  const size_t HW = (size_t)H * W;
  char* p = reinterpret_cast<char*>(base);
  size_t o = (size_t)T * B * HW * kRecStride * sizeof(float);
  o = (o + 255) & ~(size_t)255;
  *rec = reinterpret_cast<float*>(p);
  if (hgh) *hgh = reinterpret_cast<float*>(p + o);
  o += (size_t)T * B * HW * kHghStride * sizeof(float);
  *masks = reinterpret_cast<uint32_t*>(p + o);
  o += (size_t)T * B * 3 * kMaskWords * sizeof(uint32_t);
  *stats = reinterpret_cast<float*>(p + o);
}

// a stack of n_models runs wgrad_blocks_per_model blocks per model: at most kMaxWgradBlocks in all, and at least one each
static int wgrad_blocks_per_model(int T, int per, int n_models) {
  const int seg = T * per, cap = kMaxWgradBlocks / n_models;
  const int n = seg < cap ? seg : cap;
  return n < 1 ? 1 : n;
}

size_t rep_bwd_workspace_bytes(const gnca_model& m, int B, int H, int W, int n_models) {
  const size_t HW = (size_t)H * W, C = m.C;
  size_t f = (size_t)B * HW * C /*GZ*/ + (size_t)B * HW * 64 /*RG*/ + (size_t)B * 8 * 2 * C;
  const gnca_layout L = make_layout(m);
  f += (size_t)(n_models > kMaxWgradBlocks ? n_models : kMaxWgradBlocks) * (size_t)L.total;
  return f * sizeof(float) + 1024;
}

// cluster size / tile size / shared memory of k_rep_bwd for a batch: the largest NC in {8,4,2,1} whose bands start at a
// quad boundary, that fits shared memory (220 KB dynamic + ~4 KB static) and keeps all B clusters co-resident; else the
// smallest NC that fits (waves).  Returns false when nothing fits.
static bool pick_rep_bwd_config(int B, int HW, cudaStream_t st, int* out_nc, int* out_gmax, size_t* out_smem,
                                bool zp = false) {
  const int C = 16;
  // the zero-padded-shift instantiation carries the attention-backward scratch behind the plain carve
  const size_t zsm = zp ? (size_t)kZpSmemFloats * sizeof(float) : 0;
  const void* kfn = zp ? (const void*)k_rep_bwd<16, false, true> : (const void*)k_rep_bwd<16, false, false>;
  const char* env_nc = getenv("GNCA_RESIDENT_NC");
  const int cands[4] = {8, 4, 2, 1};
  int pick = -1, pick_gmax = 8;
  size_t pick_smem = 0;
  for (int pass = 0; pass < 2 && pick < 0; ++pass) {
    for (int ci = (pass == 0 ? 0 : 3); ci >= 0 && ci < 4; ci += (pass == 0 ? 1 : -1)) {
      const int NC = cands[ci];
      if (env_nc && atoi(env_nc) != NC) continue;
      if ((HW % (4 * NC)) != 0) continue;                 // bands start at a quad boundary
      int gmax = 8;
      size_t smem = rep_bwd_smem_bytes(C, HW, NC, gmax) + zsm;
      if (smem > 220 * 1024) { gmax = 4; smem = rep_bwd_smem_bytes(C, HW, NC, gmax) + zsm; }
      if (smem > 220 * 1024) continue;
      if (cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        cudaGetLastError();
        continue;
      }
      cudaLaunchConfig_t q{};
      q.gridDim = dim3(B * NC); q.blockDim = dim3(kQT); q.dynamicSmemBytes = smem; q.stream = st;
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = NC; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
      q.attrs = qa; q.numAttrs = 1;
      int ncl = 0;
      if (cudaOccupancyMaxActiveClusters(&ncl, kfn, &q) != cudaSuccess || ncl < 1) {
        cudaGetLastError();
        continue;
      }
      if (pass == 0 && B > ncl && !env_nc) continue;
      pick = NC; pick_smem = smem; pick_gmax = gmax;
      break;
    }
  }
  if (pick < 0) return false;
  *out_nc = pick; *out_gmax = pick_gmax; *out_smem = pick_smem;
  return true;
}

bool rep_bwd_supported(const gnca_model& m, int B, int H, int W, int k, bool zp) {
  if (rep_bptt_bytes(m, B, H, W, 1) == 0 || k > 16) return false;
  int nc, gmax;
  size_t smem;
  return pick_rep_bwd_config(B, H * W, nullptr, &nc, &gmax, &smem, zp && k > 0);
}

static inline size_t zp_al(size_t v) { return (v + 255) & ~(size_t)255; }

size_t rep_bptt_zp_bytes(const gnca_model& m, int B, int H, int W, int T) {
  if (!(m.flags & GNCA_F_GRAPH) || (m.flags & GNCA_F_TORUS) || m.d_model < 1 || m.d_model > 32) return 0;
  const size_t base = rep_bptt_bytes(m, B, H, W, T);
  if (base == 0) return 0;
  const size_t HW = (size_t)H * W, C = m.C, np = 2 * (size_t)m.d_model * C + 2 * (size_t)m.d_model + 1;
  return zp_al(base) + zp_al((size_t)(T + 1) * B * C * HW * 4) + zp_al((size_t)T * B * 16 * 4) +
         zp_al((size_t)T * B * C * H * 4) + zp_al((size_t)B * HW * 4) + zp_al((size_t)B * np * 4);
}

void rep_bptt_zp_carve(void* base, const gnca_model& m, int B, int H, int W, int T, float** x, ZpRec* rec, ZpBwd* bwd) {
  const size_t HW = (size_t)H * W, C = m.C;
  char* p = reinterpret_cast<char*>(base);
  size_t o = zp_al(rep_bptt_bytes(m, B, H, W, T));
  float* xs = reinterpret_cast<float*>(p + o); o += zp_al((size_t)(T + 1) * B * C * HW * 4);
  float* w = reinterpret_cast<float*>(p + o); o += zp_al((size_t)T * B * 16 * 4);
  float* rs = reinterpret_cast<float*>(p + o); o += zp_al((size_t)T * B * C * H * 4);
  float* bg = reinterpret_cast<float*>(p + o); o += zp_al((size_t)B * HW * 4);
  float* pw = reinterpret_cast<float*>(p + o);
  if (x) *x = xs;
  if (rec) *rec = ZpRec{w, rs};
  if (bwd) *bwd = ZpBwd{xs, w, rs, bg, pw, m.d_model};
}

int run_rep_bwd(const gnca_model& m, const Packed& P, const float* packed, int B, int H, int W,
                const gnca_schedule& sched, void* bptt, const float* gT, float* g0, float* gparams, void* workspace,
                cudaStream_t st, const float* g_frames, int every, int t0, const ZpBwd* zp, bool gT_frame,
                ModelStack ms) {
  const bool graph = (m.flags & GNCA_F_GRAPH) != 0;
  if (rep_bptt_bytes(m, B, H, W, sched.T) == 0) return GNCA_ERR_UNSUPPORTED;
  if (ms.stride && g_frames) return GNCA_ERR_UNSUPPORTED;      // a stack has no frame gradients
  const int k = graph ? sched.k : 0;
  if (graph && k > 0 && !(m.flags & GNCA_F_TORUS) && !zp) return GNCA_ERR_UNSUPPORTED;
  if (k > 16) return GNCA_ERR_UNSUPPORTED;
  const bool zpk = zp && graph && k > 0 && !(m.flags & GNCA_F_TORUS);   // the attention backward runs
  const int C = 16, HW = H * W;
  float *rec, *stats, *hgh;
  uint32_t* masks;
  rep_bptt_carve(bptt, B, H, W, sched.T, &rec, &masks, &stats, &hgh);
  const gnca_layout L = make_layout(m);
  float* ws = reinterpret_cast<float*>(workspace);
  float* GZ = ws; ws += (size_t)B * HW * C;
  float* RG = ws; ws += (size_t)B * HW * 64;
  float* affpart = ws; ws += (size_t)B * 8 * 2 * C;
  float* wpart = ws;

  RepBwdArgs R{};
  fill_step_args(R.s, m, B, H, W);
  R.s.k = k;
  R.s.message_gain_dev = sched.message_gain;
  R.s.offsets_dev = sched.offsets;
  R.s.steps = sched.steps;
  R.T = sched.T;
  R.t0 = t0;
  R.gT_frame = gT_frame ? 1 : 0;
  R.inv_n = (float)(1.0 / ((double)C * (double)H * (double)W));
  R.rec = rec; R.hgh = hgh; R.masks = masks; R.stats = stats; R.gT = gT; R.g0 = g0; R.GZ = GZ; R.RG = RG;
  R.affpart = affpart;
  R.damage = DamageView{sched.damage, sched.damage_layout}; R.damage_step = sched.damage_step;

  int pick = -1, pick_gmax = 8;
  size_t pick_smem = 0;
  if (!pick_rep_bwd_config(B, HW, st, &pick, &pick_gmax, &pick_smem, zpk)) pick = -1;
  if (pick < 0) return GNCA_ERR_UNSUPPORTED;
  R.NC = pick; R.gmax = pick_gmax;
  if (getenv("GNCA_DEBUG")) fprintf(stderr, "[gnca] resident bwd: B=%d NC=%d smem=%zu\n", B, pick, pick_smem);
  // the frame-gradient instantiation has the register budget and shared memory of the plain one (same launch bounds,
  // same carve), so the configuration picked for the plain kernel holds for it
  // so does the stacked one (MS)
  const auto kern = ms.stride ? (zpk ? k_rep_bwd<16, false, true, true> : k_rep_bwd<16, false, false, true>)
                  : zpk ? (g_frames ? k_rep_bwd<16, true, true> : k_rep_bwd<16, false, true>)
                        : (g_frames ? k_rep_bwd<16, true, false> : k_rep_bwd<16, false, false>);
  const ZpBwd Z = zpk ? *zp : ZpBwd{};
  const int np = 2 * m.d_model * C + 2 * m.d_model + 1;
  if (zpk) GNCA_CHECK_CUDA(cudaMemsetAsync(Z.pw, 0, (size_t)B * np * sizeof(float), st));
  GNCA_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pick_smem));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(B * pick);
  cfg.blockDim = dim3(kQT);
  cfg.dynamicSmemBytes = pick_smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = pick; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  static unsigned long long* dbg_buf = nullptr;
  if (getenv("GNCA_PHASE_TIMING")) {
    if (!dbg_buf) cudaMalloc(&dbg_buf, 16 * sizeof(unsigned long long));
    cudaMemsetAsync(dbg_buf, 0, 16 * sizeof(unsigned long long), st);
    R.dbg = dbg_buf;
    R.dbg_cta = atoi(getenv("GNCA_PHASE_TIMING"));
  }
  prof_begin(PROF_RESIDENT_BWD, st);
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, R, P, packed, g_frames, every, Z, ms);
  prof_end(PROF_RESIDENT_BWD, st);
  if (e != cudaSuccess) return (int)e;
  GNCA_LAUNCH_CHECK();
  if (R.dbg) {
    unsigned long long h[16];
    cudaStreamSynchronize(st);
    cudaMemcpy(h, dbg_buf, sizeof(h), cudaMemcpyDeviceToHost);
    const char* names[10] = {"loop top", "masks+list", "A0 inactive sums", "A gz (band)", "S reduce+push", "barrier1", "B tiles",
                             "barrier2", "C gather", "(sum n_my)"};
    fprintf(stderr, "[gnca rep bwd phase cycles, CTA%d, T=%d]", R.dbg_cta, R.T);
    for (int i = 0; i < 10; ++i) fprintf(stderr, " %s=%llu", names[i], h[i]);
    fprintf(stderr, "\n");
  }

  // weight gradients from the records
  WgradArgs A{};
  A.rec = rec; A.hgh = hgh; A.masks = masks; A.steps = sched.steps; A.T = sched.T; A.t0 = t0; A.B = B; A.HW = HW; A.NW = (HW + 31) >> 5;
  A.flags = m.flags; A.wpart = wpart; A.wtotal = L.total; A.L = L;
  // a stack: one group of blocks per model, each group summing that model's segments only (one model: the whole batch)
  const int n_models = ms.stride ? B / ms.per_model : 1;
  A.per = ms.stride ? ms.per_model : B;
  A.nbm = wgrad_blocks_per_model(sched.T, A.per, n_models);
  const int nblk = n_models * A.nbm;
  GNCA_CHECK_CUDA(cudaMemsetAsync(wpart, 0, (size_t)nblk * L.total * sizeof(float), st));
  const size_t wsmem = 2 * (size_t)kWNB * (kRecStride + kHghStride) * sizeof(float);
  const auto wkern = ms.stride ? k_rep_wgrad<16, true> : k_rep_wgrad<16, false>;
  GNCA_CHECK_CUDA(cudaFuncSetAttribute(wkern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem));
  prof_begin(PROF_BWD_MLP, st);
  wkern<<<nblk, kWT, wsmem, st>>>(A);
  prof_end(PROF_BWD_MLP, st);
  GNCA_LAUNCH_CHECK();
  const auto rkern = ms.stride ? k_rep_wreduce<true> : k_rep_wreduce<false>;
  rkern<<<dim3((unsigned)((L.total + 255) / 256), n_models), 256, 0, st>>>(A.nbm, L.total, wpart, A.per * pick, C,
                                                                          affpart, L, gparams);
  GNCA_LAUNCH_CHECK();
  if (zpk) return run_attn_param_reduce(m, B, AttnBwdScratch{nullptr, nullptr, Z.pw}, gparams, st, n_models);
  return 0;
}

}  // namespace gnca
