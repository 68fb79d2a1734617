// Streaming ("any shape") forward of the graph-NCA step: two launches per step, state in HBM/L2.
//   k_update : per-cell alive & fire test, compaction of the ACTIVE cells of a chunk, perception + MLP + graph
//              message on active cells only (inactive cells have pre-norm update 0, ncagraph.py:144-150),
//              masked pre-norm update u -> HBM, deterministic partial sums for the per-sample GroupNorm.
//   k_apply  : finish GroupNorm(1,C) statistics, x~ = x + gain*tanh(gn(u)), post-alive max-pool on the
//              UPDATED alpha (recomputed on a 1-cell halo so no extra launch), alpha gate, store.
// The cluster-resident multi-step kernel lives in gnca_resident.cu.
#include "gnca_common.cuh"
#include "gnca_internal.h"
#include "gnca_tc.cuh"
#include <cstdio>
#include <vector>
#include <utility>

namespace gnca {

std::atomic<unsigned long long> g_launches{0};

static bool g_prof_on = false;
static std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_prof_ev[PROF_COUNT];

void prof_begin(int id, cudaStream_t st) {
  if (!g_prof_on) return;
  cudaEvent_t a, b;
  cudaEventCreate(&a); cudaEventCreate(&b);
  cudaEventRecord(a, st);
  g_prof_ev[id].push_back({a, b});
}
void prof_end(int id, cudaStream_t st) {
  if (!g_prof_on || g_prof_ev[id].empty()) return;
  cudaEventRecord(g_prof_ev[id].back().second, st);
}

constexpr int kChunk = 1024;    // cells per k_update block (large problems)
constexpr int kChunkSmall = 256; // ... when the grid would otherwise not fill the 148 SMs
constexpr int kThreads = 256;
constexpr int kTileW = 32, kTileH = 8;

template <int C> struct CellsPerThread { static constexpr int value = (C <= 16) ? 2 : 1; };

// ------------------------------------------------------------------------------------------------
// pack: canonical flat params -> kernel-side buffer
// ------------------------------------------------------------------------------------------------
__global__ void k_pack(gnca_layout L, Packed P, int C, int hid, int d, const float* __restrict__ src, float* __restrict__ dst) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
  for (int i = tid; i < P.total; i += nth) dst[i] = 0.f;
  __syncthreads();  // (single-block launch: zero fill of the pad slots completes before the copies below)
  const int C3 = 3 * C;
  for (int i = tid; i < hid * C3; i += nth) {
    int j = i / C3, k = i % C3;
    float v = src[L.w1 + i];
    dst[P.w1 + i] = v;
    dst[P.w1t + k * hid + j] = v;
  }
  for (int i = tid; i < hid; i += nth) dst[P.b1 + i] = src[L.b1 + i];
  for (int i = tid; i < C * hid; i += nth) {
    int c = i / hid, j = i % hid;
    float v = src[L.w2 + i];
    dst[P.w2 + i] = v;
    dst[P.w2t + j * C + c] = v;
  }
  for (int i = tid; i < C; i += nth) { dst[P.gamma + i] = src[L.gamma + i]; dst[P.beta + i] = src[L.beta + i]; }
  if ((C & 7) == 0 && (hid & 7) == 0) {      // tf32 (hi, lo) split of both MLP weights in the UMMA operand layout
    for (int i = tid; i < hid * C3; i += nth) {
      const int j = i / C3, k = i % C3;
      const float v = src[L.w1 + i], hi = __uint_as_float(tc::tf32_rna(v)), lo = __uint_as_float(tc::tf32_rna(v - hi));
      dst[P.w1c + tc::canon_idx(j, k, C3)] = hi;
      dst[P.w1c + hid * C3 + tc::canon_idx(j, k, C3)] = lo;
    }
    for (int i = tid; i < C * hid; i += nth) {
      const int c = i / hid, j = i % hid;
      const float v = src[L.w2 + i], hi = __uint_as_float(tc::tf32_rna(v)), lo = __uint_as_float(tc::tf32_rna(v - hi));
      dst[P.w2c + tc::canon_idx(c, j, hid)] = hi;
      dst[P.w2c + C * hid + tc::canon_idx(c, j, hid)] = lo;
    }
  }
  if (P.wm >= 0) {
    for (int i = tid; i < C * C; i += nth) {
      int co = i / C, ci = i % C;
      float v = src[L.wm + i];
      dst[P.wm + i] = v;
      dst[P.wmt + ci * C + co] = v;
    }
    for (int i = tid; i < C; i += nth) dst[P.bm + i] = src[L.bm + i];
    for (int i = tid; i < d * C; i += nth) { dst[P.wq + i] = src[L.wq + i]; dst[P.wk + i] = src[L.wk + i]; }
    for (int i = tid; i < d; i += nth) { dst[P.bq + i] = src[L.bq + i]; dst[P.bk + i] = src[L.bk + i]; }
    if (tid == 0) dst[P.scaling] = src[L.scaling];
  }
}

// ------------------------------------------------------------------------------------------------
// zero-padded-shift attention weights (graph_augmentation.py:114,126,136-138,150-154).
// Q_pooled = Wq mean(x) + bq ; mean(shift_dy K) = (Wk * sum_{rows kept} rowsum(x) + n_rows*W*bk) / (H*W)
// ------------------------------------------------------------------------------------------------
__global__ void k_rowsum(int BCH, int W, const float* __restrict__ x, float* __restrict__ rs) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= BCH) return;
  const float* p = x + (size_t)row * W;
  float s = 0.f;
  for (int i = threadIdx.x & 31; i < W; i += 32) s += p[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) rs[row] = s;
}

// one block per sample; blockDim = 128.  Writes attn_w[b][k].  The sample's row sums are staged in shared memory once
// (stage != 0; the serial `s += rs[..]` chains over global memory cost 20 us per launch at 40x40x16) and the (offset,
// channel) / (offset, feature) pairs run in parallel; every sum keeps its sequential order.
__global__ void k_attn_weights(StepArgs a, Packed P, int C, int d, const float* __restrict__ packed,
                               const float* __restrict__ rowsum, float* __restrict__ attn_w, int stage) {
  extern __shared__ float sm[];
  const int b = blockIdx.x, H = a.H, W = a.W, k = a.k;
  float* xsum = sm;            // [C]
  float* qp = xsum + C;        // [d]
  float* S = qp + d;           // [k][C] row-range sums
  float* KP = S + k * C;       // [k][d]
  float* logit = KP + k * d;   // [k]
  int* rlo = reinterpret_cast<int*>(logit + k);   // [k]
  int* rhi = rlo + k;                              // [k]
  float* swq = reinterpret_cast<float*>(rhi + k);  // [d][C] query_proj / key_proj weights and biases (the dot-product
  float* swk = swq + d * C;                        // loops below would otherwise chain L2 round trips)
  float* sbq = swk + d * C;
  float* sbk = sbq + d;
  float* rss = sbk + d;                            // [C][H] when staged
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
  }
  __syncthreads();
  for (int c = tid; c < C; c += nt) {
    float s = 0.f;
    for (int y = 0; y < H; ++y) s += rs[c * H + y];
    xsum[c] = s;
  }
  for (int idx = tid; idx < k * C; idx += nt) {
    const int i = idx / C, c = idx - i * C;
    float s = 0.f;
    for (int y = rlo[i]; y < rhi[i]; ++y) s += rs[c * H + y];
    S[idx] = s;
  }
  __syncthreads();
  for (int j = tid; j < d; j += nt) {
    float s = 0.f;
    for (int c = 0; c < C; ++c) s = fmaf(swq[j * C + c], xsum[c] * invHW, s);
    qp[j] = s + sbq[j];
  }
  for (int idx = tid; idx < k * d; idx += nt) {
    const int i = idx / d, j = idx - i * d;
    float s = 0.f;
    for (int c = 0; c < C; ++c) s = fmaf(swk[j * C + c], S[i * C + c], s);
    KP[idx] = (s + (float)(rhi[i] - rlo[i]) * (float)W * sbk[j]) * invHW;
  }
  __syncthreads();
  for (int i = tid; i < k; i += nt) {
    float s = 0.f;
    for (int j = 0; j < d; ++j) s = fmaf(qp[j], KP[i * d + j], s);
    logit[i] = s;
  }
  __syncthreads();
  if (tid == 0) {
    float mx = -INFINITY;
    for (int i = 0; i < k; ++i) mx = fmaxf(mx, logit[i]);
    const float denom = fabsf(packed[P.scaling]) + 1e-6f;
    float se = 0.f;
    for (int i = 0; i < k; ++i) { float e = expf((logit[i] - mx) / denom); logit[i] = e; se += e; }
    for (int i = 0; i < k; ++i) attn_w[(size_t)b * k + i] = logit[i] / se;
  }
}

// rowsum + per-sample softmax weights of the zero-padded shift; leaves a.attn_w pointing at ws.attn_w
int run_attn_prepass(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a, const FwdWorkspace& ws,
                     cudaStream_t st) {
  const int rows = a.B * m.C * a.H;
  k_rowsum<<<(rows + 7) / 8, 256, 0, st>>>(rows, a.W, a.x_in, ws.rowsum);
  GNCA_LAUNCH_CHECK();
  const int stage = (size_t)m.C * a.H * sizeof(float) <= 32 * 1024;
  const size_t sm = (size_t)(m.C + m.d_model + a.k * (m.C + m.d_model) + 3 * a.k + 4 + 2 * m.d_model * (m.C + 1) + (stage ? m.C * a.H : 0)) * sizeof(float);
  if (sm > 48 * 1024) GNCA_CHECK_CUDA(cudaFuncSetAttribute(k_attn_weights, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  k_attn_weights<<<a.B, 128, sm, st>>>(a, P, m.C, m.d_model, packed, ws.rowsum, ws.attn_w, stage);
  GNCA_LAUNCH_CHECK();
  a.attn_w = ws.attn_w;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// k_update
// ------------------------------------------------------------------------------------------------
template <int C>
struct UpdateSmem {
  static size_t bytes(int hid, bool graph) {
    size_t f = (size_t)3 * C * hid + pad4(hid) + (size_t)hid * C;
    if (graph) f += C * C + C;
    return f * sizeof(float) + kChunk * sizeof(uint16_t) + 64 * sizeof(double);
  }
};

// BAL (large problems): the active cells of the whole sample were compacted by k_compact / k_scan into a global list;
// block j takes the active cells of rank [j*RANGE, (j+1)*RANGE) -- full rounds of NT cells whatever their position.
// (With per-chunk compaction a chunk of 1024 cells holds ~150-300 active ones: one full round of 256 threads and one
// nearly empty one, and chunks outside the alive region do nothing; measured 25 % FMA-pipe utilisation at 256x256x32.)
constexpr int kMaxBalChunks = 1024;
constexpr int kThreadsBal = 384;

// actbits (optional): the active bit of every cell, one word per 32 consecutive cells -- k_apply reads them for its tile +
// halo instead of recomputing alive_at (nine alpha loads) and the Philox draw of every halo cell
template <int CH>
__global__ void __launch_bounds__(kThreads) k_compact(StepArgs a, int C, uint16_t* __restrict__ glist, int* __restrict__ cnt,
                                                      uint32_t* __restrict__ actbits = nullptr,
                                                      uint32_t* __restrict__ alivebits = nullptr) {
  const int b = blockIdx.y, chunk = blockIdx.x;
  const int H = a.H, W = a.W, HW = H * W;
  __shared__ int swcount[kThreads / 32], swbase[kThreads / 32 + 1];
  if (!sample_active(a, b)) { if (threadIdx.x == 0) cnt[(size_t)b * a.nchunks + chunk] = 0; return; }
  const float fr = step_fire_rate(a);
  const float* alpha = a.x_in + (size_t)b * C * HW + 3 * HW;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int kPerWarp = CH / (kThreads / 32);
  const int cell0 = chunk * CH;
  uint32_t bal[kPerWarp / 32];
  int n = 0;
  // the 3x3 alpha windows of all the thread's cells are requested before the first use, from clamped coordinates (a
  // duplicated tap never changes a maximum): one L2 round trip instead of one per cell and edge test
  float win[kPerWarp / 32][9];
#pragma unroll
  for (int it = 0; it < kPerWarp / 32; ++it) {
    const int cell = min(cell0 + warp * kPerWarp + it * 32 + lane, HW - 1);
    const int y = cell / W, x = cell - y * W;
    const int ru = (y > 0 ? y - 1 : y) * W, rc = y * W, rd = (y < H - 1 ? y + 1 : y) * W;
    const int xl = x > 0 ? x - 1 : x, xr = x < W - 1 ? x + 1 : x;
    win[it][0] = __ldg(alpha + ru + xl); win[it][1] = __ldg(alpha + ru + x); win[it][2] = __ldg(alpha + ru + xr);
    win[it][3] = __ldg(alpha + rc + xl); win[it][4] = __ldg(alpha + rc + x); win[it][5] = __ldg(alpha + rc + xr);
    win[it][6] = __ldg(alpha + rd + xl); win[it][7] = __ldg(alpha + rd + x); win[it][8] = __ldg(alpha + rd + xr);
  }
#pragma unroll
  for (int it = 0; it < kPerWarp / 32; ++it) {
    const int cell = cell0 + warp * kPerWarp + it * 32 + lane;
    bool act = false, sal = false;
    if (cell < HW) {
      float mx = win[it][0];
#pragma unroll
      for (int q = 1; q < 9; ++q) mx = fmaxf(mx, win[it][q]);   // one window maximum serves both thresholds
      act = mx > a.alpha_thr && fires(a, fr, b, cell);
      sal = mx > a.graph_alpha_thr;
    }
    bal[it] = __ballot_sync(0xffffffffu, act);
    n += __popc(bal[it]);
    const size_t word = (size_t)b * ((HW + 31) >> 5) + ((cell0 + warp * kPerWarp + it * 32) >> 5);
    if (actbits && lane == 0 && cell0 + warp * kPerWarp + it * 32 < HW) actbits[word] = bal[it];
    if (alivebits) {        // the step's sender-alive bits: k_update_tc tests one bit instead of nine alpha loads per sender
      const uint32_t sb = __ballot_sync(0xffffffffu, sal);
      if (lane == 0 && cell0 + warp * kPerWarp + it * 32 < HW) alivebits[word] = sb;
    }
  }
  if (lane == 0) swcount[warp] = n;
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int w = 0; w < kThreads / 32; ++w) { swbase[w] = s; s += swcount[w]; }
    cnt[(size_t)b * a.nchunks + chunk] = s;
  }
  __syncthreads();
  int base = swbase[warp];
  uint16_t* dst = glist + (size_t)b * HW + cell0;            // chunk-local compact list (same order as k_update's own)
#pragma unroll
  for (int it = 0; it < kPerWarp / 32; ++it) {
    if (bal[it] & (1u << lane)) dst[base + __popc(bal[it] & ((1u << lane) - 1u))] = (uint16_t)(warp * kPerWarp + it * 32 + lane);
    base += __popc(bal[it]);
  }
}

// exclusive prefix of the per-chunk counts of every sample: prefix[b][0..nchunks], one warp per sample
__global__ void k_scan(int nchunks, const int* __restrict__ cnt, int* __restrict__ prefix) {
  const int b = blockIdx.x, lane = threadIdx.x;
  int carry = 0;
  for (int i0 = 0; i0 < nchunks; i0 += 32) {
    const int i = i0 + lane;
    const int v = i < nchunks ? cnt[(size_t)b * nchunks + i] : 0;
    int inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
    if (i < nchunks) prefix[(size_t)b * (nchunks + 1) + i] = carry + inc - v;
    carry += __shfl_sync(0xffffffffu, inc, 31);
  }
  if (lane == 0) prefix[(size_t)b * (nchunks + 1) + nchunks] = carry;
}

template <int C, int CH, bool BAL = false, int NT = kThreads, int JU = 4>
__global__ void __launch_bounds__(NT) k_update(StepArgs a, Packed P, int hid, const float* __restrict__ packed,
                                               const uint16_t* __restrict__ glist = nullptr,
                                               const int* __restrict__ prefix = nullptr) {
  static_assert(BAL || NT == kThreads, "the in-kernel compaction is written for kThreads threads");
  constexpr int PC = CellsPerThread<C>::value;
  const int b = blockIdx.y, chunk = blockIdx.x;
  const int H = a.H, W = a.W, HW = H * W;
  if (!sample_active(a, b)) return;
  __shared__ int s_pf[BAL ? kMaxBalChunks + 1 : 1];
  int r_lo = 0, r_hi = 0;
  if constexpr (BAL) {
    const int* pf = prefix + (size_t)b * (a.nchunks + 1);
    const int total = pf[a.nchunks];
    constexpr int RANGE = (CH + NT - 1) / NT * NT;      // active cells per block: whole rounds of NT (>= CH: nchunks blocks cover them)
    r_lo = chunk * RANGE;
    r_hi = min(r_lo + RANGE, total);
    if (r_lo >= total) {                       // no work: this block's GroupNorm partial is zero
      if (threadIdx.x == 0) {
        a.partials[((size_t)b * a.nchunks + chunk) * 2] = 0.0;
        a.partials[((size_t)b * a.nchunks + chunk) * 2 + 1] = 0.0;
      }
      return;
    }
    for (int i = threadIdx.x; i <= a.nchunks; i += NT) s_pf[i] = pf[i];
  }
  const bool graph = (a.flags & GNCA_F_GRAPH) != 0;
  const float gain_m = graph ? step_message_gain(a) : 0.f;
  const float fr = step_fire_rate(a);

  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* sW1T = reinterpret_cast<float*>(smem_raw);
  float* sb1 = sW1T + 3 * C * hid;
  float* sW2T = sb1 + pad4(hid);
  float* sWmT = sW2T + hid * C;
  float* sbm = sWmT + (graph ? C * C : 0);
  float* endf = sbm + (graph ? C : 0);
  double* sred = reinterpret_cast<double*>(endf);            // [64]
  uint16_t* slist = reinterpret_cast<uint16_t*>(sred + 64);  // [kChunk]
  __shared__ int swcount[kThreads / 32], swbase[kThreads / 32 + 1];

  block_copy(sW1T, packed + P.w1t, 3 * C * hid);
  block_copy(sb1, packed + P.b1, pad4(hid));
  block_copy(sW2T, packed + P.w2t, hid * C);
  if (graph) { block_copy(sWmT, packed + P.wmt, C * C); block_copy(sbm, packed + P.bm, C); }

  // ---- active-cell compaction (deterministic order: warp-major, then cell order) -----------------
  const float* xs_base = a.x_in + (size_t)b * C * HW;
  const float* alpha = xs_base + 3 * HW;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int kPerWarp = CH / (kThreads / 32);      // cells per warp
  const int cell0 = chunk * CH;
  int nact = 0;
  if constexpr (!BAL) {
  uint32_t bal[kPerWarp / 32];
  int cnt = 0;
#pragma unroll
  for (int it = 0; it < kPerWarp / 32; ++it) {
    const int cell = cell0 + warp * kPerWarp + it * 32 + lane;
    bool act = false;
    if (cell < HW) {
      const int y = cell / W, x = cell - y * W;
      act = alive_at(alpha, y, x, H, W, a.alpha_thr) && fires(a, fr, b, cell);
    }
    bal[it] = __ballot_sync(0xffffffffu, act);
    cnt += __popc(bal[it]);
  }
  if (lane == 0) swcount[warp] = cnt;
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int w = 0; w < kThreads / 32; ++w) { swbase[w] = s; s += swcount[w]; }
    swbase[kThreads / 32] = s;
  }
  __syncthreads();
  {
    int base = swbase[warp];
#pragma unroll
    for (int it = 0; it < kPerWarp / 32; ++it) {
      if (bal[it] & (1u << lane))
        slist[base + __popc(bal[it] & ((1u << lane) - 1u))] = (uint16_t)(warp * kPerWarp + it * 32 + lane);
      base += __popc(bal[it]);
    }
  }
  __syncthreads();
  nact = swbase[kThreads / 32];
  } else {
    __syncthreads();                            // weights and the prefix table are in shared memory
    nact = r_hi - r_lo;
  }
  // rank -> cell through the per-chunk prefix (BAL) or this block's own list
  auto cell_of = [&](int li) -> int {
    if constexpr (BAL) {
      const int rank = r_lo + li;
      int lo = 0, hi = a.nchunks;                // s_pf[lo] <= rank < s_pf[hi]
      while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (s_pf[mid] <= rank) lo = mid; else hi = mid; }
      return lo * CH + (int)glist[(size_t)b * HW + (size_t)lo * CH + (rank - s_pf[lo])];
    } else {
      return cell0 + (int)slist[li];
    }
  };

  // ---- perception + MLP + message on active cells ------------------------------------------------
  float s1 = 0.f, s2 = 0.f;
#ifdef GNCA_PHASE_COUNTERS          /* development: where a round's cycles go (one thread of one working block prints) */
  long long ph_t = clock64(), ph[3] = {0, 0, 0};
#define UPD_MARK(i) do { const long long n_ = clock64(); ph[i] += n_ - ph_t; ph_t = n_; } while (0)
#else
#define UPD_MARK(i) do { } while (0)
#endif
  for (int base = 0; base < nact; base += NT * PC) {
    float yv[PC][3 * C];
    float dxv[PC][C];
    int cells[PC];
#pragma unroll
    for (int p = 0; p < PC; ++p) {
      const int li = base + p * NT + threadIdx.x;
      cells[p] = li < nact ? cell_of(li) : -1;
      if (cells[p] >= 0) {
        const int y = cells[p] / W, x = cells[p] - y * W;
        perceive<C>(xs_base, y, x, H, W, yv[p]);
      } else {
#pragma unroll
        for (int k = 0; k < 3 * C; ++k) yv[p][k] = 0.f;
      }
    }
    UPD_MARK(0);
    mlp_forward<C, PC, JU>(yv, dxv, sW1T, sb1, sW2T, hid);
    UPD_MARK(1);
#pragma unroll
    for (int p = 0; p < PC; ++p) {
      if (cells[p] < 0) continue;
      const int y = cells[p] / W, x = cells[p] - y * W;
      if (graph && gain_m != 0.f && a.k > 0) {
        float xsnd[C], agg[C], as;
        gather_senders<C>(a, xs_base, b, y, x, xsnd, as);
        msg_project<C>(xsnd, as, sWmT, sbm, agg);
        const int c_lo = ((a.flags & GNCA_F_HIDDEN_ONLY) && C >= 4) ? 4 : 0;
#pragma unroll
        for (int c = 0; c < C; ++c)
          if (c >= c_lo) dxv[p][c] = fmaf(tanhf(agg[c]), gain_m, dxv[p][c]);
      }
      float* up = a.u + (size_t)b * C * HW + cells[p];
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const float v = dxv[p][c];
        up[(size_t)c * HW] = v;
        s1 += v;
        s2 = fmaf(v, v, s2);
      }
    }
    UPD_MARK(2);
  }
#ifdef GNCA_PHASE_COUNTERS
  if (BAL && blockIdx.x == 2 && blockIdx.y == 0 && (threadIdx.x == 0 || threadIdx.x == NT - 1) && a.t == 2)
    printf("[k_update phases, block (2,0) thread %d, %d active cells] lookup+perception %lld  mlp %lld  message+store %lld cycles\n",
           (int)threadIdx.x, nact, ph[0], ph[1], ph[2]);
#endif
#undef UPD_MARK
  // ---- deterministic block reduction of (sum u, sum u^2) ------------------------------------------
  double d1 = warp_sum((double)s1), d2 = warp_sum((double)s2);
  if (lane == 0) { sred[warp * 2] = d1; sred[warp * 2 + 1] = d2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t1 = 0.0, t2 = 0.0;
    for (int w = 0; w < NT / 32; ++w) { t1 += sred[w * 2]; t2 += sred[w * 2 + 1]; }
    a.partials[((size_t)b * a.nchunks + chunk) * 2] = t1;
    a.partials[((size_t)b * a.nchunks + chunk) * 2 + 1] = t2;
  }
}

// (sum u, sum u^2) of sample b from the chunk partials, by ONE WARP: lane l adds chunks l, l+32, ... in order, then a
// fixed shuffle tree -- the same arithmetic wherever the statistics are finished (k_apply, k_finalize_stats), and one
// L2 round trip instead of nchunks dependent ones (k_apply starts every tile with this reduction).
__device__ __forceinline__ void warp_reduce_partials(const StepArgs& a, int b, int lane, double& t1, double& t2) {
  double s1 = 0.0, s2 = 0.0;
  for (int i = lane; i < a.npart; i += 32) {
    s1 += a.partials[((size_t)b * a.npart + i) * 2];
    s2 += a.partials[((size_t)b * a.npart + i) * 2 + 1];
  }
  t1 = warp_sum(s1);
  t2 = warp_sum(s2);
}

// ------------------------------------------------------------------------------------------------
// k_apply
// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(kThreads) k_apply(StepArgs a, Packed P, const float* __restrict__ packed) {
  const int b = blockIdx.y;
  const int H = a.H, W = a.W, HW = H * W;
  const int tiles_x = (W + kTileW - 1) / kTileW;
  const int ty0 = (blockIdx.x / tiles_x) * kTileH, tx0 = (blockIdx.x % tiles_x) * kTileW;
  const int lx = threadIdx.x % kTileW, ly = threadIdx.x / kTileW;
  const int y = ty0 + ly, x = tx0 + lx;
  const bool inside = y < H && x < W;
  const float* xs_base = a.x_in + (size_t)b * C * HW;
  float* xo_base = a.x_out + (size_t)b * C * HW;

  if (!sample_active(a, b)) {  // frozen sample: state passes through (train...:306-321 `state[mask] = ...`)
    if (inside && a.x_out != a.x_in) {
#pragma unroll
      for (int c = 0; c < C; ++c) xo_base[c * HW + y * W + x] = xs_base[c * HW + y * W + x];
    }
    return;
  }

  __shared__ float s_sc[C], s_bi[C], s_idle[C];
  __shared__ float s_alpha[kTileH + 2][kTileW + 2 + 1];
  __shared__ unsigned char s_act[kTileH + 2][kTileW + 2];
  __shared__ float s_stat[2];
  const float fr = step_fire_rate(a);
  const bool gn = (a.flags & GNCA_F_GROUPNORM) != 0;

  if (threadIdx.x < 32) {
    float mu = 0.f, rstd = 1.f;
    if (gn) {
      double t1, t2;
      warp_reduce_partials(a, b, threadIdx.x, t1, t2);
      const double n = (double)C * (double)HW;
      const double m = t1 / n;
      double var = t2 / n - m * m;
      if (var < 0.0) var = 0.0;
      mu = (float)m;
      rstd = (float)(1.0 / sqrt(var + (double)a.gn_eps));
    }
    if (threadIdx.x == 0) {
      s_stat[0] = mu; s_stat[1] = rstd;
      if (blockIdx.x == 0 && a.stats) { a.stats[b * 2] = mu; a.stats[b * 2 + 1] = rstd; }
    }
  }
  __syncthreads();
  if (threadIdx.x < C) {
    const int c = threadIdx.x;
    float sc = 1.f, bi = 0.f;
    if (gn) {  // ATen: y = x*(rstd*gamma) + (beta - mean*rstd*gamma)
      sc = s_stat[1] * packed[P.gamma + c];
      bi = packed[P.beta + c] - s_stat[0] * sc;
    }
    s_sc[c] = sc; s_bi[c] = bi;
    s_idle[c] = __fmul_rn(tanhf(bi), a.update_gain);   // update of a cell whose masked pre-norm update is 0
  }
  __syncthreads();

  // ---- updated alpha (pre-gate) on the tile + 1-cell halo --------------------------------------------
  const float* alpha = xs_base + 3 * HW;
  const float* u3 = a.u + (size_t)b * C * HW + 3 * HW;
  for (int i = threadIdx.x; i < (kTileH + 2) * (kTileW + 2); i += kThreads) {
    const int hy = i / (kTileW + 2), hx = i % (kTileW + 2);
    const int yy = ty0 + hy - 1, xx = tx0 + hx - 1;
    float v = -INFINITY;
    unsigned char act = 0;
    if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
      const int cell = yy * W + xx;
      act = a.actbits ? (unsigned char)((a.actbits[(size_t)b * ((HW + 31) >> 5) + (cell >> 5)] >> (cell & 31)) & 1u)
                      : (unsigned char)(alive_at(alpha, yy, xx, H, W, a.alpha_thr) && fires(a, fr, b, cell));
      const float uu = act ? u3[cell] : 0.f;
      v = updated_alpha(alpha[cell], act, uu, s_sc[3], s_bi[3], s_idle[3], a.update_gain);
    }
    s_alpha[hy][hx] = v;
    s_act[hy][hx] = act;
  }
  __syncthreads();
  if (!inside) return;

  const int cell = y * W + x;
  const bool act = s_act[ly + 1][lx + 1] != 0;
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) mx = fmaxf(mx, s_alpha[ly + i][lx + j]);
  const bool post = mx > a.alpha_thr;
  const float* up = a.u + (size_t)b * C * HW + cell;
  // all loads of a group of channels are issued before the first use: the kernel is a pure HBM stream and a warp that
  // keeps only a few loads in flight (the compiler's choice at 32 registers) leaves it latency-bound
  constexpr int CG = C < 16 ? C : 16;
#pragma unroll
  for (int c0 = 0; c0 < C; c0 += CG) {
    float xin[CG], uu[CG];
#pragma unroll
    for (int j = 0; j < CG; ++j) {
      const int c = c0 + j;
      xin[j] = (c == 3) ? 0.f : __ldg(xs_base + (size_t)c * HW + cell);
      uu[j] = (act && c != 3) ? __ldg(up + (size_t)c * HW) : 0.f;
    }
#pragma unroll
    for (int j = 0; j < CG; ++j) {
      const int c = c0 + j;
      float v;
      if (c == 3) {
        v = post ? s_alpha[ly + 1][lx + 1] : 0.f;     // x~_3 * post_alive (ncagraph.py:158-166)
      } else {
        v = xin[j] + (act ? tanhf(fmaf(uu[j], s_sc[c], s_bi[c])) * a.update_gain : s_idle[c]);
      }
      xo_base[(size_t)c * HW + cell] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// attention map (graph_augmentation.py:160-167): attn = sum_i w_i * mean_c |M(q_i) A(q_i)|, min-max per sample
// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void k_absmean_msg(StepArgs a, Packed P, const float* __restrict__ packed, float* __restrict__ S) {
  const int b = blockIdx.y, H = a.H, W = a.W, HW = H * W;
  const int cell = blockIdx.x * blockDim.x + threadIdx.x;
  if (cell >= HW) return;
  const float* xs_base = a.x_in + (size_t)b * C * HW;
  const int y = cell / W, x = cell - y * W;
  float s = 0.f;
  if (!(a.flags & GNCA_F_ALIVE_TO_ALIVE) || alive_at(xs_base + 3 * HW, y, x, H, W, a.graph_alpha_thr)) {
    float xv[C];
#pragma unroll
    for (int c = 0; c < C; ++c) xv[c] = xs_base[c * HW + cell];
    for (int co = 0; co < C; ++co) {
      float m = packed[P.bm + co];
#pragma unroll
      for (int ci = 0; ci < C; ++ci) m = fmaf(packed[P.wm + co * C + ci], xv[ci], m);
      s += fabsf(m);
    }
    s *= (1.0f / (float)C);
  }
  S[(size_t)b * HW + cell] = s;
}

// one block per sample: gather + min/max + normalise
__global__ void k_attn_map(StepArgs a, const float* __restrict__ S, float* __restrict__ attn) {
  const int b = blockIdx.x, H = a.H, W = a.W, HW = H * W;
  const bool torus = (a.flags & GNCA_F_TORUS) != 0;
  __shared__ float smin[32], smax[32];
  const float wuni = a.k > 0 ? 1.0f / (float)a.k : 0.f;
  float lo = INFINITY, hi = -INFINITY;
  for (int cell = threadIdx.x; cell < HW; cell += blockDim.x) {
    const int y = cell / W, x = cell - y * W;
    float v = 0.f;
    for (int i = 0; i < a.k; ++i) {
      int dy, dx, qy, qx;
      step_offset(a, i, dy, dx);
      if (!sender_of(y, x, dy, dx, H, W, torus, qy, qx)) continue;
      const float w = a.attn_w ? a.attn_w[(size_t)b * a.k + i] : wuni;
      v = fmaf(w, S[(size_t)b * HW + qy * W + qx], v);
    }
    attn[(size_t)b * HW + cell] = v;
    lo = fminf(lo, v); hi = fmaxf(hi, v);
  }
  for (int o = 16; o > 0; o >>= 1) {
    lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if ((threadIdx.x & 31) == 0) { smin[threadIdx.x >> 5] = lo; smax[threadIdx.x >> 5] = hi; }
  __syncthreads();
  lo = INFINITY; hi = -INFINITY;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { lo = fminf(lo, smin[w]); hi = fmaxf(hi, smax[w]); }
  if (a.k == 0) { lo = 0.f; hi = 0.f; }
  const float inv = 1.0f / (hi - lo + 1e-8f);
  __syncthreads();
  for (int cell = threadIdx.x; cell < HW; cell += blockDim.x) {
    const size_t i = (size_t)b * HW + cell;
    attn[i] = (a.k == 0) ? 0.f : (attn[i] - lo) * inv;
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

FwdWorkspace carve_fwd_workspace(void* base, const gnca_model& m, int B, int H, int W) {
  FwdWorkspace ws;
  const int nchunks = (H * W + kChunkSmall - 1) / kChunkSmall;   // sized for the small chunk
  size_t o = 0;
  char* p = reinterpret_cast<char*>(base);
  ws.partials = reinterpret_cast<double*>(p + o); o = align_up(o + (size_t)B * nchunks * 2 * sizeof(double), 256);
  ws.rowsum = reinterpret_cast<float*>(p + o); o = align_up(o + (size_t)B * m.C * H * sizeof(float), 256);
  ws.attn_w = reinterpret_cast<float*>(p + o); o = align_up(o + (size_t)B * GNCA_MAX_K * sizeof(float), 256);
  ws.absmean = reinterpret_cast<float*>(p + o); o = align_up(o + (size_t)B * H * W * sizeof(float), 256);
  ws.actbits = reinterpret_cast<uint32_t*>(p + o); o = align_up(o + (size_t)B * ((H * W + 31) / 32) * sizeof(uint32_t), 256);
  ws.alivebits = reinterpret_cast<uint32_t*>(p + o); o = align_up(o + (size_t)B * ((H * W + 31) / 32) * sizeof(uint32_t), 256);
  ws.bytes = o;
  return ws;
}

void fill_step_args(StepArgs& a, const gnca_model& m, int B, int H, int W) {
  a = StepArgs{};
  a.B = B; a.H = H; a.W = W;
  a.flags = m.flags;
  a.update_gain = m.update_gain; a.alpha_thr = m.alpha_thr; a.graph_alpha_thr = m.graph_alpha_thr; a.gn_eps = m.gn_eps;
  // small chunks when 1024-cell chunks would leave SMs idle (launch-latency-bound small grids)
  a.chunk = ((long long)B * ((H * W + kChunk - 1) / kChunk) < 2 * 148) ? kChunkSmall : kChunk;
  a.nchunks = (H * W + a.chunk - 1) / a.chunk;
  a.npart = a.nchunks;
}

// k_update launch: per-chunk compaction inside the kernel (small problems) or the balanced global list (large ones).
// The global list lives in ws.absmean (one uint16 per cell; the attention-map kernels that own that buffer run after
// k_apply), the per-chunk counts and their prefix in the part of ws.partials that only small-chunk runs use.
template <int C>
static int launch_update(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a, const FwdWorkspace& ws,
                         cudaStream_t st) {
  const bool graph = (m.flags & GNCA_F_GRAPH) != 0;
  const size_t smem = UpdateSmem<C>::bytes(m.hidden, graph);
  dim3 g1(a.nchunks, a.B);
  a.actbits = nullptr;
  a.alivebits = nullptr;
  if (a.chunk == kChunkSmall) {
    a.npart = a.nchunks;
    GNCA_CHECK_CUDA(cudaFuncSetAttribute(k_update<C, kChunkSmall>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_update<C, kChunkSmall><<<g1, kThreads, smem, st>>>(a, P, m.hidden, packed);
    return 0;
  }
  const int HW = a.H * a.W;
  const int n_small = (HW + kChunkSmall - 1) / kChunkSmall;
  static_assert(kChunk == kTcChunk, "k_update_tc reads the chunk-local lists of k_compact<kChunk>");
  // Which k_update runs (read per launch so that one process can compare them: tests/test_gpu_scale.py):
  //   default        k_update_tc   compacted 128-cell tiles on the tensor cores (gnca_update_tc.cu)
  //   GNCA_NO_TC=1   k_update      the round-1 FFMA kernel
  const bool no_tc = getenv("GNCA_NO_TC") != nullptr;
  const bool use_tc = !no_tc && update_tc_supported(m, a);
  a.npart = use_tc ? 3 * a.nchunks : a.nchunks;
  const size_t used = (size_t)a.B * a.npart * 2 * sizeof(double), have = (size_t)a.B * n_small * 2 * sizeof(double);
  const size_t need = ((size_t)a.B * a.nchunks + (size_t)a.B * (a.nchunks + 1)) * sizeof(int);
  if (a.nchunks <= kMaxBalChunks && used + need <= have) {
    int* cnt = reinterpret_cast<int*>(reinterpret_cast<char*>(ws.partials) + used);
    int* prefix = cnt + (size_t)a.B * a.nchunks;
    uint16_t* glist = reinterpret_cast<uint16_t*>(ws.absmean);
    const bool want_alive = use_tc && graph && (a.flags & GNCA_F_ALIVE_TO_ALIVE) && a.k > 0 && !getenv("GNCA_NO_ALIVEBITS");
    k_compact<kChunk><<<g1, kThreads, 0, st>>>(a, C, glist, cnt, ws.actbits, want_alive ? ws.alivebits : nullptr);
    a.actbits = ws.actbits;
    a.alivebits = want_alive ? ws.alivebits : nullptr;
    k_scan<<<a.B, 32, 0, st>>>(a.nchunks, cnt, prefix);
    if (use_tc) {
      g_launches += 2;
      return launch_update_tc(m, P, packed, a, glist, prefix, st);
    }
    if constexpr (C >= 16) {
      // 384 threads (168 registers, no spills): 12 warps per SM instead of 8 hide the perception / sender loads better
      // (measured at 256x256x32: 9.99 -> 9.31 ms per 20 steps; 8 hidden units per pass and 256 threads were slower)
      GNCA_CHECK_CUDA(cudaFuncSetAttribute(k_update<C, kChunk, true, kThreadsBal>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      k_update<C, kChunk, true, kThreadsBal><<<g1, kThreadsBal, smem, st>>>(a, P, m.hidden, packed, glist, prefix);
    } else {
      GNCA_CHECK_CUDA(cudaFuncSetAttribute(k_update<C, kChunk, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      k_update<C, kChunk, true><<<g1, kThreads, smem, st>>>(a, P, m.hidden, packed, glist, prefix);
    }
    g_launches += 2;
    return 0;
  }
  a.npart = a.nchunks;
  GNCA_CHECK_CUDA(cudaFuncSetAttribute(k_update<C, kChunk>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_update<C, kChunk><<<g1, kThreads, smem, st>>>(a, P, m.hidden, packed);
  return 0;
}

template <int C>
int launch_step_fwd(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a, const FwdWorkspace& ws,
                    float* attn_out, cudaStream_t st) {
  const bool graph = (m.flags & GNCA_F_GRAPH) != 0;
  const bool torus = (m.flags & GNCA_F_TORUS) != 0;
  a.partials = ws.partials;
  a.attn_w = nullptr;
  if (graph && !torus && a.k > 0) {   // per-sample softmax weights (zero-padded shift)
    int rc = run_attn_prepass(m, P, packed, a, ws, st);
    if (rc) return rc;
  }
  prof_begin(PROF_UPDATE, st);
  { const int rc = launch_update<C>(m, P, packed, a, ws, st); if (rc) return rc; }
  prof_end(PROF_UPDATE, st);
  GNCA_LAUNCH_CHECK();
  const int tiles = ((a.W + kTileW - 1) / kTileW) * ((a.H + kTileH - 1) / kTileH);
  dim3 g2(tiles, a.B);
  prof_begin(PROF_APPLY, st);
  k_apply<C><<<g2, kThreads, 0, st>>>(a, P, packed);
  prof_end(PROF_APPLY, st);
  GNCA_LAUNCH_CHECK();
  if (attn_out) {
    if (!graph) return GNCA_ERR_ARG;
    dim3 g3((a.H * a.W + 255) / 256, a.B);
    k_absmean_msg<C><<<g3, 256, 0, st>>>(a, P, packed, ws.absmean);
    GNCA_LAUNCH_CHECK();
    k_attn_map<<<a.B, 256, 0, st>>>(a, ws.absmean, attn_out);
    GNCA_LAUNCH_CHECK();
  }
  return 0;
}

template <int C>
static int launch_attn_map(const Packed& P, const float* packed, StepArgs& a, const FwdWorkspace& ws, float* attn_out,
                           cudaStream_t st) {
  dim3 g3((a.H * a.W + 255) / 256, a.B);
  k_absmean_msg<C><<<g3, 256, 0, st>>>(a, P, packed, ws.absmean);
  GNCA_LAUNCH_CHECK();
  k_attn_map<<<a.B, 256, 0, st>>>(a, ws.absmean, attn_out);
  GNCA_LAUNCH_CHECK();
  return 0;
}

int run_attn_map(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a, const FwdWorkspace& ws,
                 float* attn_out, cudaStream_t st) {
  switch (m.C) {
    case 4: return launch_attn_map<4>(P, packed, a, ws, attn_out, st);
    case 8: return launch_attn_map<8>(P, packed, a, ws, attn_out, st);
    case 16: return launch_attn_map<16>(P, packed, a, ws, attn_out, st);
    case 32: return launch_attn_map<32>(P, packed, a, ws, attn_out, st);
  }
  return GNCA_ERR_UNSUPPORTED;
}

int dispatch_step_fwd(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a, const FwdWorkspace& ws,
                      float* attn_out, cudaStream_t st) {
  switch (m.C) {
    case 4: return launch_step_fwd<4>(m, P, packed, a, ws, attn_out, st);
    case 8: return launch_step_fwd<8>(m, P, packed, a, ws, attn_out, st);
    case 16: return launch_step_fwd<16>(m, P, packed, a, ws, attn_out, st);
    case 32: return launch_step_fwd<32>(m, P, packed, a, ws, attn_out, st);
  }
  return GNCA_ERR_UNSUPPORTED;
}

// (mean, rstd) from the chunk partials -- used when only u is recomputed (backward of a rollout)
__global__ void k_finalize_stats(StepArgs a, int C) {       // one warp per sample
  const int b = blockIdx.x, lane = threadIdx.x;
  if (b >= a.B || !a.stats) return;
  float mu = 0.f, rstd = 1.f;
  if (a.flags & GNCA_F_GROUPNORM) {
    double t1, t2;
    warp_reduce_partials(a, b, lane, t1, t2);
    const double n = (double)C * (double)a.H * (double)a.W;
    const double m = t1 / n;
    double var = t2 / n - m * m;
    if (var < 0.0) var = 0.0;
    mu = (float)m;
    rstd = (float)(1.0 / sqrt(var + (double)a.gn_eps));
  }
  if (lane != 0) return;
  a.stats[b * 2] = mu; a.stats[b * 2 + 1] = rstd;
}

template <int C>
int launch_step_recompute(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a, const FwdWorkspace& ws,
                          cudaStream_t st) {
  const bool graph = (m.flags & GNCA_F_GRAPH) != 0;
  a.partials = ws.partials;
  a.attn_w = nullptr;
  if (graph && !(m.flags & GNCA_F_TORUS) && a.k > 0) {
    int rc = run_attn_prepass(m, P, packed, a, ws, st);
    if (rc) return rc;
  }
  { const int rc = launch_update<C>(m, P, packed, a, ws, st); if (rc) return rc; }
  GNCA_LAUNCH_CHECK();
  k_finalize_stats<<<a.B, 32, 0, st>>>(a, C);
  GNCA_LAUNCH_CHECK();
  return 0;
}

int dispatch_step_recompute(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a,
                            const FwdWorkspace& ws, cudaStream_t st) {
  switch (m.C) {
    case 4: return launch_step_recompute<4>(m, P, packed, a, ws, st);
    case 8: return launch_step_recompute<8>(m, P, packed, a, ws, st);
    case 16: return launch_step_recompute<16>(m, P, packed, a, ws, st);
    case 32: return launch_step_recompute<32>(m, P, packed, a, ws, st);
  }
  return GNCA_ERR_UNSUPPORTED;
}

int set_host_offsets(StepArgs& a, const int32_t* offsets_host, int k) {
  if (k < 0 || k > GNCA_MAX_K) return GNCA_ERR_UNSUPPORTED;
  if (k > 0 && !offsets_host) return GNCA_ERR_ARG;
  a.k = k;
  for (int i = 0; i < k; ++i) {
    const int dy = offsets_host[2 * i], dx = offsets_host[2 * i + 1];
    if (dy < -127 || dy > 127 || dx < -127 || dx > 127) return GNCA_ERR_UNSUPPORTED;
    a.off.dy[i] = (int8_t)dy; a.off.dx[i] = (int8_t)dx;
  }
  return 0;
}

}  // namespace gnca

using namespace gnca;

extern "C" {

int gnca_version(void) { return GNCA_VERSION; }

unsigned long long gnca_launch_count(void) { return g_launches.load(); }

int gnca_profile_enable(int on) {
  g_prof_on = on != 0;
  return 0;
}

int gnca_profile_read(int kernel_id, double* total_ms, unsigned long long* launches) {
  if (kernel_id < 0 || kernel_id >= PROF_COUNT || !total_ms || !launches) return GNCA_ERR_ARG;
  double tot = 0.0;
  unsigned long long n = 0;
  for (auto& ev : g_prof_ev[kernel_id]) {
    GNCA_CHECK_CUDA(cudaEventSynchronize(ev.second));
    float ms = 0.f;
    GNCA_CHECK_CUDA(cudaEventElapsedTime(&ms, ev.first, ev.second));
    tot += ms; ++n;
    cudaEventDestroy(ev.first); cudaEventDestroy(ev.second);
  }
  g_prof_ev[kernel_id].clear();
  *total_ms = tot; *launches = n;
  return 0;
}

const char* gnca_error_string(int code) {
  if (code == 0) return "ok";
  if (code == GNCA_ERR_ARG) return "gnca: invalid argument";
  if (code == GNCA_ERR_UNSUPPORTED) return "gnca: unsupported configuration (no kernel, and no fallback by design)";
  if (code == GNCA_ERR_WORKSPACE) return "gnca: workspace too small";
  if (code > 0) return cudaGetErrorString((cudaError_t)code);
  return "gnca: unknown error";
}

int gnca_param_layout(const gnca_model* m, gnca_layout* out) {
  if (!m || !out) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  *out = make_layout(*m);
  return 0;
}

int gnca_pack_weights(const gnca_model* m, const float* params_dev, float* packed_dev, void* stream) {
  if (!m || !params_dev || !packed_dev) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  const bool graph = (m->flags & GNCA_F_GRAPH) != 0;
  k_pack<<<1, 1024, 0, (cudaStream_t)stream>>>(make_layout(*m), make_packed(m->C, m->hidden, m->d_model, graph), m->C,
                                               m->hidden, m->d_model, params_dev, packed_dev);
  GNCA_LAUNCH_CHECK();
  return 0;
}

size_t gnca_step_workspace_bytes(const gnca_model* m, int B, int H, int W) {
  if (!m || B <= 0 || H <= 0 || W <= 0) return 0;
  // forward part + backward part (see gnca_bwd.cu); the backward carve starts after the forward one
  const size_t bw = bwd_workspace_bytes(*m, B, H, W);
  const size_t gw = (m->flags & GNCA_F_GRAPH) ? graph_workspace_bytes(*m, B, H, W) : 0;
  return carve_fwd_workspace(nullptr, *m, B, H, W).bytes + (bw > gw ? bw : gw);
}

int gnca_step_fwd(const gnca_model* m, const float* packed_dev, int B, int H, int W, const float* x_in_dev,
                  float* x_out_dev, const float* fire_u_dev, float fire_rate, const int32_t* offsets_host, int k,
                  float message_gain, float* u_dev, float* stats_dev, float* attn_dev, void* workspace_dev,
                  size_t workspace_bytes, void* stream) {
  if (!m || !packed_dev || !x_in_dev || !x_out_dev || !u_dev || !workspace_dev) return GNCA_ERR_ARG;
  if (B <= 0 || H <= 0 || W <= 0) return GNCA_ERR_ARG;
  if (!model_supported(*m)) return GNCA_ERR_UNSUPPORTED;
  if (fire_rate < 1.0f && !fire_u_dev) return GNCA_ERR_ARG;
  if (x_in_dev == x_out_dev) return GNCA_ERR_ARG;
  const bool graph = (m->flags & GNCA_F_GRAPH) != 0;
  FwdWorkspace ws = carve_fwd_workspace(workspace_dev, *m, B, H, W);
  if (ws.bytes > workspace_bytes) return GNCA_ERR_WORKSPACE;
  StepArgs a;
  fill_step_args(a, *m, B, H, W);
  int rc = set_host_offsets(a, offsets_host, graph ? k : 0);
  if (rc) return rc;
  a.fire_rate = fire_rate; a.message_gain = message_gain;
  a.fire_u = fire_u_dev;
  a.x_in = x_in_dev; a.x_out = x_out_dev; a.u = u_dev; a.stats = stats_dev;
  const Packed P = make_packed(m->C, m->hidden, m->d_model, graph);
  return dispatch_step_fwd(*m, P, packed_dev, a, ws, attn_dev, (cudaStream_t)stream);
}

}  // extern "C"
