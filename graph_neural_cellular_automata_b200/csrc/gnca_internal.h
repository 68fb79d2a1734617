// Internal (non-ABI) declarations shared between the translation units of libgnca.so.
#pragma once
#include <stddef.h>
#include "gnca_common.cuh"

namespace gnca {

struct FwdWorkspace {
  double* partials;   // [B][nchunks][2]
  float* rowsum;      // [B][C][H]
  float* attn_w;      // [B][MAX_K]
  float* absmean;     // [B][H][W]
  uint32_t* actbits;  // [B][ceil(HW/32)] active bits of the step (k_compact -> k_apply)
  uint32_t* alivebits;   // [B][ceil(HW/32)] sender-alive bits of the step (k_compact -> k_update_tc)
  size_t bytes;
};

// Largest dynamic shared memory a launch of `kfn` may ask for on the current device: the opt-in limit per block less the
// kernel's static shared memory, at most 226 KB.  Cached per (kernel, device); 0 when the attributes cannot be read.
size_t dynamic_smem_cap(const void* kfn);

FwdWorkspace carve_fwd_workspace(void* base, const gnca_model& m, int B, int H, int W);
void fill_step_args(StepArgs& a, const gnca_model& m, int B, int H, int W);
int set_host_offsets(StepArgs& a, const int32_t* offsets_host, int k);
int dispatch_step_fwd(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a, const FwdWorkspace& ws,
                      float* attn_out, cudaStream_t st);
// recompute only the masked pre-norm update u (+ statistics) of a step: the forward half the backward needs
int dispatch_step_recompute(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a,
                            const FwdWorkspace& ws, cudaStream_t st);

int run_attn_prepass(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a, const FwdWorkspace& ws,
                     cudaStream_t st);
int run_attn_map(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a, const FwdWorkspace& ws,
                 float* attn_out, cudaStream_t st);
// zero-padded-shift attention backward (gnca_graph.cu): softmax / logits / pooled Q,K -> gparams (wq,bq,wk,bk,
// scaling) and the per-(b,c,row) additive term `grow` of dL/dx.  gw_part: [B][nparts][k] partial sums of
// dL/dw_i; rowsum / a.attn_w from run_attn_prepass on the same x.
struct AttnBwdScratch {
  float* gw_part;   // [B][nparts][GNCA_MAX_K]
  float* grow;      // [B][C][H]
  float* pw;        // [B][2*d*C + 2*d + 1]
};
size_t attn_bwd_scratch_bytes(const gnca_model& m, int B, int H, int nparts);
AttnBwdScratch carve_attn_bwd(void* base, const gnca_model& m, int B, int H, int nparts);
int run_attn_bwd(const gnca_model& m, const Packed& P, const float* packed, const StepArgs& a, const float* rowsum,
                 const AttnBwdScratch& sc, int nparts, float* gparams, cudaStream_t st, bool defer_reduce);
// n_models > 1: a stack (B / n_models samples per model), model i's sum into gparams + i * layout.total
int run_attn_param_reduce(const gnca_model& m, int B, const AttnBwdScratch& sc, float* gparams, cudaStream_t st,
                          int n_models = 1);

size_t graph_workspace_bytes(const gnca_model& m, int B, int H, int W);
size_t bwd_workspace_bytes(const gnca_model& m, int B, int H, int W);
// Backward of one step.  `a` describes the step (x_in, u, schedule...).  Weight-gradient partials live in the
// workspace: zero_partials clears them first, reduce_partials folds them into gparams at the end (a rollout
// clears at its first step and reduces after its last).  gframe (optional, [B][C][H][W]) is added to gx: the gradient
// of a recorded frame that is x_in itself.
int run_step_bwd(const gnca_model& m, const Packed& P, const float* packed, const StepArgs& a, const float* stats,
                 const float* gout, float* gx, float* gparams, const FwdWorkspace& fws, void* bwd_ws, bool zero_partials,
                 bool reduce_partials, cudaStream_t st, const float* gframe = nullptr);

// tensor-core k_update (gnca_update_tc.cu): the balanced large-problem path for C in {16, 32}, hidden 128.
// glist / prefix: the global active list of k_compact / k_scan.  Sets a.npart (3 partial slots per chunk).
constexpr int kTcChunk = 1024;
bool update_tc_supported(const gnca_model& m, const StepArgs& a);
int launch_update_tc(const gnca_model& m, const Packed& P, const float* packed, StepArgs& a, const uint16_t* glist,
                     const int* prefix, cudaStream_t st);

// Per-frame metrics of gnca_rollout_metrics, written by the forward kernels at every step t % every == 0 (and at T when
// T % every == 0): one partial of 4 doubles per (frame, sample, part) -- part = the CTA's rank in the cluster kernels,
// a block of k_frame_metrics on the streaming path -- summed over the parts in part order by run_metrics_reduce.
struct FrameMetrics {
  const float* target;   // [4][H][W] premultiplied RGBA ([n_models][4][H][W] with a target stride)
  double* part;          // [F][B][P][4] (gnca_metrics_scratch_bytes)
  double* sums;          // [F][B][2] premultiplied-RGBA and clipped-RGB squared-error sums
  int* counts;           // [F][B][2] pixel-perfect and alive cells
  float eps;
  int every;
};
// sums / counts of `rows` (frame, sample) pairs from their P partials (gnca_rollout.cu)
int run_metrics_reduce(int rows, int P, const double* part, double* sums, int* counts, cudaStream_t st);

// SSIM of the same frames (gnca_rollout_metrics_ssim): one double partial per (frame, sample, part), the sum of ssim_cell
// (gnca_metrics.cuh) over the part's interior cells, reduced in part order by run_ssim_reduce into ssim[F][B].  The
// cluster kernels take `part` as a trailing kernel parameter of their SSIM instantiations.
struct SsimFrames {
  double* part;          // [F][B][P] (cluster kernels) or [B][P] (streaming path, one frame at a time)
  double* ssim;          // [F][B]
};
int run_ssim_reduce(int rows, int P, const double* part, double* ssim, int H, int W, cudaStream_t st);

// A stack of same-architecture models in one launch of the cluster kernels (gnca_rollout_record_models /
// gnca_rollout_metrics_models): `packed` is [n_models][stride] and sample b runs model b / per_model.  Each kernel
// rebases `packed` once, before staging the weights into shared memory.  stride = 0: one model for the whole batch.
// A stack's metrics may take one target per model (gnca_rollout_metrics_targets): the forward entry points then take
// target_stride, the floats between two models' targets in FrameMetrics::target (0 = one target for every sample), and
// sample b measures against target + (b / per_model) * target_stride.  It is an argument of its own, not a field: both
// FrameMetrics and ModelStack are kernel parameters by value ahead of or in the plain kernels' parameter lists, and a
// larger struct would change the code of those kernels.
struct ModelStack {
  int stride;      // floats between two models' packed buffers (Packed::total)
  int per_model;   // samples per model (B / n_models)
};

// cluster-resident forward rollout (gnca_resident.cu); GNCA_ERR_UNSUPPORTED when the configuration has no
// resident kernel (zero-padded graph shift, sample too large for the cluster's shared memory).
// hist: x_t of every step t % hist_every == 0 goes to slot t / hist_every ([T/hist_every+1][B][C][H][W]).
int run_resident_fwd(const gnca_model& m, const Packed& P, const float* packed, int B, int H, int W,
                     const gnca_schedule& sched, const float* x0, float* xT, float* hist, float* stats_hist,
                     float* u_hist, float* ping, float* pong, float* alpha_tmp, cudaStream_t st, int hist_every = 1,
                     const FrameMetrics* met = nullptr, ModelStack ms = ModelStack{0, 0},
                     const SsimFrames* ss = nullptr, int target_stride = 0);

// replicated-state cluster rollout (gnca_rep.cu): every CTA of a sample's cluster holds the whole sample; first
// choice of the resident path.  scratch: >= B*C*H*W floats of device memory (overflow of the in-smem u buffer).
// t0: absolute step of the launch's first step, for a `sched` rebased to the launch (a checkpoint segment); only
// sched.steps stays absolute.  The launch configuration depends on B and H*W only, so a segment launch reproduces the
// steps of a whole-rollout launch bit for bit.
// zp (zero-padded graph shift only): with records, also the attention weights and row sums of every message step
// met: the per-frame metrics of the steps t % met->every == 0 (a whole rollout, t0 = 0)
// ms: a stack of models, one per block of ms.per_model samples, with or without records
// ss (with met only): the SSIM of the same frames, by the kernel's SSIM instantiation (run_resident_fwd likewise)
// target_stride (with met and ms only): per-model targets, see ModelStack (run_resident_fwd likewise)
struct ZpRec;
struct ZpBwd;
int run_rep_fwd(const gnca_model& m, const Packed& P, const float* packed, int B, int H, int W,
                const gnca_schedule& sched, const float* x0, float* xT, float* hist, float* stats_hist,
                float* u_hist, float* rec, uint32_t* masks, float* scratch, cudaStream_t st, int hist_every = 1,
                int t0 = 0, const ZpRec* zp = nullptr, const FrameMetrics* met = nullptr,
                ModelStack ms = ModelStack{0, 0}, const SsimFrames* ss = nullptr, int target_stride = 0);
// resident BPTT on the records of run_rep_fwd (gnca_rep_bwd.cu).  g_frames (optional, [F][B][C][H][W]): dL/dx_{f*every}
// added at step f * every (gnca_rollout_bwd_bptt_frames)
size_t rep_bptt_bytes(const gnca_model& m, int B, int H, int W, int T);     // 0: configuration not supported
void rep_bptt_carve(void* base, int B, int H, int W, int T, float** rec, uint32_t** masks, float** stats,
                    float** hgh = nullptr);
// n_models: the weight-gradient partials of a stack (at least one block per model)
size_t rep_bwd_workspace_bytes(const gnca_model& m, int B, int H, int W, int n_models = 1);
// a launch configuration of k_rep_bwd exists (zp: of the zero-padded-shift instantiation)
bool rep_bwd_supported(const gnca_model& m, int B, int H, int W, int k, bool zp = false);
// zp: the zero-padded graph shift's buffers (records of run_rep_fwd with a ZpRec); its Q/K/scaling gradients are
// reduced into gparams after the sweep.  gT_frame = false: g_frames' frame at sched.T is not added to gT (a checkpoint
// segment, where it is the next segment's first frame)
// ms: a stack of models (no frame gradients): gparams is [n_models][layout.total], model i's gradients in row i
int run_rep_bwd(const gnca_model& m, const Packed& P, const float* packed, int B, int H, int W,
                const gnca_schedule& sched, void* bptt, const float* gT, float* g0, float* gparams, void* workspace,
                cudaStream_t st, const float* g_frames = nullptr, int every = 1, int t0 = 0, const ZpBwd* zp = nullptr,
                bool gT_frame = true, ModelStack ms = ModelStack{0, 0});
// zero-padded graph shift: the records of rep_bptt_bytes followed by x_t, the softmax weights, the row sums, bm . gm of
// the active cells and the per-sample Q/K gradients (0: not supported)
size_t rep_bptt_zp_bytes(const gnca_model& m, int B, int H, int W, int T);
void rep_bptt_zp_carve(void* base, const gnca_model& m, int B, int H, int W, int T, float** x, ZpRec* rec, ZpBwd* bwd);

}  // namespace gnca
