// dqn.cu -- C ABI of the IDQN / VDN learner (marl_dqn_*), host-side orchestration of the fused kernels.
//
// Replaces marlbase/dqn/model.py: QNetwork (14-196) and VDNetwork (199-269) -- act's forward pass, _compute_loss,
// update (zero_grad/backward/clip/Adam), update_target/hard_update/soft_update -- and ReplayBuffer.sample's index
// draw + gather (marlbase/dqn/train.py:94-124).
#include "learner.cuh"
#include "retms.cuh"
#include "qmix.cuh"
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

namespace marl {

// ---- replay sampling: np.random.randint(0, len(rb), batch) with replacement (dqn/train.py:95) ------------------
__global__ void replay_sample_kernel(uint64_t seed, uint64_t update_idx, int batch, int n_valid, int32_t* idx) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  pdl_wait();
  pdl_launch_dependents();
  if (i >= batch) return;
  const u32x4 b = philox4x32_10((uint32_t)update_idx, (uint32_t)(update_idx >> 32), (uint32_t)(i >> 2), 0u, (uint32_t)seed, (uint32_t)(seed >> 32) ^ kTagSample);
  idx[i] = (int32_t)bounded(pick(b, i & 3), (uint32_t)n_valid);
}

// ---- VDN: agent-coupled TD error (marlbase/dqn/model.py:224-269) ------------------------------------------------
struct VdnTdParams {
  const float* q; const float* tq;  // [N][B][T+1][A]
  TrajView traj; const int32_t* idx; int B, N, A; float gamma; int double_q;
  float* td;         // [B][T] = 2 * delta * filled
  float* loss_part;  // [gridDim][4]
};

__global__ void __launch_bounds__(256) vdn_td_kernel(VdnTdParams p) {
  __shared__ float red[512];
  const int T = p.traj.T, i = blockIdx.x * 256 + threadIdx.x;
  float loss = 0.f, fill = 0.f;
  if (i < p.B * T) {
    const int b = i / T, t = i - b * T;
    const size_t ep = (size_t)p.idx[b];
    float chosen = 0.f, tsum = 0.f;
    for (int a = 0; a < p.N; ++a) {
      const size_t row = ((size_t)a * p.B + b) * (T + 1) + t;
      const float* q0 = p.q + row * p.A; const float* q1 = q0 + p.A; const float* t1 = p.tq + (row + 1) * p.A;
      chosen += q0[p.traj.act[(ep * p.N + a) * T + t]];
      if (p.double_q) {
        int best = 0; float bv = q1[0];
        for (int o = 1; o < p.A; ++o) if (q1[o] > bv) { bv = q1[o]; best = o; }
        tsum += t1[best];
      } else {
        float m = t1[0];
        for (int o = 1; o < p.A; ++o) m = fmaxf(m, t1[o]);
        tsum += m;
      }
    }
    const float filled = (float)p.traj.filled[ep * T + t];
    const float y = p.traj.rew[(ep * p.N + 0) * T + t] + p.gamma * tsum * (1.f - (float)p.traj.done[ep * (T + 1) + t + 1]);
    const float delta = chosen - y;
    loss = delta * delta * filled; fill = filled;
    p.td[i] = 2.f * delta * filled;
  }
  red[threadIdx.x] = loss; red[256 + threadIdx.x] = fill;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) { red[threadIdx.x] += red[threadIdx.x + s]; red[256 + threadIdx.x] += red[256 + threadIdx.x + s]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { p.loss_part[4 * blockIdx.x] = red[0]; p.loss_part[4 * blockIdx.x + 1] = red[256]; p.loss_part[4 * blockIdx.x + 2] = 0.f; p.loss_part[4 * blockIdx.x + 3] = 0.f; }
}

// ---- cfg.standardise_returns (dqn/model.py:147-158, VDN 256-264): the TD target needs statistics of the whole batch's returns before any loss ----
// 1. returns[c][b][t] = r + gamma * (target_qs * sqrt(var) + mean) * (1 - done[t + 1]) and chosen[c][b][t] = Q(o_t)[a_t] (VDN: both summed over the
//    agents, c = 0); every (b, t), filled or not, as the reference.  Columns of the statistics: one per agent (IDQN); the reference's VDN reshapes
//    its (E, B) returns with reshape(-1, B), i.e. one column per batch entry -- stat_per_b selects that.
// 2. RunningMeanStd step (retms.cuh): statistics absorb the returns, returns are standardised in place.
// 3. td[c][b][t] = 2 (chosen - returns) filled  +  the loss statistics.
struct StdRetParams {
  const float* q; const float* tq;  // [N][B][T+1][A]
  TrajView traj; const int32_t* idx; int B, N, A, vdn; float gamma; int double_q;
  const float* ret_ms; int n_stat, stat_per_b;   // mean[n_stat] | var[n_stat]
  float* ret; float* chosen; float* td;          // [C][B][T], C = vdn ? 1 : N
  float* loss_part;
};
__global__ void __launch_bounds__(256) std_returns_kernel(StdRetParams p) {
  const int T = p.traj.T, C = p.vdn ? 1 : p.N, i = blockIdx.x * 256 + threadIdx.x;
  if (i >= C * p.B * T) return;
  const int c = i / (p.B * T), rem = i - c * p.B * T, b = rem / T, t = rem - b * T;
  const size_t ep = (size_t)p.idx[b];
  float chosen = 0.f, tsel = 0.f;
  for (int a = (p.vdn ? 0 : c); a < (p.vdn ? p.N : c + 1); ++a) {
    const size_t row = ((size_t)a * p.B + b) * (T + 1) + t;
    const float* q0 = p.q + row * p.A; const float* q1 = q0 + p.A; const float* t1 = p.tq + (row + 1) * p.A;
    chosen += q0[p.traj.act[(ep * p.N + a) * T + t]];
    if (p.double_q) {
      int best = 0; float bv = q1[0];
      for (int o = 1; o < p.A; ++o) if (q1[o] > bv) { bv = q1[o]; best = o; }
      tsel += t1[best];
    } else {
      float m = t1[0];
      for (int o = 1; o < p.A; ++o) m = fmaxf(m, t1[o]);
      tsel += m;
    }
  }
  const int col = p.stat_per_b ? b : c;
  tsel = __fadd_rn(__fmul_rn(tsel, sqrtf(p.ret_ms[p.n_stat + col])), p.ret_ms[col]);     // target_qs * sqrt(var) + mean
  const float rew = p.traj.rew[(ep * p.N + (p.vdn ? 0 : c)) * T + t];
  const float y = __fadd_rn(rew, __fmul_rn(__fmul_rn(p.gamma, tsel), 1.f - (float)p.traj.done[ep * (T + 1) + t + 1]));
  // the statistics' columns must be contiguous: [col][...]
  const size_t o = p.stat_per_b ? ((size_t)b * T + t) : (size_t)i;
  p.ret[o] = y; p.chosen[o] = chosen;
}
__global__ void __launch_bounds__(256) std_td_kernel(StdRetParams p) {
  __shared__ float red[512];
  const int T = p.traj.T, C = p.vdn ? 1 : p.N, i = blockIdx.x * 256 + threadIdx.x;
  float loss = 0.f, fill = 0.f;
  if (i < C * p.B * T) {
    const int c = i / (p.B * T), rem = i - c * p.B * T, b = rem / T, t = rem - b * T;
    const float filled = (float)p.traj.filled[(size_t)p.idx[b] * T + t];
    const float delta = p.chosen[i] - p.ret[i];
    loss = delta * delta * filled; fill = c == 0 ? filled : 0.f;
    p.td[i] = 2.f * delta * filled;
  }
  red[threadIdx.x] = loss; red[256 + threadIdx.x] = fill;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) { red[threadIdx.x] += red[threadIdx.x + s]; red[256 + threadIdx.x] += red[256 + threadIdx.x + s]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { p.loss_part[4 * blockIdx.x] = red[0]; p.loss_part[4 * blockIdx.x + 1] = red[256]; p.loss_part[4 * blockIdx.x + 2] = 0.f; p.loss_part[4 * blockIdx.x + 3] = 0.f; }
}

}  // namespace marl

using namespace marl;

struct marl_dqn {
  NetSet ns;
  marl_dqn_hp hp;
  int device = 0, n_sm = 148, max_batch = 0, max_T = 0;
  int64_t n_params = 0;  // n_nets * P
  int scratch_pitch = 0;
  float *theta = nullptr, *theta_tgt = nullptr, *m = nullptr, *v = nullptr, *grad = nullptr;
  float *scratch = nullptr, *loss_part = nullptr, *tq = nullptr, *q_all = nullptr, *td = nullptr, *loss_dev = nullptr, *sumsq = nullptr;
  bool grads_are_local = false;  // set by update_grads, cleared when the caller may have all-reduced grad
  int32_t* idx = nullptr;
  uint8_t* image = nullptr;      // packed weight images for the tensor-core forward path (scratch, rebuilt per call)
  uint8_t* image_tgt = nullptr;  // image of theta_tgt, rebuilt only when the target network changed
  uint8_t* image_bwd = nullptr;  // MN-major image of W2 (online net) for the tensor-core backward
  float *tc_h1 = nullptr, *tc_h2 = nullptr, *tc_dh1 = nullptr, *tc_rec = nullptr, *tc_x = nullptr;
  bool tgt_image_current = false;
  unsigned long long* grid_barrier = nullptr; unsigned long long grid_epoch = 0;   // arrival counter of the fused reduce + Adam kernel
  unsigned long long push_epoch = 0;   // arrival counter of the push kernel (split exchange)
  bool tq_ahead = false;               // the target forward of the NEXT update has already been launched (between push and finish)
  // gradient exchange over peer memory (several ranks, one process per GPU): own buffer + the peers' buffers opened through CUDA IPC
  XchgParams xchg = {}; float* xbuf = nullptr; void* peer_base[kMaxRanks] = {};
  // online images: valid = a full pack happened and every later change of theta came from adam_kernel (which updates them in place)
  bool image_current = false, bwd_image_current = false;
  int64_t updates = 0, last_target_update = 0;
  RowPlan train_plan; int n_loss_parts = 0;
  // optional CUDA-event timing of the training kernel (bench.py's roofline leg)
  // measurement hook: 4 events per timed update (before the training pass, after each of its kernels; the FP32 path uses 0 and 3)
  bool timing = false; std::vector<cudaEvent_t> ev; int ev_used = 0; bool ev_split = false;
  // cfg.standardise_returns: RunningMeanStd over the TD targets (mean[n] | var[n], count, partial sums, returns / chosen-Q scratch)
  int standardise = 0, n_stat = 0; float *ret_ms = nullptr, *ret = nullptr, *chosen = nullptr; double *ret_count = nullptr, *ret_part = nullptr;
  // QMIX (hp.mixer == 2): the mixing network's parameters / Adam state / gradient (+ 4 statistics), per-sample records, chunked partial sums, tile list
  QmixLayout ql = {}; float *mix = nullptr, *mix_tgt = nullptr, *mix_m = nullptr, *mix_v = nullptr, *mix_grad = nullptr, *mix_rec = nullptr, *mix_part = nullptr, *mix_img = nullptr, *mix_img_tgt = nullptr;
  QmixTile* mix_tiles = nullptr; int mix_n_tiles = 0; QmixMicro* mix_micro = nullptr; int mix_n_micro = 0; bool mix_wgrad_tiles = false;
};
static const int kTimingPairs = 1024;

static int dqn_alloc(float** p, size_t n_floats) { return dev_alloc_zero(p, n_floats); }

extern "C" {

int marl_dqn_create(const marl_mlp_cfg* cfg, const marl_dqn_hp* hp, int32_t max_batch, int32_t max_T, int32_t device, marl_dqn** out) {
  MARL_REQUIRE(cfg && hp && out, "marl_dqn_create: NULL argument");
  *out = nullptr;
  MARL_REQUIRE(cfg->n_agents >= 1 && cfg->n_agents <= MARL_MAX_AGENTS, "marl_dqn_create: n_agents out of range");
  MARL_REQUIRE(cfg->n_nets >= 1 && cfg->n_nets <= cfg->n_agents, "marl_dqn_create: n_nets out of range");
  MARL_REQUIRE(cfg->hidden == kHidden, "marl_dqn_create: only layers=[128,128] is implemented on the B200 path (got hidden=%d)", cfg->hidden);
  MARL_REQUIRE(cfg->out_dim >= 1 && cfg->out_dim <= kOutPad, "marl_dqn_create: n_actions %d not supported (1..%d)", cfg->out_dim, kOutPad);
  MARL_REQUIRE(max_batch >= 1 && max_T >= 1, "marl_dqn_create: max_batch/max_T must be >= 1");
  MARL_REQUIRE(hp->mixer >= 0 && hp->mixer <= 2, "marl_dqn_create: mixer must be 0 (independent), 1 (VDN) or 2 (QMIX)");
  for (int a = 0; a < cfg->n_agents; ++a) MARL_REQUIRE(cfg->agent_net[a] >= 0 && cfg->agent_net[a] < cfg->n_nets, "marl_dqn_create: agent_net[%d] out of range", a);
  if (int rc = check_device(device)) return rc;
  marl_dqn* h = new marl_dqn();
  h->ns.n_agents = cfg->n_agents; h->ns.n_nets = cfg->n_nets; h->ns.in = cfg->in_dim; h->ns.out = cfg->out_dim;
  memcpy(h->ns.agent_net, cfg->agent_net, sizeof(int) * MARL_MAX_AGENTS);
  h->ns.lay = NetLayout::make(cfg->in_dim, cfg->out_dim);
  h->hp = *hp; h->device = device; h->max_batch = max_batch; h->max_T = max_T;
  cudaDeviceProp prop; cudaGetDeviceProperties(&prop, device); h->n_sm = prop.multiProcessorCount;
  h->n_params = (int64_t)cfg->n_nets * h->ns.lay.P;
  h->scratch_pitch = (h->ns.lay.P + 3) & ~3;
  const size_t rows = (size_t)cfg->n_agents * max_batch * (max_T + 1);
  int rc = 0;
  rc |= dqn_alloc(&h->theta, h->n_params); rc |= dqn_alloc(&h->theta_tgt, h->n_params);
  rc |= dqn_alloc(&h->m, h->n_params); rc |= dqn_alloc(&h->v, h->n_params); rc |= dqn_alloc(&h->grad, h->n_params + 4);
  rc |= dqn_alloc(&h->scratch, (size_t)h->n_sm * h->scratch_pitch);
  rc |= dqn_alloc(&h->loss_part, 4 * ((size_t)h->n_sm + (size_t)max_batch * max_T / 256 + 2));
  rc |= dqn_alloc(&h->tq, rows * cfg->out_dim);
  rc |= dqn_alloc(&h->loss_dev, 8);
  rc |= dqn_alloc(&h->sumsq, (size_t)(h->n_params + 63) / 64 + 1);
  rc |= dqn_alloc(reinterpret_cast<float**>(&h->grid_barrier), 4);   // two zero-initialised 64-bit counters (grid barrier, push arrivals)
  if (hp->mixer == 1) { rc |= dqn_alloc(&h->q_all, rows * cfg->out_dim); rc |= dqn_alloc(&h->td, (size_t)max_batch * max_T); }
  if (hp->mixer == 2) { rc |= dqn_alloc(&h->q_all, rows * cfg->out_dim); rc |= dqn_alloc(&h->td, (size_t)cfg->n_agents * max_batch * max_T); }
  rc |= dqn_alloc(reinterpret_cast<float**>(&h->idx), max_batch);
  rc |= dqn_alloc(reinterpret_cast<float**>(&h->image), (size_t)cfg->n_nets * tc_image_bytes() / 4 + 4);
  rc |= dqn_alloc(reinterpret_cast<float**>(&h->image_tgt), (size_t)cfg->n_nets * tc_image_bytes() / 4 + 4);
  if (rc) { marl_dqn_destroy(h); return MARL_ENOMEM; }
  if (int rc2 = learner_kernels_init(cfg->in_dim)) { marl_dqn_destroy(h); return rc2; }
  if (int rc2 = tc_forward_init()) { marl_dqn_destroy(h); return rc2; }
  if (int rc2 = tc_train_init()) { marl_dqn_destroy(h); return rc2; }
  *out = h;
  return MARL_OK;
}

int marl_dqn_destroy(marl_dqn* h) {
  if (!h) return MARL_OK;
  cudaSetDevice(h->device);
  cudaFree(h->theta); cudaFree(h->theta_tgt); cudaFree(h->m); cudaFree(h->v); cudaFree(h->grad); cudaFree(h->scratch);
  cudaFree(h->loss_part); cudaFree(h->tq); cudaFree(h->q_all); cudaFree(h->td); cudaFree(h->loss_dev); cudaFree(h->sumsq); cudaFree(h->idx); cudaFree(h->image); cudaFree(h->image_tgt); cudaFree(h->image_bwd); cudaFree(h->tc_h1); cudaFree(h->tc_h2); cudaFree(h->tc_dh1); cudaFree(h->tc_rec); cudaFree(h->tc_x); cudaFree(h->grid_barrier);
  for (int r = 0; r < kMaxRanks; ++r) if (h->peer_base[r] != nullptr && r != h->xchg.rank) cudaIpcCloseMemHandle(h->peer_base[r]);
  cudaFree(h->mix); cudaFree(h->mix_tgt); cudaFree(h->mix_m); cudaFree(h->mix_v); cudaFree(h->mix_grad); cudaFree(h->mix_rec); cudaFree(h->mix_part); cudaFree(h->mix_tiles); cudaFree(h->mix_micro); cudaFree(h->mix_img); cudaFree(h->mix_img_tgt);
  cudaFree(h->xbuf); cudaFree(h->ret_ms); cudaFree(h->ret); cudaFree(h->chosen); cudaFree(h->ret_count); cudaFree(h->ret_part);
  for (auto& e : h->ev) cudaEventDestroy(e);
  delete h;
  return MARL_OK;
}

/* cfg.standardise_returns (dqn/model.py:82-84, 221-222): RunningMeanStd over the TD targets, one column per agent (VDN: per batch entry, see the
 * kernels above); mean 0, var 1, count 1e-4 on first enable. */
int marl_dqn_standardise_returns(marl_dqn* h, int32_t enable) {
  MARL_REQUIRE(h != nullptr, "marl_dqn_standardise_returns: NULL handle");
  MARL_REQUIRE(h->hp.mixer != 2 || !enable, "marl_dqn_standardise_returns: not implemented for QMIX (qmix.yaml inherits standardise_returns: False)");
  MARL_CUDA_TRY(cudaSetDevice(h->device));
  if (enable && !h->ret_ms) {
    const int n = h->hp.mixer == 1 ? h->max_batch : h->ns.n_agents, C = h->hp.mixer == 1 ? 1 : h->ns.n_agents;
    const size_t rows = (size_t)h->ns.n_agents * h->max_batch * (h->max_T + 1);
    std::vector<float> init(2 * n, 0.f);
    for (int a = 0; a < n; ++a) init[n + a] = 1.f;
    const double c0 = 1e-4;
    int rc = 0;
    rc |= dqn_alloc(&h->ret_ms, 2 * n); rc |= dqn_alloc(&h->ret, (size_t)C * h->max_batch * h->max_T); rc |= dqn_alloc(&h->chosen, (size_t)C * h->max_batch * h->max_T);
    if (!h->q_all) rc |= dqn_alloc(&h->q_all, rows * h->ns.out);
    if (!h->td || h->hp.mixer == 0) { cudaFree(h->td); h->td = nullptr; rc |= dqn_alloc(&h->td, (size_t)C * h->max_batch * h->max_T); }
    if (rc) return MARL_ENOMEM;
    MARL_CUDA_TRY(cudaMalloc(&h->ret_count, sizeof(double))); MARL_CUDA_TRY(cudaMalloc(&h->ret_part, (size_t)kRetBlocks * n * 2 * sizeof(double)));
    MARL_CUDA_TRY(cudaMemcpy(h->ret_ms, init.data(), 2 * n * sizeof(float), cudaMemcpyHostToDevice));
    MARL_CUDA_TRY(cudaMemcpy(h->ret_count, &c0, sizeof(double), cudaMemcpyHostToDevice));
    h->n_stat = n;
    // the per-update loss statistics of this path come from one block per 256 (c, b, t) entries
    cudaFree(h->loss_part); h->loss_part = nullptr;
    if (dqn_alloc(&h->loss_part, 4 * ((size_t)h->n_sm + (size_t)C * h->max_batch * h->max_T / 256 + 2))) return MARL_ENOMEM;
  }
  h->standardise = enable ? 1 : 0;
  return MARL_OK;
}
int marl_dqn_ret_ms_ptrs(marl_dqn* h, float** ret_ms, double** count, int32_t* n_stat) {
  MARL_REQUIRE(h != nullptr, "marl_dqn_ret_ms_ptrs: NULL handle");
  if (ret_ms) *ret_ms = h->ret_ms; if (count) *count = h->ret_count; if (n_stat) *n_stat = h->n_stat;
  return MARL_OK;
}

/* QMixNetwork.__init__ (dqn/model.py:365-379): the mixing network over the concatenated observations (state_dim = N * in_dim).  Parameters are
 * initialised by the caller through marl_dqn_qmix_ptrs (nn.Linear defaults), then marl_dqn_sync_target copies them to the target mixer. */
int marl_dqn_qmix_init(marl_dqn* h, int32_t embed_dim, int32_t hypernet_layers, int32_t hypernet_embed) {
  MARL_REQUIRE(h != nullptr && h->hp.mixer == 2, "marl_dqn_qmix_init: the learner was not created with mixer = 2");
  MARL_REQUIRE(h->mix == nullptr, "marl_dqn_qmix_init: already initialised");
  MARL_REQUIRE(hypernet_layers == 2, "marl_dqn_qmix_init: hypernet_layers = %d: only the shipped two-layer hypernetworks (qmix.yaml) are implemented", hypernet_layers);
  MARL_REQUIRE(embed_dim >= 4 && embed_dim <= kQmixEmbedMax && embed_dim % 4 == 0, "marl_dqn_qmix_init: embed_dim %d not supported (multiple of 4, <= %d)", embed_dim, kQmixEmbedMax);
  MARL_REQUIRE(hypernet_embed >= 4 && hypernet_embed <= kQmixHypMax && hypernet_embed % 4 == 0, "marl_dqn_qmix_init: hypernet_embed %d not supported (multiple of 4, <= %d)", hypernet_embed, kQmixHypMax);
  const int N = h->ns.n_agents, S = N * h->ns.in;
  MARL_REQUIRE(S <= kQmixStateMax && N <= kQmixAgentsMax, "marl_dqn_qmix_init: state_dim %d (<= %d) or n_agents %d (<= %d) too large", S, kQmixStateMax, N, kQmixAgentsMax);
  MARL_CUDA_TRY(cudaSetDevice(h->device));
  h->ql = qmix_layout(N, S, embed_dim, hypernet_embed);
  const size_t n = (size_t)h->ql.n, samples = (size_t)h->max_batch * h->max_T;
  MARL_REQUIRE(qm_smem_bytes(h->ql) <= 227 * 1024, "marl_dqn_qmix_init: the mixer's %zu parameters + a 32-sample tile (%zu bytes) do not fit shared memory", n, qm_smem_bytes(h->ql));
  std::vector<QmixTile> tiles(kQmixMaxTiles);
  const int nt = qmix_tiles(h->ql, tiles.data());
  MARL_REQUIRE(nt > 0, "marl_dqn_qmix_init: too many weight-gradient tiles");
  int rc = 0;
  rc |= dqn_alloc(&h->mix, n); rc |= dqn_alloc(&h->mix_tgt, n); rc |= dqn_alloc(&h->mix_m, n); rc |= dqn_alloc(&h->mix_v, n); rc |= dqn_alloc(&h->mix_grad, n + 4);
  rc |= dqn_alloc(&h->mix_rec, (size_t)h->ql.R * samples); rc |= dqn_alloc(&h->mix_part, (size_t)(2 * h->n_sm > kQmixChunks ? 2 * h->n_sm : kQmixChunks) * n);
  rc |= dqn_alloc(reinterpret_cast<float**>(&h->mix_tiles), (size_t)nt * sizeof(QmixTile) / 4);
  rc |= dqn_alloc(&h->mix_img, (n + 3) & ~(size_t)3); rc |= dqn_alloc(&h->mix_img_tgt, (n + 3) & ~(size_t)3);
  cudaFree(h->loss_part); h->loss_part = nullptr;   // one block of statistics per tile of kQmTS samples
  rc |= dqn_alloc(&h->loss_part, 4 * ((size_t)h->n_sm + samples / kQmTS + 2));
  if (rc) return MARL_ENOMEM;
  MARL_CUDA_TRY(cudaMemcpy(h->mix_tiles, tiles.data(), (size_t)nt * sizeof(QmixTile), cudaMemcpyHostToDevice));
  h->mix_n_tiles = nt;
  std::vector<QmixMicro> micro(1 << 14);
  const int nm = qmix_micro_tiles(h->ql, micro.data(), (int)micro.size());
  MARL_REQUIRE(nm > 0, "marl_dqn_qmix_init: too many weight-gradient micro-tiles");
  if (dqn_alloc(reinterpret_cast<float**>(&h->mix_micro), (size_t)nm * sizeof(QmixMicro) / 4)) return MARL_ENOMEM;
  MARL_CUDA_TRY(cudaMemcpy(h->mix_micro, micro.data(), (size_t)nm * sizeof(QmixMicro), cudaMemcpyHostToDevice));
  h->mix_n_micro = nm;
  static size_t mix_limits[64] = {}, wg_limits[64] = {};   // per device (one process normally drives one GPU)
  size_t& mix_smem_limit = mix_limits[h->device & 63]; size_t& wg_smem_limit = wg_limits[h->device & 63];
  const size_t wg_smem = (size_t)(h->ql.R + 2) * kQmP * sizeof(float);
  const char* ev = getenv("MARL_QMIX_WGRAD_TILES");
  h->mix_wgrad_tiles = (ev != nullptr && ev[0] == '1') || wg_smem > 110 * 1024;   // the single-read form needs all record fields of 32 samples in shared memory
  if (!h->mix_wgrad_tiles && wg_smem > wg_smem_limit) {
    MARL_CUDA_TRY(cudaFuncSetAttribute(qmix_wgrad2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wg_smem));
    wg_smem_limit = wg_smem;
  }
  // the attribute is per function, process-wide: only ever raise it (a second learner with a smaller mixer must not lower the first one's limit)
  if (qm_smem_bytes(h->ql) > mix_smem_limit) {
    MARL_CUDA_TRY(cudaFuncSetAttribute(qmix_mix_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)qm_smem_bytes(h->ql)));
    mix_smem_limit = qm_smem_bytes(h->ql);
  }
  return MARL_OK;
}
/* Host-only self-check of the QMIX weight-gradient decompositions (no device needed): counts[0 .. n) = how many micro-tile entries of the single-read
 * kernel write parameter j, counts[n .. 2n) = the same for the 32 x 32 tile form; both must be 1 everywhere.  Returns n through n_params. */
int marl_debug_qmix_coverage(int32_t n_agents, int32_t state_dim, int32_t embed_dim, int32_t hypernet_embed, int32_t* counts, int64_t cap, int64_t* n_params) {
  MARL_REQUIRE(n_agents >= 1 && state_dim >= 1 && embed_dim >= 4 && hypernet_embed >= 4 && n_params != nullptr, "marl_debug_qmix_coverage: bad argument");
  const QmixLayout L = qmix_layout(n_agents, state_dim, embed_dim, hypernet_embed);
  *n_params = L.n;
  if (counts == nullptr) return MARL_OK;
  MARL_REQUIRE(cap >= 2 * (int64_t)L.n, "marl_debug_qmix_coverage: counts needs 2 x %d entries", L.n);
  for (int j = 0; j < 2 * L.n; ++j) counts[j] = 0;
  std::vector<QmixMicro> micro(1 << 16);
  const int nm = qmix_micro_tiles(L, micro.data(), (int)micro.size());
  MARL_REQUIRE(nm > 0, "marl_debug_qmix_coverage: too many micro-tiles");
  for (int m = 0; m < nm; ++m) {
    const QmixMicro& mt = micro[m];
    for (int oo = 0; oo < mt.n_o; ++oo)
      for (int ii = 0; ii < 8; ++ii) {
        const int o = mt.o0 + oo, i = mt.i0 + ii;
        if (i < mt.I) counts[mt.woff + o * mt.I + i] += 1;
        else if (i == mt.I) counts[mt.boff + o] += 1;
      }
  }
  std::vector<QmixTile> tiles(kQmixMaxTiles);
  const int nt = qmix_tiles(L, tiles.data());
  MARL_REQUIRE(nt > 0, "marl_debug_qmix_coverage: too many tiles");
  for (int t = 0; t < nt; ++t) {
    const QmixTile& tl = tiles[t];
    for (int oo = 0; oo < 32; ++oo)
      for (int ii = 0; ii < 32; ++ii) {
        const int o = tl.o0 + oo, i = tl.i0 + ii;
        if (o >= tl.O) continue;
        if (i < tl.I) counts[L.n + tl.woff + o * tl.I + i] += 1;
        else if (i == tl.I) counts[L.n + tl.boff + o] += 1;
      }
  }
  return MARL_OK;
}

int marl_dqn_qmix_ptrs(marl_dqn* h, float** mix, float** mix_tgt, float** adam_m, float** adam_v, float** grad, int64_t* n_params) {
  MARL_REQUIRE(h != nullptr && h->mix != nullptr, "marl_dqn_qmix_ptrs: no mixer (marl_dqn_qmix_init)");
  if (mix) *mix = h->mix; if (mix_tgt) *mix_tgt = h->mix_tgt; if (adam_m) *adam_m = h->mix_m; if (adam_v) *adam_v = h->mix_v;
  if (grad) *grad = h->mix_grad; if (n_params) *n_params = h->ql.n;
  return MARL_OK;
}

int marl_dqn_param_ptrs(marl_dqn* h, float** theta, float** theta_tgt, float** adam_m, float** adam_v, float** grad, int64_t* n_params) {
  MARL_REQUIRE(h != nullptr, "marl_dqn_param_ptrs: NULL handle");
  if (theta) *theta = h->theta; if (theta_tgt) *theta_tgt = h->theta_tgt; if (adam_m) *adam_m = h->m; if (adam_v) *adam_v = h->v;
  if (grad) *grad = h->grad; if (n_params) *n_params = h->n_params;
  return MARL_OK;
}

int marl_dqn_sync_target(marl_dqn* h, void* stream) {
  MARL_REQUIRE(h != nullptr, "marl_dqn_sync_target: NULL handle");
  MARL_CUDA_TRY(cudaSetDevice(h->device));
  MARL_CUDA_TRY(cudaMemcpyAsync(h->theta_tgt, h->theta, h->n_params * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (h->mix) MARL_CUDA_TRY(cudaMemcpyAsync(h->mix_tgt, h->mix, (size_t)h->ql.n * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));   // dqn/model.py:438-443
  h->tgt_image_current = false;
  return MARL_OK;
}

int marl_dqn_forward(marl_dqn* h, const float* obs, int32_t n_envs, int32_t use_target, float* q_out, void* stream) {
  MARL_REQUIRE(h && obs && q_out && n_envs >= 1, "marl_dqn_forward: bad argument");
  MARL_CUDA_TRY(cudaSetDevice(h->device));
  const RowPlan plan = make_plan(h->ns, n_envs, 1, h->n_sm, 32);
  RowSource src; memset(&src, 0, sizeof(src));
  src.mode = 0; src.dense = obs; src.E = n_envs; src.N = h->ns.n_agents; src.D = h->ns.in;
  bool& current = use_target ? h->tgt_image_current : h->image_current;
  const int rc = forward_any(h->ns, plan, src, use_target ? h->theta_tgt : h->theta, use_target ? h->image_tgt : h->image, q_out, (cudaStream_t)stream, current);
  if (rc == MARL_OK) current = tc_forward_for(h->ns);
  return rc;
}

int marl_replay_sample(uint64_t seed, uint64_t update_idx, int32_t batch, int32_t n_valid, int32_t* idx_out, void* stream) {
  MARL_REQUIRE(idx_out && batch >= 1 && n_valid >= 1, "marl_replay_sample: bad argument");
  MARL_CUDA_TRY(launch_pdl(replay_sample_kernel, dim3((batch + 255) / 256), dim3(256), 0, (cudaStream_t)stream, seed, update_idx, (int)batch, (int)n_valid, idx_out));
  return MARL_OK;
}

// Gradient half of an update.  rp_out == NULL: the per-CTA partials are reduced into grad[] (grad_reduce_kernel); otherwise the
// reduction is left to the caller (fused reduce + Adam tail) and its parameters are returned.
static int dqn_grads(marl_dqn* h, const marl_traj_view* traj, const int32_t* episode_idx, int32_t batch, void* stream, ReduceParams* rp_out) {
  MARL_REQUIRE(h && traj && episode_idx, "marl_dqn_update_grads: NULL argument");
  MARL_REQUIRE(batch >= 1 && batch <= h->max_batch, "marl_dqn_update_grads: batch %d exceeds max_batch %d", batch, h->max_batch);
  MARL_REQUIRE(traj->T >= 1 && traj->T <= h->max_T, "marl_dqn_update_grads: T %d exceeds max_T %d", traj->T, h->max_T);
  MARL_REQUIRE(traj->n_agents == h->ns.n_agents && traj->obs_dim == h->ns.in, "marl_dqn_update_grads: trajectory shape mismatch");
  MARL_CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int T = traj->T;
  const int min_units = (64 + T) / (T + 1) > 0 ? (64 + T) / (T + 1) : 1;
  const RowPlan plan = make_plan(h->ns, batch, T + 1, h->n_sm, min_units);
  RowSource src; memset(&src, 0, sizeof(src));
  src.mode = 1; src.traj = to_view(traj); src.idx = episode_idx; src.N = h->ns.n_agents; src.D = h->ns.in;
  // target network on every gathered row (dqn/model.py:132-134); several ranks: the previous update launched it between its push and its finish
  if (h->tq_ahead) {
    h->tq_ahead = false;
  } else {
    if (int rc = forward_any(h->ns, plan, src, h->theta_tgt, h->image_tgt, h->tq, st, h->tgt_image_current)) return rc;
    h->tgt_image_current = tc_forward_for(h->ns);
  }
  int n_loss_parts = plan.cta_begin[plan.n_nets];
  const float* td_ext = nullptr;
  float* loss_part = h->loss_part;
  int td_agent_stride = 0;
  if (h->standardise) {
    // online Q-values of every row, returns + chosen Q, RunningMeanStd step, TD error (dqn/model.py:147-158 / 256-264)
    MARL_REQUIRE(h->hp.mixer == 0 || batch == h->n_stat, "marl_dqn_update: VDN's standardise_returns keeps one statistic per batch entry (the reference's reshape(-1, B)): "
                 "batch %d must stay at max_batch %d", batch, h->n_stat);
    if (int rc = forward_any(h->ns, plan, src, h->theta, h->image, h->q_all, st, h->image_current)) return rc;
    h->image_current = tc_forward_for(h->ns);
    const int C = h->hp.mixer == 1 ? 1 : h->ns.n_agents;
    StdRetParams sp; memset(&sp, 0, sizeof(sp));
    sp.q = h->q_all; sp.tq = h->tq; sp.traj = src.traj; sp.idx = episode_idx; sp.B = batch; sp.N = h->ns.n_agents; sp.A = h->ns.out; sp.vdn = h->hp.mixer == 1;
    sp.gamma = h->hp.gamma; sp.double_q = h->hp.double_q; sp.ret_ms = h->ret_ms; sp.n_stat = h->n_stat; sp.stat_per_b = h->hp.mixer == 1;
    sp.ret = h->ret; sp.chosen = h->chosen; sp.td = h->td;
    const int vb = (C * batch * T + 255) / 256;
    sp.loss_part = h->loss_part + 4 * (size_t)n_loss_parts;
    std_returns_kernel<<<vb, 256, 0, st>>>(sp);
    RetMsParams rp; rp.ret = h->ret; rp.part = h->ret_part; rp.ret_ms = h->ret_ms; rp.count = h->ret_count; rp.T = T;
    if (h->hp.mixer == 1) { rp.N = batch; rp.P = 1; } else { rp.N = C; rp.P = batch; }
    MARL_CUDA_TRY(ret_ms_step(rp, st));
    std_td_kernel<<<vb, 256, 0, st>>>(sp);
    MARL_CUDA_TRY(cudaGetLastError());
    n_loss_parts += vb;
    td_ext = h->td;
    td_agent_stride = h->hp.mixer == 1 ? 0 : batch * T;
  } else if (h->hp.mixer == 1) {  // VDN: online Q-values of all agents first, then the agent-summed TD error
    if (int rc = forward_any(h->ns, plan, src, h->theta, h->image, h->q_all, st, h->image_current)) return rc;
    h->image_current = tc_forward_for(h->ns);
    VdnTdParams vp; vp.q = h->q_all; vp.tq = h->tq; vp.traj = src.traj; vp.idx = episode_idx; vp.B = batch; vp.N = h->ns.n_agents; vp.A = h->ns.out;
    vp.gamma = h->hp.gamma; vp.double_q = h->hp.double_q; vp.td = h->td;
    const int vb = (batch * T + 255) / 256;
    vp.loss_part = h->loss_part + 4 * (size_t)n_loss_parts;  // the train kernel's parts read as zero in this mode
    vdn_td_kernel<<<vb, 256, 0, st>>>(vp);
    MARL_CUDA_TRY(cudaGetLastError());
    n_loss_parts += vb;
    td_ext = h->td;
  } else if (h->hp.mixer == 2) {  // QMIX: the mixer turns the agents' Q-values into the TD error and hands dL/dq_a back per agent (qmix.cuh)
    MARL_REQUIRE(h->mix != nullptr, "marl_dqn_update: QMIX needs marl_dqn_qmix_init first");
    if (int rc = forward_any(h->ns, plan, src, h->theta, h->image, h->q_all, st, h->image_current)) return rc;
    h->image_current = tc_forward_for(h->ns);
    QmixParams qp; memset(&qp, 0, sizeof(qp));
    qp.L = h->ql; qp.q = h->q_all; qp.tq = h->tq; qp.traj = src.traj; qp.idx = episode_idx; qp.B = batch; qp.A = h->ns.out; qp.D = h->ns.in;
    qp.gamma = h->hp.gamma; qp.double_q = h->hp.double_q; qp.mix = h->mix; qp.mix_tgt = h->mix_tgt; qp.rec = h->mix_rec; qp.td = h->td;
    qp.loss_part = h->loss_part + 4 * (size_t)n_loss_parts;
    const int Sn = batch * T, qb = (Sn + kQmTS - 1) / kQmTS, n = h->ql.n;
    qmix_pack_kernel<<<dim3((n + 255) / 256, 2), 256, 0, st>>>(h->ql, h->mix, h->mix_tgt, h->mix_img, h->mix_img_tgt);
    qmix_mix_kernel<<<qb, kQmWarps * 32, qm_smem_bytes(h->ql), st>>>(qp, h->mix_img, h->mix_img_tgt);
    const int want = h->mix_wgrad_tiles ? kQmixChunks : 2 * h->n_sm;
    const int chunk_len = (((Sn + want - 1) / want) + 31) & ~31, chunks = (Sn + chunk_len - 1) / chunk_len;
    if (h->mix_wgrad_tiles) {
      qmix_wgrad_kernel<<<dim3(h->mix_n_tiles, chunks), 256, 0, st>>>(h->mix_rec, Sn, h->mix_tiles, chunk_len, h->mix_part, n);
    } else {
      for (int round = 0; round * kQmMicroPerRound < h->mix_n_micro; ++round)
        qmix_wgrad2_kernel<<<chunks, 256, (size_t)(h->ql.R + 2) * kQmP * sizeof(float), st>>>(h->mix_rec, Sn, h->ql.R, h->mix_micro, h->mix_n_micro, round, chunk_len, h->mix_part, n);
    }
    qmix_reduce_kernel<<<(n + 255) / 256, 256, 0, st>>>(h->mix_part, chunks, n, h->mix_grad, qp.loss_part, qb);
    MARL_CUDA_TRY(cudaGetLastError());
    n_loss_parts += qb;
    td_ext = h->td;
    td_agent_stride = batch * T;
  }
  TrainParams tp; memset(&tp, 0, sizeof(tp));
  tp.plan = plan; tp.src = src; tp.theta = h->theta; tp.lay = h->ns.lay; tp.tq = h->tq; tp.td_ext = td_ext; tp.td_agent_stride = td_agent_stride;
  tp.gamma = h->hp.gamma; tp.double_q = h->hp.double_q; tp.scratch = h->scratch; tp.scratch_pitch = h->scratch_pitch; tp.loss_part = loss_part;
  const bool rec = h->timing && h->ev_used < kTimingPairs;
  if (rec) cudaEventRecord(h->ev[4 * h->ev_used], st);
  if (tc_backward_enabled() && h->ns.in < kTcObsDim) {
    if (!h->tc_h1) {  // intermediates of the tensor-core pipeline, allocated on first use
      const size_t rows = (size_t)h->ns.n_agents * h->max_batch * (h->max_T + 1);
      int rc = 0;
      rc |= dqn_alloc(&h->tc_h1, rows * kHidden); rc |= dqn_alloc(&h->tc_h2, rows * kHidden);
      rc |= dqn_alloc(&h->tc_dh1, rows * kHidden); rc |= dqn_alloc(&h->tc_rec, rows * 16 /* kRowRec */); rc |= dqn_alloc(&h->tc_x, rows * kTcObsDim);
      rc |= dqn_alloc(reinterpret_cast<float**>(&h->image_bwd), (size_t)h->ns.n_nets * tc_bwd_image_bytes() / 4 + 4);
      if (rc) return MARL_ENOMEM;
    }
    if (!h->image_current || !h->bwd_image_current) {
      if (int rc = launch_pack_weights(h->theta, h->ns.lay, h->ns.n_nets, h->image, st, h->image_bwd)) return rc;
      h->image_current = h->bwd_image_current = true;
    }
    TcBuffers tb; tb.image = h->image; tb.bwd_image = h->image_bwd; tb.h1 = h->tc_h1; tb.h2 = h->tc_h2; tb.dh1 = h->tc_dh1; tb.rec = h->tc_rec; tb.x = h->tc_x; tb.rows = (size_t)h->ns.n_agents * h->max_batch * (h->max_T + 1);
    if (int rc = launch_tc_dqn_train(tp, tb, st, rec ? &h->ev[4 * h->ev_used + 1] : nullptr)) return rc;
    if (rec) h->ev_split = true;
  } else {
    if (int rc = launch_train(tp, kHeadDqn, st)) return rc;
  }
  if (rec) { cudaEventRecord(h->ev[4 * h->ev_used + 3], st); h->ev_used += 1; }
  ReduceParams rp; rp.scratch = h->scratch; rp.loss_part = h->loss_part; rp.n_nets = h->ns.n_nets; rp.P = h->ns.lay.P; rp.scratch_pitch = h->scratch_pitch;
  memcpy(rp.cta_begin, plan.cta_begin, sizeof(rp.cta_begin));
  rp.n_loss_parts = n_loss_parts; rp.grad = h->grad; rp.stats = h->grad + h->n_params; rp.stats_accumulate = 0; rp.sumsq_part = h->sumsq;
  if (rp_out != nullptr) { *rp_out = rp; return MARL_OK; }
  return launch_grad_reduce(rp, st);
}

int marl_dqn_update_grads(marl_dqn* h, const marl_traj_view* traj, const int32_t* episode_idx, int32_t batch, void* stream) {
  return dqn_grads(h, traj, episode_idx, batch, stream, nullptr);
}

// Optimiser-step parameters of the next update (advances the update counters)
static void dqn_adam_params(marl_dqn* h, float* loss_out, AdamParams& ap) {
  h->updates += 1;
  memset(&ap, 0, sizeof(ap)); ap.theta = h->theta; ap.theta_tgt = h->theta_tgt; ap.m = h->m; ap.v = h->v; ap.grad = h->grad; ap.n = (int)h->n_params;
  ap.lr = h->hp.lr; ap.beta1 = h->hp.beta1; ap.beta2 = h->hp.beta2; ap.eps = h->hp.eps; ap.grad_clip = h->hp.grad_clip;
  ap.bc1 = (float)(1.0 - pow((double)h->hp.beta1, (double)h->updates));
  ap.bc2_sqrt = (float)sqrt(1.0 - pow((double)h->hp.beta2, (double)h->updates));
  // update_target (dqn/model.py:176-185)
  const float tu = h->hp.target_update_interval_or_tau;
  ap.target_mode = 0; ap.tau = tu; ap.tgt_begin = 0; ap.tgt_n = (int)h->n_params;
  if (tu > 1.0f && (float)(h->updates - h->last_target_update) >= tu) { ap.target_mode = 1; h->last_target_update = h->updates; }
  else if (tu < 1.0f) ap.target_mode = 2;
  if (ap.target_mode != 0) h->tgt_image_current = false;  // theta_tgt changes in this launch
  ap.loss_out = loss_out ? loss_out : h->loss_dev;
  ap.sumsq_part = h->grads_are_local ? h->sumsq : nullptr; ap.n_sumsq = (int)((h->n_params + 63) / 64);
  h->grads_are_local = false;
  if (h->image != nullptr && tc_forward_for(h->ns)) {  // valid images stay valid: adam_kernel rewrites the entries of every parameter it steps (a wide network has none)
    ap.image = h->image; ap.bwd_image = h->image_bwd; ap.img_lay = h->ns.lay; ap.img_nets = h->ns.n_nets;
    ap.image_bytes = tc_image_bytes(); ap.bwd_image_bytes = tc_bwd_image_bytes();
    if (h->image_bwd == nullptr) h->bwd_image_current = false;
  } else {
    h->image_current = h->bwd_image_current = false;
  }
}

// QMIX: the mixer's share of the single Adam step (same step count, learning rate and target update as the agents' networks; no clipping:
// clip_grad_norm_ covers self.critic.parameters() only, dqn/model.py:169-170)
static int qmix_adam(marl_dqn* h, const AdamParams& main, cudaStream_t st) {
  if (h->hp.mixer != 2) return MARL_OK;
  AdamParams ap = main;
  ap.theta = h->mix; ap.theta_tgt = h->mix_tgt; ap.m = h->mix_m; ap.v = h->mix_v; ap.grad = h->mix_grad; ap.n = h->ql.n; ap.tgt_begin = 0; ap.tgt_n = h->ql.n;
  ap.grad_clip = 0.f; ap.loss_out = nullptr; ap.sumsq_part = nullptr; ap.n_sumsq = 0; ap.image = nullptr; ap.bwd_image = nullptr; ap.img_nets = 0;
  return launch_adam(ap, st);
}

int marl_dqn_update_apply(marl_dqn* h, float* loss_out, void* stream) {
  MARL_REQUIRE(h != nullptr, "marl_dqn_update_apply: NULL handle");
  MARL_CUDA_TRY(cudaSetDevice(h->device));
  AdamParams ap;
  dqn_adam_params(h, loss_out, ap);
  if (int rc = launch_adam(ap, (cudaStream_t)stream)) return rc;
  return qmix_adam(h, ap, (cudaStream_t)stream);
}

// one update; `next` (optional): replay indices of the following update, drawn inside the fused tail kernel; *fused_out says whether it was
static int dqn_update(marl_dqn* h, const marl_traj_view* traj, const int32_t* episode_idx, int32_t batch, float* loss_out, void* stream, const SampleParams* next,
                      bool* fused_out) {
  if (fused_out) *fused_out = false;
  ReduceParams rp;
  if (int rc = dqn_grads(h, traj, episode_idx, batch, stream, &rp)) return rc;
  h->grads_are_local = true;  // nobody touches grad between the two halves: the clip can use the per-block sums of squares
  AdamParams ap;
  dqn_adam_params(h, loss_out, ap);
  // one kernel for reduce + clip + Adam when its grid fits the GPU in one wave, else the two kernels
  SampleParams sp; memset(&sp, 0, sizeof(sp));
  if (next != nullptr) sp = *next;
  // Several ranks: the exchange costs a round trip over NVLink (push, flags, poll: 7-10 us per update when exposed).  Split it -- push the local sums
  // first, then launch the NEXT update's target forward (it needs theta_tgt and the next indices, which the push kernel draws, not this update's Adam
  // step), then wait for the peers and finish: the wait hides under ~17 us of forward.  Not when this step rewrites theta_tgt.  Off by default: on two
  // GPUs the extra launch (prologue, second pass over the Adam state) cost more than the hidden wait saved (120.9 vs 116.8 us per update).
  if (h->xchg.world > 1 && tc_split_exchange_enabled()) {
    if (launch_reduce_push(rp, ap, &h->xchg, sp, h->grid_barrier, &h->push_epoch, h->n_sm, (cudaStream_t)stream) == MARL_OK) {
      if (next != nullptr && ap.target_mode == 0 && !h->standardise && h->hp.mixer == 0) {
        const int T = traj->T;
        const int min_units = (64 + T) / (T + 1) > 0 ? (64 + T) / (T + 1) : 1;
        const RowPlan plan = make_plan(h->ns, batch, T + 1, h->n_sm, min_units);
        RowSource src; memset(&src, 0, sizeof(src));
        src.mode = 1; src.traj = to_view(traj); src.idx = next->idx; src.N = h->ns.n_agents; src.D = h->ns.in;
        if (int rc = forward_any(h->ns, plan, src, h->theta_tgt, h->image_tgt, h->tq, (cudaStream_t)stream, h->tgt_image_current)) return rc;
        h->tgt_image_current = tc_forward_for(h->ns);
        h->tq_ahead = true;
      }
      if (int rc = launch_adam_finish(rp, ap, &h->xchg, h->grid_barrier, &h->grid_epoch, h->n_sm, (cudaStream_t)stream)) return rc;
      if (fused_out) *fused_out = true;
      return MARL_OK;
    }
  }
  if (launch_reduce_adam(rp, ap, &h->xchg, sp, h->grid_barrier, &h->grid_epoch, h->n_sm, (cudaStream_t)stream) == MARL_OK) {
    if (fused_out) *fused_out = true;
    return qmix_adam(h, ap, (cudaStream_t)stream);
  }
  MARL_REQUIRE(h->xchg.world <= 1, "marl_dqn_update: the peer-memory exchange needs the fused tail kernel (parameter count too large for one wave)");
  if (int rc = launch_grad_reduce(rp, (cudaStream_t)stream)) return rc;
  if (int rc = launch_adam(ap, (cudaStream_t)stream)) return rc;
  return qmix_adam(h, ap, (cudaStream_t)stream);
}

int marl_dqn_update(marl_dqn* h, const marl_traj_view* traj, const int32_t* episode_idx, int32_t batch, float* loss_out, void* stream) {
  return dqn_update(h, traj, episode_idx, batch, loss_out, stream, nullptr, nullptr);
}

/* n_updates back-to-back updates with on-device replay sampling: the `rb.sample(); model.update()` pair of
 * marlbase/dqn/train.py:308-311 repeated, without returning to Python in between. */
int marl_dqn_update_n(marl_dqn* h, const marl_traj_view* traj, int32_t batch, int32_t n_valid, uint64_t seed, uint64_t first_update_idx,
                      int32_t n_updates, float* loss_out, void* stream) {
  MARL_REQUIRE(h && traj && n_updates >= 0, "marl_dqn_update_n: bad argument");
  MARL_REQUIRE(n_valid >= 1 && n_valid <= traj->capacity, "marl_dqn_update_n: n_valid %d out of range", n_valid);
  bool have_idx = false;   // the previous update's tail kernel already drew this update's indices
  for (int u = 0; u < n_updates; ++u) {
    if (!have_idx)
      if (int rc = marl_replay_sample(seed, first_update_idx + (uint64_t)u, batch, n_valid, h->idx, stream)) return rc;
    SampleParams next; next.seed = seed; next.update_idx = first_update_idx + (uint64_t)u + 1; next.batch = batch; next.n_valid = n_valid; next.idx = h->idx;
    bool fused = false;
    if (int rc = dqn_update(h, traj, h->idx, batch, loss_out, stream, u + 1 < n_updates ? &next : nullptr, &fused)) return rc;
    have_idx = fused && u + 1 < n_updates;
  }
  return MARL_OK;
}

/* CUDA-event timing of dqn_train_kernel launches: enable=1 starts recording (first 1024 launches), enable=0 stops, synchronises
 * the recorded events and returns their summed duration and count. */
int marl_dqn_timing(marl_dqn* h, int32_t enable, float* total_ms, int32_t* count) {
  MARL_REQUIRE(h != nullptr, "marl_dqn_timing: NULL handle");
  MARL_CUDA_TRY(cudaSetDevice(h->device));
  if (enable) {
    if (h->ev.empty()) { h->ev.resize(4 * kTimingPairs); for (auto& e : h->ev) MARL_CUDA_TRY(cudaEventCreate(&e)); }
    h->ev_used = 0; h->timing = true; h->ev_split = false;
    return MARL_OK;
  }
  h->timing = false;
  float tot = 0.f;
  for (int i = 0; i < h->ev_used; ++i) {
    MARL_CUDA_TRY(cudaEventSynchronize(h->ev[4 * i + 3]));
    float ms = 0.f; MARL_CUDA_TRY(cudaEventElapsedTime(&ms, h->ev[4 * i], h->ev[4 * i + 3]));
    tot += ms;
  }
  if (total_ms) *total_ms = tot;
  if (count) *count = h->ev_used;
  return MARL_OK;
}

/* Tell the library that the caller wrote to the parameter buffers returned by marl_dqn_param_ptrs (cached derived data --
 * the packed tensor-core images of the online and target networks -- is rebuilt on next use). */
int marl_dqn_params_changed(marl_dqn* h) {
  MARL_REQUIRE(h != nullptr, "marl_dqn_params_changed: NULL handle");
  h->tgt_image_current = false; h->image_current = false; h->bwd_image_current = false;
  return MARL_OK;
}

/* Per-kernel split of the launches timed by the last marl_dqn_timing(1) .. marl_dqn_timing(0) window: summed CUDA-event durations of
 * the three kernels of the tensor-core training pass (online forward + TD head, dH1, weight gradients).  *count = 0 when the window
 * ran the single fused FP32 kernel instead. */
int marl_dqn_timing_kernels(marl_dqn* h, float* ms3, int32_t* count) {
  MARL_REQUIRE(h != nullptr && ms3 != nullptr, "marl_dqn_timing_kernels: NULL argument");
  MARL_REQUIRE(!h->timing, "marl_dqn_timing_kernels: call marl_dqn_timing(q, 0, ...) first");
  MARL_CUDA_TRY(cudaSetDevice(h->device));
  ms3[0] = ms3[1] = ms3[2] = 0.f;
  if (count) *count = h->ev_split ? h->ev_used : 0;
  if (!h->ev_split) return MARL_OK;
  for (int i = 0; i < h->ev_used; ++i) {
    MARL_CUDA_TRY(cudaEventSynchronize(h->ev[4 * i + 3]));
    for (int k = 0; k < 3; ++k) {
      float ms = 0.f; MARL_CUDA_TRY(cudaEventElapsedTime(&ms, h->ev[4 * i + k], h->ev[4 * i + k + 1]));
      ms3[k] += ms;
    }
  }
  return MARL_OK;
}

/* ---- gradient exchange over NVLink peer memory (one process per GPU) ---------------------------------------------------------------
 * marl_dqn_peer_handle: allocates this rank's exchange buffer (2 slots of [n_params + 4] floats + a flag) and writes its 64-byte
 * cudaIpcMemHandle_t to handle_out; the caller gathers the handles of all ranks (any transport) and passes them, rank-ordered, to
 * marl_dqn_peer_attach.  From then on marl_dqn_update / marl_dqn_update_n perform the all-rank gradient sum inside the fused
 * reduce + Adam kernel (every rank must make the same sequence of update calls); the two-call form with an external all-reduce
 * between marl_dqn_update_grads and marl_dqn_update_apply keeps working. */
static size_t xbuf_data_bytes(const marl_dqn* h) { return (size_t)2 * kMaxRanks * h->xchg.slot_floats * sizeof(float); }

int marl_dqn_peer_handle(marl_dqn* h, void* handle_out) {
  MARL_REQUIRE(h != nullptr && handle_out != nullptr, "marl_dqn_peer_handle: NULL argument");
  MARL_CUDA_TRY(cudaSetDevice(h->device));
  if (h->xbuf == nullptr) {   // sized for the largest world: [2 parities][kMaxRanks sources][slot] floats + kMaxRanks flags
    h->xchg.slot_floats = (int)((h->n_params + 4 + 63) / 64 * 64);
    MARL_CUDA_TRY(cudaMalloc(&h->xbuf, xbuf_data_bytes(h) + 256));
    MARL_CUDA_TRY(cudaMemset(h->xbuf, 0, xbuf_data_bytes(h) + 256));
  }
  cudaIpcMemHandle_t mh;
  MARL_CUDA_TRY(cudaIpcGetMemHandle(&mh, h->xbuf));
  memcpy(handle_out, &mh, sizeof(mh));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size is part of the ABI");
  return MARL_OK;
}

int marl_dqn_peer_attach(marl_dqn* h, int32_t rank, int32_t world, const void* handles) {
  MARL_REQUIRE(h != nullptr && handles != nullptr, "marl_dqn_peer_attach: NULL argument");
  MARL_REQUIRE(world >= 2 && world <= kMaxRanks && rank >= 0 && rank < world, "marl_dqn_peer_attach: rank %d / world %d out of range (2..%d ranks)", rank, world, kMaxRanks);
  MARL_REQUIRE(h->xbuf != nullptr && h->xchg.world <= 1, "marl_dqn_peer_attach: call marl_dqn_peer_handle first, attach once");
  MARL_REQUIRE(h->hp.mixer != 2, "marl_dqn_peer_attach: the mixer's gradient is not part of the peer exchange: QMIX runs on one GPU");
  MARL_CUDA_TRY(cudaSetDevice(h->device));
  {  // the exchange lives inside the fused reduce + Adam kernel: refuse here, before any update mutates counters, when that kernel cannot
     // cover this parameter count with one co-resident wave (a later fallback to the two-kernel tail would dead-lock the peers' polls)
    int pb = 0, ns = 0;
    MARL_REQUIRE(reduce_adam_shape((int)h->n_params, h->n_sm, true, &pb, &ns) == MARL_OK,
                 "marl_dqn_peer_attach: %lld parameters do not fit the fused reduce + Adam kernel on %d SMs; use the all-reduce between marl_dqn_update_grads and _apply",
                 (long long)h->n_params, h->n_sm);
  }
  for (int r = 0; r < world; ++r) {
    void* base = h->xbuf;
    if (r != rank) {
      cudaIpcMemHandle_t mh;
      memcpy(&mh, static_cast<const char*>(handles) + 64 * (size_t)r, sizeof(mh));
      MARL_CUDA_TRY(cudaIpcOpenMemHandle(&base, mh, cudaIpcMemLazyEnablePeerAccess));
    }
    h->peer_base[r] = base;
    h->xchg.peers[r] = static_cast<float*>(base);
    h->xchg.peer_flags[r] = reinterpret_cast<unsigned long long*>(static_cast<char*>(base) + xbuf_data_bytes(h));
  }
  h->xchg.own_flags = h->xchg.peer_flags[rank];
  h->xchg.timed_out = reinterpret_cast<int*>(static_cast<char*>(h->peer_base[rank]) + xbuf_data_bytes(h) + 128);   // behind the 8 flags, zeroed with the buffer
  h->xchg.rank = rank; h->xchg.world = world; h->xchg.epoch = 0;
  return MARL_OK;
}

/* 0 = healthy.  1 = some update's exchange gave up waiting for a peer's flag (a rank died, skipped an update or fell out of step): every
 * result since is invalid.  Synchronises the device. */
int marl_dqn_peer_status(marl_dqn* h, int32_t* timed_out) {
  MARL_REQUIRE(h != nullptr && timed_out != nullptr, "marl_dqn_peer_status: NULL argument");
  *timed_out = 0;
  if (h->xchg.world <= 1) return MARL_OK;
  MARL_CUDA_TRY(cudaSetDevice(h->device));
  int v = 0;
  MARL_CUDA_TRY(cudaMemcpy(&v, h->xchg.timed_out, sizeof(int), cudaMemcpyDeviceToHost));
  *timed_out = v;
  return MARL_OK;
}

int marl_dqn_counters(marl_dqn* h, int64_t* updates, int64_t* last_target_update) {
  MARL_REQUIRE(h != nullptr, "marl_dqn_counters: NULL handle");
  if (updates) *updates = h->updates;
  if (last_target_update) *last_target_update = h->last_target_update;
  return MARL_OK;
}

int marl_dqn_set_counters(marl_dqn* h, int64_t updates, int64_t last_target_update) {
  MARL_REQUIRE(h != nullptr, "marl_dqn_set_counters: NULL handle");
  h->updates = updates; h->last_target_update = last_target_update;
  return MARL_OK;
}

}  // extern "C"
