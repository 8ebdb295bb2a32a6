// learner.cuh -- kernels shared by the DQN-family and actor-critic learners: gathered MLP forward, fused
// forward+loss-head+backward training pass, deterministic gradient reduction, clip + Adam + target update.
#pragma once
#include "mlp.cuh"
#include <string.h>

namespace marl {

constexpr int kMaxObsDim = 128;  // FP32 FFMA kernels: KP = 16 or 32 float input tiles, KP = kKpWide (K-chunked layer 1) above 32
constexpr int kTcObsDim = 32;    // tensor-core kernels: the staged input width (one 32-feature W1 panel, the `xg` row pitch); wider networks use FFMA

struct TrajView {  // device view of marl_traj_view
  const float* obs; const int32_t* act; const float* rew; const uint8_t* done; const uint8_t* filled;
  int capacity, N, T, D;
};

// Which rows a launch covers and how CTAs split them.  A "unit" is an indivisible run of rows that must stay inside
// one CTA: one sampled episode (T+1 rows) for training passes, one row for plain inference.
struct RowPlan {
  int n_nets;
  int cta_begin[MARL_MAX_AGENTS + 1];   // CTAs [cta_begin[k], cta_begin[k+1]) work on net k
  int slot_begin[MARL_MAX_AGENTS + 1];  // agents of net k = slot_agent[slot_begin[k] .. slot_begin[k+1])
  int slot_agent[MARL_MAX_AGENTS];
  int unit_rows;                        // rows per unit
  int units_per_agent;                  // B (episodes) or E (envs)
};

struct RowSource {
  // 0: dense obs float[E][N][D];  1: gather from the trajectory store through episode indices;
  // 2 / 3: JOINT observation rows float[units][unit_rows][D] shared by all agents (centralised critic, ac/model.py:62-65,156-157: every agent's critic
  //        sees the concatenation of all agents' observations; D = their total width): 2 = outputs laid out like mode 1 ([agent][unit][row], loss
  //        scalars from the trajectory store), 3 = like mode 0 ([unit][agent]; `joint` is then simply the dense obs array read as [E][N * D_agent])
  int mode;
  const float* dense; int E, N, D;
  TrajView traj; const int32_t* idx;  // idx[B] ring slots (device)
  const float* joint;
};
__host__ __device__ __forceinline__ bool src_dense_out(int mode) { return mode == 0 || mode == 3; }

__device__ __forceinline__ void cta_rows(const RowPlan& p, int& net, int& row_begin, int& row_end) {
  net = 0;
  while (net + 1 < p.n_nets && (int)blockIdx.x >= p.cta_begin[net + 1]) ++net;
  const int ncta = p.cta_begin[net + 1] - p.cta_begin[net], c = (int)blockIdx.x - p.cta_begin[net];
  const long long units = (long long)(p.slot_begin[net + 1] - p.slot_begin[net]) * p.units_per_agent;
  row_begin = (int)(units * c / ncta) * p.unit_rows;
  row_end = (int)(units * (c + 1) / ncta) * p.unit_rows;
}

// virtual row of net -> (agent, unit index within agent, offset within unit)
__device__ __forceinline__ void decode_row(const RowPlan& p, int net, int vr, int& agent, int& unit, int& off) {
  const int rpa = p.units_per_agent * p.unit_rows;
  const int slot = vr / rpa, rem = vr - slot * rpa;
  agent = p.slot_agent[p.slot_begin[net] + slot];
  unit = rem / p.unit_rows;
  off = rem - unit * p.unit_rows;
}

__device__ __forceinline__ const float* row_ptr(const RowSource& s, int agent, int unit, int off) {
  if (s.mode == 0) return s.dense + ((size_t)unit * s.N + agent) * s.D;
  if (s.mode >= 2) return s.joint + ((size_t)unit * (s.mode == 2 ? s.traj.T + 1 : 1) + off) * s.D;   // (unit_rows: T + 1 when training, 1 for plain inference)
  const size_t ep = (size_t)s.idx[unit];
  return s.traj.obs + ((ep * s.traj.N + agent) * (size_t)(s.traj.T + 1) + off) * s.traj.D;
}

// Per-tile row metadata staged in shared memory by the first 128 threads (one row each): the source pointer of the
// row's observation and, for training passes, the scalars the loss head needs.  Two dependent global latencies per tile
// (episode index, then its fields) instead of a dependent chain per element / per head.
struct RowMeta {
  const float* src[kTileRows];
  int act[kTileRows];
  float rew[kTileRows];
  int flags[kTileRows];  // bit 0: filled[t], bit 1: done[t+1]
  static constexpr int kBytes = kTileRows * (8 + 4 + 4 + 4);
};

template <bool kWithScalars>
__device__ __forceinline__ void setup_rows(RowMeta* m, const RowPlan& p, const RowSource& s, int net, int vr0, int nrows) {
  const int r = threadIdx.x;
  if (r >= kTileRows) return;
  const float* src = nullptr; int act = 0, flags = 0; float rew = 0.f;
  if (r < nrows) {
    int agent, unit, off;
    decode_row(p, net, vr0 + r, agent, unit, off);
    if (s.mode == 0) {
      src = s.dense + ((size_t)unit * s.N + agent) * s.D;
    } else if (s.mode == 3) {
      src = s.joint + ((size_t)unit * p.unit_rows + off) * s.D;
    } else {
      const size_t ep = (size_t)s.idx[unit];
      const TrajView& tv = s.traj;
      src = s.mode == 2 ? s.joint + ((size_t)unit * p.unit_rows + off) * s.D : tv.obs + ((ep * tv.N + agent) * (size_t)(tv.T + 1) + off) * tv.D;
      if (kWithScalars && off < tv.T) {
        act = tv.act[(ep * tv.N + agent) * tv.T + off];
        rew = tv.rew[(ep * tv.N + agent) * tv.T + off];
        flags = (int)tv.filled[ep * tv.T + off] | ((int)tv.done[ep * (tv.T + 1) + off + 1] << 1);
      }
    }
  }
  m->src[r] = src; m->act[r] = act; m->rew[r] = rew; m->flags[r] = flags;
}

// Fill the [128][KP] input tile from the staged row pointers (asynchronous copies; zero padding in both directions).
// KP = kKpWide: only the ceil(D / kW1Chunk) * kW1Chunk leading columns the K-chunks read, one row per warp and pass.
// Caller: cp_async_wait_all() + __syncthreads() before the tile is read.
template <int KP>
__device__ __forceinline__ void gather_tile_async(float* X, const RowMeta* m, int D) {
  if constexpr (KP == kKpWide) {
    const int cols = (D + kW1Chunk - 1) / kW1Chunk * kW1Chunk, lane = threadIdx.x & 31;
#pragma unroll 2
    for (int r = threadIdx.x >> 5; r < kTileRows; r += kMlpThreads / 32) {
      const float* src = m->src[r];
      for (int k = lane; k < cols; k += 32) {
        if (src != nullptr && k < D) cp_async4(&at1<KP>(X, r, k), src + k);
        else at1<KP>(X, r, k) = 0.f;
      }
    }
  } else {
#pragma unroll 4
    for (int i = threadIdx.x; i < kTileRows * KP; i += kMlpThreads) {
      const int r = i / KP, k = i - r * KP;
      const float* src = m->src[r];
      if (src != nullptr && k < D) cp_async4(&at1<KP>(X, r, k), src + k);
      else at1<KP>(X, r, k) = 0.f;
    }
  }
}

struct FwdParams {
  RowPlan plan; RowSource src;
  const float* theta;   // [n_nets][P]
  NetLayout lay;
  float* out;           // mode 0: [E][N][out]; mode 1: [N][B][T+1][out]
};

// Loss heads of the fused training kernel (what happens between the forward and the backward of a tile).
enum TrainHead { kHeadDqn = 0, kHeadA2cCritic = 1, kHeadA2cActor = 2 };

struct TrainParams {
  RowPlan plan; RowSource src;
  const float* theta; NetLayout lay;
  float* scratch;         // [gridDim][pitch] per-CTA gradient sums (un-normalised); pitch = P rounded up to 4 floats
  int scratch_pitch;
  float* loss_part;       // [gridDim][4] per-CTA loss statistics, meaning depends on the head (see below)
  // kHeadDqn: parts = (sum delta^2*filled, sum filled on agent 0, 0, 0)
  const float* tq;        // target-net Q-values of every gathered row, [N][B][T+1][out] (from the forward kernel)
  const float* td_ext;    // precomputed 2*delta*filled (VDN: per (b, t), [B][T]; standardise_returns: per (agent, b, t) with td_agent_stride = B*T); NULL: the head computes it
  int td_agent_stride;
  float gamma; int double_q;
  // kHeadA2cCritic: parts = (0, sum filled on agent 0, 0, sum adv^2*filled); writes adv = returns - V
  const float* returns;   // [N][B][T] n-step returns
  float* adv_out;         // [N][B][T]
  float value_coef;
  // kHeadA2cActor: parts = (sum -logp*adv*filled, 0, sum entropy*filled, 0)
  const float* adv;       // [N][B][T]
  float entropy_coef;
  // PPO (ac/model.py:305-321): old_logp != NULL switches the actor head to the clipped surrogate -min(ratio adv, clip(ratio, 1 -+ ppo_clip) adv),
  // ratio = exp(logp - old_logp); parts[0] = sum of that term * filled
  const float* old_logp;  // [N][B][T] log-probabilities of the taken actions under the policy the batch was collected with
  float ppo_clip;
};

struct ReduceParams {
  const float* scratch; const float* loss_part; int n_nets; int cta_begin[MARL_MAX_AGENTS + 1]; int P; int scratch_pitch;
  int n_loss_parts;
  float* grad;       // [n_nets*P] gradient sums of this network set
  float* stats;      // [4] sums of the loss parts (NULL: skip)
  int stats_accumulate;  // add to stats instead of overwriting (second pass of an actor-critic update)
  float* sumsq_part;     // [ceil(n_nets*P / 64)] per-block sum of squares of the reduced gradients (NULL: skip)
};

struct AdamParams {
  float* theta; float* theta_tgt; float* m; float* v;
  const float* grad;   // [n] gradient sums followed by 4 statistics: (loss numerator, filled count, aux0, aux1)
  int n;               // trainable floats
  int tgt_begin, tgt_n;  // theta[tgt_begin .. tgt_begin+tgt_n) is mirrored by theta_tgt[0 .. tgt_n)
  float lr, beta1, beta2, eps, bc1, bc2_sqrt, grad_clip;  // grad_clip <= 0: off
  int target_mode;  // 0 none, 1 hard copy, 2 polyak
  float tau;
  float* loss_out;  // [6]: stats[0]/filled, grad norm, stats[2]/filled, stats[3]/filled, filled, 0
  const float* sumsq_part; int n_sumsq;  // optional per-block sums of squares of grad[0..n) (local gradients only: single GPU)
  // optional packed tensor-core images of theta[0 .. img_nets * img_lay.P), kept current parameter by parameter (NULL: none)
  uint8_t* image; uint8_t* bwd_image; NetLayout img_lay; int img_nets; size_t image_bytes, bwd_image_bytes;
};

// host-side launchers (defined next to the kernels in learner_kernels.cu); return MARL_* codes
int learner_kernels_init(int in_dim);                       // opt in to > 48 KB dynamic shared memory
int launch_mlp_forward(const FwdParams& p, cudaStream_t st);
int launch_train(const TrainParams& p, int head, cudaStream_t st);
int launch_grad_reduce(const ReduceParams& p, cudaStream_t st);
// Gradient exchange over NVLink peer memory (reduce_adam_kernel<true>): every rank owns an exchange buffer
// [2 parities][world source ranks][slot_floats] floats + [world] 64-bit flags, opened by the other ranks through CUDA IPC.
constexpr int kMaxRanks = 8;
struct XchgParams {
  int world, rank, slot_floats;
  unsigned long long epoch;                        // number of exchanges so far, this one included
  float* peers[kMaxRanks];                         // every rank's buffer (own included)
  unsigned long long* peer_flags[kMaxRanks];       // every rank's flag array (own included): flag[source rank]
  const unsigned long long* own_flags;             // = peer_flags[rank]
  int* timed_out;                                  // device flag (sticky): a peer's epoch flag did not arrive within the spin bound
};
// replay indices for the next update, drawn by the fused tail kernel (idx == NULL: none); same stream as replay_sample_kernel
struct SampleParams { uint64_t seed, update_idx; int batch, n_valid; int32_t* idx; };
int launch_reduce_adam(const ReduceParams& rp, const AdamParams& ap, XchgParams* xp, const SampleParams& sp, unsigned long long* barrier, unsigned long long* epoch,
                       int n_sm, cudaStream_t st);
int launch_reduce_push(const ReduceParams& rp, const AdamParams& ap, XchgParams* xp, const SampleParams& sp, unsigned long long* barrier, unsigned long long* push_epoch,
                       int n_sm, cudaStream_t st);
int launch_adam_finish(const ReduceParams& rp, const AdamParams& ap, XchgParams* xp, unsigned long long* barrier, unsigned long long* epoch, int n_sm, cudaStream_t st);
int launch_adam(const AdamParams& p, cudaStream_t st);
// can the fused tail cover n parameters with one co-resident wave on n_sm SMs?  (pb, ns: the block shape it would use)
int reduce_adam_shape(int n, int n_sm, bool xchg, int* pb, int* ns);

template <int KP>
constexpr size_t forward_smem_bytes() { return sizeof(float) * (WeightSmem<KP>::kFloats + 2 * kTileRows * kPitchH + kTileRows * kOutPad + 48) + RowMeta::kBytes; }
template <int KP>
constexpr size_t train_smem_bytes() { return forward_smem_bytes<KP>(); }

// ---- host-side planning -----------------------------------------------------------------------------------------
struct NetSet {
  int n_agents = 0, n_nets = 0, in = 0, out = 0;
  int agent_net[MARL_MAX_AGENTS];
  NetLayout lay;
};

// Split `n_cta_max` CTAs over the networks in proportion to their row counts; every CTA gets >= min_units units.
inline RowPlan make_plan(const NetSet& ns, int units_per_agent, int unit_rows, int n_cta_max, int min_units) {
  RowPlan p; memset(&p, 0, sizeof(p));
  p.n_nets = ns.n_nets; p.unit_rows = unit_rows; p.units_per_agent = units_per_agent;
  int s = 0;
  for (int k = 0; k < ns.n_nets; ++k) {
    p.slot_begin[k] = s;
    for (int a = 0; a < ns.n_agents; ++a) if (ns.agent_net[a] == k) p.slot_agent[s++] = a;
  }
  p.slot_begin[ns.n_nets] = s;
  long long total = (long long)ns.n_agents * units_per_agent;
  int c = 0;
  for (int k = 0; k < ns.n_nets; ++k) {
    const long long units = (long long)(p.slot_begin[k + 1] - p.slot_begin[k]) * units_per_agent;
    long long want = (long long)n_cta_max * units / (total > 0 ? total : 1);
    const long long cap = (units + min_units - 1) / min_units;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    p.cta_begin[k] = c;
    c += (int)want;
  }
  p.cta_begin[ns.n_nets] = c;
  return p;
}

inline TrajView to_view(const marl_traj_view* t) {
  TrajView v; v.obs = t->obs; v.act = t->act; v.rew = t->rew; v.done = t->done; v.filled = t->filled;
  v.capacity = t->capacity; v.N = t->n_agents; v.T = t->T; v.D = t->obs_dim;
  return v;
}


inline int dev_alloc_zero(float** p, size_t n_floats) {
  cudaError_t e = cudaMalloc((void**)p, n_floats * sizeof(float));
  if (e == cudaSuccess) e = cudaMemset(*p, 0, n_floats * sizeof(float));
  if (e != cudaSuccess) { set_error("cudaMalloc(%zu floats) failed: %s", n_floats, cudaGetErrorString(e)); return MARL_ENOMEM; }
  return MARL_OK;
}

inline int launch_forward(const NetSet& ns, const RowPlan& plan, const RowSource& src, const float* theta, float* out, cudaStream_t st) {
  FwdParams fp; fp.plan = plan; fp.src = src; fp.theta = theta; fp.lay = ns.lay; fp.out = out;
  return launch_mlp_forward(fp, st);
}

// ---- tensor-core forward path (tc_forward.cu) -----------------------------------------------------------------------------
size_t tc_image_bytes();
int tc_forward_init();
size_t tc_bwd_image_bytes();
int launch_pack_weights(const float* theta, const NetLayout& lay, int n_nets, uint8_t* image, cudaStream_t st, uint8_t* bwd_image = nullptr);
int launch_tc_forward(const FwdParams& p, const uint8_t* images, cudaStream_t st);
// ---- tensor-core training pipeline (tc_train.cu) ----------------------------------------------------------------------------
struct TcBuffers {
  uint8_t* image; uint8_t* bwd_image;       // packed online-network images (forward K-major, backward K-major W2^T)
  float *h1, *h2, *dh1;                     // [32][rows][4] (chunk-major) activations and hidden-layer gradient
  float* rec;                               // [rows][16] row records (tc_train.cu)
  float* x;                                 // [rows][kTcObsDim] gathered observation rows
  size_t rows;                              // allocated rows
};
int tc_train_init();
int launch_tc_dqn_train(const TrainParams& tp, const TcBuffers& buf, cudaStream_t st, cudaEvent_t* between = nullptr);  // between[2]: recorded after kernels 1 and 2
// tc_forward_enabled(): process-wide switch (marl_set_option("tensor_core_forward", 0|1)), declared in common.cuh
// Does a forward of this network set run on the tensor cores?  Only up to kTcObsDim inputs: a wider network (a MAPPO learner's centralised
// critic next to its narrow actor, say) always takes the FFMA kernels, and no packed image is ever built or kept for it.
inline bool tc_forward_for(const NetSet& ns) { return tc_forward_enabled() && ns.in <= kTcObsDim; }

// Forward pass through whichever implementation is selected.  `image` is scratch for the packed weights (n_nets images);
// it is rebuilt from `theta` on every call (3 us) so that it can never go stale against direct parameter writes.
inline int forward_any(const NetSet& ns, const RowPlan& plan, const RowSource& src, const float* theta, uint8_t* image, float* out, cudaStream_t st,
                       bool image_is_current = false) {
  if (tc_forward_for(ns) && image != nullptr) {
    if (!image_is_current)
      if (int rc = launch_pack_weights(theta, ns.lay, ns.n_nets, image, st)) return rc;
    FwdParams fp; fp.plan = plan; fp.src = src; fp.theta = theta; fp.lay = ns.lay; fp.out = out;
    return launch_tc_forward(fp, image, st);
  }
  return launch_forward(ns, plan, src, theta, out, st);
}

inline int check_mlp_cfg(const marl_mlp_cfg* cfg, const char* who) {
  MARL_REQUIRE(cfg != nullptr, "%s: NULL network config", who);
  MARL_REQUIRE(cfg->n_agents >= 1 && cfg->n_agents <= MARL_MAX_AGENTS, "%s: n_agents out of range", who);
  MARL_REQUIRE(cfg->n_nets >= 1 && cfg->n_nets <= cfg->n_agents, "%s: n_nets out of range", who);
  MARL_REQUIRE(cfg->hidden == kHidden, "%s: only layers=[128,128] is implemented on the B200 path (got hidden=%d)", who, cfg->hidden);
  MARL_REQUIRE(cfg->in_dim >= 1 && cfg->in_dim <= kMaxObsDim, "%s: obs dim %d not supported (1..%d)", who, cfg->in_dim, kMaxObsDim);
  MARL_REQUIRE(cfg->out_dim >= 1 && cfg->out_dim <= kOutPad, "%s: output width %d not supported (1..%d)", who, cfg->out_dim, kOutPad);
  for (int a = 0; a < cfg->n_agents; ++a) MARL_REQUIRE(cfg->agent_net[a] >= 0 && cfg->agent_net[a] < cfg->n_nets, "%s: agent_net[%d] out of range", who, a);
  return MARL_OK;
}

inline NetSet to_netset(const marl_mlp_cfg* cfg) {
  NetSet ns; ns.n_agents = cfg->n_agents; ns.n_nets = cfg->n_nets; ns.in = cfg->in_dim; ns.out = cfg->out_dim;
  memcpy(ns.agent_net, cfg->agent_net, sizeof(int) * MARL_MAX_AGENTS);
  ns.lay = NetLayout::make(cfg->in_dim, cfg->out_dim);
  return ns;
}

}  // namespace marl
