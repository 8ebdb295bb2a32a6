// learner_kernels.cu -- the fused learner kernels (sm_100a).
//
//  mlp_forward_kernel   per-agent MLP inference on gathered rows: model.act's critic/actor forward
//                       (marlbase/dqn/model.py:99, marlbase/ac/model.py:148-149) and the target-network pass of the
//                       learner (marlbase/dqn/model.py:132-134, marlbase/ac/model.py:190-193).  Replay gather
//                       (marlbase/dqn/train.py:94-124) is fused into the tile load.
//  train_kernel         (head DQN) QNetwork._compute_loss + loss.backward() (marlbase/dqn/model.py:118-168): gather, online
//                       forward, double-Q TD target, MSE, masked mean numerator, full backward; every CTA keeps its
//                       network's weights resident in shared memory and walks its episodes tile by tile.
//  grad_reduce_kernel   deterministic sum of the per-CTA gradient partials (+ loss / filled sums).
//  adam_kernel          clip_grad_norm_ + Adam.step + update_target (marlbase/dqn/model.py:169-196).
//
// Persistent CTAs, one per SM (148 on B200) split across networks; FP32 FFMA register-tiled GEMMs (see mlp.cuh).
#include "tc_common.cuh"

namespace marl {

// ------------------------------------------------------------------------------------------------------------
template <int KP>
__global__ void __launch_bounds__(kMlpThreads, 1) mlp_forward_kernel(FwdParams p) {
  extern __shared__ __align__(16) float smem[];
  WeightSmem<KP> w(smem);
  float* H1 = smem + WeightSmem<KP>::kFloats;
  float* H2 = H1 + kTileRows * kPitchH;
  float* X = H2;  // the input tile lives in the H2 region until layer 2 overwrites it
  float* Q = H2 + kTileRows * kPitchH;
  RowMeta* meta = reinterpret_cast<RowMeta*>(Q + kTileRows * kOutPad + 48);
  const ThreadCoord tc;
  int net, row_begin, row_end;
  cta_rows(p.plan, net, row_begin, row_end);
  if (row_begin >= row_end) return;
  const float* theta = p.theta + (size_t)net * p.lay.P;
  w.load_async(theta, p.lay);
  for (int vr0 = row_begin; vr0 < row_end; vr0 += kTileRows) {
    const int nrows = min(kTileRows, row_end - vr0);
    __syncthreads();
    setup_rows<false>(meta, p.plan, p.src, net, vr0, nrows);
    __syncthreads();
    gather_tile_async<KP>(X, meta, p.src.D);
    if constexpr (KP == kKpWide) w.load_w1_chunk_async(theta, p.lay, 0);
    cp_async_wait_all();
    __syncthreads();
    if constexpr (KP == kKpWide) mlp_forward_tile_wide(X, H1, H2, Q, w, theta, p.lay, tc);
    else mlp_forward_tile<KP>(X, H1, H2, Q, w, tc);
    __syncthreads();
    for (int i = threadIdx.x; i < nrows * p.lay.out; i += kMlpThreads) {
      const int r = i / p.lay.out, o = i - r * p.lay.out;
      int agent, unit, off;
      decode_row(p.plan, net, vr0 + r, agent, unit, off);
      const size_t dst = src_dense_out(p.src.mode) ? ((size_t)unit * p.src.N + agent)
                                         : (((size_t)agent * p.plan.units_per_agent + unit) * p.plan.unit_rows + off);
      p.out[dst * p.lay.out + o] = Q[r * kOutPad + o];
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// per-CTA gradient partial: first tile stores, later tiles accumulate (plain loads/stores: the region is private)
// (the accumulation is a RED: no value returns to the SM, so nothing waits on the L2 round trip; one thread per address
// and tiles in program order keep the sum order fixed)
__device__ __forceinline__ void rmw(float* dst, float v, bool first) {
  if (first) *dst = v; else atomicAdd(dst, v);
}
__device__ __forceinline__ void rmw4(float* dst, float4 v, bool first) {
  if (first) *reinterpret_cast<float4*>(dst) = v; else atomicAdd(reinterpret_cast<float4*>(dst), v);
}

// Backward of one tile.  On entry: X, H1, H2 hold the forward activations, DQ[128][8] holds dLoss/dq (zero rows
// beyond the valid ones).  gs = this CTA's gradient partial [P].  Uses DQ as scratch after it is consumed.
template <int KP>
__device__ __forceinline__ void mlp_backward_tile(float* X, float* H1, float* H2, float* DQ, const WeightSmem<KP>& w, const NetLayout& lay,
                                                  float* gs, bool first, const ThreadCoord& tc, const RowMeta* meta, int obs_dim, float* part) {
  const int t = threadIdx.x;
  // ---- dW3[o][j] = sum_r dq[r][o] * h2[r][j];  db3[o] = sum_r dq[r][o] --------------------------------------
  {
    const int j = t & (kHidden - 1), o0 = (t >> 7) * 4;
    float g[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};  // two interleaved chains per output: half the FMA latency chain
#pragma unroll 4
    for (int r = 0; r < kTileRows; r += 2) {
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const float h = at1<kHidden>(H2, r + u, j);
        const float4 d = *reinterpret_cast<const float4*>(DQ + (r + u) * kOutPad + o0);
        g[u][0] = fmaf(d.x, h, g[u][0]); g[u][1] = fmaf(d.y, h, g[u][1]); g[u][2] = fmaf(d.z, h, g[u][2]); g[u][3] = fmaf(d.w, h, g[u][3]);
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (o0 + q < lay.out) rmw(gs + lay.w3 + (o0 + q) * kHidden + j, g[0][q] + g[1][q], first);
    // db3: one row per lane of the first four warps, shuffle-reduced, four partials combined after the barrier
    if (t < kTileRows) {
      const float4 d0 = *reinterpret_cast<const float4*>(DQ + t * kOutPad), d1 = *reinterpret_cast<const float4*>(DQ + t * kOutPad + 4);
      float v[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
      for (int o = 0; o < 8; ++o) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v[o] += __shfl_xor_sync(0xFFFFFFFFu, v[o], off);
      }
      if ((t & 31) == 0) {
#pragma unroll
        for (int o = 0; o < 8; ++o) part[(t >> 5) * 8 + o] = v[o];
      }
    }
  }
  __syncthreads();
  if (t < lay.out) rmw(gs + lay.b3 + t, (part[t] + part[8 + t]) + (part[16 + t] + part[24 + t]), first);
  // ---- dh2[r][j] = (sum_o dq[r][o] * W3[o][j]) * (h2[r][j] > 0), in place over H2; db2 partials ----------------
  float4 colsum = make_float4(0.f, 0.f, 0.f, 0.f);
  {
    const int c = t & 31, rbase = t >> 5;
    float4 wv[kOutPad];
#pragma unroll
    for (int o = 0; o < kOutPad; ++o) wv[o] = reinterpret_cast<const float4*>(w.w3 + o * kHidden)[c];
#pragma unroll 2
    for (int it = 0; it < kTileRows / 8; ++it) {
      const int r = rbase + 8 * it;
      const float4 d0 = *reinterpret_cast<const float4*>(DQ + r * kOutPad), d1 = *reinterpret_cast<const float4*>(DQ + r * kOutPad + 4);
      const float dv[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
      float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int o = 0; o < kOutPad; ++o) {
        g.x = fmaf(dv[o], wv[o].x, g.x); g.y = fmaf(dv[o], wv[o].y, g.y); g.z = fmaf(dv[o], wv[o].z, g.z); g.w = fmaf(dv[o], wv[o].w, g.w);
      }
      float4& h = at4<kHidden>(H2, r, c);
      g.x = h.x > 0.f ? g.x : 0.f; g.y = h.y > 0.f ? g.y : 0.f; g.z = h.z > 0.f ? g.z : 0.f; g.w = h.w > 0.f ? g.w : 0.f;
      h = g;
      colsum.x += g.x; colsum.y += g.y; colsum.z += g.z; colsum.w += g.w;
    }
  }
  __syncthreads();  // dq fully consumed -> reuse DQ as the [8][128] reduction buffer
  *reinterpret_cast<float4*>(DQ + (t >> 5) * kHidden + (t & 31) * 4) = colsum;
  __syncthreads();
  if (t < kHidden) {
    float s = 0.f;
#pragma unroll
    for (int wq = 0; wq < 8; ++wq) s += DQ[wq * kHidden + t];
    rmw(gs + lay.b2 + t, s, first);
  }
  // ---- dW2[m][n] = sum_r dh2[r][m] * h1[r][n] ------------------------------------------------------------------
  {
    float acc[8][8];
    zero_acc(acc);
    gemm_tn<kHidden, kHidden>(H2, H1, kTileRows, tc, acc);
#pragma unroll
    for (int mi = 0; mi < 8; ++mi) {
      float* row = gs + lay.w2 + tn_row(tc, mi) * kHidden;
      rmw4(row + tn_col(tc, 0), make_float4(acc[mi][0], acc[mi][1], acc[mi][2], acc[mi][3]), first);
      rmw4(row + tn_col(tc, 4), make_float4(acc[mi][4], acc[mi][5], acc[mi][6], acc[mi][7]), first);
    }
  }
  __syncthreads();  // H1 no longer needed as a GEMM operand; DQ reduction buffer consumed
  // ---- dh1[r][n] = (sum_k dh2[r][k] * W2[k][n]) * (h1[r][n] > 0), in place over H1; db1 ----------------------------
  {
    float acc[8][8];
    zero_acc(acc);
    gemm_nn(H2, w.w2, tc, acc);
    const int r0 = tc.wy * 32 + tc.ty, nc = tc.wx * 16 + tc.tx;
    float cs[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float4& h0 = at4<kHidden>(H1, r0 + 4 * i, nc);
      float4& h1 = at4<kHidden>(H1, r0 + 4 * i, nc + 8);
      float4 g0, g1;
      g0.x = h0.x > 0.f ? acc[i][0] : 0.f; g0.y = h0.y > 0.f ? acc[i][1] : 0.f; g0.z = h0.z > 0.f ? acc[i][2] : 0.f; g0.w = h0.w > 0.f ? acc[i][3] : 0.f;
      g1.x = h1.x > 0.f ? acc[i][4] : 0.f; g1.y = h1.y > 0.f ? acc[i][5] : 0.f; g1.z = h1.z > 0.f ? acc[i][6] : 0.f; g1.w = h1.w > 0.f ? acc[i][7] : 0.f;
      h0 = g0; h1 = g1;
      cs[0] += g0.x; cs[1] += g0.y; cs[2] += g0.z; cs[3] += g0.w; cs[4] += g1.x; cs[5] += g1.y; cs[6] += g1.z; cs[7] += g1.w;
    }
    // sum over the four ty lanes (lane bits 3,4), then one partial per row-warp into DQ[wy][n]
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      cs[j] += __shfl_xor_sync(0xFFFFFFFFu, cs[j], 8);
      cs[j] += __shfl_xor_sync(0xFFFFFFFFu, cs[j], 16);
    }
    if (tc.ty == 0) {
#pragma unroll
      for (int j = 0; j < 8; ++j) DQ[tc.wy * kHidden + tn_col(tc, j)] = cs[j];
    }
  }
  __syncthreads();  // dh2 (H2 region) is dead from here on: bring the input tile back into it for dW1
  gather_tile_async<KP>(X, meta, obs_dim);
  if (t < kHidden) rmw(gs + lay.b1 + t, DQ[t] + DQ[kHidden + t] + DQ[2 * kHidden + t] + DQ[3 * kHidden + t], first);
  cp_async_wait_all();
  __syncthreads();
  // ---- dW1[m][i] = sum_r dh1[r][m] * x[r][i] ---------------------------------------------------------------------
  if constexpr (KP == kKpWide) {
    // one pass per K-chunk of the input (the narrow tiles' two-column-group register block), dH1 re-read from shared memory per pass:
    // a single 128-column pass would hold 64 more accumulators than the register budget has
    const int mg = t >> 4, i0 = t & 15, n_chunks = (lay.in + kW1Chunk - 1) / kW1Chunk;
#pragma unroll 1
    for (int c = 0; c < n_chunks; ++c) {
      float acc[kW1Chunk / 16][8];
#pragma unroll
      for (int ii = 0; ii < kW1Chunk / 16; ++ii)
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[ii][q] = 0.f;
#pragma unroll 4
      for (int r = 0; r < kTileRows; ++r) {
        const float4 a0 = at4<kHidden>(H1, r, 2 * mg), a1 = at4<kHidden>(H1, r, 2 * mg + 1);
#pragma unroll
        for (int ii = 0; ii < kW1Chunk / 16; ++ii) {
          const float x = at1<KP>(X, r, c * kW1Chunk + i0 + 16 * ii);
          acc[ii][0] = fmaf(a0.x, x, acc[ii][0]); acc[ii][1] = fmaf(a0.y, x, acc[ii][1]); acc[ii][2] = fmaf(a0.z, x, acc[ii][2]); acc[ii][3] = fmaf(a0.w, x, acc[ii][3]);
          acc[ii][4] = fmaf(a1.x, x, acc[ii][4]); acc[ii][5] = fmaf(a1.y, x, acc[ii][5]); acc[ii][6] = fmaf(a1.z, x, acc[ii][6]); acc[ii][7] = fmaf(a1.w, x, acc[ii][7]);
        }
      }
#pragma unroll
      for (int ii = 0; ii < kW1Chunk / 16; ++ii) {
        const int i = c * kW1Chunk + i0 + 16 * ii;
        if (i < lay.in) {
#pragma unroll
          for (int q = 0; q < 8; ++q) rmw(gs + lay.w1 + (mg * 8 + q) * lay.in + i, acc[ii][q], first);
        }
      }
    }
  } else {
    const int mg = t >> 4, i0 = t & 15;
    float acc[KP / 16][8];
#pragma unroll
    for (int ii = 0; ii < KP / 16; ++ii)
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[ii][q] = 0.f;
#pragma unroll 4
    for (int r = 0; r < kTileRows; ++r) {
      const float4 a0 = at4<kHidden>(H1, r, 2 * mg), a1 = at4<kHidden>(H1, r, 2 * mg + 1);
#pragma unroll
      for (int ii = 0; ii < KP / 16; ++ii) {
        const float x = at1<KP>(X, r, i0 + 16 * ii);
        acc[ii][0] = fmaf(a0.x, x, acc[ii][0]); acc[ii][1] = fmaf(a0.y, x, acc[ii][1]); acc[ii][2] = fmaf(a0.z, x, acc[ii][2]); acc[ii][3] = fmaf(a0.w, x, acc[ii][3]);
        acc[ii][4] = fmaf(a1.x, x, acc[ii][4]); acc[ii][5] = fmaf(a1.y, x, acc[ii][5]); acc[ii][6] = fmaf(a1.z, x, acc[ii][6]); acc[ii][7] = fmaf(a1.w, x, acc[ii][7]);
      }
    }
#pragma unroll
    for (int ii = 0; ii < KP / 16; ++ii) {
      const int i = i0 + 16 * ii;
      if (i < lay.in) {
#pragma unroll
        for (int q = 0; q < 8; ++q) rmw(gs + lay.w1 + (mg * 8 + q) * lay.in + i, acc[ii][q], first);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------
// Loss heads: one thread per row of the tile.  `q` = this row's network outputs, `qn` = next row's (same episode),
// results: dq[0..7] = dLoss/d(output) un-normalised, st[0..3] += loss statistics.
struct RowCtx { int agent, b, tt, T, A, B; int act; float rew, filled, done1; };

__device__ __forceinline__ void head_dqn(const TrainParams& p, const RowCtx& c, const float* q, const float* qn, float (&dq)[kOutPad], float (&st)[4]) {
  const int act = c.act;
  const float filled = c.filled;
  float g;
  if (p.td_ext) {  // VDN: the agent-coupled TD error was computed by vdn_td_kernel
    g = p.td_ext[(size_t)c.agent * p.td_agent_stride + (size_t)c.b * c.T + c.tt];
  } else {
    const float rew = c.rew, done1 = c.done1;
    const float* tq = p.tq + (((size_t)c.agent * c.B + c.b) * (c.T + 1) + c.tt + 1) * c.A;
    float tsel;
    if (p.double_q) {  // dqn/model.py:138-143
      int best = 0; float bv = qn[0];
      for (int o = 1; o < c.A; ++o) if (qn[o] > bv) { bv = qn[o]; best = o; }
      tsel = tq[best];
    } else {
      tsel = tq[0];
      for (int o = 1; o < c.A; ++o) tsel = fmaxf(tsel, tq[o]);
    }
    const float y = rew + p.gamma * tsel * (1.f - done1);   // dqn/model.py:152
    const float delta = q[act] - y;
    st[0] += delta * delta * filled;                        // dqn/model.py:160-163
    if (c.agent == 0) st[1] += filled;
    g = 2.f * delta * filled;
  }
#pragma unroll
  for (int o = 0; o < kOutPad; ++o) dq[o] = (o == act) ? g : 0.f;
}

__device__ __forceinline__ void head_a2c_critic(const TrainParams& p, const RowCtx& c, const float* q, float (&dq)[kOutPad], float (&st)[4]) {
  const size_t i = ((size_t)c.agent * c.B + c.b) * c.T + c.tt;
  const float filled = c.filled;
  const float adv = p.returns[i] - q[0];                    // ac/model.py:214
  p.adv_out[i] = adv;
  st[3] += adv * adv * filled;                              // ac/model.py:221-222
  if (c.agent == 0) st[1] += filled;
  dq[0] = -2.f * adv * filled * p.value_coef;               // d(value_loss_coef * (R - V)^2)/dV
}

__device__ __forceinline__ void head_a2c_actor(const TrainParams& p, const RowCtx& c, const float* q, float (&dq)[kOutPad], float (&st)[4]) {
  const size_t i = ((size_t)c.agent * c.B + c.b) * c.T + c.tt;
  const int act = c.act;
  const float filled = c.filled;
  const float adv = p.adv[i];
  float m = q[0];
  for (int o = 1; o < c.A; ++o) m = fmaxf(m, q[o]);
  float s = 0.f;
  for (int o = 0; o < c.A; ++o) s += expf(q[o] - m);
  const float lse = m + logf(s);
  float ent = 0.f, pr[kOutPad], ls[kOutPad];
#pragma unroll
  for (int o = 0; o < kOutPad; ++o) {
    ls[o] = o < c.A ? q[o] - lse : 0.f;                     // Categorical(logits) normalisation (ac/model.py:142-144)
    pr[o] = o < c.A ? expf(ls[o]) : 0.f;
    ent -= pr[o] * ls[o];
  }
  float w = adv;   // dLoss/dlogp[act] = -w
  if (p.old_logp != nullptr) {
    // PPO clipped surrogate (ac/model.py:309-321).  torch.min sends the gradient to the smaller argument (half to each on a tie), clamp passes it
    // inside [1 - c, 1 + c]: d(-min(r adv, clamp(r) adv))/dlogp = -adv r k, k = 1 when the unclipped term is the minimum or r is inside the range.
    const float ratio = expf(ls[act] - p.old_logp[i]);
    const float lo = 1.f - p.ppo_clip, hi = 1.f + p.ppo_clip;
    const float surr1 = ratio * adv, surr2 = fminf(fmaxf(ratio, lo), hi) * adv;
    const float inrange = (ratio >= lo && ratio <= hi) ? 1.f : 0.f;
    const float k = surr1 < surr2 ? 1.f : (surr1 > surr2 ? inrange : 0.5f + 0.5f * inrange);
    st[0] += -fminf(surr1, surr2) * filled;
    w = adv * ratio * k;
  } else {
    st[0] += -ls[act] * adv * filled;                       // ac/model.py:216-219
  }
  st[2] += ent * filled;
#pragma unroll
  for (int o = 0; o < kOutPad; ++o)
    dq[o] = o < c.A ? filled * (w * (pr[o] - (o == act ? 1.f : 0.f)) + p.entropy_coef * pr[o] * (ls[o] + ent)) : 0.f;
}

// ------------------------------------------------------------------------------------------------------------
template <int KP, int HEAD>
__global__ void __launch_bounds__(kMlpThreads, 1) train_kernel(TrainParams p) {
  extern __shared__ __align__(16) float smem[];
  WeightSmem<KP> w(smem);
  float* H1 = smem + WeightSmem<KP>::kFloats;
  float* H2 = H1 + kTileRows * kPitchH;
  float* X = H2;  // the input tile aliases H2: live during layer 1, re-gathered for dW1 once dH2 is dead
  float* Q = H2 + kTileRows * kPitchH;  // network outputs, then dLoss/dOutput, then reduction scratch
  float* carry = Q + kTileRows * kOutPad;  // outputs of the first row of the previously processed (higher) tile
  RowMeta* meta = reinterpret_cast<RowMeta*>(carry + 48);  // carry[16] | db3 partials[32] | row metadata
  const ThreadCoord tc;
  const int t = threadIdx.x;
  int net, row_begin, row_end;
  cta_rows(p.plan, net, row_begin, row_end);
  float* gs = p.scratch + (size_t)blockIdx.x * p.scratch_pitch;
  float st[4] = {0.f, 0.f, 0.f, 0.f};
  if (row_begin >= row_end) {  // idle CTA: its partial must still read as zero
    for (int i = t; i < p.lay.P; i += kMlpThreads) gs[i] = 0.f;
    if (t < 4) p.loss_part[4 * blockIdx.x + t] = 0.f;
    return;
  }
  const float* theta = p.theta + (size_t)net * p.lay.P;
  w.load_async(theta, p.lay);
  RowCtx c; c.T = p.src.traj.T; c.A = p.lay.out; c.B = p.plan.units_per_agent;
  bool first = true;
  // tiles from the top of the chunk downwards, so that the next row's outputs of a tile's last row are already known
  for (int vr_hi = row_end; vr_hi > row_begin; vr_hi -= kTileRows) {
    const int vr0 = max(row_begin, vr_hi - kTileRows), nrows = vr_hi - vr0;
    __syncthreads();
    setup_rows<true>(meta, p.plan, p.src, net, vr0, nrows);
    __syncthreads();
    gather_tile_async<KP>(X, meta, p.src.D);
    if constexpr (KP == kKpWide) w.load_w1_chunk_async(theta, p.lay, 0);   // (the backward never reads W1: the slot is free)
    cp_async_wait_all();
    __syncthreads();
    if constexpr (KP == kKpWide) mlp_forward_tile_wide(X, H1, H2, Q, w, theta, p.lay, tc);
    else mlp_forward_tile<KP>(X, H1, H2, Q, w, tc);
    __syncthreads();
    float dq[kOutPad];
#pragma unroll
    for (int o = 0; o < kOutPad; ++o) dq[o] = 0.f;
    float q_first[kOutPad];
    if (t == 0) {
#pragma unroll
      for (int o = 0; o < kOutPad; ++o) q_first[o] = Q[o];
    }
    if (t < nrows) {
      decode_row(p.plan, net, vr0 + t, c.agent, c.b, c.tt);
      if (c.tt < c.T) {
        c.act = meta->act[t]; c.rew = meta->rew[t]; c.filled = (float)(meta->flags[t] & 1); c.done1 = (float)((meta->flags[t] >> 1) & 1);
        const float* q = Q + t * kOutPad;
        if constexpr (HEAD == kHeadDqn) head_dqn(p, c, q, (t + 1 < nrows) ? q + kOutPad : carry, dq, st);
        else if constexpr (HEAD == kHeadA2cCritic) head_a2c_critic(p, c, q, dq, st);
        else head_a2c_actor(p, c, q, dq, st);
      }
    }
    __syncthreads();
    if (t < kTileRows) {
      *reinterpret_cast<float4*>(Q + t * kOutPad) = make_float4(dq[0], dq[1], dq[2], dq[3]);
      *reinterpret_cast<float4*>(Q + t * kOutPad + 4) = make_float4(dq[4], dq[5], dq[6], dq[7]);
    }
    if (t == 0) {
#pragma unroll
      for (int o = 0; o < kOutPad; ++o) carry[o] = q_first[o];
    }
    __syncthreads();
    mlp_backward_tile<KP>(X, H1, H2, Q, w, p.lay, gs, first, tc, meta, p.src.D, carry + 16);
    first = false;
  }
  // ---- per-CTA loss statistics (fixed-order tree: deterministic) ---------------------------------------------------
  __syncthreads();
  float* red = Q;
#pragma unroll
  for (int k = 0; k < 4; ++k) red[k * kMlpThreads + t] = st[k];
  __syncthreads();
  for (int s = kMlpThreads / 2; s > 0; s >>= 1) {
    if (t < s) {
#pragma unroll
      for (int k = 0; k < 4; ++k) red[k * kMlpThreads + t] += red[k * kMlpThreads + t + s];
    }
    __syncthreads();
  }
  if (t < 4) p.loss_part[4 * blockIdx.x + t] = red[t * kMlpThreads];
}

// ------------------------------------------------------------------------------------------------------------
// 64 parameters x 16 CTA-slices per block: slice q sums the partials of CTAs c0+q, c0+q+16, ... (every load of a thread in
// flight at once: the kernel is a latency chain otherwise), the slices are combined in a fixed order through shared memory ->
// deterministic.  Each block also leaves the sum of squares of its 64 reduced gradients in sumsq_part (single-GPU fast path of
// the clip in adam_kernel).
constexpr int kReduceSlices = 16;
__global__ void __launch_bounds__(64 * kReduceSlices) grad_reduce_kernel(ReduceParams p) {
  __shared__ float part[kReduceSlices][64];
  __shared__ float sq[64];
  const int lane = threadIdx.x & 63, q = threadIdx.x >> 6;
  const int i = blockIdx.x * 64 + lane, n = p.n_nets * p.P;
  pdl_wait();
  pdl_launch_dependents();
  float s = 0.f;
  if (i < n) {
    const int net = i / p.P, j = i - net * p.P;
    const int c0 = p.cta_begin[net], c1 = p.cta_begin[net + 1];
    const float* base = p.scratch + j;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    int c = c0 + q;
    for (; c + 3 * kReduceSlices < c1; c += 4 * kReduceSlices) {
      a0 += base[(size_t)c * p.scratch_pitch]; a1 += base[(size_t)(c + kReduceSlices) * p.scratch_pitch];
      a2 += base[(size_t)(c + 2 * kReduceSlices) * p.scratch_pitch]; a3 += base[(size_t)(c + 3 * kReduceSlices) * p.scratch_pitch];
    }
    float t0 = 0.f, t1 = 0.f, t2 = 0.f;   // up to three more partials, loaded together
    if (c < c1) t0 = base[(size_t)c * p.scratch_pitch];
    if (c + kReduceSlices < c1) t1 = base[(size_t)(c + kReduceSlices) * p.scratch_pitch];
    if (c + 2 * kReduceSlices < c1) t2 = base[(size_t)(c + 2 * kReduceSlices) * p.scratch_pitch];
    s = ((a0 + a1) + (a2 + a3)) + ((t0 + t1) + t2);
  }
  part[q][lane] = s;
  __syncthreads();
  if (q == 0) {
    float g = 0.f;
#pragma unroll
    for (int k = 0; k < kReduceSlices; k += 4) g += (part[k][lane] + part[k + 1][lane]) + (part[k + 2][lane] + part[k + 3][lane]);
    if (i < n) p.grad[i] = g;
    sq[lane] = (i < n) ? g * g : 0.f;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = sq[threadIdx.x] + sq[threadIdx.x + 32];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, off);
    if (threadIdx.x == 0 && p.sumsq_part) p.sumsq_part[blockIdx.x] = v;
  }
  // the four loss statistics: one warp each (a serial walk over the per-CTA parts was this kernel's critical path), fixed order
  if (blockIdx.x == 0 && threadIdx.x >= 64 && threadIdx.x < 192 && p.stats) {
    const int which = (threadIdx.x - 64) >> 5, l = threadIdx.x & 31;
    float t = 0.f;
    for (int c = l; c < p.n_loss_parts; c += 32) t += p.loss_part[4 * c + which];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xFFFFFFFFu, t, off);
    if (l == 0) p.stats[which] = (p.stats_accumulate ? p.stats[which] : 0.f) + t;
  }
}

// grad holds un-normalised sums followed by 4 statistics (loss numerator, filled count, aux, aux) -- possibly
// all-reduced over ranks.
// Every CTA recomputes the global norm in the same order (bit-identical clip coefficient on every CTA and rank).
__global__ void __launch_bounds__(256) adam_kernel(AdamParams p) {
  __shared__ float red[256];
  pdl_wait();
  pdl_launch_dependents();
  const float inv_fill = 1.f / p.grad[p.n + 1];
  float clip = 1.f, norm = 0.f;
  if (p.sumsq_part) {  // single-GPU: grad_reduce_kernel already left per-block sums of squares (fixed-order combine)
    float s = 0.f;
    for (int i = threadIdx.x; i < p.n_sumsq; i += 256) s += p.sumsq_part[i];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int k = 128; k > 0; k >>= 1) { if (threadIdx.x < k) red[threadIdx.x] += red[threadIdx.x + k]; __syncthreads(); }
    norm = sqrtf(red[0]) * inv_fill;
    if (p.grad_clip > 0.f) clip = fminf(p.grad_clip / (norm + 1e-6f), 1.f);
  } else {
    float s = 0.f;
    const int n4 = p.n >> 2;
    const float4* g4 = reinterpret_cast<const float4*>(p.grad);
#pragma unroll 4
    for (int i = threadIdx.x; i < n4; i += 256) {
      const float4 g = g4[i];
      const float a = g.x * inv_fill, b = g.y * inv_fill, c = g.z * inv_fill, d = g.w * inv_fill;
      s = fmaf(a, a, s); s = fmaf(b, b, s); s = fmaf(c, c, s); s = fmaf(d, d, s);
    }
    for (int i = 4 * n4 + threadIdx.x; i < p.n; i += 256) { const float g = p.grad[i] * inv_fill; s = fmaf(g, g, s); }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int k = 128; k > 0; k >>= 1) { if (threadIdx.x < k) red[threadIdx.x] += red[threadIdx.x + k]; __syncthreads(); }
    norm = sqrtf(red[0]);
    if (p.grad_clip > 0.f) clip = fminf(p.grad_clip / (norm + 1e-6f), 1.f);  // torch.nn.utils.clip_grad_norm_
  }
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < p.n) {
    const float g = p.grad[i] * inv_fill * clip;
    float m = p.m[i], v = p.v[i], th = p.theta[i];
    m = m + (g - m) * (1.f - p.beta1);                       // exp_avg.lerp_(grad, 1 - beta1)
    v = v * p.beta2 + g * g * (1.f - p.beta2);               // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    const float denom = sqrtf(v) / p.bc2_sqrt + p.eps;
    th = th - (p.lr / p.bc1) * (m / denom);
    p.m[i] = m; p.v[i] = v; p.theta[i] = th;
    if (p.image != nullptr && i < p.img_nets * p.img_lay.P) {  // keep the packed tensor-core images of theta current
      const int net = i / p.img_lay.P;
      pack_param(p.img_lay, i - net * p.img_lay.P, th, p.image + (size_t)net * p.image_bytes, p.bwd_image ? p.bwd_image + (size_t)net * p.bwd_image_bytes : nullptr);
    }
    const int j = i - p.tgt_begin;
    if (j >= 0 && j < p.tgt_n) {
      if (p.target_mode == 1) p.theta_tgt[j] = th;
      else if (p.target_mode == 2) p.theta_tgt[j] = (1.f - p.tau) * p.theta_tgt[j] + p.tau * th;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && p.loss_out) {
    p.loss_out[0] = p.grad[p.n] * inv_fill; p.loss_out[1] = norm; p.loss_out[2] = p.grad[p.n + 2] * inv_fill;
    p.loss_out[3] = p.grad[p.n + 3] * inv_fill; p.loss_out[4] = p.grad[p.n + 1]; p.loss_out[5] = 0.f;
  }
}

// ------------------------------------------------------------------------------------------------------------
// The tail of an update in ONE kernel: grad_reduce_kernel's deterministic partial sums, (several ranks: the gradient exchange over
// NVLink peer memory,) a grid-wide barrier, then adam_kernel's clip + Adam step on the gradient each thread still holds in a register.
// 256 parameters x 4 CTA-slices per block, every load of a thread in flight at once, one wave (the launcher guarantees that all blocks
// are co-resident, which the hand-made barrier needs; `barrier` counts block arrivals across launches and is never reset, `target` is
// its value once this launch has fully arrived -- a second arrival round follows when XCHG).  grad[] and the statistics are still
// published: metrics and the two-call API read them.
//
// XCHG (one process per GPU, buffers opened through CUDA IPC): a push exchange.  Every rank's buffer holds, per epoch parity, one copy
// of [gradient | 4 statistics] PER SOURCE RANK plus one flag per source rank.  A rank stores its local sums into its own copy on every
// rank (posted remote stores over NVLink), makes them visible system-wide, and writes `epoch` into its flag on every rank; a block
// then polls only LOCAL flags and reads only LOCAL memory, adding the ranks' values of its parameter in rank order -- the same order on
// every rank, so the replicated parameters stay bit-identical without a second exchange.  Two parities suffice: a rank pushes epoch
// e + 1 only after its kernel of epoch e has completed (it has read everything of epoch e), and nobody pushes parity e & 1 again before
// having seen e + 1 from everybody.
constexpr long long kPeerSpinCycles = 20LL * 1000 * 1000 * 1000;   // ~10 s at 2 GHz: far beyond any healthy exchange (~10 us)
constexpr int kFusedMaxParams = 512, kFusedMaxSlices = 4, kFusedThreads = 1024;   // block shape is chosen at launch: pb parameters x ns slices

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ float ld_relaxed_sys(const float* p) {   // peer memory: never from a stale L1 line
  float v;
  asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}
// block-wide arrival at the grid barrier; returns once `target` arrivals have been counted (thread 0 spins, the block waits on it)
__device__ __forceinline__ void grid_barrier(unsigned long long* barrier, unsigned long long target, bool system_scope) {
  __syncthreads();
  if (threadIdx.x == 0) {
    if (system_scope) __threadfence_system(); else __threadfence();
    atomicAdd(barrier, 1ULL);
    while (*reinterpret_cast<volatile unsigned long long*>(barrier) < target) {}
    __threadfence();
  }
  __syncthreads();
}

TSG_DEFINE(g_ts_adam)
TSG_GETTER(tsg_adam, g_ts_adam)
// MODE 0: one GPU.  1: several ranks, exchange inside this kernel (push, grid barrier, flags, poll, sum).  2 + 3: the same exchange split over two
// launches so that the wait for the peers hides under other work (the next update's target forward runs between them): 2 = reduce + push; the LAST
// block to finish its pushes publishes this rank's epoch flags (an arrival counter, nobody spins) and the next update's replay indices are drawn here;
// 3 = poll the local flags, sum the ranks' copies, clip + Adam.
template <int MODE>
__global__ void __launch_bounds__(kFusedThreads) reduce_adam_kernel(ReduceParams rp, AdamParams ap, XchgParams xp, SampleParams sp, int pb, int ns,
                                                                    unsigned long long* barrier, unsigned long long target) {
  constexpr bool XCHG = MODE != 0;
  __shared__ float part[kFusedMaxSlices][kFusedMaxParams];
  __shared__ float red[32];
  __shared__ float stats_sh[4];
  // pb parameters (a multiple of 32) x ns CTA-slices per block, blockDim.x = pb * ns
  const int t = threadIdx.x, q = t / pb, lane = t - q * pb;
  const int i = blockIdx.x * pb + lane, n = rp.n_nets * rp.P;
  TSG(g_ts_adam, 0);
  pdl_wait();
  pdl_launch_dependents();
  TSG(g_ts_adam, 1);
  float s = 0.f;
  if (MODE != 3 && i < n) {
    const int net = i / rp.P, j = i - net * rp.P;
    const int c0 = rp.cta_begin[net], c1 = rp.cta_begin[net + 1];
    const float* base = rp.scratch + j;
    for (int cb = c0 + q; cb < c1; cb += 20 * ns) {   // 74 CTAs per network / 3 slices: two rounds of up to 20 loads in flight
      float v[20];
#pragma unroll
      for (int k = 0; k < 20; ++k) { const int c = cb + k * ns; v[k] = c < c1 ? base[(size_t)c * rp.scratch_pitch] : 0.f; }
      float u[5];
#pragma unroll
      for (int k = 0; k < 5; ++k) u[k] = (v[4 * k] + v[4 * k + 1]) + (v[4 * k + 2] + v[4 * k + 3]);
      s += ((u[0] + u[1]) + (u[2] + u[3])) + u[4];
    }
  }
  // this thread's optimiser state: the loads fly under the reductions and barriers below
  float m_i = 0.f, v_i = 0.f, th_i = 0.f;
  if (MODE != 2 && q == 0 && i < ap.n) { m_i = ap.m[i]; v_i = ap.v[i]; th_i = ap.theta[i]; }
  part[q][lane] = s;
  __syncthreads();
  TSG(g_ts_adam, 2);
  float g = 0.f;
  // this rank's copy inside rank r's buffer: base_r + ((epoch & 1) * world + rank) * slot_floats
  const size_t push_off = XCHG ? ((size_t)(xp.epoch & 1ULL) * xp.world + xp.rank) * xp.slot_floats : 0;
  if (MODE != 3 && q == 0) {
    g = part[0][lane];
    for (int k = 1; k < ns; ++k) g += part[k][lane];
    if (i >= n) g = 0.f;
    else if (XCHG) { for (int r = 0; r < xp.world; ++r) xp.peers[r][push_off + i] = g; }   // local sums -> every rank (own included)
    else rp.grad[i] = g;
  }
  // the four loss statistics: one warp each of block 0, fixed order
  if (MODE != 3 && blockIdx.x == 0 && t >= pb && t < pb + 128) {   // (the launcher guarantees ns >= 2 and pb >= 128)
    const int which = (t - pb) >> 5, l = t & 31;
    float x = 0.f;
    for (int c = l; c < rp.n_loss_parts; c += 32) x += rp.loss_part[4 * c + which];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(0xFFFFFFFFu, x, off);
    if (l == 0) {
      x += rp.stats_accumulate ? rp.stats[which] : 0.f;
      if (XCHG) { for (int r = 0; r < xp.world; ++r) xp.peers[r][push_off + n + which] = x; } else rp.stats[which] = x;
    }
  }
  if (MODE == 2) {
    // ---- push only: this block's pushes become visible system-wide, it arrives; the last block to arrive publishes the epoch.  `barrier` + 1 is this
    // kernel's own arrival counter (never reset: `target` is its value once this launch has fully arrived)
    if (sp.idx != nullptr) {   // replay indices of the NEXT update: its target forward runs before the finishing kernel
      for (int k = blockIdx.x * (int)blockDim.x + t; k < sp.batch; k += (int)(gridDim.x * blockDim.x)) {
        const u32x4 b = philox4x32_10((uint32_t)sp.update_idx, (uint32_t)(sp.update_idx >> 32), (uint32_t)(k >> 2), 0u, (uint32_t)sp.seed, (uint32_t)(sp.seed >> 32) ^ kTagSample);
        sp.idx[k] = (int32_t)bounded(pick(b, k & 3), (uint32_t)sp.n_valid);
      }
    }
    __syncthreads();
    if (t == 0) {
      __threadfence_system();
      const unsigned long long arrived = atomicAdd(barrier + 1, 1ULL) + 1ULL;
      if (arrived == target) {
        __threadfence_system();
        for (int r = 0; r < xp.world; ++r) st_release_sys(xp.peer_flags[r] + xp.rank, xp.epoch);   // my flag on every rank
      }
    }
    return;
  }
  if (XCHG) {
    // ---- exchange: local sums visible system-wide -> publish the epoch -> wait for every peer -> sum in rank order -----------------
    if (MODE == 1) {
      grid_barrier(barrier, target - gridDim.x, true);   // every block's pushes are ordered before the flags (system-scope fences)
      if (blockIdx.x == 0 && t < xp.world) st_release_sys(xp.peer_flags[t] + xp.rank, xp.epoch);   // my flag on rank t
    }
    if (t < xp.world) {   // local polling only; bounded: a rank that died / skipped an update must not hang this GPU for ever
      const long long t0 = clock64();
      while (ld_acquire_sys(xp.own_flags + t) < xp.epoch) {
        if (clock64() - t0 > kPeerSpinCycles) { atomicExch(xp.timed_out, 1); break; }   // sticky; the host raises on it (marl_dqn_peer_status)
      }
    }
    __syncthreads();
    const float* mine = xp.peers[xp.rank] + (size_t)(xp.epoch & 1ULL) * xp.world * xp.slot_floats;
    if (q == 0 && i < n) {
      g = 0.f;
      for (int r = 0; r < xp.world; ++r) g += ld_relaxed_sys(mine + (size_t)r * xp.slot_floats + i);
      rp.grad[i] = g;
    }
    if (t < 4) {
      float x = 0.f;
      for (int r = 0; r < xp.world; ++r) x += ld_relaxed_sys(mine + (size_t)r * xp.slot_floats + n + t);
      stats_sh[t] = x;
      if (blockIdx.x == 0) rp.stats[t] = x;
    }
  }
  // block sum of squares: slice 0 holds the gradients (pb / 32 warps) -> shuffle tree per warp, then the partials in order
  if (q == 0) {
    float sq = g * g;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) sq += __shfl_xor_sync(0xFFFFFFFFu, sq, off);
    if ((t & 31) == 0) red[t >> 5] = sq;
  }
  __syncthreads();
  if (t == 0) {
    float x = red[0];
    for (int k = 1; k < pb / 32; ++k) x += red[k];
    rp.sumsq_part[blockIdx.x] = x;
  }
  TSG(g_ts_adam, 3);
  grid_barrier(barrier, target, false);   // every block's sum of squares (and block 0's statistics) are visible after it
  TSG(g_ts_adam, 4);
  // ---- every block: global norm from the per-block sums (fixed order: lane k adds blocks k, k + 32, ..., then a shuffle tree) ----
  if (t < 32) {
    float x = 0.f;
    for (int k = t; k < (int)gridDim.x; k += 32) x += __ldcg(rp.sumsq_part + k);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(0xFFFFFFFFu, x, off);
    if (t == 0) red[0] = x;
  }
  __syncthreads();
  float st4[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) st4[k] = XCHG ? stats_sh[k] : __ldcg(ap.grad + ap.n + k);
  const float fill = st4[1], inv_fill = 1.f / fill;
  const float norm = sqrtf(red[0]) * inv_fill;
  float clip = 1.f;
  if (ap.grad_clip > 0.f) clip = fminf(ap.grad_clip / (norm + 1e-6f), 1.f);   // torch.nn.utils.clip_grad_norm_
  if (q == 0 && i < ap.n) {
    const float gg = g * inv_fill * clip;
    float m = m_i, v = v_i, th = th_i;
    m = m + (gg - m) * (1.f - ap.beta1);                       // exp_avg.lerp_(grad, 1 - beta1)
    v = v * ap.beta2 + gg * gg * (1.f - ap.beta2);             // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    const float denom = sqrtf(v) / ap.bc2_sqrt + ap.eps;
    th = th - (ap.lr / ap.bc1) * (m / denom);
    ap.m[i] = m; ap.v[i] = v; ap.theta[i] = th;
    if (ap.image != nullptr && i < ap.img_nets * ap.img_lay.P) {
      const int net = i / ap.img_lay.P;
      pack_param(ap.img_lay, i - net * ap.img_lay.P, th, ap.image + (size_t)net * ap.image_bytes, ap.bwd_image ? ap.bwd_image + (size_t)net * ap.bwd_image_bytes : nullptr);
    }
    const int j = i - ap.tgt_begin;
    if (j >= 0 && j < ap.tgt_n) {
      if (ap.target_mode == 1) ap.theta_tgt[j] = th;
      else if (ap.target_mode == 2) ap.theta_tgt[j] = (1.f - ap.tau) * ap.theta_tgt[j] + ap.tau * th;
    }
  }
  // replay indices of the NEXT update (marl_dqn_update_n): np.random.randint(0, len(rb), batch) from the Philox stream -- every reader of
  // the current indices has completed (this kernel runs after the weight-gradient kernel), and the next sample launch is saved
  if (MODE != 3 && sp.idx != nullptr) {
    for (int k = blockIdx.x * (int)blockDim.x + t; k < sp.batch; k += (int)(gridDim.x * blockDim.x)) {
      const u32x4 b = philox4x32_10((uint32_t)sp.update_idx, (uint32_t)(sp.update_idx >> 32), (uint32_t)(k >> 2), 0u, (uint32_t)sp.seed, (uint32_t)(sp.seed >> 32) ^ kTagSample);
      sp.idx[k] = (int32_t)bounded(pick(b, k & 3), (uint32_t)sp.n_valid);
    }
  }
  TSG(g_ts_adam, 31);
  if (blockIdx.x == 0 && t == 0 && ap.loss_out) {
    ap.loss_out[0] = st4[0] * inv_fill; ap.loss_out[1] = norm; ap.loss_out[2] = st4[2] * inv_fill;
    ap.loss_out[3] = st4[3] * inv_fill; ap.loss_out[4] = fill;
    ap.loss_out[5] = (XCHG && *reinterpret_cast<volatile int*>(xp.timed_out)) ? 1.f : 0.f;   // 1 = the peer exchange timed out: results are invalid
  }
}

// ---- launchers ------------------------------------------------------------------------------------------------
template <int KP>
static int init_kp() {
  MARL_CUDA_TRY(cudaFuncSetAttribute(mlp_forward_kernel<KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)forward_smem_bytes<KP>()));
  MARL_CUDA_TRY(cudaFuncSetAttribute(train_kernel<KP, kHeadDqn>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)train_smem_bytes<KP>()));
  MARL_CUDA_TRY(cudaFuncSetAttribute(train_kernel<KP, kHeadA2cCritic>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)train_smem_bytes<KP>()));
  MARL_CUDA_TRY(cudaFuncSetAttribute(train_kernel<KP, kHeadA2cActor>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)train_smem_bytes<KP>()));
  return MARL_OK;
}

int learner_kernels_init(int in_dim) {
  MARL_REQUIRE(in_dim >= 1 && in_dim <= kMaxObsDim, "learner kernels: observation width %d not supported (1..%d)", in_dim, kMaxObsDim);
  return in_dim <= 16 ? init_kp<16>() : in_dim <= 32 ? init_kp<32>() : init_kp<kKpWide>();
}

int launch_mlp_forward(const FwdParams& p, cudaStream_t st) {
  const int grid = p.plan.cta_begin[p.plan.n_nets];
  if (p.lay.in <= 16) mlp_forward_kernel<16><<<grid, kMlpThreads, forward_smem_bytes<16>(), st>>>(p);
  else if (p.lay.in <= 32) mlp_forward_kernel<32><<<grid, kMlpThreads, forward_smem_bytes<32>(), st>>>(p);
  else mlp_forward_kernel<kKpWide><<<grid, kMlpThreads, forward_smem_bytes<kKpWide>(), st>>>(p);
  MARL_CUDA_TRY(cudaGetLastError());
  return MARL_OK;
}

template <int KP>
static int launch_train_kp(const TrainParams& p, int head, cudaStream_t st) {
  const int grid = p.plan.cta_begin[p.plan.n_nets];
  const size_t sm = train_smem_bytes<KP>();
  if (head == kHeadDqn) train_kernel<KP, kHeadDqn><<<grid, kMlpThreads, sm, st>>>(p);
  else if (head == kHeadA2cCritic) train_kernel<KP, kHeadA2cCritic><<<grid, kMlpThreads, sm, st>>>(p);
  else if (head == kHeadA2cActor) train_kernel<KP, kHeadA2cActor><<<grid, kMlpThreads, sm, st>>>(p);
  else { set_error("launch_train: unknown head %d", head); return MARL_EINVAL; }
  MARL_CUDA_TRY(cudaGetLastError());
  return MARL_OK;
}

int launch_train(const TrainParams& p, int head, cudaStream_t st) {
  return p.lay.in <= 16 ? launch_train_kp<16>(p, head, st) : p.lay.in <= 32 ? launch_train_kp<32>(p, head, st) : launch_train_kp<kKpWide>(p, head, st);
}

int launch_grad_reduce(const ReduceParams& p, cudaStream_t st) {
  const int n = p.n_nets * p.P;
  MARL_CUDA_TRY(launch_pdl(grad_reduce_kernel, dim3((n + 63) / 64), dim3(64 * kReduceSlices), 0, st, p));
  return MARL_OK;
}

// Fused tail; returns MARL_EINVAL without launching when no co-resident grid covers the parameters (the caller then uses the two
// kernels).  The hand-made grid barrier needs every block resident at once, so the block shape follows from the device: capacity =
// SMs x (blocks of 1024 threads per SM, from the occupancy API: 1 at this kernel's register count), pb = parameters per block =
// ceil(n / capacity) rounded up to a warp multiple, ns = slices = 1024 / pb.
// xp: NULL or world == 1 -> single GPU; else the exchange over peer memory (xp->epoch is advanced here).
int reduce_adam_shape(int n, int n_sm, bool xchg, int* pb_out, int* ns_out) {
  static int occ[2] = {0, 0};
  if (occ[xchg] == 0) {
    int o = 0;
    if (xchg) {   // the split form shares the block shape: the smaller occupancy of the three variants counts
      int o1 = 0, o2 = 0, o3 = 0;
      MARL_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o1, reduce_adam_kernel<1>, kFusedThreads, 0));
      MARL_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o2, reduce_adam_kernel<2>, kFusedThreads, 0));
      MARL_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o3, reduce_adam_kernel<3>, kFusedThreads, 0));
      o = o1 < o2 ? o1 : o2; o = o < o3 ? o : o3;
    } else {
      MARL_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, reduce_adam_kernel<0>, kFusedThreads, 0));
    }
    occ[xchg] = o > 0 ? o : -1;
  }
  if (occ[xchg] < 1) return MARL_EINVAL;
  const int capacity = n_sm * occ[xchg];
  const int pb = ((n + capacity - 1) / capacity + 31) / 32 * 32;
  if (pb < 128 || pb > kFusedMaxParams) return MARL_EINVAL;
  int ns = kFusedThreads / pb;
  if (ns > kFusedMaxSlices) ns = kFusedMaxSlices;
  if (ns < 2) return MARL_EINVAL;
  *pb_out = pb; *ns_out = ns;
  return MARL_OK;
}

int launch_reduce_adam(const ReduceParams& rp, const AdamParams& ap, XchgParams* xp, const SampleParams& sp, unsigned long long* barrier, unsigned long long* epoch,
                       int n_sm, cudaStream_t st) {
  const bool xchg = xp != nullptr && xp->world > 1;
  const int n = rp.n_nets * rp.P;
  int pb = 0, ns = 0;
  if (ap.n != n || reduce_adam_shape(n, n_sm, xchg, &pb, &ns) != MARL_OK) return MARL_EINVAL;
  const int grid = (n + pb - 1) / pb;   // <= capacity by construction
  XchgParams x; memset(&x, 0, sizeof(x));
  if (xchg) {
    xp->epoch += 1;
    x = *xp;
    *epoch += 2ULL * (unsigned long long)grid;               // two arrival rounds
    MARL_CUDA_TRY(launch_pdl(reduce_adam_kernel<1>, dim3(grid), dim3(pb * ns), 0, st, rp, ap, x, sp, pb, ns, barrier, *epoch));
  } else {
    *epoch += (unsigned long long)grid;
    MARL_CUDA_TRY(launch_pdl(reduce_adam_kernel<0>, dim3(grid), dim3(pb * ns), 0, st, rp, ap, x, sp, pb, ns, barrier, *epoch));
  }
  return MARL_OK;
}

// The exchange split over two launches (several ranks): launch_reduce_push, then whatever should hide the wait for the peers, then launch_adam_finish.
// barrier[0] counts the finishing kernel's grid-barrier arrivals, barrier[1] the pushing kernel's block arrivals (epoch / push_epoch: their values once
// the respective launch has fully arrived).
int launch_reduce_push(const ReduceParams& rp, const AdamParams& ap, XchgParams* xp, const SampleParams& sp, unsigned long long* barrier, unsigned long long* push_epoch,
                       int n_sm, cudaStream_t st) {
  const int n = rp.n_nets * rp.P;
  int pb = 0, ns = 0;
  if (xp == nullptr || xp->world <= 1 || ap.n != n || reduce_adam_shape(n, n_sm, true, &pb, &ns) != MARL_OK) return MARL_EINVAL;
  const int grid = (n + pb - 1) / pb;
  xp->epoch += 1;
  *push_epoch += (unsigned long long)grid;
  MARL_CUDA_TRY(launch_pdl(reduce_adam_kernel<2>, dim3(grid), dim3(pb * ns), 0, st, rp, ap, *xp, sp, pb, ns, barrier, *push_epoch));
  return MARL_OK;
}
int launch_adam_finish(const ReduceParams& rp, const AdamParams& ap, XchgParams* xp, unsigned long long* barrier, unsigned long long* epoch, int n_sm, cudaStream_t st) {
  const int n = rp.n_nets * rp.P;
  int pb = 0, ns = 0;
  if (xp == nullptr || xp->world <= 1 || reduce_adam_shape(n, n_sm, true, &pb, &ns) != MARL_OK) return MARL_EINVAL;
  const int grid = (n + pb - 1) / pb;
  SampleParams none; memset(&none, 0, sizeof(none));
  *epoch += (unsigned long long)grid;                          // one arrival round
  MARL_CUDA_TRY(launch_pdl(reduce_adam_kernel<3>, dim3(grid), dim3(pb * ns), 0, st, rp, ap, *xp, none, pb, ns, barrier, *epoch));
  return MARL_OK;
}

int launch_adam(const AdamParams& p, cudaStream_t st) {
  MARL_CUDA_TRY(launch_pdl(adam_kernel, dim3((p.n + 255) / 256), dim3(256), 0, st, p));
  return MARL_OK;
}

}  // namespace marl
