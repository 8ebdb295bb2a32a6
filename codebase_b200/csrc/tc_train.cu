// tc_train.cu -- tensor-core (tcgen05 / TMEM, 3xTF32) training pass of the DQN-family learner as a three-kernel pipeline.
//
// Same arithmetic as train_kernel<KP, kHeadDqn> (QNetwork._compute_loss + backward, marlbase/dqn/model.py:118-168), split where
// one SM's shared memory / TMEM cannot hold every operand twice (hi / lo) at once (DESIGN.md section 6):
//   tc_dqn_fwd_kernel   online forward (A operand in TMEM, weights = K-major image), TD head in registers; stores H1, H2 (FP32,
//                        chunk-major), the gathered observation row and one 64-byte record per row: dLoss/dq[act], act, ReLU masks of H1 / H2
//   tc_dh1_kernel       dH1 = (dH2 x W2) * relu'(H1); dH2[r][j] = g_r W3[act_r][j] relu'(H2[r][j]) is rebuilt from the record (the TD
//                        loss touches one output per row), so it never travels through memory; B = K-major image of W2^T
//   tc_dw_kernel        dW2 | db2 and dW1 | db1: row-streaming TN GEMMs, both operands MN-major from shared memory, accumulators
//                        resident in TMEM across all the CTA's rows; dW3 / db3 (one non-zero dq per row) accumulate in FP32 registers.
//                        16 producer warps stage 16-row chunks into a two-deep ring, a 17th warp issues the MMAs (mbarrier ring)
// The partials feed the same grad_reduce_kernel / adam_kernel as the FP32 path.
#include "tc_common.cuh"

namespace marl {

__device__ __forceinline__ size_t dst_of(const RowPlan& plan, const RowSource& src, int net, int vr, int& agent, int& unit, int& off) {
  decode_row(plan, net, vr, agent, unit, off);
  return src.mode == 0 ? ((size_t)unit * src.N + agent) : (((size_t)agent * plan.units_per_agent + unit) * plan.unit_rows + off);
}

// issue helpers (one thread): 3xTF32, TS form, compile-time unrolled
template <int KSTEPS, int N, int PANEL_BYTES>
__device__ __forceinline__ void issue_kmajor(uint32_t tmem, uint32_t d_col, uint32_t b_hi, uint32_t b_lo, int ksteps_rt) {
  const uint32_t idesc = idesc_tf32(N);
  const uint64_t dhi = kmajor_desc(b_hi), dlo = kmajor_desc(b_lo);
#pragma unroll
  for (int term = 0; term < 3; ++term)
#pragma unroll
    for (int ks = 0; ks < KSTEPS; ++ks)
      if (ks < ksteps_rt)
        mma_tf32_ts(tmem + d_col, tmem + (term == 0 ? kColALo : kColAHi) + ks * 8,
                    (term == 1 ? dlo : dhi) + (uint32_t)(((ks >> 2) * PANEL_BYTES + (ks & 3) * 32) >> 4), idesc, (term | ks) ? 1u : 0u);
}

__device__ __forceinline__ void split16(const float (&h)[16], float (&hi)[16], float (&lo)[16]) {
#pragma unroll
  for (int j = 0; j < 16; ++j) { hi[j] = tf32_rn(h[j]); lo[j] = tf32_rn(h[j] - hi[j]); }
}

// =====================================================================================================================
// Thread layout of the first two kernels: 16 warps.  Warp w works on TMEM lane quarter lq = w & 3 (the hardware restricts a warp to
// lanes 32 (w % 4) .. +31) and on column quarter cq = w >> 2 of the 128 hidden features, so every SM sub-partition holds four
// warps whose TMEM / global latencies overlap (with one warp per sub-partition the kernels sat at 15 % issue utilisation).
// =====================================================================================================================
// 1. online forward + TD head
// =====================================================================================================================
TSG_DEFINE(g_ts_fwd)
TSG_GETTER(tsg_fwd, g_ts_fwd)
TSG_DEFINE(g_ts_dh1)
TSG_GETTER(tsg_dh1, g_ts_dh1)
TSG_DEFINE(g_ts_dw)
TSG_GETTER(tsg_dw, g_ts_dw)
__global__ void __launch_bounds__(kTrThreads, 1) tc_dqn_fwd_kernel(TcTrainParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kImageBytes);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
  float* qs = reinterpret_cast<float*>(smem + kImageBytes + 64);   // [128][8] outputs of this tile, then loss reduction scratch
  float* carry = qs + kTileRows * kOutPad;                         // [8] outputs of the first row of the previously processed (higher) tile
  const int t = threadIdx.x, warp = t >> 5, lq = warp & 3, cq = warp >> 2, r = 32 * lq + (t & 31), c0 = 32 * cq;
  int net, row_begin, row_end;
  cta_rows(p.plan, net, row_begin, row_end);
  float st[2] = {0.f, 0.f};
  if (row_begin >= row_end) {
    pdl_wait();
    if (t < 4) p.loss_part[4 * blockIdx.x + t] = 0.f;
    return;
  }
  TSG(g_ts_fwd, 0);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (t == 0) { mbar_init(bar, 1); mbar_init(bar + 2, 1); mbar_init(bar + 3, 1); mbar_init(bar + 4, 1); fence_mbar_init(); }
  pdl_wait();   // nothing above touches global memory
  pdl_launch_dependents();
  TSG(g_ts_fwd, 1);
  // the weight image is already in shared-memory layout: three TMA bulk copies (cp.async.bulk -> mbarrier, issued by one thread) in the
  // order the first tile needs them (W1 + biases, W2, W3), so that its first layer does not wait for the whole image
  // (without the tensor-core operand copies of W3: the head runs on the CUDA cores against the FP32 copy; their 16 KB hold the head partials)
  if (t == 0) tma_forward_image_nohead(smem_u32(smem), p.images + (size_t)net * kImageBytes, bar + 2);
  const float* b1 = reinterpret_cast<const float*>(smem + kOffB1);
  const float* b2 = reinterpret_cast<const float*>(smem + kOffB2);
  const float* b3 = reinterpret_cast<const float*>(smem + kOffB3);
  const float4* w3f = reinterpret_cast<const float4*>(smem + kOffW3F);
  float* part = reinterpret_cast<float*>(smem + kOffW3Hi);   // [3][128 rows][8]: head partials of column quarters 1..3
  const int D = p.src.D, A = p.lay.out, T = p.src.traj.T, B = p.plan.units_per_agent;
  const int k1steps = (D + 7) >> 3;
  const bool x_active = cq < k1steps;   // column quarter cq stages observation columns [8 cq, 8 cq + 8)

  // This thread's row of a tile is fetched one tile ahead, in two steps so that no step waits on a load it has just issued:
  // A = decode + the episode index of the sampled unit, B (issued a barrier later) = observation columns and loss-head scalars.
  struct RowKey { size_t dst; int agent, b, tt, ep; bool valid; };
  struct RowIn { size_t dst; int agent, b, tt, act; float rew; uint8_t filled, done1; float x[8]; };
  auto fetch_a = [&](int vr0, int nrows, RowKey& k) {
    k.dst = 0; k.agent = 0; k.b = 0; k.tt = 0; k.ep = 0; k.valid = r < nrows;
    if (k.valid) {
      k.dst = dst_of(p.plan, p.src, net, vr0 + r, k.agent, k.b, k.tt);
      if (p.src.mode != 0) k.ep = p.src.idx[k.b];
    }
  };
  auto fetch_b = [&](const RowKey& k, RowIn& ri) {
    ri.dst = k.dst; ri.agent = k.agent; ri.b = k.b; ri.tt = k.tt; ri.act = 0; ri.rew = 0.f; ri.filled = 0; ri.done1 = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) ri.x[j] = 0.f;
    if (k.valid) {
      const TrajView& tv = p.src.traj;
      const float* src = p.src.mode == 0 ? p.src.dense + ((size_t)k.b * p.src.N + k.agent) * D
                                         : tv.obs + (((size_t)k.ep * tv.N + k.agent) * (size_t)(T + 1) + k.tt) * D;
      if (x_active) {
#pragma unroll
        for (int j = 0; j < 8; ++j) ri.x[j] = (8 * cq + j < D) ? src[8 * cq + j] : 0.f;
      }
      if (cq == 0 && p.src.mode != 0 && k.tt < T) {
        const size_t ep = (size_t)k.ep;
        ri.act = tv.act[(ep * tv.N + k.agent) * T + k.tt];
        ri.rew = tv.rew[(ep * tv.N + k.agent) * T + k.tt];
        ri.filled = tv.filled[ep * T + k.tt];   // raw bytes: a conversion here would wait for the loads inside the prefetch
        ri.done1 = tv.done[ep * (T + 1) + k.tt + 1];
      }
    }
  };
  RowKey key_nxt;
  RowIn cur, nxt;
  {
    const int v0 = max(row_begin, row_end - kTileRows);
    fetch_a(v0, row_end - v0, key_nxt);
    fetch_b(key_nxt, cur);
  }
  nxt = cur;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot, smem_base = smem_u32(smem), lane_base = tmem + ((uint32_t)(32 * lq) << 16);
  TSG(g_ts_fwd, 2);
  int ts_tile = 0; (void)ts_tile;
  int image_groups_pending = 2;   // block-uniform: groups not yet waited for (W1 + biases + FP32 W3, then W2)
  uint32_t parity = 0;
  float carry_q[kOutPad];         // thread 0: outputs of row 0 of the tile just finished, published after the next barrier
#pragma unroll
  for (int o = 0; o < kOutPad; ++o) carry_q[o] = 0.f;

  // tiles from the top of the chunk downwards (the double-Q argmax needs the next row's outputs)
  for (int vr_hi = row_end; vr_hi > row_begin; vr_hi -= kTileRows) {
    const int vr0 = max(row_begin, vr_hi - kTileRows), nrows = vr_hi - vr0;
    const bool has_next = vr0 > row_begin;
    if (has_next) { const int nv0 = max(row_begin, vr0 - kTileRows); fetch_a(nv0, vr0 - nv0, key_nxt); }
    if (x_active) {
      float hi[8], lo[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { hi[j] = tf32_rn(cur.x[j]); lo[j] = tf32_rn(cur.x[j] - hi[j]); }
      tmem_st8(lane_base + kColAHi + 8 * cq, hi);
      tmem_st8(lane_base + kColALo + 8 * cq, lo);
      if (r < nrows) {
        float4* xo = reinterpret_cast<float4*>(p.xg + cur.dst * kTcObsDim + 8 * cq);
        xo[0] = make_float4(cur.x[0], cur.x[1], cur.x[2], cur.x[3]); xo[1] = make_float4(cur.x[4], cur.x[5], cur.x[6], cur.x[7]);
      }
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    if (image_groups_pending == 2) { mbar_wait(bar + 2, 0); image_groups_pending = 1; }   // W1 + biases + FP32 W3 have landed
    tc_fence_before();
    __syncthreads();
    TSG(g_ts_fwd, 3 + 6 * ts_tile);
    if (t == 0) {
      tc_fence_after();
      issue_kmajor<kTcObsDim / 8, kHidden, kPanelBytes>(tmem, kColD, smem_base + kOffW1Hi, smem_base + kOffW1Lo, k1steps);
      mma_commit(bar);
      if (vr_hi != row_end) {   // every thread is past the previous tile's TD head: publish its first row's outputs
#pragma unroll
        for (int o = 0; o < kOutPad; ++o) carry[o] = carry_q[o];
      }
    }
    const size_t dst_row = cur.dst;
    const int agent = cur.agent, b = cur.b, tt = cur.tt, act = cur.act;
    const float rew = cur.rew; const uint8_t filled_u8 = cur.filled, done1_u8 = cur.done1;
    mbar_wait(bar, parity); parity ^= 1;
    tc_fence_after();
    TSG(g_ts_fwd, 4 + 6 * ts_tile);
    // ---- layer-1 epilogue: bias + ReLU -> H1 (FP32, chunk-major) + its mask -> global; 3xTF32 split -> the A operand of layer 2 ---------------
    {
      const float* bias = b1 + c0;
      float4* hg = reinterpret_cast<float4*>(p.h1g) + dst_row;
      uint32_t ra[16], rb[16];
      tmem_ld16_issue(lane_base + kColD + c0, ra);
      tmem_ld16_issue(lane_base + kColD + c0 + 16, rb);
      tmem_ld_wait(ra);
      tmem_ld_wait(rb);
      uint32_t mask = 0;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t (&acc)[16] = half ? rb : ra;
        float h[16], hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          h[j] = fmaxf(__uint_as_float(acc[j]) + bias[16 * half + j], 0.f);
          mask |= (h[j] > 0.f ? 1u : 0u) << (16 * half + j);
        }
        split16(h, hi, lo);
        tmem_st16(lane_base + kColAHi + c0 + 16 * half, hi);
        tmem_st16(lane_base + kColALo + c0 + 16 * half, lo);
        if (r < nrows) {
#pragma unroll
          for (int j = 0; j < 4; ++j) hg[(size_t)(8 * cq + 4 * half + j) * p.rows] = make_float4(h[4 * j], h[4 * j + 1], h[4 * j + 2], h[4 * j + 3]);
        }
      }
      if (r < nrows) reinterpret_cast<uint32_t*>(p.rec + dst_row * kRowRec)[4 + cq] = mask;   // ReLU mask of H1
      if (image_groups_pending == 1) { mbar_wait(bar + 3, 0); image_groups_pending = 0; }   // W2
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      tc_fence_before();
      __syncthreads();
      TSG(g_ts_fwd, 5 + 6 * ts_tile);
      if (t == 0) {
        tc_fence_after();
        issue_kmajor<kHidden / 8, kHidden, kPanelBytes>(tmem, kColD, smem_base + kOffW2Hi, smem_base + kOffW2Lo, kHidden / 8);
        mma_commit(bar);
      }
      // the next (lower) tile's rows, requested under the layer-2 MMAs (the longest stretch in which the CUDA cores idle); the episode index they
      // hang off was requested at the top of this tile
      if (has_next) fetch_b(key_nxt, nxt);
      mbar_wait(bar, parity); parity ^= 1;
      tc_fence_after();
      TSG(g_ts_fwd, 6 + 6 * ts_tile);
    }
    // ---- layer-2 epilogue: H2 (FP32, chunk-major) + its mask -> global; head on the CUDA cores against the FP32 copy of W3 (packed FP32: even and
    // odd columns accumulate in the two halves of a register pair); partial sums of column quarters 1..3 -> shared --------------------------------
    float q[kOutPad];
    {
      uint32_t ra[16], rb[16];
      tmem_ld16_issue(lane_base + kColD + c0, ra);
      tmem_ld16_issue(lane_base + kColD + c0 + 16, rb);
      tmem_ld_wait(ra);
      tmem_ld_wait(rb);
      float2 q2[kOutPad];
#pragma unroll
      for (int a = 0; a < kOutPad; ++a) q2[a] = make_float2(0.f, 0.f);
      uint32_t mask = 0;
      float4* hg = reinterpret_cast<float4*>(p.h2g) + dst_row;
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        const uint32_t (&acc)[16] = g < 4 ? ra : rb;
        const int o = 4 * (g & 3);
        const float4 bb = *reinterpret_cast<const float4*>(b2 + c0 + 4 * g);
        float2 h01 = __fadd2_rn(make_float2(__uint_as_float(acc[o]), __uint_as_float(acc[o + 1])), make_float2(bb.x, bb.y));
        float2 h23 = __fadd2_rn(make_float2(__uint_as_float(acc[o + 2]), __uint_as_float(acc[o + 3])), make_float2(bb.z, bb.w));
        h01.x = fmaxf(h01.x, 0.f); h01.y = fmaxf(h01.y, 0.f); h23.x = fmaxf(h23.x, 0.f); h23.y = fmaxf(h23.y, 0.f);
        mask |= ((h01.x > 0.f ? 1u : 0u) | (h01.y > 0.f ? 2u : 0u) | (h23.x > 0.f ? 4u : 0u) | (h23.y > 0.f ? 8u : 0u)) << (4 * g);
        if (r < nrows) hg[(size_t)(8 * cq + g) * p.rows] = make_float4(h01.x, h01.y, h23.x, h23.y);
#pragma unroll
        for (int a = 0; a < kOutPad; ++a) {
          if (a < A) {
            const float4 w = w3f[a * (kHidden / 4) + (c0 >> 2) + g];
            q2[a] = __ffma2_rn(h23, make_float2(w.z, w.w), __ffma2_rn(h01, make_float2(w.x, w.y), q2[a]));
          }
        }
      }
      if (r < nrows) reinterpret_cast<uint32_t*>(p.rec + dst_row * kRowRec)[8 + cq] = mask;   // ReLU mask of H2
#pragma unroll
      for (int a = 0; a < kOutPad; ++a) q[a] = q2[a].x + q2[a].y;
      if (cq > 0) {
        float4* pp = reinterpret_cast<float4*>(part + ((size_t)(cq - 1) * kTileRows + r) * kOutPad);
        pp[0] = make_float4(q[0], q[1], q[2], q[3]); pp[1] = make_float4(q[4], q[5], q[6], q[7]);
      }
      named_bar_sync(2 + lq, 128);   // the four warps of this lane quarter; the next tile's partials are written two __syncthreads later
      TSG(g_ts_fwd, 7 + 6 * ts_tile);
    }
    // ---- outputs of this tile -> shared (next-row exchange), TD head: column quarter 0 (threads 0..127, r == t) ------------
    if (cq == 0) {
#pragma unroll
      for (int o = 0; o < kOutPad; ++o)
        q[o] = o < A ? (((q[o] + part[((size_t)0 * kTileRows + r) * kOutPad + o]) + part[((size_t)1 * kTileRows + r) * kOutPad + o]) + part[((size_t)2 * kTileRows + r) * kOutPad + o]) + b3[o] : 0.f;
      *reinterpret_cast<float4*>(qs + r * kOutPad) = make_float4(q[0], q[1], q[2], q[3]);
      *reinterpret_cast<float4*>(qs + r * kOutPad + 4) = make_float4(q[4], q[5], q[6], q[7]);
      if (t == 0) {
#pragma unroll
        for (int o = 0; o < kOutPad; ++o) carry_q[o] = q[o];
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");   // the four warps of column quarter 0 exchange their rows' outputs
      if (r < nrows) {
        float g = 0.f;
        if (p.q_out) for (int o = 0; o < A; ++o) p.q_out[dst_row * A + o] = q[o];
        if (tt < T) {
          if (p.td_ext) {
            g = p.td_ext[(size_t)agent * p.td_agent_stride + (size_t)b * T + tt];
          } else {
            const float* qn = (r + 1 < nrows) ? (qs + (r + 1) * kOutPad) : carry;
            const float* tq = p.tq + (((size_t)agent * B + b) * (T + 1) + tt + 1) * A;
            float tsel;
            if (p.double_q) {
              int best = 0; float bv = qn[0];
              for (int o = 1; o < A; ++o) if (qn[o] > bv) { bv = qn[o]; best = o; }
              tsel = tq[best];
            } else {
              tsel = tq[0];
              for (int o = 1; o < A; ++o) tsel = fmaxf(tsel, tq[o]);
            }
            const float filled = (float)filled_u8, done1 = (float)done1_u8;
            const float y = rew + p.gamma * tsel * (1.f - done1);
            float qa = q[0];
#pragma unroll
            for (int o = 1; o < kOutPad; ++o) qa = (o == act) ? q[o] : qa;
            const float delta = qa - y;
            st[0] += delta * delta * filled;
            if (agent == 0) st[1] += filled;
            g = 2.f * delta * filled;
          }
        }
        // the TD loss touches one output per row: dq[r][a] = g (a == act), 0 otherwise; rows at t == T carry g = 0
        *reinterpret_cast<int2*>(p.rec + dst_row * kRowRec) = make_int2(__float_as_int(g), act);
      }
    }
    TSG(g_ts_fwd, 8 + 6 * ts_tile);
    ts_tile += 1;
    cur = nxt;
  }
  TSG(g_ts_fwd, 29);
  // ---- per-CTA loss statistics (threads 0..127 hold them) ---------------------------------------------------------------
  __syncthreads();
  if (t < kTileRows) { qs[t] = st[0]; qs[kTileRows + t] = st[1]; }
  __syncthreads();
  for (int s = kTileRows / 2; s > 0; s >>= 1) {
    if (t < s) { qs[t] += qs[t + s]; qs[kTileRows + t] += qs[kTileRows + t + s]; }
    __syncthreads();
  }
  if (t < 4) p.loss_part[4 * blockIdx.x + t] = t < 2 ? qs[t * kTileRows] : 0.f;
  tc_fence_before();
  __syncthreads();
  TSG(g_ts_fwd, 30);
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
  TSG(g_ts_fwd, 31);
}

// =====================================================================================================================
// 2. dH1 = (dH2 x W2) * relu'(H1), dH2 rebuilt from the row records
// =====================================================================================================================
constexpr int kDh1W3 = kBwdImageBytes;                        // FP32 copy of W3 [8][128] behind the W2^T image
constexpr int kDh1Bar = kDh1W3 + kOutPad * kHidden * 4;

__global__ void __launch_bounds__(kTrThreads, 1) tc_dh1_kernel(TcTrainParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kDh1Bar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
  const float4* w3f4 = reinterpret_cast<const float4*>(smem + kDh1W3);
  const int t = threadIdx.x, warp = t >> 5, lq = warp & 3, cq = warp >> 2, r = 32 * lq + (t & 31), c0 = 32 * cq;
  int net, row_begin, row_end;
  cta_rows(p.plan, net, row_begin, row_end);
  if (row_begin >= row_end) { pdl_wait(); return; }
  TSG(g_ts_dh1, 0);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (t == 0) { mbar_init(bar, 1); mbar_init(bar + 2, 1); fence_mbar_init(); }
  pdl_wait();   // nothing above touches global memory
  pdl_launch_dependents();
  TSG(g_ts_dh1, 1);
  if (t == 0) {  // W2^T image + FP32 W3: TMA bulk copies onto one mbarrier
    mbar_expect_tx(bar + 2, (uint32_t)(kBwdImageBytes + kOutPad * kHidden * 4));
    tma_image_range(smem_u32(smem), p.bwd_images + (size_t)net * kBwdImageBytes, 0, kBwdImageBytes, bar + 2);
    tma_bulk_g2s(smem_u32(smem) + kDh1W3, p.images + (size_t)net * kImageBytes + kOffW3F, kOutPad * kHidden * 4, bar + 2);
  }
  // this thread's row record: dLoss/dq[act], act and the two mask words of its 32 columns; fetched one tile ahead
  struct Rec { long long d; float g; int act; uint32_t m1, m2; };
  auto fetch = [&](int vr0, Rec& rc) {
    rc.d = -1; rc.g = 0.f; rc.act = 0; rc.m1 = 0; rc.m2 = 0;
    if (vr0 + r < row_end) {
      int a, u, o;
      rc.d = (long long)dst_of(p.plan, p.src, net, vr0 + r, a, u, o);
      const float* rp = p.rec + rc.d * kRowRec;
      const int2 ga = *reinterpret_cast<const int2*>(rp);
      rc.g = __int_as_float(ga.x); rc.act = ga.y;
      rc.m1 = reinterpret_cast<const uint32_t*>(rp)[4 + cq];
      rc.m2 = reinterpret_cast<const uint32_t*>(rp)[8 + cq];
    }
  };
  Rec cur, nxt;
  fetch(row_begin, cur);
  nxt = cur;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  TSG(g_ts_dh1, 2);
  int ts_tile = 0; (void)ts_tile;
  mbar_wait(bar + 2, 0);   // images have landed (every thread reads the FP32 W3 rows; the tensor core reads W2^T)
  const uint32_t tmem = *tmem_slot, smem_base = smem_u32(smem), lane_base = tmem + ((uint32_t)(32 * lq) << 16);
  uint32_t parity = 0;
  for (int vr0 = row_begin; vr0 < row_end; vr0 += kTileRows) {
    TSG(g_ts_dh1, 3 + 4 * ts_tile);
    // dH2[r][j] = g W3[act][j] (H2[r][j] > 0) for this thread's 32 columns -> A operand (hi / lo)
    {
      const float4* wrow = w3f4 + cur.act * (kHidden / 4) + 8 * cq;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        float v[16], hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 w = wrow[4 * half + j];
          const uint32_t m = cur.m2 >> (16 * half + 4 * j);
          v[4 * j] = (m & 1u) ? cur.g * w.x : 0.f; v[4 * j + 1] = (m & 2u) ? cur.g * w.y : 0.f;
          v[4 * j + 2] = (m & 4u) ? cur.g * w.z : 0.f; v[4 * j + 3] = (m & 8u) ? cur.g * w.w : 0.f;
        }
        split16(v, hi, lo);
        tmem_st16(lane_base + kColAHi + c0 + 16 * half, hi);
        tmem_st16(lane_base + kColALo + c0 + 16 * half, lo);
      }
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    TSG(g_ts_dh1, 4 + 4 * ts_tile);
    if (t == 0) {
      tc_fence_after();
      // D[r][j1] = sum_{j2} dH2[r][j2] W2[j2][j1]: B = K-major image of W2^T (rows j1, features j2), the forward layers' MMA form
      issue_kmajor<kHidden / 8, kHidden, kPanelBytes>(tmem, kColD, smem_base, smem_base + 4 * kPanelBytes, kHidden / 8);
      mma_commit(bar);
    }
    if (vr0 + kTileRows < row_end) fetch(vr0 + kTileRows, nxt);
    mbar_wait(bar, parity); parity ^= 1;
    tc_fence_after();
    TSG(g_ts_dh1, 5 + 4 * ts_tile);
    {
      uint32_t ra[16], rb[16];
      tmem_ld16_issue(lane_base + kColD + c0, ra);
      tmem_ld16_issue(lane_base + kColD + c0 + 16, rb);
      tmem_ld_wait(ra);
      tmem_ld_wait(rb);
      if (cur.d >= 0) {
        float4* gout = reinterpret_cast<float4*>(p.dh1g) + cur.d;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          uint32_t (&acc)[16] = j < 4 ? ra : rb;
          const int o = 4 * (j & 3);
          const uint32_t m = cur.m1 >> (4 * j);
          float4 d;
          d.x = (m & 1u) ? __uint_as_float(acc[o]) : 0.f; d.y = (m & 2u) ? __uint_as_float(acc[o + 1]) : 0.f;
          d.z = (m & 4u) ? __uint_as_float(acc[o + 2]) : 0.f; d.w = (m & 8u) ? __uint_as_float(acc[o + 3]) : 0.f;
          gout[(size_t)(8 * cq + j) * p.rows] = d;
        }
      }
    }
    TSG(g_ts_dh1, 6 + 4 * ts_tile);
    ts_tile += 1;
    cur = nxt;
  }
  tc_fence_before();
  __syncthreads();
  TSG(g_ts_dh1, 31);
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// =====================================================================================================================
// 3. weight gradients: row-streaming TN GEMMs, accumulators in TMEM
// =====================================================================================================================
constexpr int kDwProducers = 512;                    // 16 staging warps
constexpr int kDwThreads = kDwProducers + 32;        // + the MMA-issuing warp
constexpr int kChunkRows = 16;                       // rows per staged chunk (two 8-row k-steps)
#ifndef MARL_DW_BUFS
#define MARL_DW_BUFS 3
#endif
constexpr int kDwBufs = MARL_DW_BUFS;                // depth of the chunk ring (and of the register prefetch): the producers run that many chunks ahead of the tensor core
constexpr int kChunkPanel = kChunkRows * 128;        // one 32-feature panel of a chunk
constexpr int kOpBytes = 4 * kChunkPanel;            // a [16 rows][128 features] operand (hi or lo)
// shared-memory map of one chunk buffer (bytes): dH2 hi|lo, H1 hi (+ ones panel) | lo (+ zero panel), dH1 hi|lo, X hi|lo
constexpr int kSDh2 = 0, kSH1 = kSDh2 + 2 * kOpBytes, kSDh1 = kSH1 + 2 * (kOpBytes + kChunkPanel), kSX = kSDh1 + 2 * kOpBytes;
constexpr int kSEnd = kSX + 2 * kChunkPanel;
constexpr int kDwW3 = kDwBufs * kSEnd;                         // FP32 copy of W3 [8][128]
constexpr int kDwBars = kDwW3 + kOutPad * kHidden * 4;         // full[kDwBufs], empty[kDwBufs], done, TMEM slot
constexpr int kDwSmemBytes = kDwBars + 64 + 1024;              // + alignment slack
static_assert(kSEnd % 1024 == 0, "chunk buffers must keep the 1024-byte swizzle alignment");
static_assert(kDwBufs >= 2 && kDwBufs <= 3 && kDwSmemBytes <= 227 * 1024, "chunk ring: 2 or 3 buffers of 56 KB");
// epilogue scratch (the chunk buffers are dead by then): dW3 / db3 partials of the four row groups, then one transpose tile per warp
constexpr int kDwRed3 = 0, kDwRedG = kDwRed3 + 4 * kOutPad * kHidden * 4, kDwTile = kDwRedG + 1024, kDwTileBytes = 32 * 33 * 4;
static_assert(kDwTile + 16 * kDwTileBytes <= kDwBufs * kSEnd, "epilogue scratch must fit in the chunk buffers");
// TMEM columns: dW2 | db2 [0,160), dW1 | db1 [160,192)
constexpr uint32_t kColW2 = 0, kColW1 = 160;

__device__ __forceinline__ void stage4(uint8_t* hi_img, uint8_t* lo_img, int r, int col, float4 v) {
  float4 h, l;
  h.x = tf32_rn(v.x); h.y = tf32_rn(v.y); h.z = tf32_rn(v.z); h.w = tf32_rn(v.w);
  l.x = tf32_rn(v.x - h.x); l.y = tf32_rn(v.y - h.y); l.z = tf32_rn(v.z - h.z); l.w = tf32_rn(v.w - h.w);
  const int off = mn_offset(r, col, kChunkPanel);
  *reinterpret_cast<float4*>(hi_img + off) = h;
  *reinterpret_cast<float4*>(lo_img + off) = l;
}

__global__ void __launch_bounds__(kDwThreads, 1) tc_dw_kernel(TcTrainParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + kDwBars);   // [kDwBufs] chunk buffer staged (16 producer-warp arrivals)
  uint64_t* empty = full + kDwBufs;                               // [kDwBufs] chunk buffer consumed by the tensor core (tcgen05.commit)
  uint64_t* done = full + 2 * kDwBufs;                            // every MMA retired
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(full + 2 * kDwBufs + 1);
  const float4* w3f4 = reinterpret_cast<const float4*>(smem + kDwW3);
  // staging: warp = (4-row group, 32-feature panel), lane = (float4 column within the panel, row within the group): shared-memory
  // stores of the swizzled MN-major image stay conflict-free and every global load instruction reads eight 64-byte segments
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31, rr = 4 * ((warp >> 2) & 3) + (lane & 3), c4 = 8 * (warp & 3) + (lane >> 2);
  const bool producer = warp < kDwProducers / 32;
  int net, row_begin, row_end;
  cta_rows(p.plan, net, row_begin, row_end);
  float* gs = p.scratch + (size_t)blockIdx.x * p.scratch_pitch;
  if (row_begin >= row_end) {
    pdl_wait();
    for (int i = t; i < p.lay.P; i += kDwThreads) gs[i] = 0.f;
    return;
  }
  TSG(g_ts_dw, 0);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(256));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (t == 0) {
    for (int b = 0; b < kDwBufs; ++b) { mbar_init(full + b, kDwProducers / 32); mbar_init(empty + b, 1); }   // one arrival per producer warp
    mbar_init(done, 1);
  }
  // constant panels of every buffer: ones column (n = 128) behind H1 hi, zeros behind H1 lo; W3 copy
  for (int i = t; i < kDwBufs * (kChunkPanel / 4); i += kDwThreads) {
    uint8_t* bufp = smem + (i / (kChunkPanel / 4)) * kSEnd;
    const int w = i % (kChunkPanel / 4);
    reinterpret_cast<float*>(bufp + kSH1 + kOpBytes)[w] = 0.f;
    reinterpret_cast<float*>(bufp + kSH1 + 2 * kOpBytes + kChunkPanel)[w] = 0.f;
  }
  pdl_wait();   // nothing above touches global memory
  pdl_launch_dependents();
  TSG(g_ts_dw, 1);
  {
    const float4* w3src = reinterpret_cast<const float4*>(p.images + (size_t)net * kImageBytes + kOffW3F);
    for (int i = t; i < kOutPad * kHidden / 4; i += kDwThreads) reinterpret_cast<float4*>(smem + kDwW3)[i] = w3src[i];
  }
  __syncthreads();
  if (t < kDwBufs * kChunkRows) *reinterpret_cast<float*>(smem + (t / kChunkRows) * kSEnd + kSH1 + kOpBytes + mn_offset(t % kChunkRows, 0, kChunkPanel)) = 1.0f;
  const int D = p.src.D, A = p.lay.out;
  const int n_chunks = (row_end - row_begin + kChunkRows - 1) / kChunkRows, rpa = p.plan.units_per_agent * p.plan.unit_rows;
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot, sb = smem_u32(smem);
  TSG(g_ts_dw, 2);

  float acc3[kOutPad][4];   // dW3[a][4 c4 .. 4 c4 + 3] over this thread's rows; gacc: db3 (used where c4 == 0)
  float gacc[kOutPad];
#pragma unroll
  for (int a = 0; a < kOutPad; ++a) { gacc[a] = 0.f; acc3[a][0] = acc3[a][1] = acc3[a][2] = acc3[a][3] = 0.f; }

  if (producer) {
    // a chunk's data in registers: this thread's float4 of H1 / dH1 / H2, its element of the [16][32] X panel, its row's record
    struct Pre { float4 h1, dh1, h2; float xv, g; int act; uint32_t m2; };
    int slot = row_begin / rpa, slot_end = (slot + 1) * rpa;
    long long slot_delta = (long long)(p.plan.slot_agent[p.plan.slot_begin[net] + slot] - slot) * rpa;
    auto issue_loads = [&](int chunk, Pre& pre) {
      const int vr = row_begin + chunk * kChunkRows + rr;
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      pre.h1 = z; pre.dh1 = z; pre.h2 = z; pre.xv = 0.f; pre.g = 0.f; pre.act = 0; pre.m2 = 0;
      if (vr < row_end) {
        size_t d;
        if (p.src.mode == 0) { int a, u, o; d = dst_of(p.plan, p.src, net, vr, a, u, o); }
        else {  // dst_of() without its divisions: this thread's rows only move forward, the agent slot changes every rpa rows
          while (vr >= slot_end) { ++slot; slot_end += rpa; slot_delta = (long long)(p.plan.slot_agent[p.plan.slot_begin[net] + slot] - slot) * rpa; }
          d = (size_t)(vr + slot_delta);
        }
        const float* rp = p.rec + d * kRowRec;
        const int2 head = *reinterpret_cast<const int2*>(rp);   // g, act
        pre.g = __int_as_float(head.x); pre.act = head.y;
        pre.m2 = reinterpret_cast<const uint32_t*>(rp)[8 + (c4 >> 3)];
        const size_t hi = (size_t)c4 * p.rows + d;
        pre.h1 = reinterpret_cast<const float4*>(p.h1g)[hi];
        pre.dh1 = reinterpret_cast<const float4*>(p.dh1g)[hi];
        pre.h2 = reinterpret_cast<const float4*>(p.h2g)[hi];
        pre.xv = c4 < D ? p.xg[d * kTcObsDim + c4] : (c4 == D ? 1.f : 0.f);   // [X | 1]: the ones column carries db1
      }
    };
    auto stage = [&](uint8_t* bufp, const Pre& pre) {
      // dH2 = g W3[act][.] relu'(H2) for this thread's four columns
      const float4 w = w3f4[pre.act * (kHidden / 4) + c4];
      const uint32_t m = pre.m2 >> (4 * (c4 & 7));
      float4 dh2;
      dh2.x = (m & 1u) ? pre.g * w.x : 0.f; dh2.y = (m & 2u) ? pre.g * w.y : 0.f;
      dh2.z = (m & 4u) ? pre.g * w.z : 0.f; dh2.w = (m & 8u) ? pre.g * w.w : 0.f;
      stage4(bufp + kSDh2, bufp + kSDh2 + kOpBytes, rr, 4 * c4, dh2);
      stage4(bufp + kSH1, bufp + kSH1 + kOpBytes + kChunkPanel, rr, 4 * c4, pre.h1);
      stage4(bufp + kSDh1, bufp + kSDh1 + kOpBytes, rr, 4 * c4, pre.dh1);
      const float xh = tf32_rn(pre.xv);
      *reinterpret_cast<float*>(bufp + kSX + mn_offset(rr, c4, kChunkPanel)) = xh;
      *reinterpret_cast<float*>(bufp + kSX + kChunkPanel + mn_offset(rr, c4, kChunkPanel)) = tf32_rn(pre.xv - xh);
      // dW3[a][j] += dq[r][a] H2[r][j], db3[a] += dq[r][a]: dq[r][.] is g at act, 0 elsewhere -- FP32 registers
#pragma unroll
      for (int a = 0; a < kOutPad; ++a) {
        const float ga = a == pre.act ? pre.g : 0.f;
        gacc[a] += ga;
        acc3[a][0] = fmaf(ga, pre.h2.x, acc3[a][0]); acc3[a][1] = fmaf(ga, pre.h2.y, acc3[a][1]);
        acc3[a][2] = fmaf(ga, pre.h2.z, acc3[a][2]); acc3[a][3] = fmaf(ga, pre.h2.w, acc3[a][3]);
      }
    };
    // register prefetch two chunks ahead (global / L2 latency), shared-memory ring kDwBufs deep (tensor-core + barrier latency); the loop is
    // unrolled over lcm(2, kDwBufs) chunks so that both indices are compile-time constants (pre[] stays in registers)
    constexpr int kUnroll = 2 * kDwBufs / (kDwBufs % 2 == 0 ? 2 : 1);
    Pre pre[2];
    issue_loads(0, pre[0]);
    issue_loads(1, pre[1]);   // past the end: zeros, no loads
    for (int c0 = 0; c0 < n_chunks; c0 += kUnroll) {
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) {
        const int c = c0 + u, b = u % kDwBufs, use = c0 / kDwBufs + u / kDwBufs;   // chunk c is the use-th user of buffer b
        if (c < n_chunks) {
          if ((c & 1) == 0) TSG(g_ts_dw, 3 + (c >> 1));   // every second chunk (at most 24 chunks: slots 3..14)
          if (use > 0) mbar_wait(empty + b, (use - 1) & 1);   // its previous user (chunk c - kDwBufs) has been consumed by the tensor core
          stage(smem + b * kSEnd, pre[u & 1]);
          issue_loads(c + 2, pre[u & 1]);
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) mbar_arrive(full + b);   // 16 arrivals per chunk instead of 512 serialised shared-memory atomics
        }
      }
    }
  } else {
    // ---- MMA warp: per chunk 12 MMAs (3xTF32 terms x 2 k-steps x 2 GEMMs), then a commit that frees the buffer ----------------
    const uint32_t id_w2 = idesc_tf32_major(160, 1, 1), id_w1 = idesc_tf32_major(32, 1, 1);
    for (int c = 0, b = 0, round = 0; c < n_chunks; ++c) {
      mbar_wait(full + b, round & 1);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t base = sb + b * kSEnd;
#pragma unroll
        for (int term = 0; term < 3; ++term) {
          const uint32_t a_sel = term == 0 ? 1u : 0u, b_sel = term == 1 ? 1u : 0u;  // lo*hi, hi*lo, hi*hi
#pragma unroll
          for (int ks = 0; ks < kChunkRows / 8; ++ks) {
            const uint32_t ko = ks * 1024;
            const uint32_t accf = (c || term || ks) ? 1u : 0u;
            // dW2[j2][j1 | 1] += dH2^T x [H1 | 1]
            mma_tf32_ss(tmem + kColW2, mnmajor_desc(base + kSDh2 + a_sel * kOpBytes + ko, kChunkPanel),
                        mnmajor_desc(base + kSH1 + b_sel * (kOpBytes + kChunkPanel) + ko, kChunkPanel), id_w2, accf);
            // dW1[j1][i | 1] += dH1^T x [X | 1]
            mma_tf32_ss(tmem + kColW1, mnmajor_desc(base + kSDh1 + a_sel * kOpBytes + ko, kChunkPanel),
                        mnmajor_desc(base + kSX + b_sel * kChunkPanel + ko, kChunkPanel), id_w1, accf);
          }
        }
        mma_commit(empty + b);
        if (c == n_chunks - 1) mma_commit(done);   // completes when every MMA issued above has
      }
      __syncwarp();
      if (++b == kDwBufs) { b = 0; ++round; }
    }
  }
  TSG(g_ts_dw, 24);
  mbar_wait(done, 0);
  tc_fence_after();
  TSG(g_ts_dw, 25);
  __syncthreads();   // every producer is past its last use of the chunk buffers: they become epilogue scratch
  // ---- dW3 / db3: sum over the four rows of a lane group (shuffles), then over the four row groups (fixed order) ------------
  float* red3 = reinterpret_cast<float*>(smem + kDwRed3);   // [4 row groups][8][128]
  float* redg = reinterpret_cast<float*>(smem + kDwRedG);   // [4 row groups][8]
  if (producer) {
#pragma unroll
    for (int a = 0; a < kOutPad; ++a) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float v = acc3[a][i];
        v += __shfl_xor_sync(0xFFFFFFFFu, v, 1);
        v += __shfl_xor_sync(0xFFFFFFFFu, v, 2);
        acc3[a][i] = v;
      }
      float g = gacc[a];
      g += __shfl_xor_sync(0xFFFFFFFFu, g, 1);
      g += __shfl_xor_sync(0xFFFFFFFFu, g, 2);
      gacc[a] = g;
    }
    if ((lane & 3) == 0) {
      const int grp = (warp >> 2) & 3;
#pragma unroll
      for (int a = 0; a < kOutPad; ++a) {
        *reinterpret_cast<float4*>(red3 + (grp * kOutPad + a) * kHidden + 4 * c4) = make_float4(acc3[a][0], acc3[a][1], acc3[a][2], acc3[a][3]);
        if (c4 == 0) redg[grp * kOutPad + a] = gacc[a];
      }
    }
  }
  __syncthreads();
  for (int i = t; i < A * kHidden; i += kDwThreads)
    gs[p.lay.w3 + i] = (red3[i] + red3[kOutPad * kHidden + i]) + (red3[2 * kOutPad * kHidden + i] + red3[3 * kOutPad * kHidden + i]);
  if (t < A) gs[p.lay.b3 + t] = (redg[t] + redg[kOutPad + t]) + (redg[2 * kOutPad + t] + redg[3 * kOutPad + t]);
  TSG(g_ts_dw, 26);
  // ---- flush the TMEM accumulators: lane j of lane quarter lq owns output feature j; each warp transposes its 32 x 32 block of
  // dW2 through shared memory so that every store instruction writes one 128-byte row segment ------------------------------------
  if (producer) {
    const int lq = warp & 3, cq = warp >> 2, j = 32 * lq + lane;
    const uint32_t lane_base = tmem + ((uint32_t)(32 * lq) << 16);
    float* tile = reinterpret_cast<float*>(smem + kDwTile + warp * kDwTileBytes);   // [32][33]
    float v[16];
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      tmem_ld16(lane_base + kColW2 + 32 * cq + 16 * half, v);
#pragma unroll
      for (int i = 0; i < 16; ++i) tile[lane * 33 + 16 * half + i] = v[i];
    }
    __syncwarp();
    float* w2blk = gs + p.lay.w2 + (32 * lq) * kHidden + 32 * cq + lane;
#pragma unroll 8
    for (int i = 0; i < 32; ++i) w2blk[i * kHidden] = tile[i * 33 + lane];
    if (cq == 0) {
      tmem_ld16(lane_base + kColW2 + kHidden, v);
      gs[p.lay.b2 + j] = v[0];
    } else if (cq == 1) {
      float w_hi[16];
      tmem_ld16(lane_base + kColW1, v);
      tmem_ld16(lane_base + kColW1 + 16, w_hi);
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float x = i < 16 ? v[i & 15] : w_hi[i & 15];
        if (i < D) gs[p.lay.w1 + j * D + i] = x;
        else if (i == D) gs[p.lay.b1 + j] = x;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  TSG(g_ts_dw, 31);
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(256));
}

// =====================================================================================================================
// launchers
// =====================================================================================================================
constexpr int kFwdTrainSmem = kImageBytes + 64 + (kTileRows * kOutPad + kOutPad + 8) * 4 + 1024;
constexpr int kDh1Smem = kDh1Bar + 64 + 1024;

int tc_train_init() {
  MARL_CUDA_TRY(cudaFuncSetAttribute(tc_dqn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kFwdTrainSmem));
  MARL_CUDA_TRY(cudaFuncSetAttribute(tc_dh1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDh1Smem));
  MARL_CUDA_TRY(cudaFuncSetAttribute(tc_dw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDwSmemBytes));
  if (int rc = tc_train2_init()) return rc;
  return tc_train3_init();
}

// all three kernels walk the same episode-aligned row split, so the per-CTA partials line up with ReduceParams::cta_begin
int launch_tc_dqn_train(const TrainParams& tp, const TcBuffers& buf, cudaStream_t st, cudaEvent_t* between) {
  MARL_REQUIRE(tp.lay.in < kTcObsDim, "tensor-core backward: observation width %d needs a spare column for the bias trick (max %d)", tp.lay.in, kTcObsDim - 1);
  TcTrainParams p; memset(&p, 0, sizeof(p));
  p.plan = tp.plan; p.src = tp.src; p.lay = tp.lay; p.images = buf.image; p.bwd_images = buf.bwd_image; p.q_out = nullptr;
  p.h1g = buf.h1; p.h2g = buf.h2; p.dh1g = buf.dh1; p.rec = buf.rec; p.xg = buf.x; p.rows = buf.rows;
  p.tq = tp.tq; p.td_ext = tp.td_ext; p.td_agent_stride = tp.td_agent_stride; p.gamma = tp.gamma; p.double_q = tp.double_q;
  p.scratch = tp.scratch; p.scratch_pitch = tp.scratch_pitch; p.loss_part = tp.loss_part;
  const int grid = tp.plan.cta_begin[tp.plan.n_nets];
  p.dbg = tc_debug_progress_ptr();
  if (tc_onchip_enabled()) return launch_tc_dqn_train3(p, grid, st, between);
  const bool pp_fwd = tc_pingpong_enabled(0) && p.src.mode == 1, pp_dh1 = tc_pingpong_enabled(1) && p.src.mode == 1;   // two-accumulator kernels (tc_train2.cu)
  if (pp_fwd) { if (int rc = launch_tc_dqn_fwd2(p, grid, st)) return rc; }
  else MARL_CUDA_TRY(launch_pdl(tc_dqn_fwd_kernel, dim3(grid), dim3(kTrThreads), kFwdTrainSmem, st, p));
  if (between) MARL_CUDA_TRY(cudaEventRecord(between[0], st));
  if (pp_dh1) { if (int rc = launch_tc_dh12(p, grid, st)) return rc; }
  else MARL_CUDA_TRY(launch_pdl(tc_dh1_kernel, dim3(grid), dim3(kTrThreads), kDh1Smem, st, p));
  if (between) MARL_CUDA_TRY(cudaEventRecord(between[1], st));
  MARL_CUDA_TRY(launch_pdl(tc_dw_kernel, dim3(grid), dim3(kDwThreads), kDwSmemBytes, st, p));
  return MARL_OK;
}

}  // namespace marl
