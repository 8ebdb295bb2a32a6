// tc_train3.cu -- the tensor-core training pass of the DQN-family learner with the activations kept on chip (default; tc_train.cu is the previous
// form: "tensor_core_onchip" 0).  Same arithmetic as QNetwork._compute_loss + backward (marlbase/dqn/model.py:118-168) and the same per-CTA
// gradient partials / loss statistics as tc_train.cu, but H1, H2 and dH1 never travel through global memory (3 x 27 MB written and read back per
// update at batch 1024: the weight-gradient kernel was streaming 93 MB per launch from DRAM).  What crosses kernels is 192 bytes per row: the
// gathered observation row and the 64-byte row record (dLoss/dq[act], act, ReLU masks of H1 and H2).
//   tc_dqn_fwd3_kernel   online forward, TD head, row records.  dW3 | db3 = dq^T x [H2 | 1] on the CUDA cores: the layer-2 accumulator of a tile stays
//                        in TMEM (two accumulators alternate) and is read a second time, under the layer-2 MMAs of the NEXT tile, when the tile's
//                        dq is known; 32 x 8 transposes through shared memory turn "thread = row" into "thread = column" sums.
//   tc_dh1w1_kernel      dH1 = (dH2 x W2) * relu'(H1) as before (dH2 rebuilt from the record), but the masked accumulator goes straight into
//                        shared memory as the MN-major operand of dW1 | db1 += dH1^T x [X | 1] (32-row chunks, two buffers, a 17th warp issues).
//   tc_dw2_kernel        dW2 | db2 += dH2^T x [H1 | 1] with H1 RECOMPUTED from the gathered observation rows (one 128 x 128 x 16..32 product per
//                        tile: 1 % of the pass's FLOP) and dH2 rebuilt from the record; operands staged as 32-row MN-major chunks.
// The second and third kernels only depend on the first.
#include "tc_common.cuh"

namespace marl {

// ---- 32-row chunks of the weight-gradient operands, K-major ------------------------------------------------------------------------------------------
// dW = dOut^T x In contracts over the ROWS: K = row.  The operands are staged K-major (SWIZZLE_128B, the forward layers' form: one 128-byte line per
// feature holding the chunk's 32 rows, 16-byte chunk c of feature f at position c ^ (f & 7)) -- the MN-major form ([row][feature] lines,
// SWIZZLE_128B_BASE32B) that tc_train.cu uses needs a quarter of the store instructions but its MMAs ran at ~210 cycles (N = 160) instead of ~90.
// A thread owns one row (K index k = its lane) and 32 consecutive features: 32 scalar stores per copy; a warp's store of one feature covers the
// feature's whole 128-byte line (conflict-free).
constexpr int kC3Rows = 32;                       // rows per chunk = one TMEM lane quarter = four 8-row k-steps
constexpr int kC3Panel = 32 * 128;                // 32 features x 128 bytes: 4 KB
constexpr int kC3Op = 4 * kC3Panel;               // a [128 features][32 rows] operand (hi or lo): 16 KB
template <int NF>
__device__ __forceinline__ void stage_kmajor(uint8_t* hi_img, uint8_t* lo_img, int k, int f0, const float (&v)[NF]) {   // f0: a multiple of 8
  const int kq = k >> 2, kw = (k & 3) * 4;
  uint8_t* ph = hi_img + f0 * 128 + kw;
  uint8_t* pl = lo_img + f0 * 128 + kw;
#pragma unroll
  for (int j = 0; j < NF; ++j) {
    const int off = j * 128 + ((kq ^ (j & 7)) << 4);
    float hi, lo;
    tf32_split(v[j], hi, lo);
    *reinterpret_cast<float*>(ph + off) = hi;
    *reinterpret_cast<float*>(pl + off) = lo;
  }
}
__device__ __forceinline__ void stage_row32(uint8_t* hi_img, uint8_t* lo_img, int row, int panel, const float (&v)[32]) { stage_kmajor<32>(hi_img, lo_img, row, 32 * panel, v); }
__device__ __forceinline__ void stage_row8(uint8_t* hi_panel, uint8_t* lo_panel, int row, int unit, const float (&v)[8]) { stage_kmajor<8>(hi_panel, lo_panel, row, 8 * unit, v); }

__device__ __forceinline__ size_t dst_of3(const RowPlan& plan, const RowSource& src, int net, int vr, int& agent, int& unit, int& off) {
  decode_row(plan, net, vr, agent, unit, off);
  return src.mode == 0 ? ((size_t)unit * src.N + agent) : (((size_t)agent * plan.units_per_agent + unit) * plan.unit_rows + off);
}

TSG_DEFINE(g_ts_fwd3)
TSG_GETTER(tsg_fwd3, g_ts_fwd3)
TSG_DEFINE(g_ts_dh1w1)
TSG_GETTER(tsg_dh1w1, g_ts_dh1w1)
TSG_DEFINE(g_ts_dw2)
TSG_GETTER(tsg_dw2, g_ts_dw2)

// =====================================================================================================================
// 1. online forward + TD head + dW3 | db3.  16 warps: lane quarter lq = warp & 3, column quarter cq = warp >> 2 (tc_train.cu).
// TMEM: A hi [0,128) | A lo [128,256) | D0 [256,384) | D1 [384,512): tile k accumulates both layers in D(k & 1).
// =====================================================================================================================
constexpr int kF3Part = kOffW3Hi;                                   // head partials of column quarters 1..3: [3][128][8] floats (the unused W3 operand copies)
constexpr int kF3Bars = kImageBytes;                                // 64 bytes: mbarriers + TMEM slot
constexpr int kF3Qs = kF3Bars + 64;                                 // [128][8] outputs of this tile (next-row exchange), later the loss reduction scratch
constexpr int kF3Carry = kF3Qs + kTileRows * kOutPad * 4;           // [8] outputs of the first row of the previously processed (higher) tile
constexpr int kF3G = kF3Carry + 64;                                 // [128][8] dq of the tile just finished: G[r][a] = g_r (a == act_r), 0 otherwise
constexpr int kF3Tb = kF3G + kTileRows * kOutPad * 4;               // [16 warps][32 rows][16] transpose tiles (16-byte chunks XOR-swizzled by the row pair)
constexpr int kF3TbWarp = 32 * 16 * 4;
constexpr int kF3Db = kF3Tb + 16 * kF3TbWarp;                       // [4 lane quarters][8] db3 partial sums
constexpr int kF3Smem = kF3Db + 4 * kOutPad * 4 + 1024;
static_assert(kF3Smem <= 227 * 1024, "training forward: shared-memory map");
static_assert(16 * kF3TbWarp >= 4 * kOutPad * kHidden * 4, "the transpose tiles double as the final dW3 reduction scratch [4][8][128]");

__global__ void __launch_bounds__(kTrThreads, 1) tc_dqn_fwd3_kernel(TcTrainParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kF3Bars);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 5);
  float* qs = reinterpret_cast<float*>(smem + kF3Qs);
  float* carry = reinterpret_cast<float*>(smem + kF3Carry);
  float* Gs = reinterpret_cast<float*>(smem + kF3G);
  float* dbs = reinterpret_cast<float*>(smem + kF3Db);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31, lq = warp & 3, cq = warp >> 2, r = 32 * lq + lane, c0 = 32 * cq;
  float* tb = reinterpret_cast<float*>(smem + kF3Tb + warp * kF3TbWarp);
  int net, row_begin, row_end;
  cta_rows(p.plan, net, row_begin, row_end);
  float* gs = p.scratch + (size_t)blockIdx.x * p.scratch_pitch;
  const int A = p.lay.out;
  if (row_begin >= row_end) {
    pdl_wait();
    if (t < 4) p.loss_part[4 * blockIdx.x + t] = 0.f;
    for (int i = t; i < A * kHidden; i += kTrThreads) gs[p.lay.w3 + i] = 0.f;
    if (t < A) gs[p.lay.b3 + t] = 0.f;
    return;
  }
  TSGP(g_ts_fwd3, p.dbg, 0, 0);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (t == 0) { mbar_init(bar, 1); mbar_init(bar + 2, 1); mbar_init(bar + 3, 1); fence_mbar_init(); }
  if (t < 4 * kOutPad) dbs[t] = 0.f;
  pdl_wait();   // nothing above touches global memory
  pdl_launch_dependents();
  TSGP(g_ts_fwd3, p.dbg, 0, 1);
  if (t == 0) tma_forward_image_nohead(smem_u32(smem), p.images + (size_t)net * kImageBytes, bar + 2);
  const float* b1 = reinterpret_cast<const float*>(smem + kOffB1);
  const float* b2 = reinterpret_cast<const float*>(smem + kOffB2);
  const float* b3 = reinterpret_cast<const float*>(smem + kOffB3);
  const float4* w3f = reinterpret_cast<const float4*>(smem + kOffW3F);
  float* part = reinterpret_cast<float*>(smem + kF3Part);
  const int D = p.src.D, T = p.src.traj.T, B = p.plan.units_per_agent;
  const int k1steps = (D + 7) >> 3;
  const bool x_active = cq < k1steps;   // column quarter cq stages observation columns [8 cq, 8 cq + 8)

  // This thread's row of a tile is fetched one tile ahead, in two steps so that no step waits on a load it has just issued:
  // A = decode + the episode index of the sampled unit, B (issued under the layer-2 MMAs) = observation columns and loss-head scalars.
  struct RowKey { size_t dst; int agent, b, tt, ep; bool valid; };
  struct RowIn { size_t dst; int agent, b, tt, act; float rew; uint8_t filled, done1; float x[8]; };
  auto fetch_a = [&](int vr0, int nrows, RowKey& k) {
    k.dst = 0; k.agent = 0; k.b = 0; k.tt = 0; k.ep = 0; k.valid = r < nrows;
    if (k.valid) {
      k.dst = dst_of3(p.plan, p.src, net, vr0 + r, k.agent, k.b, k.tt);
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
  TSGP(g_ts_fwd3, p.dbg, 0, 2);
  int ts_tile = 0; (void)ts_tile;
  int image_groups_pending = 2;   // block-uniform: groups not yet waited for (W1 + biases + FP32 W3, then W2)
  uint32_t parity = 0;
  float st[2] = {0.f, 0.f};
  float carry_q[kOutPad];         // thread 0: outputs of row 0 of the tile just finished, published after the next barrier
  float acc3[kOutPad];            // dW3[a][c0 + lane] over the rows of this lane quarter, all tiles
#pragma unroll
  for (int o = 0; o < kOutPad; ++o) { carry_q[o] = 0.f; acc3[o] = 0.f; }

  // dW3 of a finished tile: its layer-2 accumulator (still in TMEM column block d_col) is read again, ReLU'd, and the 32 rows x 32 columns of this
  // warp are summed over the rows per action with the tile's dq (Gs).  Two passes of 16 columns: every lane writes its row's 16 values into a
  // [32][16] tile (float4 chunk c of row r at position c ^ ((r >> 1) & 3): stores and loads are bank-conflict free), then lane (column j = lane & 15,
  // row parity hsel = lane >> 4) adds its 16 rows against their dq rows (packed FP32), one shuffle adds the two parities, and lane 16 * pass + j
  // keeps column 16 * pass + j.
  auto dw3_tile = [&](uint32_t d_col) {
    uint32_t ra[16], rb[16];
    tmem_ld16_issue(lane_base + d_col + c0, ra);
    tmem_ld16_issue(lane_base + d_col + c0 + 16, rb);
    tmem_ld_wait(ra);
    tmem_ld_wait(rb);
    const int j = lane & 15, hsel = lane >> 4;
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const uint32_t (&acc)[16] = pass ? rb : ra;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float4 bb = *reinterpret_cast<const float4*>(b2 + c0 + 16 * pass + 4 * c);
        float4 h;
        h.x = fmaxf(__uint_as_float(acc[4 * c]) + bb.x, 0.f); h.y = fmaxf(__uint_as_float(acc[4 * c + 1]) + bb.y, 0.f);
        h.z = fmaxf(__uint_as_float(acc[4 * c + 2]) + bb.z, 0.f); h.w = fmaxf(__uint_as_float(acc[4 * c + 3]) + bb.w, 0.f);
        *reinterpret_cast<float4*>(tb + 16 * lane + 4 * (c ^ ((lane >> 1) & 3))) = h;
      }
      __syncwarp();
      float2 s2[kOutPad / 2];
#pragma unroll
      for (int a = 0; a < kOutPad / 2; ++a) s2[a] = make_float2(0.f, 0.f);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int rr = 2 * i + hsel;
        const float h = tb[16 * rr + 4 * ((j >> 2) ^ (i & 3)) + (j & 3)];
        const float2 hh = make_float2(h, h);
        const float4 g0 = *reinterpret_cast<const float4*>(Gs + (32 * lq + rr) * kOutPad), g1 = *reinterpret_cast<const float4*>(Gs + (32 * lq + rr) * kOutPad + 4);
        s2[0] = __ffma2_rn(make_float2(g0.x, g0.y), hh, s2[0]); s2[1] = __ffma2_rn(make_float2(g0.z, g0.w), hh, s2[1]);
        s2[2] = __ffma2_rn(make_float2(g1.x, g1.y), hh, s2[2]); s2[3] = __ffma2_rn(make_float2(g1.z, g1.w), hh, s2[3]);
      }
#pragma unroll
      for (int a = 0; a < kOutPad / 2; ++a) {
        const float x = s2[a].x + __shfl_xor_sync(0xFFFFFFFFu, s2[a].x, 16), y = s2[a].y + __shfl_xor_sync(0xFFFFFFFFu, s2[a].y, 16);
        if (hsel == pass) { acc3[2 * a] += x; acc3[2 * a + 1] += y; }
      }
      __syncwarp();   // the tile is rewritten by the next pass
    }
  };

  // tiles from the top of the CTA's rows downwards (the double-Q argmax needs the next row's outputs)
  int k = 0;
  for (int vr_hi = row_end; vr_hi > row_begin; vr_hi -= kTileRows, ++k) {
    const int vr0 = max(row_begin, vr_hi - kTileRows), nrows = vr_hi - vr0;
    const bool has_next = vr0 > row_begin;
    const uint32_t d_cur = (k & 1) ? kColD1 : kColD0, d_prev = (k & 1) ? kColD0 : kColD1;
    if (has_next) { const int nv0 = max(row_begin, vr0 - kTileRows); fetch_a(nv0, vr0 - nv0, key_nxt); }
    if (x_active) {
      float hi[8], lo[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { hi[j] = tf32_rn(cur.x[j]); lo[j] = tf32_rn(cur.x[j] - hi[j]); }
      tmem_st8(lane_base + kColAHi + 8 * cq, hi);
      tmem_st8(lane_base + kColALo + 8 * cq, lo);
      if (r < nrows) {   // the other two kernels read the gathered row instead of chasing the episode index again
        float4* xo = reinterpret_cast<float4*>(p.xg + cur.dst * kTcObsDim + 8 * cq);
        xo[0] = make_float4(cur.x[0], cur.x[1], cur.x[2], cur.x[3]); xo[1] = make_float4(cur.x[4], cur.x[5], cur.x[6], cur.x[7]);
      }
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    if (image_groups_pending == 2) { mbar_wait(bar + 2, 0); image_groups_pending = 1; }   // W1 + biases + FP32 W3 have landed
    tc_fence_before();
    __syncthreads();
    TSGP(g_ts_fwd3, p.dbg, 0, 3 + 6 * ts_tile);
    if (t == 0) {
      tc_fence_after();
      const uint32_t idesc = idesc_tf32(kHidden);
      const uint64_t dhi = kmajor_desc(smem_base + kOffW1Hi), dlo = kmajor_desc(smem_base + kOffW1Lo);
#pragma unroll
      for (int term = 0; term < 3; ++term)
#pragma unroll
        for (int ks = 0; ks < kTcObsDim / 8; ++ks)
          if (ks < k1steps) mma_tf32_ts(tmem + d_cur, tmem + (term == 0 ? kColALo : kColAHi) + ks * 8, (term == 1 ? dlo : dhi) + (uint32_t)((ks * 32) >> 4), idesc, (term | ks) ? 1u : 0u);
      mma_commit(bar);
      if (k > 0) {   // every thread is past the previous tile's TD head: publish its first row's outputs
#pragma unroll
        for (int o = 0; o < kOutPad; ++o) carry[o] = carry_q[o];
      }
    }
    const size_t dst_row = cur.dst;
    const int agent = cur.agent, b = cur.b, tt = cur.tt, act = cur.act;
    const float rew = cur.rew; const uint8_t filled_u8 = cur.filled, done1_u8 = cur.done1;
    mbar_wait(bar, parity); parity ^= 1;
    tc_fence_after();
    TSGP(g_ts_fwd3, p.dbg, 0, 4 + 6 * ts_tile);
    // ---- layer-1 epilogue: bias + ReLU; the ReLU mask of H1 -> row record; 3xTF32 split -> the A operand of layer 2 ------------------------------
    {
      const float* bias = b1 + c0;
      uint32_t ra[16], rb[16];
      tmem_ld16_issue(lane_base + d_cur + c0, ra);
      tmem_ld16_issue(lane_base + d_cur + c0 + 16, rb);
      tmem_ld_wait(ra);
      tmem_ld_wait(rb);
      uint32_t mask = 0;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t (&acc)[16] = half ? rb : ra;
        float hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float h = fmaxf(__uint_as_float(acc[j]) + bias[16 * half + j], 0.f);
          mask |= (h > 0.f ? 1u : 0u) << (16 * half + j);
          tf32_split(h, hi[j], lo[j]);
        }
        tmem_st16(lane_base + kColAHi + c0 + 16 * half, hi);
        tmem_st16(lane_base + kColALo + c0 + 16 * half, lo);
      }
      if (r < nrows) reinterpret_cast<uint32_t*>(p.rec + dst_row * kRowRec)[4 + cq] = mask;
      if (image_groups_pending == 1) { mbar_wait(bar + 3, 0); image_groups_pending = 0; }   // W2
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      tc_fence_before();
      __syncthreads();
      TSGP(g_ts_fwd3, p.dbg, 0, 5 + 6 * ts_tile);
      if (t == 0) {
        tc_fence_after();
        issue_kmajor_ts(tmem, d_cur, smem_base + kOffW2Hi, smem_base + kOffW2Lo);
        mma_commit(bar);
      }
      // under the layer-2 MMAs (the longest stretch in which the CUDA cores would idle): the next (lower) tile's rows are requested, and the
      // previous tile's dW3 is formed from its accumulator, which the other TMEM column block still holds
      if (has_next) fetch_b(key_nxt, nxt);
      if (k > 0) dw3_tile(d_prev);
      mbar_wait(bar, parity); parity ^= 1;
      tc_fence_after();
      TSGP(g_ts_fwd3, p.dbg, 0, 6 + 6 * ts_tile);
    }
    // ---- layer-2 epilogue: the ReLU mask of H2 -> row record; head on the CUDA cores against the FP32 copy of W3 (packed FP32); partial sums of
    // column quarters 1..3 -> shared ------------------------------------------------------------------------------------------------------------
    float q[kOutPad];
    // target outputs of the next row of the same (agent, episode): requested now, selected in the TD head ~5 k cycles later (they used to be loaded after the
    // argmax, a dependent global load on the tile's critical path)
    float tqv[kOutPad];
#pragma unroll
    for (int o = 0; o < kOutPad; ++o) tqv[o] = 0.f;
    if (cq == 0 && r < nrows && tt < T && p.td_ext == nullptr) {
      const float* tqp = p.tq + (((size_t)agent * B + b) * (T + 1) + tt + 1) * A;
#pragma unroll
      for (int o = 0; o < kOutPad; ++o) if (o < A) tqv[o] = tqp[o];
    }
    {
      uint32_t ra[16], rb[16];
      tmem_ld16_issue(lane_base + d_cur + c0, ra);
      tmem_ld16_issue(lane_base + d_cur + c0 + 16, rb);
      tmem_ld_wait(ra);
      tmem_ld_wait(rb);
      float2 q2[kOutPad];
#pragma unroll
      for (int a = 0; a < kOutPad; ++a) q2[a] = make_float2(0.f, 0.f);
      uint32_t mask = 0;
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        const uint32_t (&acc)[16] = g < 4 ? ra : rb;
        const int o = 4 * (g & 3);
        const float4 bb = *reinterpret_cast<const float4*>(b2 + c0 + 4 * g);
        float2 h01 = __fadd2_rn(make_float2(__uint_as_float(acc[o]), __uint_as_float(acc[o + 1])), make_float2(bb.x, bb.y));
        float2 h23 = __fadd2_rn(make_float2(__uint_as_float(acc[o + 2]), __uint_as_float(acc[o + 3])), make_float2(bb.z, bb.w));
        h01.x = fmaxf(h01.x, 0.f); h01.y = fmaxf(h01.y, 0.f); h23.x = fmaxf(h23.x, 0.f); h23.y = fmaxf(h23.y, 0.f);
        mask |= ((h01.x > 0.f ? 1u : 0u) | (h01.y > 0.f ? 2u : 0u) | (h23.x > 0.f ? 4u : 0u) | (h23.y > 0.f ? 8u : 0u)) << (4 * g);
#pragma unroll
        for (int a = 0; a < kOutPad; ++a) {
          if (a < A) {
            const float4 w = w3f[a * (kHidden / 4) + (c0 >> 2) + g];
            q2[a] = __ffma2_rn(h23, make_float2(w.z, w.w), __ffma2_rn(h01, make_float2(w.x, w.y), q2[a]));
          }
        }
      }
      if (r < nrows) reinterpret_cast<uint32_t*>(p.rec + dst_row * kRowRec)[8 + cq] = mask;
#pragma unroll
      for (int a = 0; a < kOutPad; ++a) q[a] = q2[a].x + q2[a].y;
      if (cq > 0) {
        float4* pp = reinterpret_cast<float4*>(part + ((size_t)(cq - 1) * kTileRows + r) * kOutPad);
        pp[0] = make_float4(q[0], q[1], q[2], q[3]); pp[1] = make_float4(q[4], q[5], q[6], q[7]);
      }
      named_bar_sync(2 + lq, 128);   // the four warps of this lane quarter (they are also past their dW3 reads of Gs)
      TSGP(g_ts_fwd3, p.dbg, 0, 7 + 6 * ts_tile);
    }
    // ---- outputs of this tile -> shared (next-row exchange), TD head, dq -> Gs: column quarter 0 (threads 0..127, r == t) --------------------------
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
      float g = 0.f;
      if (r < nrows) {
        if (p.q_out) for (int o = 0; o < A; ++o) p.q_out[dst_row * A + o] = q[o];
        if (tt < T) {
          if (p.td_ext) {
            g = p.td_ext[(size_t)agent * p.td_agent_stride + (size_t)b * T + tt];
          } else {
            const float* qn = (r + 1 < nrows) ? (qs + (r + 1) * kOutPad) : carry;
            float tsel;
            if (p.double_q) {
              int best = 0; float bv = qn[0];
              for (int o = 1; o < A; ++o) if (qn[o] > bv) { bv = qn[o]; best = o; }
              tsel = tqv[0];
#pragma unroll
              for (int o = 1; o < kOutPad; ++o) tsel = (o == best) ? tqv[o] : tsel;
            } else {
              tsel = tqv[0];
#pragma unroll
              for (int o = 1; o < kOutPad; ++o) if (o < A) tsel = fmaxf(tsel, tqv[o]);
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
      // dq of this tile for the dW3 pass (padding rows: zeros), db3: the sum of dq over the 32 rows of this warp
      float gv[kOutPad];
#pragma unroll
      for (int o = 0; o < kOutPad; ++o) gv[o] = (o == act) ? g : 0.f;
      *reinterpret_cast<float4*>(Gs + r * kOutPad) = make_float4(gv[0], gv[1], gv[2], gv[3]);
      *reinterpret_cast<float4*>(Gs + r * kOutPad + 4) = make_float4(gv[4], gv[5], gv[6], gv[7]);
#pragma unroll
      for (int o = 0; o < kOutPad; ++o) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) gv[o] += __shfl_xor_sync(0xFFFFFFFFu, gv[o], off);
      }
      if (lane < kOutPad) {
        float x = gv[0];
#pragma unroll
        for (int o = 1; o < kOutPad; ++o) x = (lane == o) ? gv[o] : x;
        dbs[lq * kOutPad + lane] += x;
      }
    }
    TSGP(g_ts_fwd3, p.dbg, 0, 8 + 6 * ts_tile);
    ts_tile += 1;
    cur = nxt;
  }
  // ---- dW3 of the last tile (its accumulator block: (k - 1) & 1) ---------------------------------------------------------------------------------
  __syncthreads();   // Gs of the last tile is complete
  dw3_tile(((k - 1) & 1) ? kColD1 : kColD0);
  TSGP(g_ts_fwd3, p.dbg, 0, 29);
  // ---- per-CTA loss statistics (threads 0..127 hold them) and the dW3 | db3 partials: sum over the four lane quarters in a fixed order ------------
  float* red3 = reinterpret_cast<float*>(smem + kF3Tb);   // [4][8][128]
  __syncthreads();   // every warp is done with its transpose tile
#pragma unroll
  for (int a = 0; a < kOutPad; ++a) red3[(lq * kOutPad + a) * kHidden + c0 + lane] = acc3[a];
  if (t < kTileRows) { qs[t] = st[0]; qs[kTileRows + t] = st[1]; }
  __syncthreads();
  for (int i = t; i < A * kHidden; i += kTrThreads)
    gs[p.lay.w3 + i] = (red3[i] + red3[kOutPad * kHidden + i]) + (red3[2 * kOutPad * kHidden + i] + red3[3 * kOutPad * kHidden + i]);
  if (t < A) gs[p.lay.b3 + t] = (dbs[t] + dbs[kOutPad + t]) + (dbs[2 * kOutPad + t] + dbs[3 * kOutPad + t]);
  for (int s = kTileRows / 2; s > 0; s >>= 1) {
    if (t < s) { qs[t] += qs[t + s]; qs[kTileRows + t] += qs[kTileRows + t + s]; }
    __syncthreads();
  }
  if (t < 4) p.loss_part[4 * blockIdx.x + t] = t < 2 ? qs[t * kTileRows] : 0.f;
  tc_fence_before();
  __syncthreads();
  TSGP(g_ts_fwd3, p.dbg, 0, 30);
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
  TSGP(g_ts_fwd3, p.dbg, 0, 31);
}

// =====================================================================================================================
// 2. dH1 = (dH2 x W2) * relu'(H1) and dW1 | db1 += dH1^T x [X | 1].  17 warps: 16 epilogue warps (lq x cq) + one that issues the dW1 MMAs.
// TMEM: A hi [0,128) | A lo [128,256) | D [256,384) | dW1 | db1 [384,416).  Shared memory: W2^T image | FP32 W3 | two chunk buffers, each
// {dH1 hi | dH1 lo | X hi | X lo} for the 32 rows of one lane quarter: lane quarters 0 and 1 fill buffers 0 and 1, quarters 2 and 3 follow once the
// tensor core has consumed them.
// =====================================================================================================================
constexpr int kH3Threads = kTrThreads + 32;
constexpr int kH3W3 = kBwdImageBytes;                               // FP32 copy of W3 [8][128] behind the W2^T image
constexpr int kH3Buf = kH3W3 + kOutPad * kHidden * 4;               // 133 120: a multiple of 1024
constexpr int kH3BufBytes = 2 * kC3Op + 2 * kC3Panel;               // dH1 hi | lo, X hi | lo: 40 KB
constexpr int kH3X = 2 * kC3Op;
constexpr int kH3Bars = kH3Buf + 2 * kH3BufBytes;
constexpr int kH3Smem = kH3Bars + 128 + 1024;
constexpr uint32_t kColW1acc = 384;
static_assert(kH3Buf % 1024 == 0 && kH3BufBytes % 1024 == 0 && kH3Smem <= 227 * 1024, "dH1 + dW1: shared-memory map");

__global__ void __launch_bounds__(kH3Threads, 1) tc_dh1w1_kernel(TcTrainParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  // [0] dH1 MMAs of a tile retired, [1] images landed, [2..3] chunk buffer staged (4 warp arrivals), [4..7] the chunk of lane quarter 0..3 consumed,
  // [8] every dW1 MMA retired.  One "consumed" barrier per lane quarter (not per buffer): lane quarter lq waits for the chunk of quarter (lq + 2) & 3
  // that held its buffer before, so every barrier has ONE group of waiters that sees each of its phases in turn -- a parity wait cannot tell a
  // phase from the one two before it, and with a barrier per buffer the quarters 2 / 3 could run one phase ahead of what they were waiting for.
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kH3Bars);
  uint64_t* full = bar + 2; uint64_t* empty = bar + 4; uint64_t* done = bar + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 9);
  const float4* w3f4 = reinterpret_cast<const float4*>(smem + kH3W3);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31, lq = warp & 3, cq = (warp >> 2) & 3, r = 32 * lq + lane, c0 = 32 * cq;
  int net, row_begin, row_end;
  cta_rows(p.plan, net, row_begin, row_end);
  float* gs = p.scratch + (size_t)blockIdx.x * p.scratch_pitch;
  const int D = p.src.D;
  if (row_begin >= row_end) {
    pdl_wait();
    for (int i = t; i < kHidden * D; i += kH3Threads) gs[p.lay.w1 + i] = 0.f;
    for (int i = t; i < kHidden; i += kH3Threads) gs[p.lay.b1 + i] = 0.f;
    return;
  }
  TSGP(g_ts_dh1w1, p.dbg, 1, 0);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (t == 0) {
    mbar_init(bar, 1); mbar_init(bar + 1, 1); mbar_init(full, 4); mbar_init(full + 1, 4);
    mbar_init(empty, 1); mbar_init(empty + 1, 1); mbar_init(empty + 2, 1); mbar_init(empty + 3, 1); mbar_init(done, 1);
    fence_mbar_init();
  }
  pdl_wait();   // nothing above touches global memory
  pdl_launch_dependents();
  TSGP(g_ts_dh1w1, p.dbg, 1, 1);
  if (t == 0) {  // W2^T image + FP32 W3: TMA bulk copies onto one mbarrier
    mbar_expect_tx(bar + 1, (uint32_t)(kBwdImageBytes + kOutPad * kHidden * 4));
    tma_image_range(smem_u32(smem), p.bwd_images + (size_t)net * kBwdImageBytes, 0, kBwdImageBytes, bar + 1);
    tma_bulk_g2s(smem_u32(smem) + kH3W3, p.images + (size_t)net * kImageBytes + kOffW3F, kOutPad * kHidden * 4, bar + 1);
  }
  const int n_tiles = (row_end - row_begin + kTileRows - 1) / kTileRows;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot, smem_base = smem_u32(smem);

  if (warp == kTrThreads / 32) {
    // ---- MMA warp: dW1[j1][i | 1] += dH1^T x [X | 1] per 32-row chunk: 3 terms x 4 k-steps of M = 128, N = 32 ---------------------------------
    const uint32_t id_w1 = idesc_tf32(32);
    const int n_chunks = 4 * n_tiles;
    for (int c = 0; c < n_chunks; ++c) {
      const int b = c & 1;   // chunk c = (tile c >> 2, lane quarter c & 3) -> buffer (c & 1); its use count is c >> 1
      TSGP(g_ts_dh1w1, p.dbg, 1, 100 + c);
      mbar_wait(full + b, (uint32_t)(c >> 1) & 1u);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t base = smem_base + kH3Buf + b * kH3BufBytes;
        const uint64_t a_hi = kmajor_desc(base), a_lo = kmajor_desc(base + kC3Op), b_hi = kmajor_desc(base + kH3X), b_lo = kmajor_desc(base + kH3X + kC3Panel);
#pragma unroll
        for (int term = 0; term < 3; ++term) {   // lo*hi, hi*lo, hi*hi
#pragma unroll
          for (int ks = 0; ks < kC3Rows / 8; ++ks)
            mma_tf32_ss(tmem + kColW1acc, (term == 0 ? a_lo : a_hi) + (uint32_t)((ks * 32) >> 4), (term == 1 ? b_lo : b_hi) + (uint32_t)((ks * 32) >> 4), id_w1, (c || term || ks) ? 1u : 0u);
        }
        mma_commit(empty + (c & 3));
        if (c == n_chunks - 1) mma_commit(done);
      }
      __syncwarp();
    }
  } else {
    // ---- epilogue warps -------------------------------------------------------------------------------------------------------------------------
    const uint32_t lane_base = tmem + ((uint32_t)(32 * lq) << 16);
    // this thread's row record (dLoss/dq[act], act, the two mask words of its 32 columns) and its 8 observation columns; fetched one tile ahead
    struct Rec { long long d; float g; int act; uint32_t m1, m2; float x[8]; };
    auto fetch = [&](int vr0, Rec& rc) {
      rc.d = -1; rc.g = 0.f; rc.act = 0; rc.m1 = 0; rc.m2 = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) rc.x[j] = 0.f;
      if (vr0 + r < row_end) {
        int a, u, o;
        rc.d = (long long)dst_of3(p.plan, p.src, net, vr0 + r, a, u, o);
        const float* rp = p.rec + rc.d * kRowRec;
        const int2 ga = *reinterpret_cast<const int2*>(rp);
        rc.g = __int_as_float(ga.x); rc.act = ga.y;
        rc.m1 = reinterpret_cast<const uint32_t*>(rp)[4 + cq];
        rc.m2 = reinterpret_cast<const uint32_t*>(rp)[8 + cq];
        const float4* xp = reinterpret_cast<const float4*>(p.xg + rc.d * kTcObsDim + 8 * cq);
        const float4 x0 = xp[0], x1 = xp[1];
        rc.x[0] = x0.x; rc.x[1] = x0.y; rc.x[2] = x0.z; rc.x[3] = x0.w; rc.x[4] = x1.x; rc.x[5] = x1.y; rc.x[6] = x1.z; rc.x[7] = x1.w;
#pragma unroll
        for (int j = 0; j < 8; ++j) rc.x[j] = (8 * cq + j < D) ? rc.x[j] : ((8 * cq + j == D) ? 1.f : 0.f);   // [X | 1]: the ones column carries db1
      }
    };
    Rec cur, nxt;
    fetch(row_begin, cur);
    nxt = cur;
    TSGP(g_ts_dh1w1, p.dbg, 1, 2);
    mbar_wait(bar + 1, 0);   // images have landed (every thread reads the FP32 W3 rows; the tensor core reads W2^T)
    uint32_t parity = 0;
    uint8_t* buf = smem + kH3Buf + (lq & 1) * kH3BufBytes;
    // dH2[r][j] = g W3[act][j] (H2[r][j] > 0) for this thread's 32 columns -> A operand (hi / lo); then (everybody's part written, and everybody has
    // taken the previous tile's accumulator into registers) one thread issues D[r][j1] = sum_{j2} dH2[r][j2] W2[j2][j1]: B = K-major image of W2^T
    auto rebuild_and_issue = [&](const Rec& rc) {
      const float4* wrow = w3f4 + rc.act * (kHidden / 4) + 8 * cq;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        float v[16], hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 w = wrow[4 * half + j];
          const uint32_t m = rc.m2 >> (16 * half + 4 * j);
          v[4 * j] = (m & 1u) ? rc.g * w.x : 0.f; v[4 * j + 1] = (m & 2u) ? rc.g * w.y : 0.f;
          v[4 * j + 2] = (m & 4u) ? rc.g * w.z : 0.f; v[4 * j + 3] = (m & 8u) ? rc.g * w.w : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) tf32_split(v[j], hi[j], lo[j]);
        tmem_st16(lane_base + kColAHi + c0 + 16 * half, hi);
        tmem_st16(lane_base + kColALo + c0 + 16 * half, lo);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      tc_fence_before();
      named_bar_sync(1, kTrThreads);   // the 16 epilogue warps (the MMA warp runs its own schedule)
      if (t == 0) {
        tc_fence_after();
        issue_kmajor_ts(tmem, kColD, smem_base, smem_base + 4 * kPanelBytes);
        mma_commit(bar);
      }
    };
    TSGP(g_ts_dh1w1, p.dbg, 1, 3);
    rebuild_and_issue(cur);
    if (n_tiles > 1) fetch(row_begin + kTileRows, nxt);
    for (int tile = 0; tile < n_tiles; ++tile) {
      mbar_wait(bar, parity); parity ^= 1;
      tc_fence_after();
      TSGP(g_ts_dh1w1, p.dbg, 1, 4 + 3 * tile);
      uint32_t ra[16], rb[16];
      tmem_ld16_issue(lane_base + kColD + c0, ra);
      tmem_ld16_issue(lane_base + kColD + c0 + 16, rb);
      tmem_ld_wait(ra);
      tmem_ld_wait(rb);
      // what staging this tile still needs from its record: the H1 mask word and the [X | 1] columns
      const uint32_t m1 = cur.m1;
      float xk[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) xk[j] = cur.x[j];
      cur = nxt;
      // the next tile's MMAs start first; this tile's dH1 is masked, split and staged under them
      if (tile + 1 < n_tiles) rebuild_and_issue(cur);
      TSGP(g_ts_dh1w1, p.dbg, 1, 5 + 3 * tile);
      {
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const uint32_t a = j < 16 ? ra[j & 15] : rb[j & 15];
          v[j] = ((m1 >> j) & 1u) ? __uint_as_float(a) : 0.f;   // padding rows: m1 = 0
        }
        // chunk (tile, lq) -> buffer lq & 1; its previous user is chunk (tile, lq - 2) or (tile - 1, lq + 2)
        if (lq >= 2) mbar_wait(empty + (lq - 2), (uint32_t)tile & 1u);
        else if (tile > 0) mbar_wait(empty + (lq + 2), (uint32_t)(tile - 1) & 1u);
        stage_row32(buf, buf + kC3Op, lane, cq, v);
        stage_row8(buf + kH3X, buf + kH3X + kC3Panel, lane, cq, xk);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(full + (lq & 1));
      }
      if (tile + 2 < n_tiles) fetch(row_begin + (tile + 2) * kTileRows, nxt);
      TSGP(g_ts_dh1w1, p.dbg, 1, 6 + 3 * tile);
    }
  }
  // ---- flush dW1 | db1: lane j of lane quarter lq owns output feature j (column quarter 0 does it) -------------------------------------------------
  mbar_wait(done, 0);
  tc_fence_after();
  TSGP(g_ts_dh1w1, p.dbg, 1, 29);
  if (warp < 4) {
    const int j = 32 * lq + lane;
    const uint32_t lane_base = tmem + ((uint32_t)(32 * lq) << 16);
    float v[16], w[16];
    tmem_ld16(lane_base + kColW1acc, v);
    tmem_ld16(lane_base + kColW1acc + 16, w);
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const float x = i < 16 ? v[i & 15] : w[i & 15];
      if (i < D) gs[p.lay.w1 + j * D + i] = x;
      else if (i == D) gs[p.lay.b1 + j] = x;
    }
  }
  tc_fence_before();
  __syncthreads();
  TSGP(g_ts_dh1w1, p.dbg, 1, 31);
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// =====================================================================================================================
// 3. dW2 | db2 += dH2^T x [H1 | 1], H1 = relu(X W1^T + b1) recomputed per 128-row tile (SS form: X tile and W1 image K-major in shared memory),
// dH2 rebuilt from the row record.  17 warps as above.  TMEM: H1 accumulators of even | odd tiles [0,256) (layer 1 runs one tile ahead) | dW2 | db2 [256,416).
// Shared memory: W1 hi | lo, b1 | .. | FP32 W3 (the forward image's tail), X tile hi | lo, two chunk buffers {dH2 hi | lo, H1 hi + ones panel | H1 lo + zero panel}.
// =====================================================================================================================
constexpr int kW3Tail = 2 * kPanelBytes;                            // b1 | b2 | b3 | FP32 W3 (kTailBytes)
constexpr int kW3Xs = ((kW3Tail + kTailBytes + 1023) / 1024) * 1024;   // X tile hi | lo (K-major SWIZZLE_128B)
constexpr int kW3Buf = kW3Xs + 2 * kPanelBytes;
constexpr int kW3H1 = 2 * kC3Op;                                    // inside a buffer: dH2 hi | lo, then H1 hi (+ ones panel) | H1 lo (+ zero panel)
constexpr int kW3BufBytes = 2 * kC3Op + 2 * (kC3Op + kC3Panel);     // 72 KB
constexpr int kW3Bars = kW3Buf + 2 * kW3BufBytes;
constexpr int kW3Smem = kW3Bars + 128 + 1024;
constexpr uint32_t kColH1 = 0, kColW2acc = 256;   // H1 accumulators of even / odd tiles: [0,128) / [128,256)
static_assert(kW3Buf % 1024 == 0 && kW3BufBytes % 1024 == 0 && kW3Smem <= 227 * 1024, "dW2: shared-memory map");

__global__ void __launch_bounds__(kH3Threads, 1) tc_dw2_kernel(TcTrainParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  // [0] layer-1 MMAs of a tile retired, [1] image pieces landed, [2..3] chunk buffer staged (4 warp arrivals), [4..7] the chunk of lane quarter 0..3
  // consumed (one barrier per lane quarter: see tc_dh1w1_kernel), [8] every dW2 MMA retired
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kW3Bars);
  uint64_t* full = bar + 2; uint64_t* empty = bar + 4; uint64_t* done = bar + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 9);
  const float* b1 = reinterpret_cast<const float*>(smem + kW3Tail);
  const float4* w3f4 = reinterpret_cast<const float4*>(smem + kW3Tail + (kOffW3F - kOffB1));
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31, lq = warp & 3, cq = (warp >> 2) & 3, r = 32 * lq + lane, c0 = 32 * cq;
  int net, row_begin, row_end;
  cta_rows(p.plan, net, row_begin, row_end);
  float* gs = p.scratch + (size_t)blockIdx.x * p.scratch_pitch;
  if (row_begin >= row_end) {
    pdl_wait();
    for (int i = t; i < kHidden * kHidden; i += kH3Threads) gs[p.lay.w2 + i] = 0.f;
    for (int i = t; i < kHidden; i += kH3Threads) gs[p.lay.b2 + i] = 0.f;
    return;
  }
  TSGP(g_ts_dw2, p.dbg, 2, 0);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (t == 0) {
    mbar_init(bar, 1); mbar_init(bar + 1, 1); mbar_init(full, 8); mbar_init(full + 1, 8);   // a chunk: 4 warps stage H1, 4 warps dH2
    mbar_init(empty, 1); mbar_init(empty + 1, 1); mbar_init(empty + 2, 1); mbar_init(empty + 3, 1); mbar_init(done, 1);
    fence_mbar_init();
  }
  // constant panels of both buffers (features 128..159 of the B operand): feature 128 = ones over the chunk's 32 rows behind H1 hi (it carries db2),
  // zeros elsewhere and behind H1 lo
  for (int i = t; i < 2 * 2 * (kC3Panel / 4); i += kH3Threads) {
    const int bsel = i / (2 * (kC3Panel / 4)), w = i % (2 * (kC3Panel / 4)), which = w / (kC3Panel / 4), ww = w % (kC3Panel / 4);
    reinterpret_cast<float*>(smem + kW3Buf + bsel * kW3BufBytes + kW3H1 + kC3Op + which * (kC3Op + kC3Panel))[ww] = (which == 0 && ww < 32) ? 1.0f : 0.f;
  }
  pdl_wait();   // nothing above touches global memory
  pdl_launch_dependents();
  TSGP(g_ts_dw2, p.dbg, 2, 1);
  if (t == 0) {  // W1 hi | lo and the image's tail (biases, FP32 W3)
    const uint8_t* src = p.images + (size_t)net * kImageBytes;
    mbar_expect_tx(bar + 1, (uint32_t)(2 * kPanelBytes + kTailBytes));
    tma_image_range(smem_u32(smem), src, kOffW1Hi, kOffW2Hi, bar + 1);
    tma_bulk_g2s(smem_u32(smem) + kW3Tail, src + kOffB1, kTailBytes, bar + 1);
  }
  const int n_tiles = (row_end - row_begin + kTileRows - 1) / kTileRows;
  const int k1steps = (p.src.D + 7) >> 3;
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot, smem_base = smem_u32(smem);
  TSGP(g_ts_dw2, p.dbg, 2, 2);

  if (warp == kTrThreads / 32) {
    // ---- MMA warp: dW2[j2][j1 | 1] += dH2^T x [H1 | 1] per 32-row chunk: 3 terms x 4 k-steps of M = 128, N = 160 --------------------------------
    const uint32_t id_w2 = idesc_tf32(160);
    const int n_chunks = 4 * n_tiles;
    for (int c = 0; c < n_chunks; ++c) {
      const int b = c & 1;
      TSGP(g_ts_dw2, p.dbg, 2, 100 + c);
      mbar_wait(full + b, (uint32_t)(c >> 1) & 1u);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t base = smem_base + kW3Buf + b * kW3BufBytes;
        const uint64_t a_hi = kmajor_desc(base), a_lo = kmajor_desc(base + kC3Op), b_hi = kmajor_desc(base + kW3H1), b_lo = kmajor_desc(base + kW3H1 + kC3Op + kC3Panel);
#pragma unroll
        for (int term = 0; term < 3; ++term) {   // lo*hi, hi*lo, hi*hi
#pragma unroll
          for (int ks = 0; ks < kC3Rows / 8; ++ks)
            mma_tf32_ss(tmem + kColW2acc, (term == 0 ? a_lo : a_hi) + (uint32_t)((ks * 32) >> 4), (term == 1 ? b_lo : b_hi) + (uint32_t)((ks * 32) >> 4), id_w2, (c || term || ks) ? 1u : 0u);
        }
        mma_commit(empty + (c & 3));
        if (c == n_chunks - 1) mma_commit(done);
      }
      __syncwarp();
    }
  } else {
    // ---- epilogue warps -------------------------------------------------------------------------------------------------------------------------
    const uint32_t lane_base = tmem + ((uint32_t)(32 * lq) << 16);
    uint8_t* xs = smem + kW3Xs;
    // per tile and row: the record (dLoss/dq[act], act, this thread's H2 mask word), needed when the tile is staged, and this thread's 8 observation
    // columns, needed one tile earlier (layer 1 runs one tile ahead)
    // A warp may only read its own TMEM lane quarter, so H1 of the chunk (tile, lq) is staged by the four warps of lane quarter lq -- but dH2 comes from
    // the row records, which any thread can read: the dH2 half of a chunk is staged by the warps of the OTHER pair of lane quarters (lq ^ 2).  All sixteen
    // warps then work on the chunks of quarters 0 / 1 first and on those of quarters 2 / 3 second, instead of half of them waiting for a buffer.
    // Per tile and thread: validity of its own row (H1) and the record of the partner row 32 (lq ^ 2) + lane (dLoss/dq[act], act, this thread's H2 mask word).
    struct Rec { bool valid; float g; int act; uint32_t m2; };
    const int rp = 32 * (lq ^ 2) + lane;
    auto fetch_rec = [&](int vr0, Rec& rc) {
      rc.valid = vr0 + r < row_end; rc.g = 0.f; rc.act = 0; rc.m2 = 0;
      if (vr0 + rp < row_end) {
        int a, u, o;
        const size_t d = dst_of3(p.plan, p.src, net, vr0 + rp, a, u, o);
        const float* rpp = p.rec + d * kRowRec;
        const int2 ga = *reinterpret_cast<const int2*>(rpp);
        rc.g = __int_as_float(ga.x); rc.act = ga.y;
        rc.m2 = reinterpret_cast<const uint32_t*>(rpp)[8 + cq];
      }
    };
    auto fetch_x = [&](int vr0, float (&x)[8]) {
#pragma unroll
      for (int j = 0; j < 8; ++j) x[j] = 0.f;
      if (cq < k1steps && vr0 + r < row_end) {
        int a, u, o;
        const size_t d = dst_of3(p.plan, p.src, net, vr0 + r, a, u, o);
        const float4* xp = reinterpret_cast<const float4*>(p.xg + d * kTcObsDim + 8 * cq);
        const float4 x0 = xp[0], x1 = xp[1];
        x[0] = x0.x; x[1] = x0.y; x[2] = x0.z; x[3] = x0.w; x[4] = x1.x; x[5] = x1.y; x[6] = x1.z; x[7] = x1.w;
      }
    };
    // X tile (this thread: 8 columns of its row) -> K-major operand; everybody's part written (and everybody past its reads of the accumulator block
    // the MMAs are about to overwrite: the tile before last's) -> one thread issues layer 1 of tile `tile`
    auto stage_x_and_issue = [&](int tile, const float (&x)[8]) {
      if (cq < k1steps) stage_x_tile(xs, r, cq, x);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      tc_fence_before();
      named_bar_sync(1, kTrThreads);
      if (t == 0) {
        tc_fence_after();
        issue_l1_ss(tmem + kColH1 + (uint32_t)(tile & 1) * kHidden, smem_base + kW3Xs, smem_base + kW3Xs + kPanelBytes, smem_base + kOffW1Hi, smem_base + kOffW1Lo, k1steps);
        mma_commit(bar);
      }
    };
    Rec cur, nxt;
    float xn[8];
    fetch_rec(row_begin, cur);
    fetch_x(row_begin, xn);
    nxt = cur;
    mbar_wait(bar + 1, 0);   // W1, b1 and the FP32 W3 rows have landed
    uint32_t parity = 0;
    uint8_t* buf = smem + kW3Buf + (lq & 1) * kW3BufBytes;
    TSGP(g_ts_dw2, p.dbg, 2, 3);
    stage_x_and_issue(0, xn);
    if (n_tiles > 1) fetch_x(row_begin + kTileRows, xn);
    for (int tile = 0; tile < n_tiles; ++tile) {
      mbar_wait(bar, parity); parity ^= 1;   // layer 1 of this tile has retired: its accumulator is ready and the X tile is free
      tc_fence_after();
      TSGP(g_ts_dw2, p.dbg, 2, 4 + 3 * tile);
      // the two halves of a tile: first the chunks of lane quarters 0 / 1 (quarters 0 / 1 stage their H1, quarters 2 / 3 the matching dH2), then the
      // chunks of quarters 2 / 3 the other way round.  Both times this warp writes buffer lq & 1.
      auto stage_dh2 = [&]() {   // dH2[r'][j] = g W3[act][j] (H2[r'][j] > 0) for the partner row and this thread's 32 columns
        float v[32];
        const float4* wrow = w3f4 + cur.act * (kHidden / 4) + 8 * cq;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 w = wrow[j];
          const uint32_t m = cur.m2 >> (4 * j);
          v[4 * j] = (m & 1u) ? cur.g * w.x : 0.f; v[4 * j + 1] = (m & 2u) ? cur.g * w.y : 0.f;
          v[4 * j + 2] = (m & 4u) ? cur.g * w.z : 0.f; v[4 * j + 3] = (m & 8u) ? cur.g * w.w : 0.f;
        }
        stage_row32(buf, buf + kC3Op, lane, cq, v);
      };
      auto stage_h1 = [&]() {   // H1 = relu(accumulator + b1) of this thread's own row (padding rows: zero)
        uint32_t ra[16], rb[16];
        const uint32_t d_col = kColH1 + (uint32_t)(tile & 1) * kHidden;
        tmem_ld16_issue(lane_base + d_col + c0, ra);
        tmem_ld16_issue(lane_base + d_col + c0 + 16, rb);
        tmem_ld_wait(ra);
        tmem_ld_wait(rb);
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const uint32_t a = j < 16 ? ra[j & 15] : rb[j & 15];
          v[j] = cur.valid ? fmaxf(__uint_as_float(a) + b1[c0 + j], 0.f) : 0.f;
        }
        stage_row32(buf + kW3H1, buf + kW3H1 + kC3Op + kC3Panel, lane, cq, v);
      };
      auto publish = [&]() {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(full + (lq & 1));
      };
      // first half: chunk (tile, lq & 1); the buffer's previous user was chunk (tile - 1, (lq & 1) + 2)
      if (tile > 0) mbar_wait(empty + ((lq & 1) + 2), (uint32_t)(tile - 1) & 1u);
      if (lq < 2) stage_h1(); else stage_dh2();
      publish();
      TSGP(g_ts_dw2, p.dbg, 2, 5 + 3 * tile);
      // between the halves (the tensor core is busy with the first two chunks, whose consumption the second half waits for anyway): the next tile's
      // X tile and layer 1, the next tile's records, the X columns of the tile after it
      if (tile + 1 < n_tiles) {
        stage_x_and_issue(tile + 1, xn);
        fetch_rec(row_begin + (tile + 1) * kTileRows, nxt);
        if (tile + 2 < n_tiles) fetch_x(row_begin + (tile + 2) * kTileRows, xn);
      }
      // second half: chunk (tile, (lq & 1) + 2); previous user: chunk (tile, lq & 1)
      mbar_wait(empty + (lq & 1), (uint32_t)tile & 1u);
      if (lq < 2) stage_dh2(); else stage_h1();
      publish();
      TSGP(g_ts_dw2, p.dbg, 2, 6 + 3 * tile);
      cur = nxt;
    }
  }
  // ---- flush dW2 | db2: lane j of lane quarter lq owns output feature j; each warp transposes its 32 x 32 block through shared memory so that
  // every store instruction writes one 128-byte row segment (the chunk buffers are dead by then) --------------------------------------------------
  mbar_wait(done, 0);
  tc_fence_after();
  __syncthreads();
  TSGP(g_ts_dw2, p.dbg, 2, 29);
  if (warp < kTrThreads / 32) {
    const int j = 32 * lq + lane;
    const uint32_t lane_base = tmem + ((uint32_t)(32 * lq) << 16);
    float* tile = reinterpret_cast<float*>(smem + kW3Buf + warp * (32 * 33 * 4));   // [32][33]
    float v[16];
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      tmem_ld16(lane_base + kColW2acc + 32 * cq + 16 * half, v);
#pragma unroll
      for (int i = 0; i < 16; ++i) tile[lane * 33 + 16 * half + i] = v[i];
    }
    __syncwarp();
    float* w2blk = gs + p.lay.w2 + (32 * lq) * kHidden + 32 * cq + lane;
#pragma unroll 8
    for (int i = 0; i < 32; ++i) w2blk[i * kHidden] = tile[i * 33 + lane];
    if (cq == 0) {
      tmem_ld16(lane_base + kColW2acc + kHidden, v);
      gs[p.lay.b2 + j] = v[0];
    }
  }
  tc_fence_before();
  __syncthreads();
  TSGP(g_ts_dw2, p.dbg, 2, 31);
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// =====================================================================================================================

int tc_train3_init() {
  MARL_CUDA_TRY(cudaFuncSetAttribute(tc_dqn_fwd3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kF3Smem));
  MARL_CUDA_TRY(cudaFuncSetAttribute(tc_dh1w1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kH3Smem));
  MARL_CUDA_TRY(cudaFuncSetAttribute(tc_dw2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kW3Smem));
  return MARL_OK;
}

// all three kernels walk the same episode-aligned row split, so the per-CTA partials line up with ReduceParams::cta_begin
int launch_tc_dqn_train3(const TcTrainParams& p, int grid, cudaStream_t st, cudaEvent_t* between) {
  MARL_CUDA_TRY(launch_pdl(tc_dqn_fwd3_kernel, dim3(grid), dim3(kTrThreads), kF3Smem, st, p));
  if (between) MARL_CUDA_TRY(cudaEventRecord(between[0], st));
  MARL_CUDA_TRY(launch_pdl(tc_dh1w1_kernel, dim3(grid), dim3(kH3Threads), kH3Smem, st, p));
  if (between) MARL_CUDA_TRY(cudaEventRecord(between[1], st));
  MARL_CUDA_TRY(launch_pdl(tc_dw2_kernel, dim3(grid), dim3(kH3Threads), kW3Smem, st, p));
  return MARL_OK;
}

}  // namespace marl
