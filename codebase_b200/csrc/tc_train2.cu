// tc_train2.cu -- two-accumulator (ping-pong) versions of the first two kernels of the tensor-core training pass (tc_train.cu):
//   tc_dqn_fwd2_kernel   online forward + TD head (QNetwork._compute_loss, marlbase/dqn/model.py:118-163): same outputs as tc_dqn_fwd_kernel
//                        (H1, H2, gathered X, 64-byte row records, per-CTA loss statistics)
//   tc_dh12_kernel       dH1 = (dH2 x W2) * relu'(H1), dH2 rebuilt from the row records: same outputs as tc_dh1_kernel
// Structure (tc_forward.cu, tc_forward2_kernel): 20 warps -- 16 epilogue warps (lane quarter x column quarter of a 128 x 128 tile), one MMA-issuing
// warp, three loader warps; TMEM = A hi | A lo | D0 | D1; consecutive tiles alternate accumulators, so the CUDA-core work of one tile (bias, ReLU,
// masks, activation stores, head, TD error / dH2 rebuild, 3xTF32 split) runs under the MMAs of its neighbour; the head (6 outputs) runs on the CUDA
// cores against the FP32 copy of W3.  Selected by marl_set_option("tensor_core_pingpong", 1) (default); the weight-gradient kernel is unchanged.
#include "tc_common.cuh"

namespace marl {

constexpr int kT2Threads = kTrThreads + 128;
constexpr int kT2Loaders = 96;
constexpr int kT2ReadyArrivals = kTrThreads / 32 + kT2Loaders / 32;

// ---- shared-memory map of the forward kernel (bytes) -------------------------------------------------------------------------------------------
constexpr int kF2Xs = kOffW3Hi;                                     // X tile hi | lo (K-major SWIZZLE_128B, 2 x 16 KB)
constexpr int kF2Tail = kF2Xs + 2 * kPanelBytes;                    // b1 | b2 | b3 | FP32 W3
constexpr int kF2Part = kF2Tail + kTailBytes;                       // head partials of column quarters 1..3: [3][128][8] floats
constexpr int kF2Meta = kF2Part + 3 * kTileRows * kOutPad * 4;      // [4 tiles in flight][128 rows] x {dst, act | flags, rew, td}: 16 bytes
constexpr int kF2Qs = kF2Meta + 4 * kTileRows * 16;                 // outputs of a tile's rows for the next-row exchange: [2 parities][128][8] floats
constexpr int kF2Carry = kF2Qs + 2 * kTileRows * kOutPad * 4;       // [2 parities][8]: outputs of row 0 of the previously processed (higher) tile
constexpr int kF2Red = kF2Carry + 2 * kOutPad * 4;                  // loss statistics of the four TD warps: [4][2]
constexpr int kF2Bars = kF2Red + 64;
constexpr int kF2Smem = kF2Bars + 64 + 1024;
static_assert(kF2Xs % 1024 == 0 && kF2Smem <= 227 * 1024, "ping-pong training forward: shared-memory map");

struct RowMeta4 { uint32_t dst; uint32_t act_flags; float rew; float td; };   // act_flags: bits 0..7 act, bit 8 filled, bit 9 done[t+1], bit 10 t < T, bit 11 agent == first

__device__ __forceinline__ uint32_t relu_mask32(const float (&h)[32]) {
  uint32_t m = 0;
#pragma unroll
  for (int j = 0; j < 32; ++j) m |= (h[j] > 0.f ? 1u : 0u) << j;
  return m;
}

// =====================================================================================================================
// 1. online forward + TD head.  Tiles are taken from the top of the CTA's row range downwards (the double-Q argmax of a row needs the NEXT row's
// outputs): tile k covers virtual rows [row_end - 128 (k + 1), row_end - 128 k); row r of a tile is virtual row row_end - 128 (k + 1) + r, rows below
// row_begin (only in the last tile, at its LOW r) are padding.
// =====================================================================================================================
__global__ void __launch_bounds__(kT2Threads, 1) tc_dqn_fwd2_kernel(TcTrainParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  // [0] layer-1 MMAs retired, [1] layer-2 MMAs retired, [2] W1 + tail landed, [3] W2 landed, [4] operands ready (19 warp arrivals)
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kF2Bars);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 5);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  int net, row_begin, row_end;
  cta_rows(p.plan, net, row_begin, row_end);
  if (row_begin >= row_end) {
    pdl_wait();
    if (t < 4) p.loss_part[4 * blockIdx.x + t] = 0.f;
    return;
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (t == 0) { mbar_init(bar, 1); mbar_init(bar + 1, 1); mbar_init(bar + 2, 1); mbar_init(bar + 3, 1); mbar_init(bar + 4, kT2ReadyArrivals); fence_mbar_init(); }
  pdl_wait();   // nothing above touches global memory
  pdl_launch_dependents();
  const uint32_t smem_base = smem_u32(smem);
  if (t == 0) {
    const uint8_t* src = p.images + (size_t)net * kImageBytes;
    mbar_expect_tx(bar + 2, (uint32_t)(kOffW2Hi + kTailBytes));
    tma_image_range(smem_base, src, 0, kOffW2Hi, bar + 2);
    tma_bulk_g2s(smem_base + kF2Tail, src + kOffB1, kTailBytes, bar + 2);
    mbar_expect_tx(bar + 3, (uint32_t)(kOffW3Hi - kOffW2Hi));
    tma_image_range(smem_base, src, kOffW2Hi, kOffW3Hi, bar + 3);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int D = p.src.D, A = p.lay.out, T = p.src.traj.T, B = p.plan.units_per_agent, k1steps = (D + 7) >> 3;
  const int n_tiles = (row_end - row_begin + kTileRows - 1) / kTileRows;
  RowMeta4* meta = reinterpret_cast<RowMeta4*>(smem + kF2Meta);

  if (warp == kTrThreads / 32) {
    // ---- MMA warp ---------------------------------------------------------------------------------------------------------------------------
    mbar_wait(bar + 2, 0);
    for (int k = -1; k < n_tiles; ++k) {
      mbar_wait(bar + 4, (uint32_t)(k + 1) & 1u);
      tc_fence_after();
      if (k == 0) mbar_wait(bar + 3, 0);
      if (lane == 0) {
        const uint32_t d_next = ((k + 1) & 1) ? kColD1 : kColD0, d_cur = (k & 1) ? kColD1 : kColD0;
        if (k + 1 < n_tiles) {
          issue_l1_ss(tmem + d_next, smem_base + kF2Xs, smem_base + kF2Xs + kPanelBytes, smem_base + kOffW1Hi, smem_base + kOffW1Lo, k1steps);
          mma_commit(bar);
        }
        if (k >= 0) {
          issue_kmajor_ts(tmem, d_cur, smem_base + kOffW2Hi, smem_base + kOffW2Lo);
          mma_commit(bar + 1);
        }
      }
      __syncwarp();
    }
  } else if (warp > kTrThreads / 32) {
    // ---- loader warps: thread i owns rows i and i + 96 (the latter for i < 32) of every tile: observation row -> X tile (hi | lo) and the gathered
    // copy the weight-gradient kernel reads; the row's output index and loss-head scalars -> shared.  Row decode: divisions once, then -128 rows per tile.
    const int i = t - (kTrThreads + 32);
    uint8_t* xs = smem + kF2Xs;
    const int urows = p.plan.unit_rows, q128 = kTileRows / urows, r128 = kTileRows % urows;
    struct RowState { int slot, unit, off; };
    RowState rs[2];
#pragma unroll
    for (int m = 0; m < 2; ++m) {   // virtual row of (tile 0, row i + 96 m); may be below row_begin (padding) or even negative
      const int vr = row_end - kTileRows + i + m * kT2Loaders, rpa = B * urows;
      const int vrc = vr < 0 ? 0 : vr;
      rs[m].slot = vrc / rpa;
      const int rem = vrc - rs[m].slot * rpa;
      rs[m].unit = rem / urows; rs[m].off = rem - rs[m].unit * urows;
    }
    float xv[2][kTcObsDim];
    RowMeta4 mt[2];
    auto fetch = [&](int tile) {
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const int row = i + m * kT2Loaders;
        mt[m].dst = 0xFFFFFFFFu; mt[m].act_flags = 0; mt[m].rew = 0.f; mt[m].td = 0.f;
#pragma unroll
        for (int j = 0; j < kTcObsDim; ++j) xv[m][j] = 0.f;
        const int vr = row_end - (tile + 1) * kTileRows + row;
        if (row < kTileRows && vr >= row_begin) {
          const int agent = p.plan.slot_agent[p.plan.slot_begin[net] + rs[m].slot], b = rs[m].unit, tt = rs[m].off;
          const TrajView& tv = p.src.traj;
          const size_t ep = (size_t)p.src.idx[b];
          const float* src = tv.obs + ((ep * tv.N + agent) * (size_t)(T + 1) + tt) * D;
          mt[m].dst = (uint32_t)(((size_t)agent * B + b) * urows + tt);
#pragma unroll
          for (int j = 0; j < kTcObsDim; ++j) if (j < D) xv[m][j] = src[j];
          uint32_t fl = 0u;
          if (tt < T) {
            const uint32_t act = (uint32_t)tv.act[(ep * tv.N + agent) * T + tt];
            mt[m].rew = tv.rew[(ep * tv.N + agent) * T + tt];
            fl = (act & 0xFFu) | ((uint32_t)tv.filled[ep * T + tt] << 8) | ((uint32_t)tv.done[ep * (T + 1) + tt + 1] << 9) | (1u << 10);
            if (p.td_ext) mt[m].td = p.td_ext[(size_t)agent * p.td_agent_stride + (size_t)b * T + tt];
          }
          if (agent == 0) fl |= 1u << 11;
          mt[m].act_flags = fl;
        }
        // next tile: - 128 rows
        rs[m].off -= r128; rs[m].unit -= q128;
        if (rs[m].off < 0) { rs[m].off += urows; rs[m].unit -= 1; }
        while (rs[m].unit < 0 && rs[m].slot > 0) { rs[m].unit += B; rs[m].slot -= 1; }
      }
    };
    auto stage = [&](int rnd) {
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const int row = i + m * kT2Loaders;
        if (row < kTileRows) {
          float x8[8];
#pragma unroll
          for (int ch = 0; ch < kTcObsDim / 8; ++ch) {
            if (ch < k1steps) {
#pragma unroll
              for (int j = 0; j < 8; ++j) x8[j] = xv[m][8 * ch + j];
              stage_x_tile(xs, row, ch, x8);
              if (mt[m].dst != 0xFFFFFFFFu) {   // the weight-gradient kernel reads the gathered row instead of chasing the episode index again
                float4* xo = reinterpret_cast<float4*>(p.xg + (size_t)mt[m].dst * kTcObsDim + 8 * ch);
                xo[0] = make_float4(x8[0], x8[1], x8[2], x8[3]); xo[1] = make_float4(x8[4], x8[5], x8[6], x8[7]);
              }
            }
          }
          meta[(rnd & 3) * kTileRows + row] = mt[m];
        }
      }
    };
    fetch(0);
    stage(0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0) mbar_arrive(bar + 4);   // round 0
    if (n_tiles > 1) fetch(1);
    for (int rnd = 1; rnd <= n_tiles; ++rnd) {
      if (rnd < n_tiles) {
        mbar_wait(bar, (uint32_t)(rnd - 1) & 1u);   // layer 1 of tile rnd - 1 has retired: the X tile is free (and arrival round rnd - 1 is complete)
        stage(rnd);
        if (rnd + 1 < n_tiles) fetch(rnd + 1);
      } else {
        mbar_wait(bar + 4, (uint32_t)(rnd - 1) & 1u);   // never two arrivals of one warp in the same phase
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(bar + 4);
    }
  } else {
    // ---- epilogue warps -----------------------------------------------------------------------------------------------------------------------
    const int lq = warp & 3, cq = warp >> 2, r = 32 * lq + lane, c0 = 32 * cq;
    const uint32_t lane_base = tmem + ((uint32_t)(32 * lq) << 16);
    const float* b1 = reinterpret_cast<const float*>(smem + kF2Tail);
    const float* b2 = b1 + kHidden;
    const float* b3 = b2 + kHidden;
    const float4* w3f = reinterpret_cast<const float4*>(smem + kF2Tail + (kOffW3F - kOffB1));
    float* part = reinterpret_cast<float*>(smem + kF2Part);
    float* qs = reinterpret_cast<float*>(smem + kF2Qs);
    float* carry = reinterpret_cast<float*>(smem + kF2Carry);
    float st0 = 0.f, st1 = 0.f;   // loss statistics of this thread's rows (column quarter 0 only)
    auto arrive_ready = [&]() {
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar + 4);
    };
    // layer-2 epilogue of tile `tile` from the drained accumulator: H2 (FP32, chunk-major) + its ReLU mask -> global, head partials -> shared, then
    // (column quarter 0) outputs, next-row exchange, TD error -> row record
    auto epilogue2 = [&](int tile, const uint32_t (&ra)[16], const uint32_t (&rb)[16]) {
      const RowMeta4 mt = meta[(tile & 3) * kTileRows + r];
      const bool valid = mt.dst != 0xFFFFFFFFu;
      float2 q2[kOutPad];
#pragma unroll
      for (int a = 0; a < kOutPad; ++a) q2[a] = make_float2(0.f, 0.f);
      uint32_t mask = 0;
      float4* hg = reinterpret_cast<float4*>(p.h2g) + (valid ? mt.dst : 0);
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        const uint32_t (&acc)[16] = g < 4 ? ra : rb;
        const int o = 4 * (g & 3);
        const float4 bb = *reinterpret_cast<const float4*>(b2 + c0 + 4 * g);
        float2 h01 = __fadd2_rn(make_float2(__uint_as_float(acc[o]), __uint_as_float(acc[o + 1])), make_float2(bb.x, bb.y));
        float2 h23 = __fadd2_rn(make_float2(__uint_as_float(acc[o + 2]), __uint_as_float(acc[o + 3])), make_float2(bb.z, bb.w));
        h01.x = fmaxf(h01.x, 0.f); h01.y = fmaxf(h01.y, 0.f); h23.x = fmaxf(h23.x, 0.f); h23.y = fmaxf(h23.y, 0.f);
        mask |= ((h01.x > 0.f ? 1u : 0u) | (h01.y > 0.f ? 2u : 0u) | (h23.x > 0.f ? 4u : 0u) | (h23.y > 0.f ? 8u : 0u)) << (4 * g);
        if (valid) hg[(size_t)(8 * cq + g) * p.rows] = make_float4(h01.x, h01.y, h23.x, h23.y);
#pragma unroll
        for (int a = 0; a < kOutPad; ++a) {
          if (a < A) {
            const float4 w = w3f[a * (kHidden / 4) + (c0 >> 2) + g];
            q2[a] = __ffma2_rn(h23, make_float2(w.z, w.w), __ffma2_rn(h01, make_float2(w.x, w.y), q2[a]));
          }
        }
      }
      if (valid) reinterpret_cast<uint32_t*>(p.rec + (size_t)mt.dst * kRowRec)[8 + cq] = mask;
      float q[kOutPad];
#pragma unroll
      for (int a = 0; a < kOutPad; ++a) q[a] = q2[a].x + q2[a].y;
      named_bar_sync(1 + lq, 128);   // the previous tile's partials have been read
      if (cq > 0) {
        float4* pp = reinterpret_cast<float4*>(part + ((size_t)(cq - 1) * kTileRows + r) * kOutPad);
        pp[0] = make_float4(q[0], q[1], q[2], q[3]); pp[1] = make_float4(q[4], q[5], q[6], q[7]);
      }
      named_bar_sync(1 + lq, 128);
      if (cq == 0) {
        const int par = tile & 1;
#pragma unroll
        for (int a = 0; a < kOutPad; ++a)
          q[a] = a < A ? (((q[a] + part[((size_t)0 * kTileRows + r) * kOutPad + a]) + part[((size_t)1 * kTileRows + r) * kOutPad + a]) + part[((size_t)2 * kTileRows + r) * kOutPad + a]) + b3[a] : 0.f;
        float4* qo = reinterpret_cast<float4*>(qs + ((size_t)par * kTileRows + r) * kOutPad);
        qo[0] = make_float4(q[0], q[1], q[2], q[3]); qo[1] = make_float4(q[4], q[5], q[6], q[7]);
        if (r == 0) {   // row 0 of this tile is the "next row" of the last row of the tile below
          float4* co = reinterpret_cast<float4*>(carry + par * kOutPad);
          co[0] = make_float4(q[0], q[1], q[2], q[3]); co[1] = make_float4(q[4], q[5], q[6], q[7]);
        }
        named_bar_sync(5, 128);   // the four warps of column quarter 0 exchange their rows' outputs
        if (valid) {
          const int act = (int)(mt.act_flags & 0xFFu);
          float g = 0.f;
          if (p.q_out) for (int o = 0; o < A; ++o) p.q_out[(size_t)mt.dst * A + o] = q[o];
          if (mt.act_flags & (1u << 10)) {   // t < T
            if (p.td_ext) {
              g = mt.td;
            } else {
              const float* qn = (r + 1 < kTileRows) ? (qs + ((size_t)par * kTileRows + r + 1) * kOutPad) : (carry + (par ^ 1) * kOutPad);
              const float* tq = p.tq + ((size_t)mt.dst + 1) * A;   // target outputs of the next row of the same (agent, episode)
              float tsel;
              if (p.double_q) {
                int best = 0; float bv = qn[0];
                for (int o = 1; o < A; ++o) if (qn[o] > bv) { bv = qn[o]; best = o; }
                tsel = tq[best];
              } else {
                tsel = tq[0];
                for (int o = 1; o < A; ++o) tsel = fmaxf(tsel, tq[o]);
              }
              const float filled = (mt.act_flags >> 8) & 1u ? 1.f : 0.f, done1 = (mt.act_flags >> 9) & 1u ? 1.f : 0.f;
              const float y = mt.rew + p.gamma * tsel * (1.f - done1);
              float qa = q[0];
#pragma unroll
              for (int o = 1; o < kOutPad; ++o) qa = (o == act) ? q[o] : qa;
              const float delta = qa - y;
              st0 += delta * delta * filled;
              if (mt.act_flags & (1u << 11)) st1 += filled;
              g = 2.f * delta * filled;
            }
          }
          // the TD loss touches one output per row: dq[r][a] = g (a == act), 0 otherwise; rows at t == T carry g = 0
          *reinterpret_cast<int2*>(p.rec + (size_t)mt.dst * kRowRec) = make_int2(__float_as_int(g), act);
        }
      }
    };

    arrive_ready();          // round 0 belongs to the loaders
    mbar_wait(bar + 2, 0);   // biases + FP32 W3 have landed
    uint32_t ph1 = 0, ph2 = 0;
    for (int k = 0; k < n_tiles; ++k) {
      const uint32_t d_cur = (k & 1) ? kColD1 : kColD0, d_prev = (k & 1) ? kColD0 : kColD1;
      // ---- layer-1 epilogue of tile k: bias + ReLU into 32 registers, H1 + its mask -> global ----------------------------------------------------
      mbar_wait(bar, ph1); ph1 ^= 1;
      tc_fence_after();
      float h1[32];
      {
        uint32_t ra[16], rb[16];
        tmem_ld16_issue(lane_base + d_cur + c0, ra);
        tmem_ld16_issue(lane_base + d_cur + c0 + 16, rb);
        tmem_ld_wait(ra);
        tmem_ld_wait(rb);
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const float4 bb = *reinterpret_cast<const float4*>(b1 + c0 + 4 * g);
          const uint32_t (&acc)[16] = g < 4 ? ra : rb;
          const int o = 4 * (g & 3);
          h1[4 * g] = fmaxf(__uint_as_float(acc[o]) + bb.x, 0.f); h1[4 * g + 1] = fmaxf(__uint_as_float(acc[o + 1]) + bb.y, 0.f);
          h1[4 * g + 2] = fmaxf(__uint_as_float(acc[o + 2]) + bb.z, 0.f); h1[4 * g + 3] = fmaxf(__uint_as_float(acc[o + 3]) + bb.w, 0.f);
        }
      }
      {
        const uint32_t dst = meta[(k & 3) * kTileRows + r].dst;
        if (dst != 0xFFFFFFFFu) {
          float4* hg = reinterpret_cast<float4*>(p.h1g) + dst;
#pragma unroll
          for (int g = 0; g < 8; ++g) hg[(size_t)(8 * cq + g) * p.rows] = make_float4(h1[4 * g], h1[4 * g + 1], h1[4 * g + 2], h1[4 * g + 3]);
          reinterpret_cast<uint32_t*>(p.rec + (size_t)dst * kRowRec)[4 + cq] = relu_mask32(h1);
        }
      }
      // ---- A columns free once the layer-2 MMAs of tile k - 1 have retired; their accumulator comes out in the same breath ----------------
      if (k > 0) { mbar_wait(bar + 1, ph2); ph2 ^= 1; tc_fence_after(); }
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        float hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) tf32_split(h1[16 * half + j], hi[j], lo[j]);
        tmem_st16(lane_base + kColAHi + c0 + 16 * half, hi);
        tmem_st16(lane_base + kColALo + c0 + 16 * half, lo);
      }
      uint32_t r2a[16], r2b[16];
      if (k > 0) {
        tmem_ld16_issue(lane_base + d_prev + c0, r2a);
        tmem_ld16_issue(lane_base + d_prev + c0 + 16, r2b);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      if (k > 0) { tmem_ld_wait(r2a); tmem_ld_wait(r2b); }
      arrive_ready();   // round k + 1: layer 1 of tile k + 1 and layer 2 of tile k may go
      if (k > 0) epilogue2(k - 1, r2a, r2b);
    }
    // ---- last tile -----------------------------------------------------------------------------------------------------------------------------
    mbar_wait(bar + 1, ph2);
    tc_fence_after();
    {
      const uint32_t d_last = ((n_tiles - 1) & 1) ? kColD1 : kColD0;
      uint32_t r2a[16], r2b[16];
      tmem_ld16_issue(lane_base + d_last + c0, r2a);
      tmem_ld16_issue(lane_base + d_last + c0 + 16, r2b);
      tmem_ld_wait(r2a);
      tmem_ld_wait(r2b);
      epilogue2(n_tiles - 1, r2a, r2b);
    }
    // ---- per-CTA loss statistics: the four warps of column quarter 0 hold them ----------------------------------------------------------------------
    if (cq == 0) {
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) { st0 += __shfl_xor_sync(0xFFFFFFFFu, st0, off); st1 += __shfl_xor_sync(0xFFFFFFFFu, st1, off); }
      float* red = reinterpret_cast<float*>(smem + kF2Red);
      if (lane == 0) { red[2 * lq] = st0; red[2 * lq + 1] = st1; }
      named_bar_sync(5, 128);
      if (t < 4) p.loss_part[4 * blockIdx.x + t] = t < 2 ? ((red[t] + red[2 + t]) + (red[4 + t] + red[6 + t])) : 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// =====================================================================================================================
// 2. dH1 = (dH2 x W2) * relu'(H1), dH2[r][j] = g_r W3[act_r][j] relu'(H2[r][j]) rebuilt from the row records.  Two accumulators: the rebuild of
// tile k (into registers, FP32) runs under the MMAs of tile k - 1, its 3xTF32 split + TMEM store follow the moment they retire, and the masked
// store of tile k - 1 runs under the MMAs of tile k.  The three extra warps prefetch the row records (dst, g, act, both mask rows: 48 of the 64
// bytes) into shared memory up to two tiles ahead.
// =====================================================================================================================
constexpr int kH2W3 = kBwdImageBytes;                               // FP32 copy of W3 [8][128] behind the W2^T image
constexpr int kH2Rec = kH2W3 + kOutPad * kHidden * 4;               // [4 tiles in flight][128 rows] x 12 words {dst, g, act, -, mask1[4], mask2[4]}
constexpr int kH2Bars = kH2Rec + 4 * kTileRows * 48;
constexpr int kH2Smem = kH2Bars + 64 + 1024;
static_assert(kH2Smem <= 227 * 1024, "ping-pong dH1: shared-memory map");

TSG_DEFINE(g_ts_dh12)
TSG_GETTER(tsg_dh12, g_ts_dh12)
__global__ void __launch_bounds__(kT2Threads, 1) tc_dh12_kernel(TcTrainParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  // [1] MMAs of a tile retired, [2] images landed, [4] A operand ready (16 warp arrivals), [6] / [7] records of an even / odd tile in shared memory (3 arrivals)
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kH2Bars);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 5);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  int net, row_begin, row_end;
  cta_rows(p.plan, net, row_begin, row_end);
  if (row_begin >= row_end) { pdl_wait(); return; }
  TSG(g_ts_dh12, 0);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (t == 0) { mbar_init(bar + 1, 1); mbar_init(bar + 2, 1); mbar_init(bar + 4, kTrThreads / 32); mbar_init(bar + 6, kT2Loaders / 32); mbar_init(bar + 7, kT2Loaders / 32); fence_mbar_init(); }
  pdl_wait();   // nothing above touches global memory
  pdl_launch_dependents();
  TSG(g_ts_dh12, 1);
  const uint32_t smem_base = smem_u32(smem);
  if (t == 0) {
    mbar_expect_tx(bar + 2, (uint32_t)(kBwdImageBytes + kOutPad * kHidden * 4));
    tma_image_range(smem_base, p.bwd_images + (size_t)net * kBwdImageBytes, 0, kBwdImageBytes, bar + 2);
    tma_bulk_g2s(smem_base + kH2W3, p.images + (size_t)net * kImageBytes + kOffW3F, kOutPad * kHidden * 4, bar + 2);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int n_tiles = (row_end - row_begin + kTileRows - 1) / kTileRows;
  uint32_t* recs = reinterpret_cast<uint32_t*>(smem + kH2Rec);   // 12 words per row

  if (warp == kTrThreads / 32) {
    // ---- MMA warp: D_k = dH2_k x W2 (B = K-major image of W2^T) -----------------------------------------------------------------------------------
    mbar_wait(bar + 2, 0);
    for (int k = 0; k < n_tiles; ++k) {
      mbar_wait(bar + 4, (uint32_t)k & 1u);
      tc_fence_after();
      if (lane == 0) {
        issue_kmajor_ts(tmem, (k & 1) ? kColD1 : kColD0, smem_base, smem_base + 4 * kPanelBytes);
        mma_commit(bar + 1);
      }
      __syncwarp();
    }
  } else if (warp > kTrThreads / 32) {
    // ---- record prefetch: thread i owns rows i and i + 96 (i < 32) of every tile ------------------------------------------------------------------
    const int i = t - (kTrThreads + 32);
    const int urows = p.plan.unit_rows, B = p.plan.units_per_agent;
    uint32_t w[2][12];
    auto fetch = [&](int tile) {
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const int row = i + m * kT2Loaders, vr = row_begin + tile * kTileRows + row;
#pragma unroll
        for (int j = 0; j < 12; ++j) w[m][j] = 0u;
        w[m][0] = 0xFFFFFFFFu;
        if (row < kTileRows && vr < row_end) {
          int agent, unit, off;
          decode_row(p.plan, net, vr, agent, unit, off);
          const uint32_t dst = (uint32_t)(p.src.mode == 0 ? ((size_t)unit * p.src.N + agent) : (((size_t)agent * B + unit) * urows + off));
          const uint4* rp = reinterpret_cast<const uint4*>(p.rec + (size_t)dst * kRowRec);
          const uint4 a = rp[0], m1 = rp[1], m2 = rp[2];
          w[m][0] = dst; w[m][1] = a.x; w[m][2] = a.y;
          w[m][4] = m1.x; w[m][5] = m1.y; w[m][6] = m1.z; w[m][7] = m1.w; w[m][8] = m2.x; w[m][9] = m2.y; w[m][10] = m2.z; w[m][11] = m2.w;
        }
      }
    };
    fetch(0);
    for (int rnd = 0; rnd < n_tiles; ++rnd) {
      // slot rnd & 3 last held tile rnd - 4 (read for the last time while the MMAs of tile rnd - 3 ran); and a waiter of the even / odd barrier may
      // be at most one phase behind: both hold once the MMAs of tile rnd - 2 have retired
      if (rnd >= 2) mbar_wait(bar + 1, (uint32_t)(rnd - 2) & 1u);
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const int row = i + m * kT2Loaders;
        if (row < kTileRows) {
          uint4* d = reinterpret_cast<uint4*>(recs + ((size_t)(rnd & 3) * kTileRows + row) * 12);
          d[0] = make_uint4(w[m][0], w[m][1], w[m][2], w[m][3]); d[1] = make_uint4(w[m][4], w[m][5], w[m][6], w[m][7]); d[2] = make_uint4(w[m][8], w[m][9], w[m][10], w[m][11]);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar + 6 + (rnd & 1));
      if (rnd + 1 < n_tiles) fetch(rnd + 1);
    }
  } else {
    // ---- epilogue warps -----------------------------------------------------------------------------------------------------------------------------
    const int lq = warp & 3, cq = warp >> 2, r = 32 * lq + lane, c0 = 32 * cq;
    const uint32_t lane_base = tmem + ((uint32_t)(32 * lq) << 16);
    const float4* w3f4 = reinterpret_cast<const float4*>(smem + kH2W3);
    TSG(g_ts_dh12, 2);
    mbar_wait(bar + 2, 0);   // FP32 W3 rows
    uint32_t ph = 0;
    for (int k = 0; k <= n_tiles; ++k) {
      // ---- dH2 of tile k for this thread's 32 columns, FP32, in registers (the MMAs of tile k - 1 may still be reading the A columns) ----------------
      float v[32];
      TSG(g_ts_dh12, 3 + 4 * k);
      if (k < n_tiles) {
        mbar_wait(bar + 6 + (k & 1), (uint32_t)(k >> 1) & 1u);   // the records of tile k are in shared memory
        const uint32_t* pr = recs + ((size_t)(k & 3) * kTileRows + r) * 12;
        const float g = __uint_as_float(pr[1]);
        const int act = (int)pr[2];
        const uint32_t m2w = pr[8 + cq];
        const float4* wrow = w3f4 + act * (kHidden / 4) + 8 * cq;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 w = wrow[j];
          const uint32_t m = m2w >> (4 * j);
          v[4 * j] = (m & 1u) ? g * w.x : 0.f; v[4 * j + 1] = (m & 2u) ? g * w.y : 0.f;
          v[4 * j + 2] = (m & 4u) ? g * w.z : 0.f; v[4 * j + 3] = (m & 8u) ? g * w.w : 0.f;
        }
      }
      TSG(g_ts_dh12, 4 + 4 * k);
      if (k > 0) { mbar_wait(bar + 1, ph); ph ^= 1; tc_fence_after(); }   // MMAs of tile k - 1 retired: A free, D_{(k-1)&1} holds its result
      TSG(g_ts_dh12, 5 + 4 * k);
      if (k < n_tiles) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          float hi[16], lo[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) tf32_split(v[16 * half + j], hi[j], lo[j]);
          tmem_st16(lane_base + kColAHi + c0 + 16 * half, hi);
          tmem_st16(lane_base + kColALo + c0 + 16 * half, lo);
        }
      }
      // ---- drain the accumulator of tile k - 1 ---------------------------------------------------------------------------------------------------
      uint32_t ra[16], rb[16];
      if (k > 0) {
        const uint32_t d_prev = ((k - 1) & 1) ? kColD1 : kColD0;
        tmem_ld16_issue(lane_base + d_prev + c0, ra);
        tmem_ld16_issue(lane_base + d_prev + c0 + 16, rb);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      if (k > 0) { tmem_ld_wait(ra); tmem_ld_wait(rb); }
      if (k < n_tiles) {   // round k: the MMAs of tile k may go
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar + 4);
      }
      TSG(g_ts_dh12, 6 + 4 * k);
      // ---- dH1 of tile k - 1: mask with relu'(H1) and store (chunk-major) ------------------------------------------------------------------------------
      if (k > 0) {
        const uint32_t* pr = recs + ((size_t)((k - 1) & 3) * kTileRows + r) * 12;
        const uint32_t dst = pr[0], m1w = pr[4 + cq];
        if (dst != 0xFFFFFFFFu) {
          float4* gout = reinterpret_cast<float4*>(p.dh1g) + dst;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint32_t (&acc)[16] = j < 4 ? ra : rb;
            const int o = 4 * (j & 3);
            const uint32_t m = m1w >> (4 * j);
            float4 d;
            d.x = (m & 1u) ? __uint_as_float(acc[o]) : 0.f; d.y = (m & 2u) ? __uint_as_float(acc[o + 1]) : 0.f;
            d.z = (m & 4u) ? __uint_as_float(acc[o + 2]) : 0.f; d.w = (m & 8u) ? __uint_as_float(acc[o + 3]) : 0.f;
            gout[(size_t)(8 * cq + j) * p.rows] = d;
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  TSG(g_ts_dh12, 31);
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// =====================================================================================================================

int tc_train2_init() {
  MARL_CUDA_TRY(cudaFuncSetAttribute(tc_dqn_fwd2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kF2Smem));
  MARL_CUDA_TRY(cudaFuncSetAttribute(tc_dh12_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kH2Smem));
  return MARL_OK;
}

int launch_tc_dqn_fwd2(const TcTrainParams& p, int grid, cudaStream_t st) {
  MARL_CUDA_TRY(launch_pdl(tc_dqn_fwd2_kernel, dim3(grid), dim3(kT2Threads), kF2Smem, st, p));
  return MARL_OK;
}
int launch_tc_dh12(const TcTrainParams& p, int grid, cudaStream_t st) {
  MARL_CUDA_TRY(launch_pdl(tc_dh12_kernel, dim3(grid), dim3(kT2Threads), kH2Smem, st, p));
  return MARL_OK;
}

}  // namespace marl
