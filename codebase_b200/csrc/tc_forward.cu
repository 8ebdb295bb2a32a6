// tc_forward.cu -- tcgen05 / TMEM implementation of the forward-only MLP pass (sm_100a).
//
// Same contract as mlp_forward_kernel (model.act's network pass, the target-network / target-critic pass of the
// learners; marlbase/dqn/model.py:99,132-134, marlbase/ac/model.py:148-149,190-193) but the three GEMMs of each 128-row
// tile run on the 5th-generation tensor cores:
//   * activations never touch shared memory: row r of a tile = TMEM lane r, 16 warps each own a lane quarter x column quarter;
//     the A operand of every layer is written with tcgen05.st, the accumulator is read back with tcgen05.ld, bias + ReLU
//     happen in registers;
//   * weights are the B operand, resident in shared memory as a pre-packed image (K-major, 128-byte swizzle, one
//     16-KB panel per 32 input features) built by pack_weights_kernel and kept current by the optimiser step (pack_param);
//   * FP32 parity (<= 1e-5, SURVEY H3) is kept with the error-compensated 3xTF32 split: every operand is stored as
//     hi = tf32(x) and lo = tf32(x - hi) and each product is accumulated as lo*hi + hi*lo + hi*hi in the FP32 TMEM
//     accumulator (measured 4e-7 relative on a 128x128x128 product, tools/tc_probe.cu).
// One elected thread issues tcgen05.mma (kind::tf32, cta_group::1, M = 128, N = 128 or 16); completion reaches the
// other threads through tcgen05.commit -> mbarrier.
#include "tc_common.cuh"

namespace marl {

size_t tc_image_bytes() { return kImageBytes; }
size_t tc_bwd_image_bytes() { return kBwdImageBytes; }

// Whole images from the flat parameters: the padding (observation columns >= in, head rows >= out) is zeroed, everything else goes
// through pack_param (tc_common.cuh).
__global__ void pack_weights_kernel(const float* __restrict__ theta, NetLayout lay, int n_nets, uint8_t* __restrict__ image, uint8_t* __restrict__ bwd_image) {
  const int net = blockIdx.y;
  if (net >= n_nets) return;
  const float* th = theta + (size_t)net * lay.P;
  uint8_t* img = image + (size_t)net * kImageBytes;
  uint8_t* bwd = bwd_image ? bwd_image + (size_t)net * kBwdImageBytes : nullptr;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < kHidden * 32 && (i & 31) >= lay.in) {  // W1 [128][32]: zero columns beyond in
    const int o = panel_offset(i >> 5, i & 31, kPanelBytes);
    *reinterpret_cast<float*>(img + kOffW1Hi + o) = 0.f; *reinterpret_cast<float*>(img + kOffW1Lo + o) = 0.f;
  }
  if (i < kHeadRows * kHidden && (i >> 7) >= lay.out) {  // W3 [16][128]: zero rows beyond out (also in the FP32 copy [8][128])
    const int o = panel_offset(i >> 7, i & 127, kHeadPanelBytes);
    *reinterpret_cast<float*>(img + kOffW3Hi + o) = 0.f; *reinterpret_cast<float*>(img + kOffW3Lo + o) = 0.f;
    if (i < kOutPad * kHidden) reinterpret_cast<float*>(img + kOffW3F)[i] = 0.f;
  }
  if (i < kHeadRows && i >= lay.out) reinterpret_cast<float*>(img + kOffB3)[i] = 0.f;
  if (i < lay.P) pack_param(lay, i, th[i], img, bwd);
}


// 3xTF32: D (+)= A_lo*B_hi + A_hi*B_lo + A_hi*B_hi over KSTEPS steps of 8 features; issued by one thread.
// Fully unrolled: every operand address is base + compile-time constant (the descriptor's address field counts
// 16-byte units, so advancing by b bytes is desc + (b >> 4)); the issuing thread spends a handful of instructions per
// MMA and the tensor pipe, not the issue loop, sets the pace.
template <int KSTEPS, int N, int PANEL_BYTES>
__device__ __forceinline__ void issue_layer(uint32_t tmem, uint32_t d_col, uint32_t b_hi_addr, uint32_t b_lo_addr, int ksteps_rt) {
  const uint32_t idesc = idesc_tf32(N);
  const uint64_t dhi = kmajor_desc(b_hi_addr), dlo = kmajor_desc(b_lo_addr);
  const uint32_t d = tmem + d_col, ahi = tmem + kColAHi, alo = tmem + kColALo;
#pragma unroll
  for (int term = 0; term < 3; ++term) {
#pragma unroll
    for (int ks = 0; ks < KSTEPS; ++ks) {
      if (ks < ksteps_rt) {
        constexpr int kDummy = 0; (void)kDummy;
        const uint32_t off16 = (uint32_t)(((ks >> 2) * PANEL_BYTES + (ks & 3) * 32) >> 4);
        mma_tf32_ts(d, (term == 0 ? alo : ahi) + ks * 8, (term == 1 ? dlo : dhi) + off16, idesc, (term | ks) ? 1u : 0u);
      }
    }
  }
}

TSG_DEFINE(g_ts_forward)
TSG_GETTER(tsg_forward, g_ts_forward)
// 16 warps: warp w owns TMEM lane quarter (w & 3) -- rows 32 (w & 3) .. +31 of the tile -- and column quarter (w >> 2) of the
// 128 hidden features, so that four warps per SM sub-partition overlap their TMEM / shared / global latencies.
__global__ void __launch_bounds__(kTrThreads, 1) tc_forward_kernel(FwdParams p, const uint8_t* __restrict__ images) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);  // swizzle atoms need 1024-byte alignment
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kImageBytes);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
  const int t = threadIdx.x, warp = t >> 5, lq = warp & 3, cq = warp >> 2, r = 32 * lq + (t & 31), c0 = 32 * cq;
  int net, row_begin, row_end;
  cta_rows(p.plan, net, row_begin, row_end);
  if (row_begin >= row_end) { pdl_wait(); return; }
  TSG(g_ts_forward, 0);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (t == 0) { mbar_init(bar, 1); mbar_init(bar + 2, 1); mbar_init(bar + 3, 1); mbar_init(bar + 4, 1); fence_mbar_init(); }
  pdl_wait();   // nothing above touches global memory (PDL contract, common.cuh)
  pdl_launch_dependents();
  TSG(g_ts_forward, 1);
  // the weight image is already in shared-memory layout: three TMA bulk copies (cp.async.bulk -> mbarrier, issued by one thread) in the
  // order the first tile needs them (W1 + biases, W2, W3), so that its first layer does not wait for the whole image
  // (the tensor-core operand copies of W3 are not loaded: the 6-wide head runs on the CUDA cores against the FP32 copy, and their 16 KB hold
  // the head partials of column quarters 1..3)
  if (t == 0) tma_forward_image_nohead(smem_u32(smem), images + (size_t)net * kImageBytes, bar + 2);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t lane_base = tmem + ((uint32_t)(32 * lq) << 16);
  const float* b1 = reinterpret_cast<const float*>(smem + kOffB1);
  const float* b2 = reinterpret_cast<const float*>(smem + kOffB2);
  const float* b3 = reinterpret_cast<const float*>(smem + kOffB3);
  const float4* w3f = reinterpret_cast<const float4*>(smem + kOffW3F);
  float* part = reinterpret_cast<float*>(smem + kOffW3Hi);   // [3][128 rows][8]
  const int D = p.src.D, out = p.lay.out;
  const int k1steps = (D + 7) >> 3;
  const bool x_active = cq < k1steps;   // column quarter cq stages observation columns [8 cq, 8 cq + 8)
  int image_groups_pending = 2;         // block-uniform: W1 + biases + FP32 W3, then W2
  uint32_t parity = 0;
  // this thread's 8 observation columns of its row (prefetched one tile ahead) and where the row's outputs go
  // (two steps, a barrier apart, so that neither waits on a load it has just issued: A = decode + episode index, B = the columns)
  float xin[8], xnext[8];
  size_t dst_row = 0, dst_next = 0;
  struct RowKey { int agent, unit, off, ep; bool valid; };
  auto fetch_a = [&](int vr0, int nrows, RowKey& k, size_t& dst) {
    k.agent = 0; k.unit = 0; k.off = 0; k.ep = 0; k.valid = r < nrows;
    if (k.valid) {
      decode_row(p.plan, net, vr0 + r, k.agent, k.unit, k.off);
      dst = src_dense_out(p.src.mode) ? ((size_t)k.unit * p.src.N + k.agent) : (((size_t)k.agent * p.plan.units_per_agent + k.unit) * p.plan.unit_rows + k.off);
      if (p.src.mode == 1) k.ep = p.src.idx[k.unit];
    }
  };
  auto fetch_b = [&](const RowKey& k, float (&x)[8]) {
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = 0.f;
    if (k.valid && x_active) {
      const TrajView& tv = p.src.traj;
      const float* src = p.src.mode == 0 ? p.src.dense + ((size_t)k.unit * p.src.N + k.agent) * D
                         : p.src.mode == 1 ? tv.obs + (((size_t)k.ep * tv.N + k.agent) * (size_t)(tv.T + 1) + k.off) * D
                                           : p.src.joint + ((size_t)k.unit * p.plan.unit_rows + k.off) * D;   // joint rows (centralised critic)
#pragma unroll
      for (int j = 0; j < 8; ++j) x[j] = (8 * cq + j < D) ? src[8 * cq + j] : 0.f;
    }
  };
  RowKey key_nxt;
  fetch_a(row_begin, min(kTileRows, row_end - row_begin), key_nxt, dst_row);
  fetch_b(key_nxt, xin);
  TSG(g_ts_forward, 2);
  int ts_tile = 0; (void)ts_tile;

  // Two accumulator blocks alternate between tiles (TMEM: A hi | A lo | D0 | D1): the head of tile k - 1 (CUDA cores) runs under the layer-2 MMAs of tile k.
  auto head_tile = [&](uint32_t d_col, size_t dst, int nr) {
    // layer-2 epilogue + head: relu(D + b2) of this thread's 32 columns against the FP32 copy of W3; the partial sums of column quarters 1..3 travel
    // through shared memory and column quarter 0 adds them in a fixed order
    uint32_t ra[16], rb[16];
    tmem_ld16_issue(lane_base + d_col + c0, ra);
    tmem_ld16_issue(lane_base + d_col + c0 + 16, rb);
    tmem_ld_wait(ra);
    tmem_ld_wait(rb);
    float q[kOutPad];
    head_partial(ra, rb, b2 + c0, w3f + (c0 >> 2), out, q);
    if (cq > 0) {
      float4* pp = reinterpret_cast<float4*>(part + ((size_t)(cq - 1) * kTileRows + r) * kOutPad);
      pp[0] = make_float4(q[0], q[1], q[2], q[3]); pp[1] = make_float4(q[4], q[5], q[6], q[7]);
    }
    named_bar_sync(1 + lq, 128);   // the four warps of this lane quarter
    if (cq == 0 && r < nr) {
      float* dstp = p.out + dst * out;
#pragma unroll
      for (int o = 0; o < kOutPad; ++o)
        if (o < out) dstp[o] = (((q[o] + part[((size_t)0 * kTileRows + r) * kOutPad + o]) + part[((size_t)1 * kTileRows + r) * kOutPad + o]) + part[((size_t)2 * kTileRows + r) * kOutPad + o]) + b3[o];
    }
    // the next head's partials are written at least two __syncthreads later: no second barrier needed
  };
  int k = 0, prev_nrows = 0;
  size_t prev_dst = 0;
  for (int vr0 = row_begin; vr0 < row_end; vr0 += kTileRows, ++k) {
    const int nrows = min(kTileRows, row_end - vr0);
    const bool has_next = vr0 + kTileRows < row_end;
    const uint32_t d_cur = (k & 1) ? kColD1 : kColD0, d_prev = (k & 1) ? kColD0 : kColD1;
    if (has_next) fetch_a(vr0 + kTileRows, min(kTileRows, row_end - vr0 - kTileRows), key_nxt, dst_next);
    // ---- input row -> A operand (hi / lo), zero padded to k1steps * 8 features -----------------------------------
    if (x_active) {
      float hi[8], lo[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) tf32_split(xin[j], hi[j], lo[j]);
      tmem_st8(lane_base + kColAHi + 8 * cq, hi);
      tmem_st8(lane_base + kColALo + 8 * cq, lo);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    if (image_groups_pending == 2) { mbar_wait(bar + 2, 0); image_groups_pending = 1; }   // W1 + biases + FP32 W3 have landed
    tc_fence_before();
    __syncthreads();
    TSG(g_ts_forward, 3 + 6 * ts_tile);
    // ---- layer 1 -------------------------------------------------------------------------------------------------
    if (t == 0) {
      tc_fence_after();
      issue_layer<kTcObsDim / 8, kHidden, kPanelBytes>(tmem, d_cur, smem_base + kOffW1Hi, smem_base + kOffW1Lo, k1steps);
      mma_commit(bar);
    }
    mbar_wait(bar, parity); parity ^= 1;
    tc_fence_after();
    TSG(g_ts_forward, 4 + 6 * ts_tile);
    // ---- layer-1 epilogue: bias + ReLU, 3xTF32 split -> the A operand of layer 2 (this thread's 32 columns) ---------------------
    {
      const float* bias = b1 + c0;
      uint32_t ra[16], rb[16];
      tmem_ld16_issue(lane_base + d_cur + c0, ra);
      tmem_ld16_issue(lane_base + d_cur + c0 + 16, rb);
      tmem_ld_wait(ra);
      tmem_ld_wait(rb);
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t (&acc)[16] = half ? rb : ra;
        float hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float h = fmaxf(__uint_as_float(acc[j]) + bias[16 * half + j], 0.f);
          tf32_split(h, hi[j], lo[j]);
        }
        tmem_st16(lane_base + kColAHi + c0 + 16 * half, hi);
        tmem_st16(lane_base + kColALo + c0 + 16 * half, lo);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      if (image_groups_pending == 1) { mbar_wait(bar + 3, 0); image_groups_pending = 0; }   // W2
      tc_fence_before();
      __syncthreads();
      TSG(g_ts_forward, 5 + 6 * ts_tile);
      if (t == 0) {
        tc_fence_after();
        issue_layer<kHidden / 8, kHidden, kPanelBytes>(tmem, d_cur, smem_base + kOffW2Hi, smem_base + kOffW2Lo, kHidden / 8);
        mma_commit(bar);
      }
      // under the layer-2 MMAs (the longest stretch in which the CUDA cores would idle): the next tile's rows are requested (the episode index they
      // hang off was requested at the top of this tile), and the previous tile's head runs on its accumulator block
      if (has_next) fetch_b(key_nxt, xnext);
      if (k > 0) head_tile(d_prev, prev_dst, prev_nrows);
      mbar_wait(bar, parity); parity ^= 1;
      tc_fence_after();
      TSG(g_ts_forward, 6 + 6 * ts_tile);
    }
    prev_dst = dst_row; prev_nrows = nrows;
    TSG(g_ts_forward, 8 + 6 * ts_tile);
    ts_tile += 1;
    dst_row = dst_next;
#pragma unroll
    for (int j = 0; j < 8; ++j) xin[j] = xnext[j];
    // the next tile's first MMAs write D / read A only after the __syncthreads that follows its operand staging, by which time
    // every warp has finished reading this tile's accumulators
  }
  head_tile(((k - 1) & 1) ? kColD1 : kColD0, prev_dst, prev_nrows);   // the last tile's head
  tc_fence_before();
  __syncthreads();
  TSG(g_ts_forward, 30);
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
  TSG(g_ts_forward, 31);
}

// =====================================================================================================================
// Ping-pong variant (default; marl_set_option("tensor_core_pingpong", 0) selects the kernel above).
//
// The kernel above runs one 128-row tile at a time: stage -> MMA -> epilogue -> MMA -> epilogue -> MMA -> output, and while the tensor core
// works the 16 warps wait (and vice versa): both units sat at 20-30 % (profiles/r1_tc_pipeline.md).  TMEM cannot hold a second tile's A operand
// (hi | lo = 256 of 512 columns), but it can hold a second ACCUMULATOR once the head leaves the tensor core:
//     A hi [0,128) | A lo [128,256) | D0 [256,384) | D1 [384,512)
// so consecutive tiles alternate accumulators and the CUDA-core work of one tile runs under the MMAs of its neighbour:
//   * layer 1 reads its A operand from a shared-memory X tile (SS form, K-major SWIZZLE_128B, hi | lo), so its MMAs can be queued while the A
//     columns still hold the previous tile's hidden layer;
//   * the epilogue of layer 1 (bias, ReLU, 3xTF32 split) computes tile k's next A operand INTO REGISTERS under the layer-2 MMAs of tile k - 1
//     and stores it to TMEM the moment those retire;
//   * the layer-2 accumulator of tile k - 1 is pulled into registers in the same breath (tcgen05.ld), which frees its columns for the layer-1
//     MMAs of tile k + 1; the head (out <= 8 columns: 6 x 32 FMAs per thread against the FP32 copy of W3, partials of the four column quarters
//     summed in a fixed order through shared memory) and the output stores then run under the layer-1 (k + 1) + layer-2 (k) MMAs.
// One __syncthreads per tile; MMA completion reaches the warps through two mbarriers (layer 1, layer 2).
// =====================================================================================================================
constexpr int kP2Xs = kOffW3Hi;                                     // X tile hi | lo (2 x 16 KB): where the head panels of the full image would sit
constexpr int kP2Tail = kP2Xs + 2 * kPanelBytes;
constexpr int kP2Part = kP2Tail + kTailBytes;                       // head partials [4 column quarters][128 rows][8]
constexpr int kP2Dst = kP2Part + 4 * kTileRows * kOutPad * 4;      // [4][128] output row indices (a loader may be three tiles ahead of the head that reads them)
constexpr int kP2Bars = kP2Dst + 4 * kTileRows * 4;
constexpr int kP2Smem = kP2Bars + 64 + kTsBytes + 1024;
static_assert(kP2Xs % 1024 == 0 && kP2Smem <= 227 * 1024, "ping-pong forward: shared-memory map");

constexpr int kP2Threads = kTrThreads + 128;   // 16 epilogue warps + one more warpgroup: the MMA-issuing warp and three loader warps
constexpr int kP2Loaders = 96;                 // threads of warps 17..19
constexpr int kP2ReadyArrivals = kTrThreads / 32 + kP2Loaders / 32;

// Warp roles (20 warps).
//   * warp 16 issues every MMA.  tcgen05.mma issue is NOT fire-and-forget: the issuing thread advances at the tensor pipe's pace (measured: 48
//     layer-2 MMAs keep it busy for ~3.7 k cycles, 77 per MMA), so an epilogue warp that also issues is the critical path of every tile.  It waits
//     on the `ready` mbarrier (one arrival per epilogue warp: A operand stored, previous accumulator drained; one per loader warp: X tile staged),
//     queues layer 1 of tile k + 1 and layer 2 of tile k, and commits each group to its own mbarrier.  (A 17-warp block -- the issuer alone in a
//     partial warpgroup -- faults with "illegal memory access" at the first tcgen05.mma; a full warpgroup does not.  Measured, not documented.)
//   * warps 17..19 (loaders) gather the observation rows of the next tile, split them (hi | lo) into the shared-memory X tile as soon as the
//     layer-1 MMAs that read the previous one have retired, and publish each row's output offset: no address arithmetic, no global loads and
//     no decode registers in the epilogue warps.
//   * warps 0..15: epilogues (lane quarter x column quarter of the 128 x 128 tile), head on the CUDA cores.  No block-wide barrier in the loop.
__global__ void __launch_bounds__(kP2Threads, 1) tc_forward2_kernel(FwdParams p, const uint8_t* __restrict__ images) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = align_smem_1024(smem_raw);
  // [0] layer-1 MMAs retired, [1] layer-2 MMAs retired, [2] W1 + tail landed, [3] W2 landed, [4] operands ready (19 warp arrivals)
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kP2Bars);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 5);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  int net, row_begin, row_end;
  cta_rows(p.plan, net, row_begin, row_end);
  if (row_begin >= row_end) { pdl_wait(); return; }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (t == 0) { mbar_init(bar, 1); mbar_init(bar + 1, 1); mbar_init(bar + 2, 1); mbar_init(bar + 3, 1); mbar_init(bar + 4, kP2ReadyArrivals); fence_mbar_init(); }
  pdl_wait();   // nothing above touches global memory (PDL contract, common.cuh)
  pdl_launch_dependents();
  const uint32_t smem_base = smem_u32(smem);
  if (t == 0) {  // TMA bulk copies: W1 + tail first (the first layer-1 MMAs and epilogue need them), then W2
    const uint8_t* src = images + (size_t)net * kImageBytes;
    mbar_expect_tx(bar + 2, (uint32_t)(kOffW2Hi + kTailBytes));
    tma_image_range(smem_base, src, 0, kOffW2Hi, bar + 2);
    tma_bulk_g2s(smem_base + kP2Tail, src + kOffB1, kTailBytes, bar + 2);
    mbar_expect_tx(bar + 3, (uint32_t)(kOffW3Hi - kOffW2Hi));
    tma_image_range(smem_base, src, kOffW2Hi, kOffW3Hi, bar + 3);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int D = p.src.D, out = p.lay.out, k1steps = (D + 7) >> 3;
  const int n_tiles = (row_end - row_begin + kTileRows - 1) / kTileRows;
  uint32_t* dst_s = reinterpret_cast<uint32_t*>(smem + kP2Dst);   // [4][128] output row index of every row of the tiles in flight (0xFFFFFFFF: no row)

  if (warp == kTrThreads / 32) {
    // ---- MMA warp ---------------------------------------------------------------------------------------------------------------------------
    mbar_wait(bar + 2, 0);   // W1 in shared memory
    for (int k = -1; k < n_tiles; ++k) {
      mbar_wait(bar + 4, (uint32_t)(k + 1) & 1u);   // arrival round k + 1
      tc_fence_after();
      if (k == 0) mbar_wait(bar + 3, 0);            // W2 in shared memory
      if (lane == 0) {
        const uint32_t d_next = ((k + 1) & 1) ? kColD1 : kColD0, d_cur = (k & 1) ? kColD1 : kColD0;
        if (k + 1 < n_tiles) {   // tile k + 1's layer 1 goes first: its epilogue then runs under the (long) layer-2 MMAs queued behind it
          issue_l1_ss(tmem + d_next, smem_base + kP2Xs, smem_base + kP2Xs + kPanelBytes, smem_base + kOffW1Hi, smem_base + kOffW1Lo, k1steps);
          mma_commit(bar);
        }
        if (k >= 0) {
          issue_layer<kHidden / 8, kHidden, kPanelBytes>(tmem, d_cur, smem_base + kOffW2Hi, smem_base + kOffW2Lo, kHidden / 8);
          mma_commit(bar + 1);
        }
      }
      __syncwarp();
    }
  } else if (warp > kTrThreads / 32) {
    // ---- loader warps: thread i owns rows i and i + 96 (the latter for i < 32) of every tile.  The row -> (agent slot, unit, offset) decode is done
    // once, with divisions, for tile 0 and then advanced by 128 rows per tile with additions only. --------------------------------------------
    const int i = t - (kTrThreads + 32);
    uint8_t* xs = smem + kP2Xs;
    const int rpa_units = p.plan.units_per_agent, urows = p.plan.unit_rows, q128 = kTileRows / urows, r128 = kTileRows % urows;
    const int n_slots = p.plan.slot_begin[net + 1] - p.plan.slot_begin[net];
    struct RowState { int slot, unit, off; };
    RowState rs[2];
#pragma unroll
    for (int m = 0; m < 2; ++m) {   // virtual row row_begin + i + 96 m of this network
      const int vr = row_begin + i + m * kP2Loaders, rpa = rpa_units * urows;
      rs[m].slot = vr / rpa;
      const int rem = vr - rs[m].slot * rpa;
      rs[m].unit = rem / urows; rs[m].off = rem - rs[m].unit * urows;
    }
    float xv[2][kTcObsDim];
    uint32_t dst[2];
    auto fetch = [&](int tile) {   // registers <- this thread's rows of `tile` (loads stay in flight until they are staged); advances the row state
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const int row = i + m * kP2Loaders;
        dst[m] = 0xFFFFFFFFu;
#pragma unroll
        for (int j = 0; j < kTcObsDim; ++j) xv[m][j] = 0.f;
        if (row < kTileRows && row_begin + tile * kTileRows + row < row_end && rs[m].slot < n_slots) {
          const int agent = p.plan.slot_agent[p.plan.slot_begin[net] + rs[m].slot];
          const TrajView& tv = p.src.traj;
          const float* src;
          if (p.src.mode == 0) { src = p.src.dense + ((size_t)rs[m].unit * p.src.N + agent) * D; dst[m] = (uint32_t)((size_t)rs[m].unit * p.src.N + agent); }
          else {
            src = tv.obs + (((size_t)p.src.idx[rs[m].unit] * tv.N + agent) * (size_t)(tv.T + 1) + rs[m].off) * D;
            dst[m] = (uint32_t)(((size_t)agent * rpa_units + rs[m].unit) * urows + rs[m].off);
          }
#pragma unroll
          for (int j = 0; j < kTcObsDim; ++j) if (j < D) xv[m][j] = src[j];
        }
        // next tile: + 128 rows
        rs[m].off += r128; rs[m].unit += q128;
        if (rs[m].off >= urows) { rs[m].off -= urows; rs[m].unit += 1; }
        while (rs[m].unit >= rpa_units) { rs[m].unit -= rpa_units; rs[m].slot += 1; }
      }
    };
    auto stage = [&](int rnd) {
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const int row = i + m * kP2Loaders;
        if (row < kTileRows) {
          float x8[8];
#pragma unroll
          for (int ch = 0; ch < kTcObsDim / 8; ++ch) {
            if (ch < k1steps) {
#pragma unroll
              for (int j = 0; j < 8; ++j) x8[j] = xv[m][8 * ch + j];
              stage_x_tile(xs, row, ch, x8);
            }
          }
          dst_s[(rnd & 3) * kTileRows + row] = dst[m];
        }
      }
    };
    __syncwarp();
    if (lane == 0) mbar_arrive(bar + 4);   // round 0: tile 0 is staged by the (otherwise idle) epilogue warps, 256 threads with one unit each
    fetch(0);                              // (advances the row state past tile 0; its values are not used)
    if (n_tiles > 1) fetch(1);
    for (int rnd = 1; rnd <= n_tiles; ++rnd) {   // round rnd: X(rnd) staged (if any), then one arrival per warp
      if (rnd < n_tiles) {
        mbar_wait(bar, (uint32_t)(rnd - 1) & 1u);   // layer 1 of tile rnd - 1 has retired: the X tile is free (and arrival round rnd - 1 is complete)
        stage(rnd);
        if (rnd + 1 < n_tiles) fetch(rnd + 1);
      } else {
        mbar_wait(bar + 4, (uint32_t)(rnd - 1) & 1u);   // never two arrivals of one warp in the same phase
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // X tile: written through the generic proxy, read by the tensor core
      __syncwarp();
      if (lane == 0) mbar_arrive(bar + 4);
    }
  } else {
    // ---- epilogue warps -----------------------------------------------------------------------------------------------------------------------
    const int lq = warp & 3, cq = warp >> 2, r = 32 * lq + lane, c0 = 32 * cq;
    const uint32_t lane_base = tmem + ((uint32_t)(32 * lq) << 16);
    const float* b1 = reinterpret_cast<const float*>(smem + kP2Tail);
    const float* b2 = b1 + kHidden;
    const float* b3 = b2 + kHidden;
    const float4* w3f = reinterpret_cast<const float4*>(smem + kP2Tail + (kOffW3F - kOffB1));
    float* part = reinterpret_cast<float*>(smem + kP2Part);
    auto arrive_ready = [&]() {   // this warp's share of the next MMA group's operands is in place
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar + 4);
    };
    // outputs of tile `tile`: partials -> shared, the lane quarter's four warps meet, column quarter 0 adds them in order and stores
    auto head_and_store = [&](int tile, const uint32_t (&ra)[16], const uint32_t (&rb)[16]) {
      float q[kOutPad];
      head_partial(ra, rb, b2 + c0, w3f + (c0 >> 2), out, q);
      named_bar_sync(1 + lq, 128);   // the previous tile's partials have been read
      float4* pp = reinterpret_cast<float4*>(part + ((size_t)cq * kTileRows + r) * kOutPad);
      pp[0] = make_float4(q[0], q[1], q[2], q[3]); pp[1] = make_float4(q[4], q[5], q[6], q[7]);
      named_bar_sync(1 + lq, 128);
      if (cq == 0) {
        const uint32_t dst = dst_s[(tile & 3) * kTileRows + r];
        if (dst != 0xFFFFFFFFu) {
          float* o = p.out + (size_t)dst * out;
#pragma unroll
          for (int a = 0; a < kOutPad; ++a)
            if (a < out) o[a] = (((q[a] + part[((size_t)1 * kTileRows + r) * kOutPad + a]) + part[((size_t)2 * kTileRows + r) * kOutPad + a]) + part[((size_t)3 * kTileRows + r) * kOutPad + a]) + b3[a];
        }
      }
    };
    {  // ---- prologue: tile 0's X tile from here (column quarter cq stages observation columns [8 cq, 8 cq + 8) of row r) ------------------
      const int vr = row_begin + r;
      if (cq < k1steps) {
        float x[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = 0.f;
        uint32_t dst = 0xFFFFFFFFu;
        if (vr < row_end) {
          int agent, unit, off;
          decode_row(p.plan, net, vr, agent, unit, off);
          const TrajView& tv = p.src.traj;
          const float* src;
          if (p.src.mode == 0) { src = p.src.dense + ((size_t)unit * p.src.N + agent) * D; dst = (uint32_t)((size_t)unit * p.src.N + agent); }
          else {
            src = tv.obs + (((size_t)p.src.idx[unit] * tv.N + agent) * (size_t)(tv.T + 1) + off) * D;
            dst = (uint32_t)(((size_t)agent * p.plan.units_per_agent + unit) * p.plan.unit_rows + off);
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) x[j] = (8 * cq + j < D) ? src[8 * cq + j] : 0.f;
        }
        stage_x_tile(smem + kP2Xs, r, cq, x);
        if (cq == 0) dst_s[r] = dst;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      }
    }
    arrive_ready();          // round 0
    mbar_wait(bar + 2, 0);   // biases + FP32 W3 have landed
    uint32_t ph1 = 0, ph2 = 0;
    TS_DECL(smem + kP2Bars + 64, 0, 0);
    TS();

    for (int k = 0; k < n_tiles; ++k) {
      const uint32_t d_cur = (k & 1) ? kColD1 : kColD0, d_prev = (k & 1) ? kColD0 : kColD1;
      // ---- layer-1 epilogue of tile k: bias + ReLU into 32 registers (the layer-2 MMAs of tile k - 1 may still be reading the A columns; the
      // hi | lo split -- 64 registers, this block has 96 per thread -- happens on the way into TMEM) ------------------------------------------
      mbar_wait(bar, ph1); ph1 ^= 1;
      tc_fence_after();
      TS();   // a: layer 1 of tile k retired
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
      TS();   // b: layer-1 epilogue in registers
      // ---- A columns free once the layer-2 MMAs of tile k - 1 have retired; their accumulator comes out in the same breath ----------------
      if (k > 0) { mbar_wait(bar + 1, ph2); ph2 ^= 1; tc_fence_after(); }
      TS();   // c: layer 2 of tile k - 1 retired
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
      TS();   // d: A operand stored, previous accumulator in registers, arrival posted
      if (k > 0) head_and_store(k - 1, r2a, r2b);
      TS();   // e: head + outputs of tile k - 1
    }
    // ---- last tile's outputs ------------------------------------------------------------------------------------------------------------------
    mbar_wait(bar + 1, ph2);
    tc_fence_after();
    {
      const uint32_t d_last = ((n_tiles - 1) & 1) ? kColD1 : kColD0;
      uint32_t r2a[16], r2b[16];
      tmem_ld16_issue(lane_base + d_last + c0, r2a);
      tmem_ld16_issue(lane_base + d_last + c0 + 16, r2b);
      tmem_ld_wait(r2a);
      tmem_ld_wait(r2b);
      TS();
      head_and_store(n_tiles - 1, r2a, r2b);
    }
    TS();
    TS_DUMP("fwd2 [start | per tile: a=L1 retired, b=epilogue 1 in regs, c=L2(k-1) retired, d=A stored + arrival, e=head(k-1) | tail: acc-in-regs, end]");
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// ---- launchers ----------------------------------------------------------------------------------------------------------
int tc_forward_init() {
  MARL_CUDA_TRY(cudaFuncSetAttribute(tc_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBytes));
  MARL_CUDA_TRY(cudaFuncSetAttribute(tc_forward2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kP2Smem));
  return MARL_OK;
}

int launch_pack_weights(const float* theta, const NetLayout& lay, int n_nets, uint8_t* image, cudaStream_t st, uint8_t* bwd_image) {
  dim3 grid((lay.P + 255) / 256, n_nets);   // P > 128 * 128 >= every padded extent
  pack_weights_kernel<<<grid, 256, 0, st>>>(theta, lay, n_nets, image, bwd_image);
  MARL_CUDA_TRY(cudaGetLastError());
  return MARL_OK;
}

int launch_tc_forward(const FwdParams& p, const uint8_t* images, cudaStream_t st) {
  if (tc_pingpong_enabled(0) && p.src.mode < 2) MARL_CUDA_TRY(launch_pdl(tc_forward2_kernel, dim3(p.plan.cta_begin[p.plan.n_nets]), dim3(kP2Threads), kP2Smem, st, p, images));
  else MARL_CUDA_TRY(launch_pdl(tc_forward_kernel, dim3(p.plan.cta_begin[p.plan.n_nets]), dim3(kTrThreads), kTcSmemBytes, st, p, images));
  return MARL_OK;
}

}  // namespace marl
