// mlp.cuh -- CTA-level building blocks of the fused per-agent MLP (in -> H -> H -> out) forward / backward.
//
// Restates, as hand-tiled FP32 FFMA GEMMs on shared-memory tiles, what the reference runs as three nn.Linear +
// ReLU calls and their autograd backward: marlbase/utils/models.py:14-48 (FCNetwork), :133-173
// (MultiAgentIndependentNetwork), :176-300 (MultiAgentSharedNetwork).
//
// Tile shape: R = 128 rows (one row = one observation of one agent) x H = 128 features, 256 threads, every
// thread owns an 8x8 register block.  All activations and weights are row-major [row][K] in shared memory; 128-wide
// tiles use a 132-float pitch, 16-wide tiles an XOR swizzle, so that every 128-bit shared load of the three GEMM forms
// below is bank-conflict free:
//   NT  C[r][n] = sum_k A[r][k] * B[n][k]     (forward layers: A = activations, B = nn.Linear weight [out][in])
//   TN  C[m][n] = sum_r A[r][m] * B[r][n]     (weight gradients: A = dOut, B = layer input)
//   NN  C[r][n] = sum_k A[r][k] * B[k][n]     (input gradients: B = nn.Linear weight in its native layout)
// FP32 is kept end to end (parity <= 1e-5 against the reference's float32 CPU path, SURVEY H3).
#pragma once
#include "common.cuh"

namespace marl {

constexpr int kTileRows = 128;
constexpr int kHidden = 128;
constexpr int kMlpThreads = 256;
constexpr int kOutPad = 8;

struct ThreadCoord {
  int wy, wx, ty, tx;
  __device__ ThreadCoord() {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    wy = warp >> 1; wx = warp & 1; ty = lane >> 3; tx = lane & 7;
  }
};

// Row pitch (floats) of a [rows][KP] shared-memory tile.  128-wide tiles are padded to 132 floats: linear addresses
// (base register + immediate offsets in the unrolled GEMM loops, no per-load address arithmetic) and still conflict
// free for every 128-bit access pattern below (row stride 132 words = 4 banks).  Narrow tiles (K = 16: observations,
// first-layer weights) keep a dense pitch with the 16-byte chunk index XOR-swizzled by the row.
template <int KP>
constexpr int pitch_of() { return KP == 128 ? 132 : KP; }
constexpr int kPitchH = 132;

// Wide inputs (33..128 features, KP = kKpWide): the input tile is gathered at full width into the H2 region ([128][132], like H2), but a
// resident [128][128] first-layer weight tile does not fit next to W2, H1 and H2.  Layer 1 therefore walks the input in K-chunks of
// kW1Chunk columns, staging chunk c of W1 into the [128][kW1Chunk] slot the narrow tiles keep W1 in (see mlp_forward_tile_wide).
constexpr int kKpWide = 128;
constexpr int kW1Chunk = 32;
template <int KP>
constexpr int w1_kp() { return KP == kKpWide ? kW1Chunk : KP; }   // width of the shared-memory W1 slot

// physical 16-byte chunk of logical chunk c in `row`
template <int KP>
__device__ __forceinline__ int swz(int row, int c) {
  if constexpr (KP == 128) return c;
  else if constexpr (KP >= 32) return c ^ (row & 7);
  else return c ^ ((row >> 1) & 3);
}
template <int KP>
__device__ __forceinline__ float4& at4(float* base, int row, int c) {
  return reinterpret_cast<float4*>(base + row * pitch_of<KP>())[swz<KP>(row, c)];
}
template <int KP>
__device__ __forceinline__ const float4& at4(const float* base, int row, int c) {
  return reinterpret_cast<const float4*>(base + row * pitch_of<KP>())[swz<KP>(row, c)];
}
template <int KP>
__device__ __forceinline__ float& at1(float* base, int row, int k) {
  return base[row * pitch_of<KP>() + swz<KP>(row, k >> 2) * 4 + (k & 3)];
}
template <int KP>
__device__ __forceinline__ const float& at1(const float* base, int row, int k) {
  return base[row * pitch_of<KP>() + swz<KP>(row, k >> 2) * 4 + (k & 3)];
}

// 4-byte asynchronous global->shared copy (LDGSTS): fire and forget, completion via cp_async_wait_all + barrier
__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gsrc) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

__device__ __forceinline__ void zero_acc(float (&acc)[8][8]) {
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
}

// ---- NT: acc[i][j] = sum_k A[r_i][k] * B[n_j][k];  r_i = wy*32 + 4i + ty,  n_j = wx*64 + 8j + tx ------------------
template <int KP>
__device__ __forceinline__ void gemm_nt(const float* __restrict__ A, const float* __restrict__ B, const ThreadCoord& tc, float (&acc)[8][8]) {
  const int r0 = tc.wy * 32 + tc.ty, n0 = tc.wx * 64 + tc.tx;
#pragma unroll 2
  for (int c = 0; c < KP / 4; ++c) {
    float4 a[8], b[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = at4<KP>(A, r0 + 4 * i, c);
#pragma unroll
    for (int j = 0; j < 8; ++j) b[j] = at4<KP>(B, n0 + 8 * j, c);
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        acc[i][j] = fmaf(a[i].x, b[j].x, acc[i][j]);
        acc[i][j] = fmaf(a[i].y, b[j].y, acc[i][j]);
        acc[i][j] = fmaf(a[i].z, b[j].z, acc[i][j]);
        acc[i][j] = fmaf(a[i].w, b[j].w, acc[i][j]);
      }
  }
}

// Forward-layer epilogue: out[r_i][n_j] = relu(acc + bias[n_j]) into a [128][128] swizzled tile.
__device__ __forceinline__ void store_relu_bias(float* __restrict__ out, const float* __restrict__ bias, const ThreadCoord& tc, const float (&acc)[8][8]) {
  const int r0 = tc.wy * 32 + tc.ty, n0 = tc.wx * 64 + tc.tx;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float bj = bias[n0 + 8 * j];
#pragma unroll
    for (int i = 0; i < 8; ++i) at1<kHidden>(out, r0 + 4 * i, n0 + 8 * j) = fmaxf(acc[i][j] + bj, 0.f);
  }
}

// ---- head: q[r][o] = sum_k H[r][k] * W3[o][k] + b3[o], o < 8 (rows of W3 beyond `out` are zero) ------------------
// thread t: row = t/2, outputs (t%2)*4 .. +3.  W3 is plain [8][128]; q is plain [128][8].
__device__ __forceinline__ void head_forward(const float* __restrict__ H, const float* __restrict__ W3, const float* __restrict__ b3, float* __restrict__ q) {
  const int row = threadIdx.x >> 1, o0 = (threadIdx.x & 1) * 4;
  float s[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};  // even / odd chunks accumulate separately (shorter FMA chains)
#pragma unroll 4
  for (int c = 0; c < kHidden / 4; c += 2) {
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const float4 h = at4<kHidden>(H, row, c + u);
#pragma unroll
      for (int o = 0; o < 4; ++o) {
        const float4 w = reinterpret_cast<const float4*>(W3 + (o0 + o) * kHidden)[c + u];
        s[u][o] = fmaf(h.x, w.x, s[u][o]); s[u][o] = fmaf(h.y, w.y, s[u][o]); s[u][o] = fmaf(h.z, w.z, s[u][o]); s[u][o] = fmaf(h.w, w.w, s[u][o]);
      }
    }
  }
  *reinterpret_cast<float4*>(q + row * kOutPad + o0) =
      make_float4(s[0][0] + s[1][0] + b3[o0], s[0][1] + s[1][1] + b3[o0 + 1], s[0][2] + s[1][2] + b3[o0 + 2], s[0][3] + s[1][3] + b3[o0 + 3]);
}

// ---- TN: acc[mi][nj] = sum_r A[r][m] * B[r][n];  m = wy*32 + (mi/4)*16 + ty*4 + mi%4,  n = wx*64 + (nj/4)*32 + tx*4 + nj%4
template <int KPA, int KPB>
__device__ __forceinline__ void gemm_tn(const float* __restrict__ A, const float* __restrict__ B, int rows, const ThreadCoord& tc, float (&acc)[8][8]) {
  const int mc = tc.wy * 8 + tc.ty, nc = tc.wx * 16 + tc.tx;  // chunk indices
#pragma unroll 4
  for (int r = 0; r < rows; ++r) {
    const float4 a0 = at4<KPA>(A, r, mc), a1 = at4<KPA>(A, r, mc + 4);
    const float4 b0 = at4<KPB>(B, r, nc), b1 = at4<KPB>(B, r, nc + 8);
    const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
  }
}
// global index helpers for the TN output block (dW[m][n], row pitch = ld)
__device__ __forceinline__ int tn_row(const ThreadCoord& tc, int mi) { return tc.wy * 32 + (mi >> 2) * 16 + tc.ty * 4 + (mi & 3); }
__device__ __forceinline__ int tn_col(const ThreadCoord& tc, int nj) { return tc.wx * 64 + (nj >> 2) * 32 + tc.tx * 4 + (nj & 3); }

// ---- NN: acc[i][nj] = sum_k A[r_i][k] * B[k][n];  r_i = wy*32 + 4i + ty,  n as in TN ---------------------------------
__device__ __forceinline__ void gemm_nn(const float* __restrict__ A, const float* __restrict__ B, const ThreadCoord& tc, float (&acc)[8][8]) {
  const int r0 = tc.wy * 32 + tc.ty, nc = tc.wx * 16 + tc.tx;
#pragma unroll 1
  for (int c = 0; c < kHidden / 4; ++c) {
    float4 a[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = at4<kHidden>(A, r0 + 4 * i, c);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const int k = 4 * c + kk;
      const float4 b0 = at4<kHidden>(B, k, nc), b1 = at4<kHidden>(B, k, nc + 8);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float av = kk == 0 ? a[i].x : kk == 1 ? a[i].y : kk == 2 ? a[i].z : a[i].w;
        acc[i][0] = fmaf(av, b0.x, acc[i][0]); acc[i][1] = fmaf(av, b0.y, acc[i][1]);
        acc[i][2] = fmaf(av, b0.z, acc[i][2]); acc[i][3] = fmaf(av, b0.w, acc[i][3]);
        acc[i][4] = fmaf(av, b1.x, acc[i][4]); acc[i][5] = fmaf(av, b1.y, acc[i][5]);
        acc[i][6] = fmaf(av, b1.z, acc[i][6]); acc[i][7] = fmaf(av, b1.w, acc[i][7]);
      }
    }
  }
}

// ---- parameter layout of one network, reference state_dict order (network.0.weight, .0.bias, .2.weight, ...) ------
struct NetLayout {
  int in, out;          // true dims
  int w1, b1, w2, b2, w3, b3, P;  // float offsets, P = total
  __host__ __device__ static NetLayout make(int in_, int out_) {
    NetLayout l; l.in = in_; l.out = out_;
    l.w1 = 0; l.b1 = l.w1 + kHidden * in_; l.w2 = l.b1 + kHidden; l.b2 = l.w2 + kHidden * kHidden;
    l.w3 = l.b2 + kHidden; l.b3 = l.w3 + out_ * kHidden; l.P = l.b3 + out_;
    return l;
  }
};

// Shared-memory weight block of one network.  KP = kKpWide: the W1 slot holds one [128][kW1Chunk] K-chunk at a time (load_w1_chunk_async).
template <int KP>
struct WeightSmem {
  static constexpr int kFloats = kHidden * pitch_of<w1_kp<KP>()>() + kHidden * kPitchH + kOutPad * kHidden + kHidden + kHidden + kOutPad;
  float* w1; float* w2; float* w3; float* b1; float* b2; float* b3;
  __device__ explicit WeightSmem(float* base) {
    w1 = base; w2 = w1 + kHidden * pitch_of<w1_kp<KP>()>(); w3 = w2 + kHidden * kPitchH; b1 = w3 + kOutPad * kHidden; b2 = b1 + kHidden; b3 = b2 + kHidden;
  }
  // cooperative asynchronous load from global params (native layouts) into the swizzled smem layouts; 4-byte
  // cp.async because theta + net*P is only 4-byte aligned.  Caller: cp_async_wait_all() + __syncthreads() before use.
  // (KP = kKpWide: everything but W1, whose chunks are staged per tile)
  __device__ void load_async(const float* __restrict__ theta, const NetLayout& l) {
    if constexpr (KP != kKpWide) {
      for (int i = threadIdx.x; i < kHidden * KP; i += kMlpThreads) {
        const int n = i / KP, k = i % KP;
        if (k < l.in) cp_async4(&at1<KP>(w1, n, k), theta + l.w1 + n * l.in + k);
        else at1<KP>(w1, n, k) = 0.f;
      }
    }
#pragma unroll 8
    for (int i = threadIdx.x; i < kHidden * kHidden; i += kMlpThreads) cp_async4(&at1<kHidden>(w2, i / kHidden, i % kHidden), theta + l.w2 + i);
    for (int i = threadIdx.x; i < kOutPad * kHidden; i += kMlpThreads) {
      if (i / kHidden < l.out) cp_async4(w3 + i, theta + l.w3 + i);
      else w3[i] = 0.f;
    }
    for (int i = threadIdx.x; i < kHidden; i += kMlpThreads) { cp_async4(b1 + i, theta + l.b1 + i); cp_async4(b2 + i, theta + l.b2 + i); }
    if (threadIdx.x < kOutPad) b3[threadIdx.x] = threadIdx.x < l.out ? theta[l.b3 + threadIdx.x] : 0.f;
  }
  // KP = kKpWide: W1[:, c*kW1Chunk .. +kW1Chunk) into the W1 slot (columns >= in zeroed); one warp reads 32 consecutive floats of a row.
  // Caller: the slot's previous readers are past a barrier; cp_async_wait_all() + __syncthreads() before use.
  __device__ void load_w1_chunk_async(const float* __restrict__ theta, const NetLayout& l, int c) const {
    const int k0 = c * kW1Chunk;
#pragma unroll 4
    for (int i = threadIdx.x; i < kHidden * kW1Chunk; i += kMlpThreads) {
      const int n = i / kW1Chunk, k = i % kW1Chunk;
      if (k0 + k < l.in) cp_async4(&at1<kW1Chunk>(w1, n, k), theta + l.w1 + n * l.in + k0 + k);
      else at1<kW1Chunk>(w1, n, k) = 0.f;
    }
  }
};

// ---- NT over one K-chunk of a wide input: acc[i][j] += sum_{k < kW1Chunk} X[r_i][c*kW1Chunk + k] * W1c[n_j][k] ------------------------
// X: the full-width [128][132] input tile, W1c: the staged [128][kW1Chunk] chunk (same thread mapping as gemm_nt)
__device__ __forceinline__ void gemm_nt_chunk(const float* __restrict__ X, int c, const float* __restrict__ W1c, const ThreadCoord& tc, float (&acc)[8][8]) {
  const int r0 = tc.wy * 32 + tc.ty, n0 = tc.wx * 64 + tc.tx, q0 = c * (kW1Chunk / 4);
#pragma unroll 2
  for (int q = 0; q < kW1Chunk / 4; ++q) {
    float4 a[8], b[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = at4<kKpWide>(X, r0 + 4 * i, q0 + q);
#pragma unroll
    for (int j = 0; j < 8; ++j) b[j] = at4<kW1Chunk>(W1c, n0 + 8 * j, q);
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        acc[i][j] = fmaf(a[i].x, b[j].x, acc[i][j]);
        acc[i][j] = fmaf(a[i].y, b[j].y, acc[i][j]);
        acc[i][j] = fmaf(a[i].z, b[j].z, acc[i][j]);
        acc[i][j] = fmaf(a[i].w, b[j].w, acc[i][j]);
      }
  }
}

// x -> h1 -> h2 -> q for one 128-row tile (all buffers in shared memory; caller syncs before use of q).
template <int KP>
__device__ __forceinline__ void mlp_forward_tile(const float* X, float* H1, float* H2, float* Q, const WeightSmem<KP>& w, const ThreadCoord& tc) {
  float acc[8][8];
  zero_acc(acc);
  gemm_nt<KP>(X, w.w1, tc, acc);
  store_relu_bias(H1, w.b1, tc, acc);
  __syncthreads();
  zero_acc(acc);
  gemm_nt<kHidden>(H1, w.w2, tc, acc);
  store_relu_bias(H2, w.b2, tc, acc);
  __syncthreads();
  head_forward(H2, w.w3, w.b3, Q);
}

// The same for a wide input (KP = kKpWide).  On entry X holds the tile's ceil(in / kW1Chunk) * kW1Chunk leading columns and the W1 slot
// holds chunk 0 (staged with the tile, waited for and synced by the caller).  Chunks 1.. are staged here from `theta` (this network's
// parameters, L2-resident), each after every thread is done with the previous one, into the same accumulators: layer 1 costs
// ceil(in / 32) chunk round trips per tile instead of holding a [128][128] W1 that does not fit next to W2, H1 and H2.
__device__ __forceinline__ void mlp_forward_tile_wide(const float* X, float* H1, float* H2, float* Q, const WeightSmem<kKpWide>& w, const float* theta,
                                                      const NetLayout& lay, const ThreadCoord& tc) {
  const int n_chunks = (lay.in + kW1Chunk - 1) / kW1Chunk;
  float acc[8][8];
  zero_acc(acc);
  gemm_nt_chunk(X, 0, w.w1, tc, acc);
#pragma unroll 1
  for (int c = 1; c < n_chunks; ++c) {
    __syncthreads();   // every thread is done with chunk c - 1
    w.load_w1_chunk_async(theta, lay, c);
    cp_async_wait_all();
    __syncthreads();
    gemm_nt_chunk(X, c, w.w1, tc, acc);
  }
  store_relu_bias(H1, w.b1, tc, acc);
  __syncthreads();
  zero_acc(acc);
  gemm_nt<kHidden>(H1, w.w2, tc, acc);
  store_relu_bias(H2, w.b2, tc, acc);
  __syncthreads();
  head_forward(H2, w.w3, w.b3, Q);
}

}  // namespace marl
