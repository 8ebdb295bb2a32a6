// tc_common.cuh -- tcgen05 / TMEM / mbarrier primitives and the packed weight-image layout shared by the tensor-core kernels.
// PTX forms and descriptor bit fields follow cute/arch/{mma_sm100_umma,mma_sm100_desc,copy_sm100,tmem_allocator_sm100}.hpp and
// cutlass/arch/barrier.h (vendored CUTLASS headers, read for reference only); bring-up: tools/tc_probe.cu, tools/tc_probe2.cu.
#pragma once
#include "learner.cuh"

namespace marl {


constexpr int kTrThreads = 512;   // 16 warps: lane quarter x column quarter
constexpr int kPanelBytes = kHidden * 128;         // 128 rows x 32 floats
constexpr int kHeadRows = 16;                      // head GEMM uses N = 16 (minimum for M = 128)
constexpr int kHeadPanelBytes = kHeadRows * 128;
// image layout (bytes): W1 hi | W1 lo | W2 hi (4 panels) | W2 lo | W3 hi (4 panels of 16 rows) | W3 lo | b1 | b2 | b3
constexpr int kOffW1Hi = 0, kOffW1Lo = kOffW1Hi + kPanelBytes, kOffW2Hi = kOffW1Lo + kPanelBytes, kOffW2Lo = kOffW2Hi + 4 * kPanelBytes;
constexpr int kOffW3Hi = kOffW2Lo + 4 * kPanelBytes, kOffW3Lo = kOffW3Hi + 4 * kHeadPanelBytes;
constexpr int kOffB1 = kOffW3Lo + 4 * kHeadPanelBytes, kOffB2 = kOffB1 + kHidden * 4, kOffB3 = kOffB2 + kHidden * 4;
constexpr int kOffW3F = kOffB3 + kHeadRows * 4;           // plain FP32 copy of W3 [8][128] (head gradient dH2 = dq x W3)
constexpr int kImageBytes = kOffW3F + kOutPad * kHidden * 4;
// backward image: W2^T as a K-major operand (rows = input features j1, K = output features j2), hi | lo
constexpr int kBwdImageBytes = 8 * kPanelBytes;
constexpr int kTcSmemBytes = kImageBytes + 64 + 1024;
// TMEM columns of the row-per-lane kernels: A hi [0,128), A lo [128,256), D [256,384), head D [384,400)
constexpr uint32_t kColAHi = 0, kColALo = 128, kColD = 256, kColDHead = 384;  // + mbarrier / TMEM slot, + slack for 1024-byte alignment

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// round to TF32 (10-bit mantissa), nearest with ties away from zero: what cvt.rna.tf32.f32 computes for finite inputs, in two
// integer instructions instead of the five the compiler emits for the cvt (its extra work is NaN / infinity handling)
__device__ __forceinline__ float tf32_rn(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }
// 3xTF32 operand split: x = hi + lo with both parts representable in TF32 (lo rounded too: leaving it to the tensor core's
// truncation was measured to make no speed difference)
#ifdef MARL_TF32_SPLIT_RN
__device__ __forceinline__ void tf32_split(float x, float& hi, float& lo) { hi = tf32_rn(x); lo = tf32_rn(x - hi); }
#else
// two instructions instead of five: hi = x with the 13 low mantissa bits cleared (exactly representable in TF32), lo = x - hi (exact in FP32, same sign
// as x, < 2^-10 |x|); the tensor core drops the low 13 bits of lo, i.e. at most 2^-20 |x| -- the same order as the lo*lo term that 3xTF32 omits anyway.
// Measured against the oracle: tests/test_tc_backward_gpu.py (gradient error stays ~1e-6 of the gradient scale, bar 1e-5).
__device__ __forceinline__ void tf32_split(float x, float& hi, float& lo) { hi = __uint_as_float(__float_as_uint(x) & 0xffffe000u); lo = x - hi; }
#endif
// ---- weight image --------------------------------------------------------------------------------------------------
// element (row n, feature k) of a [rows][K] K-major SWIZZLE_128B operand -> byte offset inside its panel set
__device__ __forceinline__ int panel_offset(int n, int k, int panel_bytes) {
  const int p = k >> 5, c = (k >> 2) & 7, w = k & 3;
  return p * panel_bytes + n * 128 + ((c ^ (n & 7)) << 4) + (w << 2);
}
// One parameter (flat index j of a network, value x) -> its entries of the packed forward image `img` and, when present, of the
// backward image `bwd` (W2^T).  pack_weights_kernel writes whole images with it; adam_kernel keeps valid images current.
__device__ __forceinline__ void pack_param(const NetLayout& lay, int j, float x, uint8_t* img, uint8_t* bwd) {
  const float hi = tf32_rn(x), lo = tf32_rn(x - hi);
  if (j < lay.b1) {
    const int n = (j - lay.w1) / lay.in, k = (j - lay.w1) - n * lay.in, o = panel_offset(n, k, kPanelBytes);
    *reinterpret_cast<float*>(img + kOffW1Hi + o) = hi; *reinterpret_cast<float*>(img + kOffW1Lo + o) = lo;
  } else if (j < lay.w2) {
    reinterpret_cast<float*>(img + kOffB1)[j - lay.b1] = x;
  } else if (j < lay.b2) {
    const int n = (j - lay.w2) >> 7, k = (j - lay.w2) & 127, o = panel_offset(n, k, kPanelBytes);
    *reinterpret_cast<float*>(img + kOffW2Hi + o) = hi; *reinterpret_cast<float*>(img + kOffW2Lo + o) = lo;
    if (bwd != nullptr) {  // W2^T as a K-major operand: row = input feature, K = output feature
      const int ob = panel_offset(k, n, kPanelBytes);
      *reinterpret_cast<float*>(bwd + ob) = hi; *reinterpret_cast<float*>(bwd + 4 * kPanelBytes + ob) = lo;
    }
  } else if (j < lay.w3) {
    reinterpret_cast<float*>(img + kOffB2)[j - lay.b2] = x;
  } else if (j < lay.b3) {
    const int n = (j - lay.w3) >> 7, k = (j - lay.w3) & 127, o = panel_offset(n, k, kHeadPanelBytes);
    *reinterpret_cast<float*>(img + kOffW3Hi + o) = hi; *reinterpret_cast<float*>(img + kOffW3Lo + o) = lo;
    reinterpret_cast<float*>(img + kOffW3F)[j - lay.w3] = x;
  } else if (j < lay.P) {
    reinterpret_cast<float*>(img + kOffB3)[j - lay.b3] = x;
  }
}

// ---- optional phase timestamps (profiling builds: MARL_NVCC_DEFINES=-DMARL_TC_TIMESTAMPS) ------------------------------------------
// One thread of CTA 5 records clock64() at phase boundaries into shared memory and prints the offsets when the kernel ends.
#ifdef MARL_TC_TIMESTAMPS
constexpr int kTsBytes = 1024;
#define TS_DECL(ptr, thread, slot) long long* ts_ = reinterpret_cast<long long*>(ptr) + 48 * (slot); const bool ts_on_ = (int)threadIdx.x == (thread) && blockIdx.x == 5; \
  int tsi_ = 1; if (ts_on_) { for (int i_ = 1; i_ < 48; ++i_) ts_[i_] = 0; ts_[0] = clock64(); }
#define TS() do { if (ts_on_ && tsi_ < 48) ts_[tsi_++] = clock64(); } while (0)
#define TS_DUMP(name) do { if (ts_on_) { printf("TS %s:", name); for (int i_ = 1; i_ < tsi_; ++i_) printf(" %lld", ts_[i_] - ts_[0]); printf("\n"); } } while (0)
#else
constexpr int kTsBytes = 0;
#define TS_DECL(ptr, thread, slot)
#define TS()
#define TS_DUMP(name)
#endif

// Global timeline probes of the same builds: thread 0 of every CTA stores %globaltimer (ns) and clock64() per probe slot into a per-kernel
// device buffer; tools/ts_timeline.py reads them back through marl_debug_timestamps (launch gaps, prologues, per-tile phases, tail skew).
#ifdef MARL_TC_TIMESTAMPS
constexpr int kTsgCtas = 160, kTsgSlots = 32;
#define TSG_DEFINE(name) static __device__ unsigned long long name[kTsgCtas][kTsgSlots][2];
#define TSG(name, slot) do { if (threadIdx.x == 0 && blockIdx.x < kTsgCtas && (slot) < kTsgSlots) { unsigned long long g_; \
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g_)); name[blockIdx.x][(slot)][0] = g_; name[blockIdx.x][(slot)][1] = (unsigned long long)clock64(); } } while (0)
#define TSG_GETTER(fn, name) int fn(unsigned long long* out) { return cudaMemcpyFromSymbol(out, name, sizeof(name)) == cudaSuccess ? 0 : -1; }
// the same probe plus a progress mark per WARP in host-mapped memory (dbg: [3 kernels][160 CTAs][32 warps], slot + 1 of the last probe the warp
// passed): readable from the host while a kernel hangs (tools/debug_hang.py)
#define TSGP(name, dbg, kid, slot) do { TSG(name, slot); if ((dbg) != nullptr && (threadIdx.x & 31) == 0 && blockIdx.x < kTsgCtas) { \
  *reinterpret_cast<volatile unsigned long long*>((dbg) + ((kid) * kTsgCtas + blockIdx.x) * 32 + (threadIdx.x >> 5)) = (unsigned long long)((slot) + 1); } } while (0)
#else
#define TSGP(name, dbg, kid, slot)
#define TSG_DEFINE(name)
#define TSG(name, slot)
#define TSG_GETTER(fn, name) int fn(unsigned long long*) { return -1; }
#endif
int tsg_forward(unsigned long long* out); int tsg_fwd(unsigned long long* out); int tsg_dh1(unsigned long long* out); int tsg_dw(unsigned long long* out);
int tsg_dh12(unsigned long long* out); int tsg_adam(unsigned long long* out);
int tsg_fwd3(unsigned long long* out); int tsg_dh1w1(unsigned long long* out); int tsg_dw2(unsigned long long* out);

// dynamic shared memory rounded up to 1024 bytes (swizzle atoms), keeping the pointer in the shared address space so that the
// compiler emits LDS / STS rather than generic loads and stores
__device__ __forceinline__ uint8_t* align_smem_1024(uint8_t* raw) { return raw + ((1024u - ((uint32_t)__cvta_generic_to_shared(raw) & 1023u)) & 1023u); }

// ---- tcgen05 helpers -------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start >> 4, LBO 1, SBO 1024 B,
// version 1, layout type 2
__device__ __forceinline__ uint64_t kmajor_desc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32, both K-major, M = 128
__device__ __forceinline__ uint32_t idesc_tf32(int n) { return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24); }

__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
      "}" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// MN-major tf32 operand: SWIZZLE_128B_BASE32B (layout type 1), 4-row swizzle period (SBO 512 B), LBO = byte stride between
// 32-feature panels.  Element (k, mn) lives at panel mn/32, row k (128 B), 32-byte unit ((mn % 32) / 8) ^ (k & 3), word mn % 8.
__device__ __forceinline__ uint64_t mnmajor_desc(uint32_t smem_addr, uint32_t lbo_bytes) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)(512 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)1 << 61);
}
__device__ __forceinline__ int mn_offset(int k, int mn, int panel_bytes) {
  return (mn >> 5) * panel_bytes + k * 128 + ((((mn >> 3) & 3) ^ (k & 3)) << 5) + ((mn & 7) << 2);
}
__device__ __forceinline__ uint32_t idesc_tf32_major(int n, int a_mn, int b_mn) { return idesc_tf32(n) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16); }
__device__ __forceinline__ void mma_tf32_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// ---- TMA bulk copy (cp.async.bulk, SASS UBLKCP): one thread moves a contiguous, 16-byte aligned block global -> shared; completion is
// counted in bytes on an mbarrier (expect_tx by the issuing thread).  The packed weight images are byte-for-byte shared-memory images, so
// an image (or a slice of it) is one instruction instead of a loop of per-thread cp.async, and the writes arrive through the async proxy,
// the one the tensor core reads operands through.
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem), "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// copy bytes [begin, end) of an image to the same offsets of its shared-memory copy, in pieces of at most 32 KB; the caller has armed `bar`
// with the total byte count of everything it sends to it (mbar_expect_tx, once)
__device__ __forceinline__ void tma_image_range(uint32_t smem_base, const uint8_t* src, int begin, int end, uint64_t* bar) {
  for (int o = begin; o < end; o += 32768) tma_bulk_g2s(smem_base + (uint32_t)o, src + o, (uint32_t)min(32768, end - o), bar);
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// the forward image in the order the first tile needs it: bars[0] <- W1 + biases + FP32 W3, bars[1] <- W2, bars[2] <- W3 (one thread)
__device__ __forceinline__ void tma_forward_image(uint32_t smem_base, const uint8_t* src, uint64_t* bars) {
  mbar_expect_tx(bars + 0, (uint32_t)(kOffW2Hi + (kImageBytes - kOffB1)));
  tma_image_range(smem_base, src, kOffW1Hi, kOffW2Hi, bars + 0);
  tma_image_range(smem_base, src, kOffB1, kImageBytes, bars + 0);
  mbar_expect_tx(bars + 1, (uint32_t)(kOffW3Hi - kOffW2Hi));
  tma_image_range(smem_base, src, kOffW2Hi, kOffW3Hi, bars + 1);
  mbar_expect_tx(bars + 2, (uint32_t)(kOffB1 - kOffW3Hi));
  tma_image_range(smem_base, src, kOffW3Hi, kOffB1, bars + 2);
}
// the same without the tensor-core operand copies of W3 (head on the CUDA cores): bars[0] <- W1 + biases + FP32 W3, bars[1] <- W2
__device__ __forceinline__ void tma_forward_image_nohead(uint32_t smem_base, const uint8_t* src, uint64_t* bars) {
  mbar_expect_tx(bars + 0, (uint32_t)(kOffW2Hi + (kImageBytes - kOffB1)));
  tma_image_range(smem_base, src, kOffW1Hi, kOffW2Hi, bars + 0);
  tma_image_range(smem_base, src, kOffB1, kImageBytes, bars + 0);
  mbar_expect_tx(bars + 1, (uint32_t)(kOffW3Hi - kOffW2Hi));
  tma_image_range(smem_base, src, kOffW2Hi, kOffW3Hi, bars + 1);
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(uint32_t addr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
                 "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
               : "r"(addr));
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]),
                 "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// issue only; the caller waits with tmem_ld_wait() before touching r[]
__device__ __forceinline__ void tmem_ld16_issue(uint32_t addr, uint32_t (&r)[16]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
                 "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
               : "r"(addr));
}
// the registers are in/out operands of the wait so that no use of them can be scheduled ahead of it
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]),
                 "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t addr, const float (&v)[16]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(addr),
               "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])),
               "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])),
               "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])), "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])),
               "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
               : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t addr, const float (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(addr), "r"(__float_as_uint(v[0])),
               "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])),
               "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
               : "memory");
}

// ---- the tensor-core training pass (tc_train.cu: one tile at a time; tc_train2.cu: two accumulators) -----------------------------------------------
constexpr int kRowRec = 16;  // floats per row record: [0] g, [1] act, [2..3] spare, [4..7] mask1, [8..11] mask2

struct TcTrainParams {
  RowPlan plan; RowSource src; NetLayout lay;
  const uint8_t* images;      // forward images [n_nets][kImageBytes]
  const uint8_t* bwd_images;  // backward images [n_nets][kBwdImageBytes]
  float* q_out;               // [rows][out] online outputs (optional)
  // H1, H2, dH1: [32 float4 column chunks][rows][4] -- chunk-major, so that a warp whose lanes are 32 consecutive rows writes or
  // reads 512 contiguous bytes per instruction (row-major rows of 512 B cost one cache line per lane and instruction)
  float* h1g; float* h2g; float* dh1g; size_t rows;
  float* rec;                 // [rows][kRowRec] row records
  float* xg;                  // [rows][kTcObsDim] gathered observation rows (zero padded to the staged width): the weight-gradient
                              // kernel reads them without chasing the episode index again
  const float* tq; const float* td_ext; int td_agent_stride; float gamma; int double_q;
  float* scratch; int scratch_pitch; float* loss_part;
  unsigned long long* dbg;    // profiling builds: host-mapped progress marks (NULL otherwise)
};
unsigned long long* tc_debug_progress_ptr();   // core.cu

int tc_train2_init();
int tc_train3_init();
int launch_tc_dqn_train3(const TcTrainParams& p, int grid, cudaStream_t st, cudaEvent_t* between);   // tc_train3.cu: activations stay on chip
int launch_tc_dqn_fwd2(const TcTrainParams& p, int grid, cudaStream_t st);
int launch_tc_dh12(const TcTrainParams& p, int grid, cudaStream_t st);

// ---- pieces shared by the two-accumulator (ping-pong) kernels: tc_forward2_kernel, tc_dqn_fwd2_kernel, tc_dh12_kernel ---------------------------
constexpr int kTailBytes = kImageBytes - kOffB1;                    // b1 | b2 | b3 | FP32 W3
constexpr uint32_t kColD0 = 256, kColD1 = 384;                      // TMEM: A hi [0,128) | A lo [128,256) | D0 | D1
// a 128 x 128 x 128 product in TS form (A hi | lo in the TMEM A columns, B = K-major SWIZZLE_128B hi / lo images of four 32-feature panels):
// 3 terms x 16 k-steps, fully unrolled, issued by one thread
__device__ __forceinline__ void issue_kmajor_ts(uint32_t tmem, uint32_t d_col, uint32_t b_hi, uint32_t b_lo) {
  const uint32_t idesc = idesc_tf32(kHidden);
  const uint64_t dhi = kmajor_desc(b_hi), dlo = kmajor_desc(b_lo);
#pragma unroll
  for (int term = 0; term < 3; ++term)
#pragma unroll
    for (int ks = 0; ks < kHidden / 8; ++ks)
      mma_tf32_ts(tmem + d_col, tmem + (term == 0 ? kColALo : kColAHi) + ks * 8, (term == 1 ? dlo : dhi) + (uint32_t)(((ks >> 2) * kPanelBytes + (ks & 3) * 32) >> 4), idesc,
                  (term | ks) ? 1u : 0u);
}
// layer 1 in SS form: D = X_lo*W_hi + X_hi*W_lo + X_hi*W_hi, both operands K-major SWIZZLE_128B panels of 32 features (one thread)
__device__ __forceinline__ void issue_l1_ss(uint32_t d_tmem, uint32_t xs_hi, uint32_t xs_lo, uint32_t w_hi, uint32_t w_lo, int ksteps) {
  const uint32_t idesc = idesc_tf32(kHidden);
  const uint64_t ahi = kmajor_desc(xs_hi), alo = kmajor_desc(xs_lo), bhi = kmajor_desc(w_hi), blo = kmajor_desc(w_lo);
#pragma unroll
  for (int term = 0; term < 3; ++term)
#pragma unroll
    for (int ks = 0; ks < kTcObsDim / 8; ++ks)
      if (ks < ksteps) mma_tf32_ss(d_tmem, (term == 0 ? alo : ahi) + (uint32_t)((ks * 32) >> 4), (term == 1 ? blo : bhi) + (uint32_t)((ks * 32) >> 4), idesc, (term | ks) ? 1u : 0u);
}
// this thread's 8 observation columns of its row -> the K-major SWIZZLE_128B X tile (hi | lo): 16-byte chunk c of row r sits at chunk c ^ (r & 7)
__device__ __forceinline__ void stage_x_tile(uint8_t* xs, int r, int cq, const float (&x)[8]) {
  float4 h0, h1, l0, l1;
  tf32_split(x[0], h0.x, l0.x); tf32_split(x[1], h0.y, l0.y); tf32_split(x[2], h0.z, l0.z); tf32_split(x[3], h0.w, l0.w);
  tf32_split(x[4], h1.x, l1.x); tf32_split(x[5], h1.y, l1.y); tf32_split(x[6], h1.z, l1.z); tf32_split(x[7], h1.w, l1.w);
  const int o0 = r * 128 + (((2 * cq) ^ (r & 7)) << 4), o1 = r * 128 + (((2 * cq + 1) ^ (r & 7)) << 4);
  *reinterpret_cast<float4*>(xs + o0) = h0; *reinterpret_cast<float4*>(xs + o1) = h1;
  *reinterpret_cast<float4*>(xs + kPanelBytes + o0) = l0; *reinterpret_cast<float4*>(xs + kPanelBytes + o1) = l1;
}
__device__ __forceinline__ void named_bar_sync(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }

// head on the CUDA cores: this thread's 32 columns of relu(D + b2) against the FP32 copy of W3 -> 8 partial outputs of its row.  Packed FP32
// (fma.rn.f32x2, sm_100): even and odd columns accumulate in the two halves of a register pair and are added at the end (fixed order).
__device__ __forceinline__ void head_partial(const uint32_t (&ra)[16], const uint32_t (&rb)[16], const float* b2c, const float4* w3c, int out, float (&q)[kOutPad]) {
  float2 q2[kOutPad];
#pragma unroll
  for (int a = 0; a < kOutPad; ++a) q2[a] = make_float2(0.f, 0.f);
#pragma unroll
  for (int g = 0; g < 8; ++g) {
    const uint32_t (&acc)[16] = g < 4 ? ra : rb;
    const int o = 4 * (g & 3);
    const float4 bb = *reinterpret_cast<const float4*>(b2c + 4 * g);
    float2 h01 = __fadd2_rn(make_float2(__uint_as_float(acc[o]), __uint_as_float(acc[o + 1])), make_float2(bb.x, bb.y));
    float2 h23 = __fadd2_rn(make_float2(__uint_as_float(acc[o + 2]), __uint_as_float(acc[o + 3])), make_float2(bb.z, bb.w));
    h01.x = fmaxf(h01.x, 0.f); h01.y = fmaxf(h01.y, 0.f); h23.x = fmaxf(h23.x, 0.f); h23.y = fmaxf(h23.y, 0.f);
#pragma unroll
    for (int a = 0; a < kOutPad; ++a) {
      if (a < out) {
        const float4 w = w3c[a * (kHidden / 4) + g];
        q2[a] = __ffma2_rn(h23, make_float2(w.z, w.w), __ffma2_rn(h01, make_float2(w.x, w.y), q2[a]));
      }
    }
  }
#pragma unroll
  for (int a = 0; a < kOutPad; ++a) q[a] = q2[a].x + q2[a].y;
}


}  // namespace marl
