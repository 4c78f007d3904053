// TF32 implicit-GEMM convolution on the 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM),
// operands staged by TMA, for the dense stride-1 convolutions that carry >90 % of the MACs of every
// network on the path (3x3 d=1 / d=A, 1x1; MyEfficientLFNet.py:555-565, DistgSSR.py:78-100,
// LF_InterNet.py:55, EPIT.py:24-31,76-90).
//
// GEMM view per tile:  D[128 pixels, NC couts] += A_tap[128 pixels, 32 ch] * W_tap[NC, 32 ch]^T
//   * M tile = TH x TW output pixels (TH*TW = 128). For tap (ky,kx) the A operand is ONE TMA box of the
//     NHWC input shifted by (ky*dil - pad, kx*dil - pad); out-of-image (and, with view blocking,
//     out-of-view) taps are zero-filled by the TMA unit, so padding and EPIT's per-view convs cost
//     nothing. The tensor map is 5-D (c, x-in-block, block-x, y-in-block, image*block-y).
//   * K loop = taps x 32-channel groups; each stage holds A (16 KB) and W (NC x 128 B), both K-major
//     with the 128-byte swizzle that TMA writes and the UMMA descriptors read.
//   * warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM alloc), warps 2-5 = epilogue
//     (TMEM -> registers -> bias/act/alpha/PixelShuffle/residual -> global). Two TMEM accumulator
//     stages let the epilogue of tile i overlap the MMAs of tile i+1. Persistent CTAs, one per SM.
// TF32: activations are converted by the TMA unit (tensor map type TFLOAT32), weights are rounded
// to nearest-even at pack time; accumulation is fp32.
#include <atomic>
#include <cuda.h>
#include <stdlib.h>
#include <string.h>
#include <mutex>
#include <type_traits>
#include <cuda_fp16.h>
#include "lfsr_common.cuh"

namespace lfsr {
namespace tc {

static std::atomic<uint64_t> g_lean_launches{0};   // launches that took conv_tc_lean_kernel (tests assert the path)
static std::atomic<uint64_t> g_halo_launches{0};   // launches that took conv_tc_halo_kernel
constexpr int kThreads = 320;          // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue (two warps per TMEM lane quarter)
constexpr int kEpiWarps = 8;
constexpr int kTmaWarp = 8, kMmaWarp = 9;
constexpr int kMaxStages = 8;
constexpr int kABytes = 128 * 128;     // 128 pixels x 32 floats
constexpr int kTmemCols = 512;
constexpr int kAccStride = 256;        // TMEM columns per accumulator stage
constexpr int kSmemBudget = 225 * 1024;      // stages + epilogue staging (barriers and alignment slack come on top)

// n / d for 0 <= n < 2^31 and a divisor fixed at launch: q = (umulhi(n, mul) + n) >> shift  (round-up method);
// the per-tile coordinate decode of every role would otherwise spend ~100 dependent instructions per division
struct FastDiv { uint32_t mul, shift; };
inline FastDiv make_fastdiv(int d) {
  FastDiv f;
  int s = 0;
  while ((1ll << s) < d) ++s;
  f.shift = (uint32_t)s;
  f.mul = (uint32_t)((((unsigned long long)1 << 32) * (((unsigned long long)1 << s) - (unsigned long long)d)) / (unsigned long long)d + 1);
  return f;
}
__device__ __forceinline__ int fdiv(int n, FastDiv f) { return (int)((__umulhi((uint32_t)n, f.mul) + (uint32_t)n) >> f.shift); }

// Tail-projection table (lfsr_conv_desc.tail_w_host, zero rows beyond cq) passed BY VALUE as a __grid_constant__ kernel
// parameter: the projection's FFMA2s then take each weight from the constant bank at a compile-time offset instead of a
// broadcast LDS - those LDS were about as many shared-memory wavefronts per tile as the MMAs' operand reads.
constexpr int kTailMaxC = 64;
struct TailW { float w[kTailMaxC * 12]; };
struct NoTailW {};
template <bool T> using TailArg = typename std::conditional<T, TailW, NoTailW>::type;

struct Params {
  FastDiv fd_tiles_x, fd_nbx, fd_tiles_y, fd_nby, fd_nchunks, fd_cq, fd_rx;
  int out_mode;                        // 0: fp32 output, 1: fp32 + fp16 copy, 2: fp16 only (lane-per-pixel epilogue only)
  __half* out16; int out16_ld, out16_h, out16_w;       // fp16 NHWC copy of the output (stored geometry)
  int tma_epi, OHc;                    // tma_epi: epilogue stores go through the output tensor map; OHc: conv-output rows per image
  const float* tail_w;                 // tail projection (lfsr_conv_desc.tail_w): [cq][12] in global memory, else null
  int tail_rows;                       // rows of the zero-padded copy in shared memory (cq rounded up to 32)
  int nb_total, nby, nbx, bh, bw;      // blocks: nb_total = images * nby
  int C, cgs, kh, kw, dil_h, dil_w, pad_h, pad_w;
  int cout, NC, nchunks;
  int TH, TW, tw_shift, tiles_y, tiles_x, total_tiles;
  int stages, b_stage_bytes;
  int kps;                             // K-stages (tap x 32-channel group) per smem stage / barrier round trip
  int resident, m_tiles;               // resident: all K-stages of W stay in smem for the CTA's lifetime
  TView out, res, mul;                 // mul: optional elementwise multiplier (conv-output geometry, no shuffle)
  const float* bias;
  int act, mul_act;
  float slope, alpha;
  int ry, rx, shuf_mode, cq, vec;      // vec: floats per lane in the coalesced write-out (4, 2 or 1)
  // A-operand addressing: TMA coordinate d (1..4) of tap t = base_d(tile) + tap_off[t][d-1]; `amode` picks which tile
  // variable feeds which tensor-map dimension (0: same-size conv, dims (c, x, view-x, y, image*view-y);
  // 1: stride along x, dims (c, x%s, x/s, y, image); 2: stride along y, dims (c, x, y%s, y/s, image);
  // 3: stride along both, dims (c, x%s, x/s, y%s, image*y/s))
  int amode, out_rows_per_img;
  int cta2;                            // 1: 2-CTA clusters run ONE tcgen05.mma.cta_group::2 (M = 256) per K-step: each CTA stages its own
                                       //    activation tile and HALF of the weight slice; the leader CTA issues for both
  int w_img_rows;                      // >0: per-image weight sets, this many packed rows apart (streamed B only)
  short tap_off[25][4];
  long long* dbg;                      // optional per-CTA cycle counters (profiles/ experiments), else null
  // halo-block CTA pairs (conv_tc_halo_kernel): blocks of Rout x TWo output pixels; a CTA stages its block's (Rout + 2) x P
  // input pixels (P = TWo + 2) once and each tap's A operand is that buffer read from a row-shifted descriptor, so MMA row m of
  // tile j is the flattened padded position g = 128 j + m = ty * P + tx (tx >= TWo: halo columns, never stored)
  int TWo, Rout, P, Rin, ntiles, strips_x, blocks_y, total_blocks, a_buf_bytes, pdiv_mul;
  FastDiv fd_strips, fd_blocks_y;
};

// ---- PTX wrappers ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  // bounded spin: a protocol bug must fault, not hang the GPU
  for (uint32_t it = 0; it < (1u << 26); ++it) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) return;
  }
  __trap();
}
// one lane of a CONVERGED warp (elect.sync): code under `if (elect_one())` keeps its warp-uniform operands in uniform
// registers, so a tcgen05.mma / tcgen05.commit there is ONE predicated instruction. Under `if (lane == 0)` ptxas cannot
// prove that and wraps every such instruction in an ELECT / BRA.U.ANY loop (~10 instructions, ~40 cycles per MMA).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3,
                                            int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// shared -> global tensor store (bulk async group of the issuing thread); out-of-range elements of the box are dropped
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* map, const void* src, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];"
               ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
// ---- CTA-pair (cta_group::2) forms ------------------------------------------------------------------------------------
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;      // clears the CTA-rank bit of a shared::cluster address -> the leader CTA
__device__ __forceinline__ void tmem_alloc2(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
// both CTAs of the pair issue their loads; the transaction bytes are accounted on the LEADER's mbarrier
__device__ __forceinline__ void tma_load_5d_2sm(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3,
                                                int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
template <int ACC, bool F16 = false>
__device__ __forceinline__ void umma2_tf32_c(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc) {
  if (F16) {
    if (ACC)
      asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 1;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                   ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc) : "memory");
    else
      asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                   ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc) : "memory");
    return;
  }
  if (ACC)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 1;\n\ttcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc) : "memory");
  else
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 0;\n\ttcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc) : "memory");
}
__device__ __forceinline__ void umma2_commit_mc(uint64_t* bar) {      // arrives on the barrier at this offset in BOTH CTAs
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {   // arrive on the leader CTA's barrier from either CTA
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], kind::tf32, issued by one thread
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same with the accumulate flag known at compile time (keeps the single issuing thread's instruction stream short:
// that thread retires one dependent instruction every ~5 cycles, so descriptor arithmetic is what bounds the issue rate)
template <int ACC, bool F16 = false>
__device__ __forceinline__ void umma_tf32_c(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc) {
  if (F16) {      // fp16 operands (K = 16 per instruction over the same 32 bytes per row), fp32 accumulate
    if (ACC)
      asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 1;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                   ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc) : "memory");
    else
      asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                   ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc) : "memory");
    return;
  }
  if (ACC)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 1;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc) : "memory");
  else
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc) : "memory");
}
// issue the K-steps of one (tap, channel-group) stage: descriptors advance by 32 B (= 2 in the >>4 address field)
template <bool FIRST, bool F16 = false>
__device__ __forceinline__ void umma_stage(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, int ksteps) {
  umma_tf32_c<FIRST ? 0 : 1, F16>(tmem_d, a_desc, b_desc, idesc);
  if (ksteps == 4) {
    umma_tf32_c<1, F16>(tmem_d, a_desc + 2, b_desc + 2, idesc);
    umma_tf32_c<1, F16>(tmem_d, a_desc + 4, b_desc + 4, idesc);
    umma_tf32_c<1, F16>(tmem_d, a_desc + 6, b_desc + 6, idesc);
  } else {
    for (int k = 1; k < ksteps; ++k) umma_tf32_c<1, F16>(tmem_d, a_desc + 2 * k, b_desc + 2 * k, idesc);
  }
}
// one smem stage = one tap with all its CGS channel groups (16 KB of A each, B rows b_step apart): 4*CGS MMAs
// issued back to back with nothing but 64-bit adds in between
template <int CGS, bool FIRST, bool F16>
__device__ __forceinline__ void umma_tap(uint32_t tmem_d, uint64_t a_d, uint64_t b_d, uint32_t b_step, uint32_t idesc,
                                         int ksteps_last) {
#pragma unroll
  for (int g = 0; g < CGS; ++g) {
    const uint64_t ad = a_d + (uint64_t)(g * (kABytes >> 4));
    const uint64_t bd = b_d + (uint64_t)(g * b_step);
    if (g == CGS - 1 && ksteps_last != 4) {
      if (FIRST && g == 0) umma_tf32_c<0, F16>(tmem_d, ad, bd, idesc); else umma_tf32_c<1, F16>(tmem_d, ad, bd, idesc);
      for (int k = 1; k < ksteps_last; ++k) umma_tf32_c<1, F16>(tmem_d, ad + 2 * k, bd + 2 * k, idesc);
    } else {
      if (FIRST && g == 0) umma_tf32_c<0, F16>(tmem_d, ad, bd, idesc); else umma_tf32_c<1, F16>(tmem_d, ad, bd, idesc);
      umma_tf32_c<1, F16>(tmem_d, ad + 2, bd + 2, idesc);
      umma_tf32_c<1, F16>(tmem_d, ad + 4, bd + 4, idesc);
      umma_tf32_c<1, F16>(tmem_d, ad + 6, bd + 6, idesc);
    }
  }
}
template <bool FIRST, bool F16>
__device__ __forceinline__ void umma_tap_dispatch(int cgs, uint32_t tmem_d, uint64_t a_d, uint64_t b_d, uint32_t b_step,
                                                  uint32_t idesc, int ksteps_last) {
  switch (cgs) {
    case 1: umma_tap<1, FIRST, F16>(tmem_d, a_d, b_d, b_step, idesc, ksteps_last); break;
    case 2: umma_tap<2, FIRST, F16>(tmem_d, a_d, b_d, b_step, idesc, ksteps_last); break;
    case 3: umma_tap<3, FIRST, F16>(tmem_d, a_d, b_d, b_step, idesc, ksteps_last); break;
    default: umma_tap<4, FIRST, F16>(tmem_d, a_d, b_d, b_step, idesc, ksteps_last); break;
  }
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor: rows of 128 B, 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);   // start address, 16-byte units
  d |= (uint64_t)1 << 16;                      // leading byte offset (unused for swizzled K-major) = 1
  d |= (uint64_t)(1024 >> 4) << 32;            // stride byte offset between 8-row groups
  d |= (uint64_t)1 << 46;                      // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                      // SWIZZLE_128B
  return d;
}
// instruction descriptor: D=f32, A=B=tf32, both K-major, M=128, N=n
__device__ __forceinline__ uint32_t make_idesc(int n, uint32_t fmt = 2u) {      // fmt: 2 = tf32, 0 = f16
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

struct TileCoord {
  int chunk, nb, y0, vx, x0;
};
// i-th tile of this CTA. Streaming mode: round-robin over (m-tile, cout-chunk). Resident mode: the CTA
// keeps one cout-chunk's weights in smem, so its chunk is fixed and only the m-tile advances.
__device__ __forceinline__ bool next_tile(const Params& p, int i, int& m, int& chunk) {
  if (p.cta2) {           // cluster c = blockIdx / 2 walks tile pairs; rank r of the cluster owns tile 2*pair + r
    const int pr = (int)(blockIdx.x >> 1) + i * (int)(gridDim.x >> 1);
    if (2 * pr >= p.m_tiles) return false;
    m = 2 * pr + (int)(blockIdx.x & 1);
    if (m >= p.m_tiles) m = -1;         // odd tail: the partner runs a dummy tile (loads valid data, stores nothing)
    chunk = 0;
    return true;
  }
  if (p.resident) {
    const int b = fdiv((int)blockIdx.x, p.fd_nchunks);
    chunk = (int)blockIdx.x - b * p.nchunks;
    m = b + i * fdiv((int)gridDim.x, p.fd_nchunks);
    return m < p.m_tiles;
  }
  const int t = blockIdx.x + i * gridDim.x;
  if (t >= p.total_tiles) return false;
  m = fdiv(t, p.fd_nchunks);
  chunk = t - m * p.nchunks;
  return true;
}
__device__ __forceinline__ TileCoord decode_tile(const Params& p, int t, int chunk) {
  TileCoord c;
  if (t < 0) t = p.m_tiles - 1;      // dummy tile of a CTA pair: valid coordinates, nothing is stored
  c.chunk = chunk;
  int u = fdiv(t, p.fd_tiles_x);
  c.x0 = (t - u * p.tiles_x) * p.TW; t = u;
  u = fdiv(t, p.fd_nbx);
  c.vx = t - u * p.nbx; t = u;
  u = fdiv(t, p.fd_tiles_y);
  c.y0 = (t - u * p.tiles_y) * p.TH;
  c.nb = u;
  return c;
}

// Coalesced write-out of a warp's staged [32 pixels][<=32 packed channels] block. V floats per lane.
// packed channel pc = sub*cq + c ("factor-major": the weights are packed in that order when an
// nn.PixelShuffle is fused), sub = i*rx + j selects the output pixel of the shuffle.
// Everything that does not depend on the pixel row is hoisted: the loop body is ~25 instructions.
template <int ACT>
__device__ __forceinline__ float act_t(float v, float slope) {
  if (ACT == LFSR_ACT_RELU) return fmaxf(v, 0.f);
  if (ACT == LFSR_ACT_LRELU) return v > 0.f ? v : v * slope;
  if (ACT == LFSR_ACT_SIGMOID) return __fdividef(1.f, 1.f + __expf(-v));
  if (ACT == LFSR_ACT_GELU) return 0.5f * v * (1.f + erff(v * 0.70710678118654752f));
  if (ACT == LFSR_ACT_SILU) return __fdividef(v, 1.f + __expf(-v));
  return v;
}

template <int V, bool HAS_MUL, bool HAS_RES>
__device__ __forceinline__ void epi_writeout(const Params& p, const float* stg, int lane, int q, const TileCoord& tc_, int pc0,
                                             int ncols) {
  constexpr int LPR = 32 / V;   // lanes per pixel row
  // rows handled together. The loop is written in phases (coordinates, global loads, shared loads, math, stores), each
  // over all NB rows, so that NB independent memory operations are in flight: with two epilogue warps per scheduler
  // the write-out is latency-bound, not issue-bound.
  constexpr int NB = (V == 4 && !(HAS_MUL && HAS_RES)) ? 8 : 4;
  const int r2 = p.ry * p.rx;
  const int col = (lane % LPR) * V;
  const int pc = pc0 + col;
  if (col >= ncols || pc >= p.cout) return;
  int sub = 0, c = pc;
  if (r2 > 1) { sub = fdiv(pc, p.fd_cq); c = pc - sub * p.cq; }
  const int si = r2 > 1 ? sub / p.rx : 0, sj = r2 > 1 ? sub - si * p.rx : 0;
  const bool chan_major = r2 > 1 && p.shuf_mode == LFSR_SHUF_CHANNEL_MAJOR;
  float bv[V];
#pragma unroll
  for (int e = 0; e < V; ++e) bv[e] = p.bias ? __ldg(p.bias + (chan_major ? (c + e) * r2 + sub : pc + e)) : 0.f;
  const int img = fdiv(tc_.nb, p.fd_nby);
  const int oy0 = ((tc_.nb - img * p.nby) * p.bh + tc_.y0) * p.ry + si;      // output row of tile pixel (0,0)
  const int ox0 = (tc_.vx * p.bw + tc_.x0) * p.rx + sj;
  float* const obase = p.out.p + p.out.pix(img, oy0, ox0) + c;
  const float* const rbase = HAS_RES ? p.res.p + p.res.pix(img, oy0, ox0) + c : nullptr;
  const float* const mbase = HAS_MUL ? p.mul.p + p.mul.pix(img, oy0, ox0) + c : nullptr;
  const int m_py = p.mul.w * p.mul.ld, m_px = p.mul.ld;
  const int o_py = p.ry * p.out.w * p.out.ld, o_px = p.rx * p.out.ld;         // float pitch per tile row / column
  const int r_py = p.ry * p.res.w * p.res.ld, r_px = p.rx * p.res.ld;
  const bool full = tc_.y0 + p.TH <= p.bh && tc_.x0 + p.TW <= p.bw;
  const int tw_mask = p.TW - 1;
  const int rows_valid = min(p.TH, p.bh - tc_.y0), cols_valid = min(p.TW, p.bw - tc_.x0);
  const float slope = p.slope, alpha = p.alpha;
  const bool mul_silu = p.mul_act == LFSR_ACT_SILU;   // the one multiplier activation the networks use (checked on the host)
  const int swz_hi = col >> 2, swz_lo = col & 3;
  const int lrow = lane / LPR;
#pragma unroll 1
  for (int it0 = 0; it0 < LPR; it0 += NB) {
    int tyx[NB];                       // (ty << 16) | tx of the row's tile pixel, or -1 when it lies outside the image
#pragma unroll
    for (int j = 0; j < NB; ++j) {
      const int m = q * 32 + (it0 + j) * V + lrow;
      const int ty = m >> p.tw_shift, tx = m & tw_mask;
      tyx[j] = (full || (ty < rows_valid && tx < cols_valid)) ? ((ty << 16) | tx) : -1;
    }
    // residual / multiplier operands first (longest latency). The stores below may alias `res` (in-place residuals),
    // which is why the compiler cannot hoist these itself; every lane reads exactly the addresses it later writes.
    float mv[HAS_MUL ? NB : 1][V], rv[HAS_RES ? NB : 1][V];
    if (HAS_MUL) {
#pragma unroll
      for (int j = 0; j < NB; ++j) {
#pragma unroll
        for (int e = 0; e < V; ++e) mv[j][e] = 1.f;
        if (tyx[j] >= 0) {
          const float* ms = mbase + (tyx[j] >> 16) * m_py + (tyx[j] & 0xffff) * m_px;
          if (V == 4) { const float4 t = *reinterpret_cast<const float4*>(ms); mv[j][0] = t.x; mv[j][1 % V] = t.y; mv[j][2 % V] = t.z; mv[j][3 % V] = t.w; }
          else if (V == 2) { const float2 t = *reinterpret_cast<const float2*>(ms); mv[j][0] = t.x; mv[j][1 % V] = t.y; }
          else mv[j][0] = *ms;
        }
      }
    }
    if (HAS_RES) {
#pragma unroll
      for (int j = 0; j < NB; ++j) {
#pragma unroll
        for (int e = 0; e < V; ++e) rv[j][e] = 0.f;
        if (tyx[j] >= 0) {
          const float* rs = rbase + (tyx[j] >> 16) * r_py + (tyx[j] & 0xffff) * r_px;
          if (V == 4) { const float4 t = *reinterpret_cast<const float4*>(rs); rv[j][0] = t.x; rv[j][1 % V] = t.y; rv[j][2 % V] = t.z; rv[j][3 % V] = t.w; }
          else if (V == 2) { const float2 t = *reinterpret_cast<const float2*>(rs); rv[j][0] = t.x; rv[j][1 % V] = t.y; }
          else rv[j][0] = *rs;
        }
      }
    }
    float v[NB][V];
#pragma unroll
    for (int j = 0; j < NB; ++j) {
      const int r = (it0 + j) * V + lrow;
      const float* src = stg + r * 32 + (((swz_hi ^ (r & 7)) << 2) | swz_lo);
      if (V == 4) { const float4 t = *reinterpret_cast<const float4*>(src); v[j][0] = t.x; v[j][1 % V] = t.y; v[j][2 % V] = t.z; v[j][3 % V] = t.w; }
      else if (V == 2) { const float2 t = *reinterpret_cast<const float2*>(src); v[j][0] = t.x; v[j][1 % V] = t.y; }
      else v[j][0] = *src;
    }
#define LFSR_EPI_ACT(A)                                                                  \
  _Pragma("unroll") for (int j = 0; j < NB; ++j) {                                       \
    _Pragma("unroll") for (int e = 0; e < V; ++e) v[j][e] = act_t<A>(v[j][e] + bv[e], slope); \
  }
    switch (p.act) {                   // one uniform branch per NB rows
      case LFSR_ACT_RELU: LFSR_EPI_ACT(LFSR_ACT_RELU) break;
      case LFSR_ACT_LRELU: LFSR_EPI_ACT(LFSR_ACT_LRELU) break;
      case LFSR_ACT_SIGMOID: LFSR_EPI_ACT(LFSR_ACT_SIGMOID) break;
      case LFSR_ACT_GELU: LFSR_EPI_ACT(LFSR_ACT_GELU) break;
      case LFSR_ACT_SILU: LFSR_EPI_ACT(LFSR_ACT_SILU) break;
      default: LFSR_EPI_ACT(LFSR_ACT_NONE) break;
    }
#undef LFSR_EPI_ACT
    if (HAS_MUL) {
#pragma unroll
      for (int j = 0; j < NB; ++j) {
#pragma unroll
        for (int e = 0; e < V; ++e) v[j][e] *= mul_silu ? __fdividef(mv[j][e], 1.f + __expf(-mv[j][e])) : mv[j][e];
      }
    }
#pragma unroll
    for (int j = 0; j < NB; ++j) {
#pragma unroll
      for (int e = 0; e < V; ++e) v[j][e] *= alpha;
    }
    if (HAS_RES) {
#pragma unroll
      for (int j = 0; j < NB; ++j) {
#pragma unroll
        for (int e = 0; e < V; ++e) v[j][e] += rv[j][e];
      }
    }
#pragma unroll
    for (int j = 0; j < NB; ++j) {
      if (tyx[j] >= 0) {
        float* dst = obase + (tyx[j] >> 16) * o_py + (tyx[j] & 0xffff) * o_px;
        if (V == 4) *reinterpret_cast<float4*>(dst) = make_float4(v[j][0], v[j][1 % V], v[j][2 % V], v[j][3 % V]);
        else if (V == 2) *reinterpret_cast<float2*>(dst) = make_float2(v[j][0], v[j][1 % V]);
        else *dst = v[j][0];
      }
    }
  }
}

template <int V>
__device__ __forceinline__ void epi_writeout_act(const Params& p, const float* stg, int lane, int q, const TileCoord& tc_,
                                                 int pc0, int ncols) {
  const bool m = p.mul.p != nullptr, r = p.res.p != nullptr;
  if (m && r) epi_writeout<V, true, true>(p, stg, lane, q, tc_, pc0, ncols);
  else if (m) epi_writeout<V, true, false>(p, stg, lane, q, tc_, pc0, ncols);
  else if (r) epi_writeout<V, false, true>(p, stg, lane, q, tc_, pc0, ncols);
  else epi_writeout<V, false, false>(p, stg, lane, q, tc_, pc0, ncols);
}

// TMEM accumulator (32 lanes x NC columns of this warp) -> staged transpose -> coalesced global stores
__device__ __forceinline__ void epilogue_tile(const Params& p, float* stg, uint32_t taddr, int lane, int q, const TileCoord& tc_,
                                              int g_first = 0, int g_step = 1, long long* dbg_ld = nullptr) {
  for (int g = g_first; g * 32 < p.NC; g += g_step) {
    const int ncols = p.NC - g * 32 < 32 ? p.NC - g * 32 : 32;
    float v[32];
    long long t0 = 0;
    if (dbg_ld) t0 = clock64();
    tmem_ld16(taddr + g * 32, v);
    if (ncols > 16) tmem_ld16(taddr + g * 32 + 16, v + 16);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (j * 4 < ncols)
        *reinterpret_cast<float4*>(stg + lane * 32 + ((j ^ (lane & 7)) << 2)) =
            make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    __syncwarp();
    if (dbg_ld) *dbg_ld += clock64() - t0;
    const int pc0 = tc_.chunk * p.NC + g * 32;
    if (p.vec == 4) epi_writeout_act<4>(p, stg, lane, q, tc_, pc0, ncols);
    else if (p.vec == 2) epi_writeout_act<2>(p, stg, lane, q, tc_, pc0, ncols);
    else epi_writeout_act<1>(p, stg, lane, q, tc_, pc0, ncols);
    __syncwarp();
  }
}

// Epilogue of one tile for one warp, TMA-store flavour. After tcgen05.ld a lane owns ONE pixel and 32 consecutive packed
// output channels of it, so bias / activation / multiplier / residual are applied in registers with no index math
// (the residual and multiplier runs of the lane's pixel are fetched before the accumulator is even waited for), the
// block is staged as [32 pixels][128 B] in the SWIZZLE_128B pattern and one elected lane hands it to the TMA unit:
// the output tensor map does the addressing, clips partial tiles / channel tails and expresses the PixelShuffle
// (dims (c, j, x, i, row) with packed channel = (i*rx + j)*cq + c). Blocks whose padding columns would alias real
// channels of the next cout-chunk take the per-row write-out instead.
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ void epilogue_tile_tma(const Params& p, const CUtensorMap* tmO, float* stg, uint32_t taddr, int lane, int q,
                                                  const TileCoord& tc_, int g_first, int g_step, uint64_t* tfull_bar,
                                                  uint32_t tfull_parity, long long* dbg_rd = nullptr) {
  const int tw_mask = p.TW - 1;
  const int m = q * 32 + lane;
  const int ty = m >> p.tw_shift, tx = m & tw_mask;
  const bool pix_ok = tc_.y0 + ty < p.bh && tc_.x0 + tx < p.bw;
  const int img = fdiv(tc_.nb, p.fd_nby);
  // at most one of residual / multiplier is fused here (the host sends layers that use both to the per-row write-out),
  // so one 32-register operand run per block is prefetched
  const bool is_mul = p.mul.p != nullptr;
  const float* xpix = nullptr;
  const int Y = (tc_.nb - img * p.nby) * p.bh + tc_.y0 + ty, X = tc_.vx * p.bw + tc_.x0 + tx;
  const bool shuf_res = p.res.p && p.ry * p.rx > 1;     // residual in stored-output geometry: its pixel depends on the block's sub-pixel
  if (pix_ok && (p.res.p || p.mul.p) && !shuf_res)
    xpix = is_mul ? p.mul.p + p.mul.pix(img, Y, X) : p.res.p + p.res.pix(img, Y, X);
  const int ty_w = (q * 32) >> p.tw_shift, tx_w = (q * 32) & tw_mask;      // origin of the warp's 32-pixel box in the tile
  const int r2 = p.ry * p.rx;
  const bool chan_major = r2 > 1 && p.shuf_mode == LFSR_SHUF_CHANNEL_MAJOR;
  const bool mul_silu = p.mul_act == LFSR_ACT_SILU;
  bool waited = false;
  // column blocks of <= 32 packed channels that never straddle a PixelShuffle sub-pixel run (so each is ONE tensor
  // store whose channel coordinate is >= 0 and 16-byte aligned); the two warps of a lane quarter take alternate blocks
  const int chunk_lo = tc_.chunk * p.NC;
  const int chunk_hi = chunk_lo + p.NC < p.cout ? chunk_lo + p.NC : p.cout;
  int bi = 0;
  long long tp = 0;
#define LFSR_EPI_TICK(i) if (dbg_rd) { const long long t_ = clock64(); dbg_rd[i] += t_ - tp; tp = t_; }
  for (int pc0 = chunk_lo, ncols = 0; pc0 < chunk_hi; pc0 += ncols, ++bi) {
    int sub = 0, c0 = pc0;
    if (r2 > 1) { sub = fdiv(pc0, p.fd_cq); c0 = pc0 - sub * p.cq; }
    ncols = p.cq - c0 < 32 ? p.cq - c0 : 32;
    if (chunk_hi - pc0 < ncols) ncols = chunk_hi - pc0;
    if (bi % g_step != g_first) continue;
    if (dbg_rd) tp = clock64();
    const int tcol = pc0 - chunk_lo;                           // TMEM column of the block
    // columns right of the block are clipped by the channel dim of the tensor store; fp16-only outputs are stored from
    // registers (any block shape), so they always take the lane-per-pixel path
    const bool tma_ok = p.out_mode == 2 || ncols == 32 || c0 + ncols == p.cq;
    float4 xv[8];
    float bcol = 0.f;
    if (tma_ok) {
      const float fill = is_mul ? 1.f : 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        xv[k] = make_float4(fill, fill, fill, fill);
        if (xpix && pc0 + 4 * k < p.cout) xv[k] = *reinterpret_cast<const float4*>(xpix + pc0 + 4 * k);
      }
      if (shuf_res && pix_ok) {
        const int si = fdiv(sub, p.fd_rx), sj = sub - si * p.rx;
        const float* rp = p.res.p + p.res.pix(img, Y * p.ry + si, X * p.rx + sj) + c0;
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (c0 + 4 * k < p.cq) xv[k] = *reinterpret_cast<const float4*>(rp + 4 * k);
      }
      if (p.bias) {
        const int pcl = pc0 + lane;
        if (pcl < p.cout) {
          int bi = pcl;
          if (chan_major) { const int sub = fdiv(pcl, p.fd_cq); bi = (pcl - sub * p.cq) * r2 + sub; }
          bcol = __ldg(p.bias + bi);
        }
      }
    }
    LFSR_EPI_TICK(1)
    if (!waited) { mbar_wait(tfull_bar, tfull_parity); tc_fence_after(); waited = true; }
    LFSR_EPI_TICK(2)
    float v[32];
    tmem_ld16(taddr + tcol, v);
    if (ncols > 16) tmem_ld16(taddr + tcol + 16, v + 16);
    else {
#pragma unroll
      for (int k = 16; k < 32; ++k) v[k] = 0.f;
    }
    LFSR_EPI_TICK(3)
    if (tma_ok) {
      if (p.bias) {
#pragma unroll
        for (int k = 0; k < 32; ++k) v[k] += __shfl_sync(0xffffffffu, bcol, k);
      }
      const float slope = p.slope;
#define LFSR_EPI_ACT32(A) _Pragma("unroll") for (int k = 0; k < 32; ++k) v[k] = act_t<A>(v[k], slope);
      switch (p.act) {
        case LFSR_ACT_RELU: LFSR_EPI_ACT32(LFSR_ACT_RELU) break;
        case LFSR_ACT_LRELU: LFSR_EPI_ACT32(LFSR_ACT_LRELU) break;
        case LFSR_ACT_SIGMOID: LFSR_EPI_ACT32(LFSR_ACT_SIGMOID) break;
        case LFSR_ACT_GELU: LFSR_EPI_ACT32(LFSR_ACT_GELU) break;
        case LFSR_ACT_SILU: LFSR_EPI_ACT32(LFSR_ACT_SILU) break;
        default: break;
      }
#undef LFSR_EPI_ACT32
      if (is_mul) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          float4 t = xv[k];
          if (mul_silu) {
            t.x = __fdividef(t.x, 1.f + __expf(-t.x)); t.y = __fdividef(t.y, 1.f + __expf(-t.y));
            t.z = __fdividef(t.z, 1.f + __expf(-t.z)); t.w = __fdividef(t.w, 1.f + __expf(-t.w));
          }
          v[4 * k] *= t.x; v[4 * k + 1] *= t.y; v[4 * k + 2] *= t.z; v[4 * k + 3] *= t.w;
          xv[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      const float alpha = p.alpha;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        v[4 * k] = fmaf(v[4 * k], alpha, xv[k].x); v[4 * k + 1] = fmaf(v[4 * k + 1], alpha, xv[k].y);
        v[4 * k + 2] = fmaf(v[4 * k + 2], alpha, xv[k].z); v[4 * k + 3] = fmaf(v[4 * k + 3], alpha, xv[k].w);
      }
    }
    LFSR_EPI_TICK(4)
    if (p.out_mode != 2) {
      if (lane == 0) bulk_wait_read0();        // the TMA unit has finished reading the previous block out of `stg`
      __syncwarp();
    }
    LFSR_EPI_TICK(0)
    if (p.out_mode != 2) {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        *reinterpret_cast<float4*>(stg + lane * 32 + ((j ^ (lane & 7)) << 2)) =
            make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    }
    if (p.out_mode != 0 && pix_ok) {      // fp16 copy: the lane's pixel x <= 32 channels = <= 64 contiguous bytes, straight from registers
      int Yo = Y, Xo = X;
      if (r2 > 1) { const int si = fdiv(sub, p.fd_rx), sj = sub - si * p.rx; Yo = Y * p.ry + si; Xo = X * p.rx + sj; }
      __half* dst = p.out16 + ((size_t)((size_t)img * p.out16_h + Yo) * p.out16_w + Xo) * (size_t)p.out16_ld + c0;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (8 * j < ncols)
          *reinterpret_cast<uint4*>(dst + 8 * j) =
              make_uint4(pack_h2(v[8 * j], v[8 * j + 1]), pack_h2(v[8 * j + 2], v[8 * j + 3]), pack_h2(v[8 * j + 4], v[8 * j + 5]),
                         pack_h2(v[8 * j + 6], v[8 * j + 7]));
    }
    LFSR_EPI_TICK(5)
    if (tma_ok) {
      if (p.out_mode != 2) { fence_proxy_async(); __syncwarp(); }
      if (lane == 0 && p.out_mode != 2) {
        if (r2 == 1) {
          tma_store_5d(tmO, stg, c0, tc_.x0 + tx_w, tc_.vx, tc_.y0 + ty_w, tc_.nb);
        } else {
          const int si = fdiv(sub, p.fd_rx), sj = sub - si * p.rx;
          tma_store_5d(tmO, stg, c0, sj, tc_.x0 + tx_w, si, tc_.nb * p.OHc + tc_.y0 + ty_w);
        }
        bulk_commit();
      }
    } else {
      __syncwarp();
      if (p.vec == 4) epi_writeout_act<4>(p, stg, lane, q, tc_, pc0, ncols);
      else if (p.vec == 2) epi_writeout_act<2>(p, stg, lane, q, tc_, pc0, ncols);
      else epi_writeout_act<1>(p, stg, lane, q, tc_, pc0, ncols);
      __syncwarp();
    }
    LFSR_EPI_TICK(6)
  }
#undef LFSR_EPI_TICK
  if (!waited) { mbar_wait(tfull_bar, tfull_parity); tc_fence_after(); }
}

// Epilogue of one tile for one warp when the layer ends in a tail projection (Params::tail_w): the warp owns whole
// PixelShuffle sub-pixels (alternating with its partner warp), a lane owns one pixel, and instead of storing the cq
// activated channels of that output pixel it accumulates their dot products with the <= 12 tail vectors (weights from the
// constant bank in the 16-warp kernels, else broadcast from shared memory) and stores those 12 floats - 48 bytes instead
// of 4*cq per output pixel.
// The projection of one pixel per lane (conv-output pixel (Y, X) of image img) for sub-pixels sub0 + g_first, + g_step, ...
// below sub1; taddr addresses accumulator column sub0 * cq. Shared by the per-tap and the halo-block kernels.
// CW: `tw` is the __grid_constant__ table (cq <= kTailMaxC; both 32-channel blocks unrolled so that every weight offset is
// a compile-time constant), else the zero-padded copy in shared memory.
template <bool CW>
__device__ __forceinline__ void tail_project(const Params& p, const float* tw, uint32_t taddr, int lane, int img, int Y, int X,
                                             bool pix_ok, int sub0, int sub1, int g_first, int g_step) {
  const int r2 = p.ry * p.rx;
  const bool chan_major = p.shuf_mode == LFSR_SHUF_CHANNEL_MAJOR;
  const float slope = p.slope;
  taddr -= sub0 * p.cq;                            // accumulator column of global output column pc0 is pc0 - sub0 * cq
  for (int sub = sub0 + g_first; sub < sub1; sub += g_step) {
    f32x2 rp[6];                      // 12 tap responses as 6 packed pairs: the projection is FFMA2 throughout
#pragma unroll
    for (int t = 0; t < 6; ++t) rp[t] = pack2(0.f, 0.f);
#pragma unroll
    for (int cb = 0; cb < (CW ? kTailMaxC / 32 : 1 << 20); ++cb) {
      const int c0 = cb * 32;
      if (c0 >= p.cq) break;
      const int pc0 = sub * p.cq + c0;
      float bcol = 0.f;
      if (p.bias && c0 + lane < p.cq) bcol = __ldg(p.bias + (chan_major ? (c0 + lane) * r2 + sub : pc0 + lane));
      float v[32];
      tmem_ld16(taddr + pc0, v);
      tmem_ld16(taddr + pc0 + 16, v + 16);
      if (p.bias) {
#pragma unroll
        for (int k = 0; k < 32; ++k) v[k] += __shfl_sync(0xffffffffu, bcol, k);
      }
#define LFSR_EPI_ACT32(A) _Pragma("unroll") for (int k = 0; k < 32; ++k) v[k] = act_t<A>(v[k], slope);
      switch (p.act) {
        case LFSR_ACT_RELU: LFSR_EPI_ACT32(LFSR_ACT_RELU) break;
        case LFSR_ACT_LRELU: LFSR_EPI_ACT32(LFSR_ACT_LRELU) break;
        case LFSR_ACT_SIGMOID: LFSR_EPI_ACT32(LFSR_ACT_SIGMOID) break;
        case LFSR_ACT_GELU: LFSR_EPI_ACT32(LFSR_ACT_GELU) break;
        case LFSR_ACT_SILU: LFSR_EPI_ACT32(LFSR_ACT_SILU) break;
        default: break;
      }
#undef LFSR_EPI_ACT32
      // rows >= cq of the shared-memory table are zero, so the columns a short last block shares with the next
      // sub-pixel contribute nothing - provided they are finite: past the last sub-pixel they are accumulator columns this
      // kernel's MMAs never wrote (whatever an earlier kernel left in tensor memory, possibly NaN), so they are cleared
      if (p.cq - c0 < 32) {
#pragma unroll
        for (int k = 0; k < 32; ++k)
          if (c0 + k >= p.cq) v[k] = 0.f;
      }
      const float* wt = tw + c0 * 12;
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        const float a = v[k] * p.alpha;
        const f32x2 aa = pack2(a, a);
#pragma unroll
        for (int t = 0; t < 6; ++t) rp[t] = fma2(aa, pack2(wt[12 * k + 2 * t], wt[12 * k + 2 * t + 1]), rp[t]);
      }
    }
    if (pix_ok) {
      const int si = fdiv(sub, p.fd_rx), sj = sub - si * p.rx;
      float4* dst = reinterpret_cast<float4*>(p.out.p + p.out.pix(img, Y * p.ry + si, X * p.rx + sj));
      float r[12];
#pragma unroll
      for (int t = 0; t < 6; ++t) unpack2(rp[t], r[2 * t], r[2 * t + 1]);
      dst[0] = make_float4(r[0], r[1], r[2], r[3]);
      dst[1] = make_float4(r[4], r[5], r[6], r[7]);
      dst[2] = make_float4(r[8], r[9], r[10], r[11]);
    }
  }
}

template <bool CW>
__device__ __forceinline__ void epilogue_tile_tail(const Params& p, const float* tw, uint32_t taddr, int lane, int q,
                                                   const TileCoord& tc_, int g_first, int g_step, uint64_t* tfull_bar,
                                                   uint32_t tfull_parity) {
  const int m = q * 32 + lane;
  const int ty = m >> p.tw_shift, tx = m & (p.TW - 1);
  const bool pix_ok = tc_.y0 + ty < p.bh && tc_.x0 + tx < p.bw;
  const int img = fdiv(tc_.nb, p.fd_nby);
  const int Y = (tc_.nb - img * p.nby) * p.bh + tc_.y0 + ty, X = tc_.vx * p.bw + tc_.x0 + tx;
  mbar_wait(tfull_bar, tfull_parity);
  tc_fence_after();
  // sub-pixels of this cout-chunk: all of them with one chunk, else NC / cq whole sub-pixels per chunk (host-checked)
  const int r2 = p.ry * p.rx;
  const int sub0 = p.nchunks == 1 ? 0 : tc_.chunk * (p.NC / p.cq);
  const int sub1 = p.nchunks == 1 ? r2 : min(r2, sub0 + p.NC / p.cq);
  tail_project<CW>(p, tw, taddr, lane, img, Y, X, pix_ok, sub0, sub1, g_first, g_step);
}

__device__ __forceinline__ const float* tail_w_of(const TailW& tw, const float*) { return tw.w; }
__device__ __forceinline__ const float* tail_w_of(const NoTailW&, const float* sTail) { return sTail; }

// (register files are allocated for 4-warp groups: 320 threads cost what 384 do, i.e. at most 168 registers each)
// CTA2 = true is a separate instantiation: a kernel that contains cta_group::2 instructions can only be launched in
// clusters of two, so the single-CTA paths must not see them
// DBG = false compiles the cycle counters (LFSR_TC_DBG_PTR) out of the role loops
// F16 = true: the activation tensor is fp16 NHWC (channel groups of 64 = one 128-byte row) and the weights are packed
// as fp16: kind::f16 MMAs, K = 16 per instruction over the same bytes - half the shared-memory traffic and MMA time per MAC
// T16 = true (tail-projection layers): SIXTEEN epilogue warps, one PixelShuffle sub-pixel each - the projection epilogue
// (~1.8 k dependent-latency-bound instructions per warp and tile on 8 warps) bounded the dominant kernel, not the MMAs;
// the other write-outs are compiled out, which keeps the 20 allocated warps inside 96 registers
template <bool CTA2, bool DBG, bool F16, bool T16 = false>
__global__ void __launch_bounds__(T16 ? 640 : kThreads, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmO, const Params p,
               const __grid_constant__ TailArg<T16> tw) {
  constexpr int CG = F16 ? 64 : 32;            // channels per 128-byte row / channel group
  constexpr int kEpiW = T16 ? 16 : kEpiWarps;  // epilogue warps; the TMA producer and the MMA issuer are the two warps after them
  constexpr int kTmaWarp = kEpiW, kMmaWarp = kEpiW + 1;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  uint8_t* sA = smem;
  uint8_t* sB = smem + p.stages * p.kps * kABytes;
  const int taps = p.kh * p.kw;
  const int nks = taps * p.cgs;
  float* sEpi = reinterpret_cast<float*>(sB + (CTA2 ? p.stages * p.kps * (p.b_stage_bytes >> 1)         // (half slices)
                                                      : (p.resident ? nks : p.stages * p.kps) * p.b_stage_bytes));   // 8 warps x 4 KB
  float* sTail = sEpi + kEpiWarps * 1024;                                                                  // tail_rows x 12
  uint64_t* bars = reinterpret_cast<uint64_t*>(sTail + p.tail_rows * 12);
  uint64_t* full = bars;
  uint64_t* empty = bars + kMaxStages;
  uint64_t* tfull = bars + 2 * kMaxStages;
  uint64_t* tempty = tfull + 2;
  uint64_t* bfull = tempty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bfull + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (!T16)
    for (int i = threadIdx.x; i < p.tail_rows * 12; i += (int)blockDim.x) sTail[i] = i < p.cq * 12 ? __ldg(p.tail_w + i) : 0.f;
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull + a, 1); mbar_init(tempty + a, CTA2 ? 2 * kEpiW : kEpiW); }
    mbar_init(bfull, 1);
    fence_barrier_init();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (CTA2) tma_prefetch_desc(&tmBh);
    if (p.tma_epi) tma_prefetch_desc(&tmO);
  }
  // warp roles: 0..7 epilogue, 8 TMA producer, 9 MMA issuer. The scheduler favours the highest warp id of a
  // sub-partition, so the latency-critical single-thread roles get the top ids (B300_MICROARCH: hi-wid-first).
  if (CTA2) cluster_sync_all();      // both CTAs are resident before the paired allocation is requested
  if (warp == kMmaWarp) { if (CTA2) tmem_alloc2(tmem_slot, kTmemCols); else tmem_alloc(tmem_slot, kTmemCols); }
  tc_fence_before();
  __syncthreads();
  if (CTA2) cluster_sync_all();     // the partner's barriers must be initialised before anything is multicast to them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kTmaWarp) {
    // ================= TMA producer: ONE elected lane runs the whole role loop (see elect_one()) =================
    if (elect_one()) {
      int s_ring = 0;
      uint32_t ph_ring = 0;
      const uint32_t stage_bytes = kABytes + (p.resident ? 0 : p.NC * 128);
      int m, chunk;
      if (p.resident && next_tile(p, 0, m, chunk)) {
        // one-time load of this CTA's whole weight set
        mbar_expect_tx(bfull, (uint32_t)nks * p.b_stage_bytes);
        for (int ks = 0; ks < nks; ++ks)
          tma_load_2d(sB + ks * p.b_stage_bytes, &tmB, bfull, 0, (chunk * nks + ks) * p.NC);
      }
      if (CTA2) {        // stage = {own A tile, own HALF (NC/2 rows) of one (tap, channel group) of B}; bytes land on the leader's barrier
        const int crank2 = (int)cluster_ctarank();
        const int half_rows = p.NC >> 1;
        for (int i = 0; next_tile(p, i, m, chunk); ++i) {
          const TileCoord t0 = decode_tile(p, m, 0);
          int cg = 0, tap = 0;
          for (int ks = 0; ks < nks; ks += p.kps) {           // a smem stage holds kps K-stages (fewer barrier round trips per tile)
            if (s_ring == p.stages) { s_ring = 0; ph_ring ^= 1; }
            const int s = s_ring++;
            mbar_wait(empty + s, ph_ring ^ 1);                // own barrier: the multicast commit arrives in both CTAs
            const int nsub = nks - ks < p.kps ? nks - ks : p.kps;
            if (crank2 == 0) mbar_expect_tx(full + s, (uint32_t)nsub * (2u * kABytes + (uint32_t)p.NC * 128u));   // both CTAs' loads
            for (int u = 0; u < nsub; ++u) {
              const short* to = p.tap_off[tap];
              const int slot = s * p.kps + u;
              tma_load_5d_2sm(sA + slot * kABytes, &tmA, full + s, cg * CG, t0.x0 + to[0], t0.vx + to[1], t0.y0 + to[2], t0.nb + to[3]);
              tma_load_2d_2sm(sB + slot * (p.b_stage_bytes >> 1), &tmBh, full + s, 0, (ks + u) * p.NC + crank2 * half_rows);
              if (++cg == p.cgs) { cg = 0; ++tap; }
            }
          }
        }
      } else
      for (int i = 0; next_tile(p, i, m, chunk); ++i) {
        const TileCoord tc_ = decode_tile(p, m, chunk);
        int cg = 0, tap = 0;
        int b1, b2, b3, b4;      // tile part of the TMA coordinates
        if (p.amode == 0) { b1 = tc_.x0; b2 = tc_.vx; b3 = tc_.y0; b4 = tc_.nb; }
        else if (p.amode == 1) { b1 = 0; b2 = tc_.x0; b3 = tc_.y0; b4 = tc_.nb; }
        else if (p.amode == 2) { b1 = tc_.x0; b2 = 0; b3 = tc_.y0; b4 = tc_.nb; }
        else { b1 = 0; b2 = tc_.x0; b3 = 0; b4 = tc_.nb * p.out_rows_per_img + tc_.y0; }
        const int w_row0 = tc_.chunk * nks * p.NC + (tc_.nb / p.nby) * p.w_img_rows;
        for (int ks = 0; ks < nks; ks += p.kps) {
          if (s_ring == p.stages) { s_ring = 0; ph_ring ^= 1; }
          const int s = s_ring++;
          mbar_wait(empty + s, ph_ring ^ 1);
          const int nsub = nks - ks < p.kps ? nks - ks : p.kps;
          mbar_expect_tx(full + s, (uint32_t)nsub * stage_bytes);
          for (int u = 0; u < nsub; ++u) {
            const short* to = p.tap_off[tap];
            const int slot = s * p.kps + u;
            tma_load_5d(sA + slot * kABytes, &tmA, full + s, cg * CG, b1 + to[0], b2 + to[1], b3 + to[2], b4 + to[3]);
            if (!p.resident) tma_load_2d(sB + slot * p.b_stage_bytes, &tmB, full + s, 0, w_row0 + (ks + u) * p.NC);
            if (++cg == p.cgs) { cg = 0; ++tap; }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == kMmaWarp) {
    // ================= MMA issuer =================
    // The whole role loop runs in ONE lane chosen by elect.sync, inside a single elect block: no per-stage __syncwarp /
    // re-election (probe_mma_rate2.py: leaving and re-entering the elect block costs the tensor pipe ~200 cycles per
    // stage at N = 64) and, unlike `if (lane == 0)`, ptxas keeps the tcgen05 operands in uniform registers. That lane is in
    // lock-step with the tensor pipe (the MMA queue is shallow), so everything here that is not a tcgen05.mma is overhead.
    if (elect_one()) {
      long long dbg_full_wait = 0, dbg_acc_wait = 0, dbg_mma = 0;
      const long long dbg_t0 = clock64();
      uint32_t tcount = 0;
      int s_ring = 0;
      uint32_t ph_ring = 0;
      const uint32_t idesc = make_idesc(p.NC, F16 ? 0u : 2u);
      const uint64_t a_desc0 = make_smem_desc(smem_u32(sA)), b_desc0 = make_smem_desc(smem_u32(sB));
      const int rem_last = p.C - (p.cgs - 1) * CG;
      const int ksteps_last = rem_last >= CG ? 4 : (F16 ? (rem_last + 15) >> 4 : (rem_last + 7) >> 3);
      const uint32_t b_step = (uint32_t)(p.b_stage_bytes >> 4);
      const uint32_t a_stage_step = (uint32_t)(p.kps * (kABytes >> 4)), b_stage_step = (uint32_t)p.kps * b_step;
      const bool tap_stages = p.kps == p.cgs;
      int m, chunk;
      if (p.resident && next_tile(p, 0, m, chunk)) mbar_wait(bfull, 0);
      if (CTA2) {
        if (cluster_ctarank() == 0) {        // the leader issues M = 256 MMAs for the pair; the partner's MMA warp idles
          const uint32_t idesc2 = (idesc & ~(0x1fu << 24)) | ((uint32_t)(256 >> 4) << 24);
          const uint32_t b_half_step = b_step >> 1;
          for (int i = 0; next_tile(p, i, m, chunk); ++i, ++tcount) {
            const uint32_t a = tcount & 1, aph = (tcount >> 1) & 1;
            long long tw0 = 0;
            if ((DBG && p.dbg)) tw0 = clock64();
            mbar_wait(tempty + a, aph ^ 1);               // both CTAs' epilogues have drained this accumulator stage
            if ((DBG && p.dbg)) dbg_acc_wait += clock64() - tw0;
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + a * kAccStride;
            int cg_i = 0;
            for (int ks = 0; ks < nks; ks += p.kps) {
              if (s_ring == p.stages) { s_ring = 0; ph_ring ^= 1; }
              const int s = s_ring++;
              if ((DBG && p.dbg)) tw0 = clock64();
              mbar_wait(full + s, ph_ring);
              long long tw1 = 0;
              if ((DBG && p.dbg)) { tw1 = clock64(); dbg_full_wait += tw1 - tw0; }
              tc_fence_after();
              const int nsub = nks - ks < p.kps ? nks - ks : p.kps;
              uint64_t a_d = a_desc0 + (uint64_t)(s * p.kps) * (kABytes >> 4);
              uint64_t b_d = b_desc0 + (uint64_t)(s * p.kps) * b_half_step;
              for (int u = 0; u < nsub; ++u) {
                const int ksteps = (cg_i == p.cgs - 1) ? ksteps_last : 4;
                if (ks + u == 0) umma2_tf32_c<0, F16>(d_tmem, a_d, b_d, idesc2); else umma2_tf32_c<1, F16>(d_tmem, a_d, b_d, idesc2);
                if (ksteps == 4) {
                  umma2_tf32_c<1, F16>(d_tmem, a_d + 2, b_d + 2, idesc2);
                  umma2_tf32_c<1, F16>(d_tmem, a_d + 4, b_d + 4, idesc2);
                  umma2_tf32_c<1, F16>(d_tmem, a_d + 6, b_d + 6, idesc2);
                } else {
                  for (int k = 1; k < ksteps; ++k) umma2_tf32_c<1, F16>(d_tmem, a_d + 2 * k, b_d + 2 * k, idesc2);
                }
                if (++cg_i == p.cgs) cg_i = 0;
                a_d += (uint64_t)(kABytes >> 4); b_d += (uint64_t)b_half_step;
              }
              umma2_commit_mc(empty + s);
              if (ks + p.kps >= nks) umma2_commit_mc(tfull + a);
              if ((DBG && p.dbg)) dbg_mma += clock64() - tw1;
            }
          }
        }
      } else
      for (int i = 0; next_tile(p, i, m, chunk); ++i, ++tcount) {
        const uint32_t a = tcount & 1, aph = (tcount >> 1) & 1;
        long long tw0 = 0;
        if ((DBG && p.dbg)) tw0 = clock64();
        mbar_wait(tempty + a, aph ^ 1);
        if ((DBG && p.dbg)) dbg_acc_wait += clock64() - tw0;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + a * kAccStride;
        int cg_i = 0;
        for (int ks = 0; ks < nks; ks += p.kps) {
          if (s_ring == p.stages) { s_ring = 0; ph_ring ^= 1; }
          const int s = s_ring++;
          if ((DBG && p.dbg)) tw0 = clock64();
          mbar_wait(full + s, ph_ring);
          long long tw1 = 0;
          if ((DBG && p.dbg)) { tw1 = clock64(); dbg_full_wait += tw1 - tw0; }
          tc_fence_after();
          const uint64_t a_d0 = a_desc0 + (uint64_t)(s * a_stage_step);
          const uint64_t b_d0 = b_desc0 + (uint64_t)(p.resident ? ks * b_step : s * b_stage_step);
          if (tap_stages) {              // stage == one tap with all channel groups: fully unrolled issue
            if (ks == 0) umma_tap_dispatch<true, F16>(p.cgs, d_tmem, a_d0, b_d0, b_step, idesc, ksteps_last);
            else umma_tap_dispatch<false, F16>(p.cgs, d_tmem, a_d0, b_d0, b_step, idesc, ksteps_last);
          } else if (p.kps == 1) {       // stage == one (tap, channel group)
            const int ksteps = (cg_i == p.cgs - 1) ? ksteps_last : 4;
            if (ks == 0) umma_stage<true, F16>(d_tmem, a_d0, b_d0, idesc, ksteps);
            else umma_stage<false, F16>(d_tmem, a_d0, b_d0, idesc, ksteps);
            if (++cg_i == p.cgs) cg_i = 0;
          } else {
            const int nsub = nks - ks < p.kps ? nks - ks : p.kps;
            for (int u = 0; u < nsub; ++u) {
              const int ksteps = (cg_i == p.cgs - 1) ? ksteps_last : 4;
              const uint64_t a_d = a_d0 + (uint64_t)(u * (kABytes >> 4));
              const uint64_t b_d = b_d0 + (uint64_t)(u * b_step);
              if (ks + u == 0) umma_stage<true, F16>(d_tmem, a_d, b_d, idesc, ksteps);
              else umma_stage<false, F16>(d_tmem, a_d, b_d, idesc, ksteps);
              if (++cg_i == p.cgs) cg_i = 0;
            }
          }
          umma_commit(empty + s);                            // frees the smem stage when these MMAs retire
          if (ks + p.kps >= nks) umma_commit(tfull + a);     // accumulator complete -> epilogue
          if ((DBG && p.dbg)) dbg_mma += clock64() - tw1;
        }
      }
      if ((DBG && p.dbg)) {
        p.dbg[blockIdx.x * 8 + 2] = dbg_full_wait; p.dbg[blockIdx.x * 8 + 3] = dbg_acc_wait;
        p.dbg[blockIdx.x * 8 + 4] = dbg_mma; p.dbg[blockIdx.x * 8 + 5] = clock64() - dbg_t0;
      }
    }
    __syncwarp();
  } else {
    // ================= epilogue (warps 0..7 <-> TMEM lane quarters, two warps each) =================
    // TMEM -> registers (one pixel row per lane) -> 4 KB swizzled smem transpose per warp ->
    // coalesced vector stores (consecutive lanes write consecutive bytes of a pixel's channel run).
    const int q = warp & 3;
    const int half = warp >> 2;                // the two warps of a lane quarter split the 32-column groups
    float* stg = sEpi + (T16 ? 0 : warp * 1024);
    uint32_t tcount = 0;
    int m_, chunk_;
    long long dbg_wait = 0, dbg_t0 = 0, tw0 = 0, dbg_epi = 0;
    long long dbg_seg[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long& dbg_ld = dbg_seg[0];
    if ((DBG && p.dbg)) dbg_t0 = clock64();
    for (int i = 0; next_tile(p, i, m_, chunk_); ++i, ++tcount) {
      const uint32_t a = tcount & 1, aph = (tcount >> 1) & 1;
      const TileCoord tc_ = decode_tile(p, m_, chunk_);
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + a * kAccStride;
      long long tw1 = 0;
      if (T16) {
        if (m_ >= 0) epilogue_tile_tail<T16>(p, tail_w_of(tw, sTail), taddr, lane, q, tc_, half, 4, tfull + a, aph);
        else { mbar_wait(tfull + a, aph); tc_fence_after(); }
      } else if (p.tail_w && m_ >= 0) {
        epilogue_tile_tail<false>(p, sTail, taddr, lane, q, tc_, half, 2, tfull + a, aph);
      } else if (p.tma_epi && m_ >= 0) {
        if ((DBG && p.dbg)) tw1 = clock64();
        epilogue_tile_tma(p, &tmO, stg, taddr, lane, q, tc_, half, 2, tfull + a, aph, (DBG && p.dbg) ? dbg_seg : nullptr);
        if ((DBG && p.dbg)) dbg_epi += clock64() - tw1;
      } else {
        if ((DBG && p.dbg)) tw0 = clock64();
        mbar_wait(tfull + a, aph);
        if ((DBG && p.dbg)) dbg_wait += clock64() - tw0;
        tc_fence_after();
        if ((DBG && p.dbg)) tw1 = clock64();
        if (m_ >= 0) epilogue_tile(p, stg, taddr, lane, q, tc_, half, 2, (DBG && p.dbg) ? &dbg_ld : nullptr);
        if ((DBG && p.dbg)) dbg_epi += clock64() - tw1;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { if (CTA2) mbar_arrive_leader(tempty + a); else mbar_arrive(tempty + a); }
    }
    if (p.tma_epi && lane == 0) bulk_wait0();     // all of this warp's tensor stores have landed
    if ((DBG && p.dbg) && threadIdx.x == 0) p.dbg[blockIdx.x * 8 + 0] = dbg_ld;        // TMA path: cycles waiting for the store unit to release the staging buffer
    if ((DBG && p.dbg) && threadIdx.x == 0) {
      p.dbg[blockIdx.x * 8 + 1] = dbg_epi;
      p.dbg[blockIdx.x * 8 + 6] = dbg_wait; p.dbg[blockIdx.x * 8 + 7] = clock64() - dbg_t0;
      for (int k = 1; k < 7; ++k) p.dbg[gridDim.x * 8 + blockIdx.x * 8 + k] = dbg_seg[k];     // (second table: phases inside the TMA-store epilogue)
    }
  }
  __syncthreads();
  if (CTA2) cluster_sync_all();     // no CTA may exit while its partner can still multicast into it
  if (warp == kMmaWarp) {
    __syncwarp();
    if (CTA2) tmem_dealloc2(tmem_base, kTmemCols); else tmem_dealloc(tmem_base, kTmemCols);
  }
}


// ======================= lean kernel: narrow fp16 layers, TWO CTAs per SM ===========================================
// probe_tc_roles16.py / the ncu source view of the N <= 64 layers on fp16 operands: nothing is saturated (tensor pipe 22 %,
// L2 -> SM 32 %, shared memory 32 %); a tile is a chain of dependent latencies - TMA round trip per 2-stage ring, ~300 cycles
// per stage boundary of the issuing lane, and a ~3-4 k-cycle epilogue per 32 x 32 block on 2 warps per scheduler. Two
// independent CTAs per SM overlap each other's bubbles. That needs <= 80 registers (2 x 12 allocated warps) and <= 113 KB /
// 256 TMEM columns per CTA: this kernel keeps only what those layers use - same-size / strided fp16 activations through the
// same tensor maps and stage ring, N <= 64 in one chunk, no PixelShuffle / multiplier / tail projection, bias from shared
// memory, activation none / ReLU / LeakyReLU as one select, residual prefetched before the accumulator wait, the 32-column
// block handled as two 16-column halves (16 live accumulators), output fp32 through the tensor store and / or fp16 from
// registers (OUT_MODE = lfsr_conv_desc.out_mode).
constexpr int kLeanTmemCols = 256;
constexpr int kLeanAccStride = 128;
constexpr int kLeanSmem = 112 * 1024;

// (register files are allocated per 4-warp group: the bound is stated for 384 threads so that ptxas budgets 2 x 12 warps)
template <int OUT_MODE, bool HAS_RES, bool F16>
__global__ void __launch_bounds__(384, 2)
conv_tc_lean_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmO, const Params p) {
  constexpr int CG = F16 ? 64 : 32;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  const int nks = p.kh * p.kw * p.cgs;
  uint8_t* sA = smem;
  uint8_t* sB = smem + p.stages * p.kps * kABytes;
  float* sEpi = reinterpret_cast<float*>(sB + (p.resident ? nks : p.stages * p.kps) * p.b_stage_bytes);
  float* sBias = sEpi + (OUT_MODE != 2 ? kEpiWarps * 1024 : 0);
  uint64_t* bars = reinterpret_cast<uint64_t*>(sBias + 64);
  uint64_t* full = bars;
  uint64_t* empty = bars + kMaxStages;
  uint64_t* tfull = bars + 2 * kMaxStages;
  uint64_t* tempty = tfull + 2;
  uint64_t* bfull = tempty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bfull + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x < 64) sBias[threadIdx.x] = (p.bias && (int)threadIdx.x < p.cout) ? __ldg(p.bias + threadIdx.x) : 0.f;
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull + a, 1); mbar_init(tempty + a, kEpiWarps); }
    mbar_init(bfull, 1);
    fence_barrier_init();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (OUT_MODE != 2) tma_prefetch_desc(&tmO);
  }
  if (warp == kMmaWarp) tmem_alloc(tmem_slot, kLeanTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int G = (int)gridDim.x;

  if (warp == kTmaWarp) {
    if (elect_one()) {
      int s_ring = 0;
      uint32_t ph_ring = 0;
      const uint32_t stage_bytes = kABytes + (p.resident ? 0 : p.NC * 128);
      if (p.resident && (int)blockIdx.x < p.m_tiles) {
        mbar_expect_tx(bfull, (uint32_t)nks * p.b_stage_bytes);
        for (int ks = 0; ks < nks; ++ks) tma_load_2d(sB + ks * p.b_stage_bytes, &tmB, bfull, 0, ks * p.NC);
      }
      for (int m = blockIdx.x; m < p.m_tiles; m += G) {
        const TileCoord tc_ = decode_tile(p, m, 0);
        int cg = 0, tap = 0;
        int b1, b2, b3, b4;
        if (p.amode == 0) { b1 = tc_.x0; b2 = tc_.vx; b3 = tc_.y0; b4 = tc_.nb; }
        else if (p.amode == 1) { b1 = 0; b2 = tc_.x0; b3 = tc_.y0; b4 = tc_.nb; }
        else if (p.amode == 2) { b1 = tc_.x0; b2 = 0; b3 = tc_.y0; b4 = tc_.nb; }
        else { b1 = 0; b2 = tc_.x0; b3 = 0; b4 = tc_.nb * p.out_rows_per_img + tc_.y0; }
        const int w_row0 = p.w_img_rows ? fdiv(tc_.nb, p.fd_nby) * p.w_img_rows : 0;       // per-image (gated) weight sets
        for (int ks = 0; ks < nks; ks += p.kps) {
          if (s_ring == p.stages) { s_ring = 0; ph_ring ^= 1; }
          const int s = s_ring++;
          mbar_wait(empty + s, ph_ring ^ 1);
          const int nsub = nks - ks < p.kps ? nks - ks : p.kps;
          mbar_expect_tx(full + s, (uint32_t)nsub * stage_bytes);
          for (int u = 0; u < nsub; ++u) {
            const short* to = p.tap_off[tap];
            const int slot = s * p.kps + u;
            tma_load_5d(sA + slot * kABytes, &tmA, full + s, cg * CG, b1 + to[0], b2 + to[1], b3 + to[2], b4 + to[3]);
            if (!p.resident) tma_load_2d(sB + slot * p.b_stage_bytes, &tmB, full + s, 0, w_row0 + (ks + u) * p.NC);
            if (++cg == p.cgs) { cg = 0; ++tap; }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == kMmaWarp) {
    if (elect_one()) {
      uint32_t tcount = 0;
      int s_ring = 0;
      uint32_t ph_ring = 0;
      const uint32_t idesc = make_idesc(p.NC, F16 ? 0u : 2u);
      const uint64_t a_desc0 = make_smem_desc(smem_u32(sA)), b_desc0 = make_smem_desc(smem_u32(sB));
      const int rem_last = p.C - (p.cgs - 1) * CG;
      const int ksteps_last = rem_last >= CG ? 4 : (F16 ? (rem_last + 15) >> 4 : (rem_last + 7) >> 3);
      const uint32_t b_step = (uint32_t)(p.b_stage_bytes >> 4);
      const uint32_t a_stage_step = (uint32_t)(p.kps * (kABytes >> 4)), b_stage_step = (uint32_t)p.kps * b_step;
      const bool tap_stages = p.kps == p.cgs;
      if (p.resident && (int)blockIdx.x < p.m_tiles) mbar_wait(bfull, 0);
      for (int m = blockIdx.x; m < p.m_tiles; m += G, ++tcount) {
        const uint32_t a = tcount & 1, aph = (tcount >> 1) & 1;
        mbar_wait(tempty + a, aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + a * kLeanAccStride;
        int cg_i = 0;
        for (int ks = 0; ks < nks; ks += p.kps) {
          if (s_ring == p.stages) { s_ring = 0; ph_ring ^= 1; }
          const int s = s_ring++;
          mbar_wait(full + s, ph_ring);
          tc_fence_after();
          const uint64_t a_d0 = a_desc0 + (uint64_t)(s * a_stage_step);
          const uint64_t b_d0 = b_desc0 + (uint64_t)(p.resident ? ks * b_step : s * b_stage_step);
          if (tap_stages) {
            if (ks == 0) umma_tap_dispatch<true, F16>(p.cgs, d_tmem, a_d0, b_d0, b_step, idesc, ksteps_last);
            else umma_tap_dispatch<false, F16>(p.cgs, d_tmem, a_d0, b_d0, b_step, idesc, ksteps_last);
          } else {
            const int nsub = nks - ks < p.kps ? nks - ks : p.kps;
            for (int u = 0; u < nsub; ++u) {
              const int ksteps = (cg_i == p.cgs - 1) ? ksteps_last : 4;
              const uint64_t a_d = a_d0 + (uint64_t)(u * (kABytes >> 4));
              const uint64_t b_d = b_d0 + (uint64_t)(u * b_step);
              if (ks + u == 0) umma_stage<true, F16>(d_tmem, a_d, b_d, idesc, ksteps);
              else umma_stage<false, F16>(d_tmem, a_d, b_d, idesc, ksteps);
              if (++cg_i == p.cgs) cg_i = 0;
            }
          }
          umma_commit(empty + s);
          if (ks + p.kps >= nks) umma_commit(tfull + a);
        }
      }
    }
    __syncwarp();
  } else {
    // ---- epilogue: warp w <-> TMEM lane quarter w & 3, column block w >> 2 (32 columns); a lane owns one pixel ----
    const int q = warp & 3;
    const int pc0 = (warp >> 2) * 32;
    const int ncols = p.cout - pc0 < 32 ? p.cout - pc0 : 32;         // <= 0: this warp only keeps the barrier phases
    float* stg = sEpi + warp * 1024;
    const int tw_mask = p.TW - 1;
    const int mpx = q * 32 + lane;
    const int ty = mpx >> p.tw_shift, tx = mpx & tw_mask;
    const int ty_w = (q * 32) >> p.tw_shift, tx_w = (q * 32) & tw_mask;
    const float slope = p.act == LFSR_ACT_NONE ? 1.f : (p.act == LFSR_ACT_RELU ? 0.f : p.slope);
    const float alpha = p.alpha;
    uint32_t tcount = 0;
    for (int m = blockIdx.x; m < p.m_tiles; m += G, ++tcount) {
      const uint32_t a = tcount & 1, aph = (tcount >> 1) & 1;
      if (ncols > 0) {
        const TileCoord tc_ = decode_tile(p, m, 0);
        const bool pix_ok = tc_.y0 + ty < p.bh && tc_.x0 + tx < p.bw;
        const int img = fdiv(tc_.nb, p.fd_nby);
        const int Y = (tc_.nb - img * p.nby) * p.bh + tc_.y0 + ty, X = tc_.vx * p.bw + tc_.x0 + tx;
        float4 xv[8];
        if (HAS_RES) {
          const float* rp = p.res.p + p.res.pix(img, Y, X) + pc0;
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            xv[k] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (pix_ok && 4 * k < ncols) xv[k] = *reinterpret_cast<const float4*>(rp + 4 * k);
          }
        }
        __half* dst16 = nullptr;
        if (OUT_MODE != 0) dst16 = p.out16 + ((size_t)((size_t)img * p.out16_h + Y) * p.out16_w + X) * (size_t)p.out16_ld + pc0;
        mbar_wait(tfull + a, aph);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + a * kLeanAccStride + pc0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          if (h * 16 < ncols) {
            float v[16];
            tmem_ld16(taddr + h * 16, v);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 b = *reinterpret_cast<const float4*>(sBias + pc0 + h * 16 + 4 * j);
              v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
            }
#pragma unroll
            for (int k = 0; k < 16; ++k) v[k] = v[k] > 0.f ? v[k] : v[k] * slope;
            if (HAS_RES) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float4 r = xv[4 * h + j];
                v[4 * j] = fmaf(v[4 * j], alpha, r.x); v[4 * j + 1] = fmaf(v[4 * j + 1], alpha, r.y);
                v[4 * j + 2] = fmaf(v[4 * j + 2], alpha, r.z); v[4 * j + 3] = fmaf(v[4 * j + 3], alpha, r.w);
              }
            } else {
#pragma unroll
              for (int k = 0; k < 16; ++k) v[k] *= alpha;
            }
            if (OUT_MODE != 2) {
              if (h == 0) {
                if (lane == 0) bulk_wait_read0();        // the TMA unit has finished reading the previous block out of `stg`
                __syncwarp();
              }
#pragma unroll
              for (int j = 0; j < 4; ++j)
                *reinterpret_cast<float4*>(stg + lane * 32 + (((4 * h + j) ^ (lane & 7)) << 2)) =
                    make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
            if (OUT_MODE != 0 && pix_ok) {
#pragma unroll
              for (int j = 0; j < 2; ++j)
                if (h * 16 + 8 * j < ncols)
                  *reinterpret_cast<uint4*>(dst16 + h * 16 + 8 * j) =
                    make_uint4(pack_h2(v[8 * j], v[8 * j + 1]), pack_h2(v[8 * j + 2], v[8 * j + 3]),
                               pack_h2(v[8 * j + 4], v[8 * j + 5]), pack_h2(v[8 * j + 6], v[8 * j + 7]));
            }
          }
        }
        if (OUT_MODE != 2) {
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_5d(&tmO, stg, pc0, tc_.x0 + tx_w, tc_.vx, tc_.y0 + ty_w, tc_.nb);
            bulk_commit();
          }
        }
      } else {
        mbar_wait(tfull + a, aph);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty + a);
    }
    if (OUT_MODE != 2 && lane == 0) bulk_wait0();
  }
  __syncthreads();
  if (warp == kMmaWarp) {
    __syncwarp();
    tmem_dealloc(tmem_base, kLeanTmemCols);
  }
}

// ======================= halo-block CTA-pair kernel: fp16 3x3 "same" convs with 128 < N <= 256 ===========================
// The per-tap kernel stages a 16 KB activation tile and a half weight slice per tap: ~270 KB written to shared memory per
// 128-pixel tile, which (with the MMA operand reads) is what bounds the upsampler convs. Here each CTA of a pair
//   * keeps ITS HALF of all 9 taps' weights resident (loaded once),
//   * stages its block's haloed input ONCE per block: one TMA box of (Rout + 2) x P pixels x 64 fp16 channels, out-of-image
//     pixels zero-filled (the conv padding); tap (ky, kx) of MMA tile j reads that buffer from the descriptor start row
//     128 j + ky P + kx (SWIZZLE_128B is a function of the absolute address, so any 128-byte row works as a start),
//   * runs tcgen05.mma.cta_group::2 (M = 256: 128 rows from each CTA's own block at the same offsets), taps and K-steps in
//     the per-tap kernel's order, so every fp32 sum is the same,
// with two input buffers and two TMEM accumulator stages, and 16 epilogue warps (four per TMEM lane quarter, each owning
// whole PixelShuffle sub-pixels / column blocks). TAIL: the layer ends in the head-conv tap projection (epilogue of the
// T16 kernel), else it writes its fp16 output only.
constexpr int kHaloEpiW = 16;
constexpr int kHaloThreads = (kHaloEpiW + 2) * 32;

struct BlockCoord { int img, y0, x0; };
// cluster c walks block pairs c, c + clusters, ...; rank r of the pair owns block 2 * pair + r (an odd tail: a dummy block
// that loads valid data and stores nothing, so both CTAs step through the same barrier phases)
__device__ __forceinline__ bool next_block(const Params& p, int i, int& b) {
  const int pr = (int)(blockIdx.x >> 1) + i * (int)(gridDim.x >> 1);
  if (2 * pr >= p.total_blocks) return false;
  b = 2 * pr + (int)(blockIdx.x & 1);
  if (b >= p.total_blocks) b = -1;
  return true;
}
__device__ __forceinline__ BlockCoord decode_block(const Params& p, int b) {
  if (b < 0) b = p.total_blocks - 1;
  BlockCoord c;
  const int u = fdiv(b, p.fd_strips);
  c.x0 = (b - u * p.strips_x) * p.TWo;
  c.img = fdiv(u, p.fd_blocks_y);
  c.y0 = (u - c.img * p.blocks_y) * p.Rout;
  return c;
}

// fp16-only write-out of one pixel per lane (what epilogue_tile_tma does with out_mode 2 and no residual / multiplier):
// column blocks of <= 32 packed channels that never straddle a sub-pixel run, g_first, + g_step, ... of them
__device__ __forceinline__ void halo_store_f16(const Params& p, uint32_t taddr, int lane, int img, int Y, int X, bool pix_ok,
                                               int g_first, int g_step) {
  const int r2 = p.ry * p.rx;
  const bool chan_major = r2 > 1 && p.shuf_mode == LFSR_SHUF_CHANNEL_MAJOR;
  const float slope = p.slope, alpha = p.alpha;
  int bi = 0;
  for (int pc0 = 0, ncols = 0; pc0 < p.cout; pc0 += ncols, ++bi) {
    int sub = 0, c0 = pc0;
    if (r2 > 1) { sub = fdiv(pc0, p.fd_cq); c0 = pc0 - sub * p.cq; }
    ncols = p.cq - c0 < 32 ? p.cq - c0 : 32;
    if (p.cout - pc0 < ncols) ncols = p.cout - pc0;
    if (bi % g_step != g_first) continue;
    float bcol = 0.f;
    if (p.bias) {
      const int pcl = pc0 + lane;
      if (pcl < p.cout) {
        int bidx = pcl;
        if (chan_major) { const int s_ = fdiv(pcl, p.fd_cq); bidx = (pcl - s_ * p.cq) * r2 + s_; }
        bcol = __ldg(p.bias + bidx);
      }
    }
    float v[32];
    tmem_ld16(taddr + pc0, v);
    if (ncols > 16) tmem_ld16(taddr + pc0 + 16, v + 16);
    else {
#pragma unroll
      for (int k = 16; k < 32; ++k) v[k] = 0.f;
    }
    if (p.bias) {
#pragma unroll
      for (int k = 0; k < 32; ++k) v[k] += __shfl_sync(0xffffffffu, bcol, k);
    }
#define LFSR_EPI_ACT32(A) _Pragma("unroll") for (int k = 0; k < 32; ++k) v[k] = act_t<A>(v[k], slope);
    switch (p.act) {
      case LFSR_ACT_RELU: LFSR_EPI_ACT32(LFSR_ACT_RELU) break;
      case LFSR_ACT_LRELU: LFSR_EPI_ACT32(LFSR_ACT_LRELU) break;
      case LFSR_ACT_SIGMOID: LFSR_EPI_ACT32(LFSR_ACT_SIGMOID) break;
      case LFSR_ACT_GELU: LFSR_EPI_ACT32(LFSR_ACT_GELU) break;
      case LFSR_ACT_SILU: LFSR_EPI_ACT32(LFSR_ACT_SILU) break;
      default: break;
    }
#undef LFSR_EPI_ACT32
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = fmaf(v[k], alpha, 0.f);      // (as the per-tap epilogue rounds it: alpha * v + 0)
    if (pix_ok) {
      int Yo = Y, Xo = X;
      if (r2 > 1) { const int si = fdiv(sub, p.fd_rx), sj = sub - si * p.rx; Yo = Y * p.ry + si; Xo = X * p.rx + sj; }
      __half* dst = p.out16 + ((size_t)((size_t)img * p.out16_h + Yo) * p.out16_w + Xo) * (size_t)p.out16_ld + c0;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (8 * j < ncols)
          *reinterpret_cast<uint4*>(dst + 8 * j) =
              make_uint4(pack_h2(v[8 * j], v[8 * j + 1]), pack_h2(v[8 * j + 2], v[8 * j + 3]), pack_h2(v[8 * j + 4], v[8 * j + 5]),
                         pack_h2(v[8 * j + 6], v[8 * j + 7]));
    }
  }
}

// (register files are allocated per 4-warp group: the bound is stated for 20 warps so that ptxas budgets what 18 cost)
template <bool TAIL>
__global__ void __launch_bounds__(640, 1)
conv_tc_halo_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBh, const Params p,
                    const __grid_constant__ TailArg<TAIL> tw) {
  constexpr int kTmaW = kHaloEpiW, kMmaW = kHaloEpiW + 1;
  constexpr int kTaps = 9;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  const uint32_t half_bytes = (uint32_t)(p.NC >> 1) * 128u;      // this CTA's rows of one tap's weight slice
  uint8_t* sA = smem;                                              // 2 x a_buf_bytes
  uint8_t* sB = sA + 2 * p.a_buf_bytes;                            // kTaps x half_bytes
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + kTaps * half_bytes);
  uint64_t* afull = bars;
  uint64_t* aempty = bars + 2;
  uint64_t* tfull = bars + 4;
  uint64_t* tempty = bars + 6;
  uint64_t* bfull = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int k = 0; k < 2; ++k) {
      mbar_init(afull + k, 1); mbar_init(aempty + k, 1);
      mbar_init(tfull + k, 1); mbar_init(tempty + k, 2 * kHaloEpiW);
    }
    mbar_init(bfull, 1);
    fence_barrier_init();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmBh);
  }
  cluster_sync_all();                           // both CTAs are resident before the paired allocation is requested
  if (warp == kMmaW) tmem_alloc2(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                           // the partner's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t crank = cluster_ctarank();

  if (warp == kTmaW) {
    // ---- TMA producer (both CTAs): the weight halves once, then one haloed input box per block; all transaction bytes
    // land on the leader's barriers, whose MMAs read both CTAs' buffers
    if (elect_one()) {
      if (crank == 0) mbar_expect_tx(bfull, 2u * kTaps * half_bytes);
      for (int t = 0; t < kTaps; ++t)
        tma_load_2d_2sm(sB + t * half_bytes, &tmBh, bfull, 0, t * p.NC + (int)crank * (p.NC >> 1));
      const uint32_t box_bytes = (uint32_t)(p.Rin * p.P * 128);
      int b;
      for (int i = 0; next_block(p, i, b); ++i) {
        const int buf = i & 1;
        mbar_wait(aempty + buf, ((i >> 1) & 1) ^ 1);      // own barrier: the leader's commit arrives in both CTAs
        if (crank == 0) mbar_expect_tx(afull + buf, 2u * box_bytes);
        const BlockCoord bc = decode_block(p, b);
        tma_load_5d_2sm(sA + buf * p.a_buf_bytes, &tmA, afull + buf, 0, bc.x0 - 1, 0, bc.y0 - 1, bc.img);
      }
    }
    __syncwarp();
  } else if (warp == kMmaW) {
    // ---- MMA issuer: the leader's elected lane issues M = 256 for the pair; the partner's MMA warp idles
    if (crank == 0) {
      if (elect_one()) {
        const uint32_t idesc2 = (make_idesc(p.NC, 0u) & ~(0x1fu << 24)) | ((uint32_t)(256 >> 4) << 24);
        const uint64_t a_desc0 = make_smem_desc(smem_u32(sA)), b_desc0 = make_smem_desc(smem_u32(sB));
        const uint32_t row_p = (uint32_t)p.P * 8u;                 // one padded input row (P pixels x 128 B), 16-byte units
        const uint32_t b_tap = half_bytes >> 4;
        const int ksteps = p.C >= 64 ? 4 : (p.C + 15) >> 4;
        mbar_wait(bfull, 0);
        tc_fence_after();
        uint32_t tcount = 0;
        int b;
        for (int i = 0; next_block(p, i, b); ++i) {
          const int buf = i & 1;
          mbar_wait(afull + buf, (i >> 1) & 1);
          tc_fence_after();
          const uint64_t a_blk = a_desc0 + (uint64_t)buf * (uint64_t)(p.a_buf_bytes >> 4);
          for (int j = 0; j < p.ntiles; ++j, ++tcount) {
            const uint32_t a = tcount & 1;
            mbar_wait(tempty + a, ((tcount >> 1) & 1) ^ 1);          // both CTAs' epilogues have drained this stage
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + a * kAccStride;
            const uint64_t a_tile = a_blk + (uint64_t)(j * 1024);   // 128 rows x 128 B
            uint64_t b_d = b_desc0;
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
              for (int kx = 0; kx < 3; ++kx) {
                const uint64_t a_d = a_tile + (uint64_t)(ky * row_p + kx * 8);
                if (ky == 0 && kx == 0) umma2_tf32_c<0, true>(d_tmem, a_d, b_d, idesc2);
                else umma2_tf32_c<1, true>(d_tmem, a_d, b_d, idesc2);
                if (ksteps == 4) {
                  umma2_tf32_c<1, true>(d_tmem, a_d + 2, b_d + 2, idesc2);
                  umma2_tf32_c<1, true>(d_tmem, a_d + 4, b_d + 4, idesc2);
                  umma2_tf32_c<1, true>(d_tmem, a_d + 6, b_d + 6, idesc2);
                } else {
                  for (int k = 1; k < ksteps; ++k) umma2_tf32_c<1, true>(d_tmem, a_d + 2 * k, b_d + 2 * k, idesc2);
                }
                b_d += b_tap;
              }
            }
            umma2_commit_mc(tfull + a);              // accumulator complete -> both CTAs' epilogues
          }
          umma2_commit_mc(aempty + buf);             // both CTAs' input buffers may be refilled
        }
      }
      __syncwarp();
    }
  } else {
    // ---- epilogue: warp w <-> TMEM lane quarter w & 3; the four warps of a quarter take alternate sub-pixels / blocks ----
    const int q = warp & 3, grp = warp >> 2;
    uint32_t tcount = 0;
    int b;
    for (int i = 0; next_block(p, i, b); ++i) {
      const BlockCoord bc = decode_block(p, b);
      for (int j = 0; j < p.ntiles; ++j, ++tcount) {
        const uint32_t a = tcount & 1;
        const int g = j * 128 + q * 32 + lane;                     // flattened padded position of the lane's MMA row
        const int ty = (g * p.pdiv_mul) >> 16, tx = g - ty * p.P;
        const int Y = bc.y0 + ty, X = bc.x0 + tx;
        const bool pix_ok = b >= 0 && ty < p.Rout && tx < p.TWo && Y < p.bh && X < p.bw;
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + a * kAccStride;
        mbar_wait(tfull + a, (tcount >> 1) & 1);
        tc_fence_after();
        if (TAIL) tail_project<true>(p, tail_w_of(tw, nullptr), taddr, lane, bc.img, Y, X, pix_ok, 0, p.ry * p.rx, grp, 4);
        else halo_store_f16(p, taddr, lane, bc.img, Y, X, pix_ok, grp, 4);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(tempty + a);
      }
    }
  }
  __syncthreads();
  cluster_sync_all();                           // no CTA may exit while its partner can still signal it
  if (warp == kMmaW) {
    __syncwarp();
    tmem_dealloc2(tmem_base, kTmemCols);
  }
}

// ---- host side ----------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

struct Plan {
  int nchunks, NC, cgs;
};
static Plan plan_for(int cin, int cout, bool f16 = false) {
  Plan pl;
  pl.nchunks = (cout + 255) / 256;
  const int per = (cout + pl.nchunks - 1) / pl.nchunks;
  pl.NC = (per + 15) / 16 * 16;
  pl.cgs = f16 ? (cin + 63) / 64 : (cin + 31) / 32;      // channel groups = 128-byte rows of the K-major operands
  return pl;
}

static float round_tf32(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  if ((u & 0x7F800000u) == 0x7F800000u) return x;   // inf / nan
  u += 0xFFFu + ((u >> 13) & 1u);
  u &= ~0x1FFFu;
  float y;
  memcpy(&y, &u, 4);
  return y;
}

// Block geometry of conv_tc_halo_kernel for an H x W image: output blocks of Rout x TWo pixels, flattened over padded rows of
// P = TWo + 2 into ntiles MMA tiles of 128 rows. Chosen to maximise the share of MMA rows that are output pixels (halo
// columns, the unused tail of the last tile and the blocks that overhang the image are the waste), then to minimise the
// input rows staged per output pixel. Shared memory: two input buffers (each must also cover the rows the last tile's
// bottom-right tap reads: 128 ntiles + 2 P + 2) and the resident weight halves of 9 taps.
struct HaloGeom { int TWo, Rout, P, Rin, ntiles, strips_x, blocks_y, a_buf_bytes, smem, pdiv_mul; };
constexpr int kHaloSmemMax = 227 * 1024;
static int halo_smem_bytes(int a_buf_bytes, int NC) { return 1024 + 2 * a_buf_bytes + 9 * (NC / 2) * 128 + 9 * 8 + 16; }
static bool plan_halo(int H, int W, int NC, HaloGeom& g) {
  if (H < 1 || W < 1 || NC < 16 || NC > 256 || NC % 16) return false;
  double best = 0.0, best_rows = 1e30;
  bool found = false;
  for (int nt = 1; nt <= 3; ++nt)
    for (int two = W < 254 ? W : 254; two >= 1; --two) {
      const int P = two + 2;
      int rout = nt * 128 / P;
      if (rout > H) rout = H;
      if (rout > 254) rout = 254;
      if (rout < 1 || rout * P <= (nt - 1) * 128) continue;       // a tile that holds no block position
      const int rin = rout + 2;
      const int rows = rin * P > nt * 128 + 2 * P + 2 ? rin * P : nt * 128 + 2 * P + 2;
      const int a_buf = (rows * 128 + 1023) / 1024 * 1024;
      if (halo_smem_bytes(a_buf, NC) > kHaloSmemMax) continue;
      const int sx = (W + two - 1) / two, by = (H + rout - 1) / rout;
      const double eff = (double)H * W / ((double)sx * by * nt * 128);
      const double staged = (double)sx * by * rin * P / ((double)H * W);
      if (eff > best + 1e-9 || (eff > best - 1e-9 && staged < best_rows - 1e-9)) {
        best = eff; best_rows = staged; found = true;
        g.TWo = two; g.Rout = rout; g.P = P; g.Rin = rin; g.ntiles = nt; g.strips_x = sx; g.blocks_y = by;
        g.a_buf_bytes = a_buf; g.smem = halo_smem_bytes(a_buf, NC);
      }
    }
  if (!found) return false;
  g.pdiv_mul = (65536 + g.P - 1) / g.P;             // ty = (g * pdiv_mul) >> 16 == g / P for every position of a block
  for (int k = 0; k < 128 * g.ntiles; ++k)
    if (((k * g.pdiv_mul) >> 16) != k / g.P) return false;
  return true;
}

}  // namespace tc
}  // namespace lfsr

using namespace lfsr;
using namespace lfsr::tc;

// Block plan of the halo-block kernel for an h x w fp16 image (lfsr.h): geom[0..7] = TWo, Rout, P, ntiles, strips_x,
// blocks_y, input buffer bytes, dynamic shared memory bytes. Returns 1 when a plan exists.
extern "C" int lfsr_conv_tc_halo_plan(int h, int w, int cout, int* geom) {
  if (!geom || cout < 1) return 0;
  const Plan pl = plan_for(64, cout, true);
  if (pl.nchunks != 1) return 0;
  HaloGeom g;
  if (!plan_halo(h, w, pl.NC, g)) return 0;
  const int v[8] = {g.TWo, g.Rout, g.P, g.ntiles, g.strips_x, g.blocks_y, g.a_buf_bytes, g.smem};
  memcpy(geom, v, sizeof(v));
  return 1;
}

extern "C" size_t lfsr_conv2d_tc_packed_floats(int kh, int kw, int cin, int cout) {
  if (kh <= 0 || kw <= 0 || cin <= 0 || cout <= 0) return 0;
  const Plan pl = plan_for(cin, cout);
  return (size_t)pl.nchunks * kh * kw * pl.cgs * pl.NC * 32;
}

// packed[chunk][tap][cg][NC][32]: row r of chunk holds output channel chunk*NC + r (zero rows beyond cout),
// 32 consecutive input channels of group cg (zero beyond cin), TF32-rounded.
extern "C" int lfsr_pack_conv_tc(const float* w, float* packed, int kh, int kw, int cin, int cout) {
  LFSR_REQUIRE(w && packed && kh > 0 && kw > 0 && cin > 0 && cout > 0, "lfsr_pack_conv_tc: bad arguments");
  const Plan pl = plan_for(cin, cout);
  const int taps = kh * kw;
  const size_t total = lfsr_conv2d_tc_packed_floats(kh, kw, cin, cout);
  memset(packed, 0, total * sizeof(float));
  for (int co = 0; co < cout; ++co) {
    const int chunk = co / pl.NC, r = co - chunk * pl.NC;
    for (int tap = 0; tap < taps; ++tap)
      for (int ci = 0; ci < cin; ++ci) {
        const int cg = ci / 32, k = ci - cg * 32;
        const size_t dst = ((((size_t)chunk * taps + tap) * pl.cgs + cg) * pl.NC + r) * 32 + k;
        packed[dst] = round_tf32(w[((size_t)co * cin + ci) * taps + tap]);
      }
  }
  return LFSR_OK;
}

extern "C" size_t lfsr_conv2d_tc16_packed_bytes(int kh, int kw, int cin, int cout) {
  if (kh <= 0 || kw <= 0 || cin <= 0 || cout <= 0) return 0;
  const Plan pl = plan_for(cin, cout, true);
  return (size_t)pl.nchunks * kh * kw * pl.cgs * pl.NC * 128;
}

// fp16 packing for fp16 activations: packed[chunk][tap][cg][NC][64] - row r of a chunk holds output channel chunk*NC + r,
// 64 consecutive input channels of group cg (zeros beyond cin / cout), round-to-nearest-even.
extern "C" int lfsr_pack_conv_tc16(const float* w, void* packed, int kh, int kw, int cin, int cout) {
  LFSR_REQUIRE(w && packed && kh > 0 && kw > 0 && cin > 0 && cout > 0, "lfsr_pack_conv_tc16: bad arguments");
  const Plan pl = plan_for(cin, cout, true);
  const int taps = kh * kw;
  memset(packed, 0, lfsr_conv2d_tc16_packed_bytes(kh, kw, cin, cout));
  __half* out = static_cast<__half*>(packed);
  for (int co = 0; co < cout; ++co) {
    const int chunk = co / pl.NC, r = co - chunk * pl.NC;
    for (int tap = 0; tap < taps; ++tap)
      for (int ci = 0; ci < cin; ++ci) {
        const int cg = ci / 64, k = ci - cg * 64;
        const size_t dst = ((((size_t)chunk * taps + tap) * pl.cgs + cg) * pl.NC + r) * 64 + k;
        out[dst] = __float2half_rn(w[((size_t)co * cin + ci) * taps + tap]);
      }
  }
  return LFSR_OK;
}

static int floordiv(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }

namespace lfsr { namespace tc {
// out[img][row][k] = packed[row][k] * gate[img][cg(row)*32 + k]   (rows are [chunk][tap][cg][NC])
__global__ void __launch_bounds__(256)
scale_pack_kernel(const float* __restrict__ packed, const float* __restrict__ gate, long long gate_ld, float* __restrict__ out,
                  int rows, int cgs, int NC, int cin) {
  const int img = blockIdx.y;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < rows * 32; i += gridDim.x * blockDim.x) {
    const int k = i & 31, row = i >> 5;
    const int cg = (row / NC) % cgs;
    const int ci = cg * 32 + k;
    const float g = ci < cin ? __ldg(gate + (size_t)img * gate_ld + ci) : 0.f;
    out[(size_t)img * rows * 32 + i] = __ldg(packed + i) * g;
  }
}
}}  // namespace

extern "C" int lfsr_scale_pack_tc(const float* packed, const float* gate, int64_t gate_ld, float* out, int n, int kh, int kw,
                                  int cin, int cout, void* stream) {
  LFSR_REQUIRE(packed && gate && out && n > 0 && n <= 65535, "lfsr_scale_pack_tc: bad arguments");
  const lfsr::tc::Plan pl = lfsr::tc::plan_for(cin, cout);
  const int rows = pl.nchunks * kh * kw * pl.cgs * pl.NC;
  dim3 grid(ceil_div(rows * 32, 256) < 64 ? ceil_div(rows * 32, 256) : 64, n);
  lfsr::tc::scale_pack_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(packed, gate, gate_ld > 0 ? gate_ld : cin, out, rows,
                                                                       pl.cgs, pl.NC, cin);
  return check_launch("scale_pack_kernel");
}

static bool tc_geometry_ok(const lfsr_tensor* in, const lfsr_tensor* out, const lfsr_conv_desc* d) {
  if (!tensor_ok(in) || !tensor_ok(out) || !d) return false;
  if (d->in_perm || d->out_perm) return false;
  if (d->mul.ptr && ((d->shuf_ry > 1) || (d->shuf_rx > 1))) return false;      // mul is only fused for unshuffled outputs
  if (d->mul.ptr && d->mul_act != LFSR_ACT_NONE && d->mul_act != LFSR_ACT_SILU) return false;
  if (d->in_scale && d->w_batch_stride <= 0) return false;      // gates must come folded into per-image weights
  if (d->kh * d->kw > 25 || d->kh < 1 || d->kw < 1) return false;
  if (in->c < 8 || in->ld % (d->in_f16 ? 8 : 4) != 0 || ((uintptr_t)in->ptr & 15)) return false;
  if (d->in_f16 && (d->in_scale || d->w_batch_stride > 0)) return false;        // gated per-image weight sets are fp32 / tf32 only
  if (d->out_mode < 0 || d->out_mode > 2) return false;
  if (d->out_mode != 0) {      // fp16 copy of the output: through the TMA-store epilogue only (checked again at launch)
    const lfsr_tensor* o = &d->out16;
    if (!tensor_ok(o) || o->n != out->n || o->h != out->h || o->w != out->w || o->c != out->c) return false;
    if (o->ld % 8 != 0 || ((uintptr_t)o->ptr & 15) || out->c % 8 != 0 || d->tail_w || (d->res.ptr && d->mul.ptr)) return false;
  }
  const int ry = d->shuf_ry > 0 ? d->shuf_ry : 1, rx = d->shuf_rx > 0 ? d->shuf_rx : 1;
  const int sh = d->stride_h, sw = d->stride_w;
  if (sh < 1 || sw < 1 || in->h % sh || in->w % sw) return false;
  const int OH = (in->h + 2 * d->pad_h - d->dil_h * (d->kh - 1) - 1) / sh + 1;
  const int OW = (in->w + 2 * d->pad_w - d->dil_w * (d->kw - 1) - 1) / sw + 1;
  if (OH != in->h / sh || OW != in->w / sw) return false;                 // "same" geometry (per stride)
  if (out->n != in->n || out->h != OH * ry || out->w != OW * rx) return false;
  if (sh > 1 || sw > 1) {
    if (d->dil_h != 1 || d->dil_w != 1 || d->block_h > 0 || d->block_w > 0) return false;
    if (sh > 1 && sw > 1 && (d->pad_h || d->pad_w)) return false;         // image and row-block share one TMA dim there
    if (sh > 8 || sw > 8) return false;
  }
  const int cout = (d->tail_w ? d->tail_c : out->c) * ry * rx;
  if (cout < 1) return false;
  if (d->tail_w) {      // tail projection: one cout-chunk whose sub-pixel blocks stay inside a 256-column accumulator stage
    if (ry * rx < 2 || d->tail_c < 4 || d->tail_c % 4 || d->tail_taps < 1 || d->tail_taps > 12 || out->c != d->tail_taps) return false;
    if (!d->tail_w_host) return false;
    if ((cout > 256 && (d->tail_c % 32 || 256 % d->tail_c)) || (cout > 240 && d->tail_c % 32) || out->ld < 12 || out->ld % 4 || ((uintptr_t)out->ptr & 15) || ((uintptr_t)d->tail_w & 15)) return false;
    if (d->res.ptr || d->mul.ptr || sh > 1 || sw > 1 || d->block_h > 0 || d->block_w > 0) return false;
  }
  const int bh = d->block_h > 0 ? d->block_h : in->h, bw = d->block_w > 0 ? d->block_w : in->w;
  if (in->h % bh || in->w % bw) return false;
  if ((long long)in->n * (in->h / bh) > 0x7fffffffLL) return false;
  return true;
}

extern "C" int lfsr_conv2d_tc_supported(const lfsr_tensor* in, const lfsr_tensor* out, const lfsr_conv_desc* d) {
  return tc_geometry_ok(in, out, d) && get_encode() != nullptr ? 1 : 0;
}

extern "C" int lfsr_conv2d_tc(const lfsr_tensor* in, const float* w_packed_tc, const lfsr_tensor* out,
                              const lfsr_conv_desc* d, void* stream) {
  LFSR_REQUIRE(w_packed_tc, "lfsr_conv2d_tc: null weights");
  LFSR_REQUIRE(tc_geometry_ok(in, out, d), "lfsr_conv2d_tc: unsupported geometry (query lfsr_conv2d_tc_supported)");
  EncodeTiledFn encode = get_encode();
  if (!encode) { set_error("lfsr_conv2d_tc: cuTensorMapEncodeTiled unavailable"); return LFSR_ERR_CUDA; }
  const int ry = d->shuf_ry > 0 ? d->shuf_ry : 1, rx = d->shuf_rx > 0 ? d->shuf_rx : 1;
  Params p;
  memset(&p, 0, sizeof(p));
  const int sh = d->stride_h, sw = d->stride_w;
  const bool strided = sh > 1 || sw > 1;
  // "block" = the region tiles may not straddle: a view (EPIT), else the whole (output-resolution) image
  p.bh = strided ? in->h / sh : (d->block_h > 0 ? d->block_h : in->h);
  p.bw = strided ? in->w / sw : (d->block_w > 0 ? d->block_w : in->w);
  p.nby = strided ? 1 : in->h / p.bh; p.nbx = strided ? 1 : in->w / p.bw;
  p.nb_total = in->n * p.nby;
  p.amode = !strided ? 0 : (sh == 1 ? 1 : (sw == 1 ? 2 : 3));
  p.out_rows_per_img = in->h / sh;
  for (int ky = 0; ky < d->kh; ++ky)
    for (int kx = 0; kx < d->kw; ++kx) {
      short* to = p.tap_off[ky * d->kw + kx];
      const int dy = ky * d->dil_h - d->pad_h, dx = kx * d->dil_w - d->pad_w;
      const int ay = floordiv(dy, sh), ry_ = dy - ay * sh, ax = floordiv(dx, sw), rx_ = dx - ax * sw;
      if (p.amode == 0) { to[0] = (short)dx; to[1] = 0; to[2] = (short)dy; to[3] = 0; }
      else if (p.amode == 1) { to[0] = (short)rx_; to[1] = (short)ax; to[2] = (short)dy; to[3] = 0; }
      else if (p.amode == 2) { to[0] = (short)dx; to[1] = (short)ry_; to[2] = (short)ay; to[3] = 0; }
      else { to[0] = (short)rx_; to[1] = (short)ax; to[2] = (short)ry_; to[3] = (short)ay; }
    }
  p.C = in->c; p.kh = d->kh; p.kw = d->kw; p.dil_h = d->dil_h; p.dil_w = d->dil_w; p.pad_h = d->pad_h; p.pad_w = d->pad_w;
  p.cout = (d->tail_w ? d->tail_c : out->c) * ry * rx;
  const bool f16 = d->in_f16 != 0;
  const Plan pl = plan_for(p.C, p.cout, f16);
  p.NC = pl.NC; p.nchunks = pl.nchunks; p.cgs = pl.cgs;
  p.out_mode = d->out_mode;
  p.out = view_of(out);
  p.res = d->res.ptr ? view_of(&d->res) : null_view();
  p.mul = d->mul.ptr ? view_of(&d->mul) : null_view();
  if (d->res.ptr)
    LFSR_REQUIRE(d->res.n == out->n && d->res.h == out->h && d->res.w == out->w && d->res.c == out->c,
                 "lfsr_conv2d_tc: res tensor geometry");
  if (d->mul.ptr)
    LFSR_REQUIRE(d->mul.n == out->n && d->mul.h == out->h && d->mul.w == out->w && d->mul.c == out->c,
                 "lfsr_conv2d_tc: mul tensor geometry");
  LFSR_REQUIRE((long long)out->h * out->w * out->ld < 0x7fffffffLL, "lfsr_conv2d_tc: output image too large for 32-bit pitches");
  p.bias = d->bias; p.act = d->act; p.slope = d->act_slope; p.alpha = d->alpha; p.mul_act = d->mul_act;
  p.ry = ry; p.rx = rx; p.shuf_mode = d->shuf_mode; p.cq = d->tail_w ? d->tail_c : out->c;
  p.tail_w = d->tail_w; p.tail_rows = d->tail_w ? (d->tail_c + 31) / 32 * 32 : 0;
  TailW tt;                                        // the table by value (kernels with 16 epilogue warps read it from there)
  memset(&tt, 0, sizeof(tt));
  if (d->tail_w && p.cq <= kTailMaxC) memcpy(tt.w, d->tail_w_host, (size_t)p.cq * 12 * sizeof(float));
  // (a short last block of a sub-pixel run reads up to 31 accumulator columns past it: keep that inside the 256-column stage)
  if (d->tail_w)
    LFSR_REQUIRE((p.nchunks == 1 && (p.NC <= 240 || p.cq % 32 == 0)) ||
                     (p.nchunks > 1 && p.cq % 32 == 0 && p.NC % p.cq == 0 && p.cout == p.nchunks * p.NC),
                 "lfsr_conv2d_tc: tail projection needs cout chunks made of whole sub-pixel channel runs");
  p.fd_cq = make_fastdiv(p.cq); p.fd_nby = make_fastdiv(p.nby); p.fd_nbx = make_fastdiv(p.nbx); p.fd_rx = make_fastdiv(rx);
  p.vec = 1;
  for (int v = 2; v <= 4; v *= 2) {
    const uintptr_t mask = (uintptr_t)v * 4 - 1;
    if ((p.cq % v == 0) && (out->ld % v == 0) && (((uintptr_t)out->ptr & mask) == 0) &&
        (!d->res.ptr || ((d->res.ld % v == 0) && (((uintptr_t)d->res.ptr & mask) == 0))) &&
        (!d->mul.ptr || ((d->mul.ld % v == 0) && (((uintptr_t)d->mul.ptr & mask) == 0))))
      p.vec = v;
    else
      break;
  }
  p.b_stage_bytes = p.NC * 128;
#ifdef LFSR_DEBUG_HOOKS      // probe build only (liblfsr_probe.so): cycle counters
  p.dbg = getenv("LFSR_TC_DBG_PTR") ? (long long*)strtoull(getenv("LFSR_TC_DBG_PTR"), nullptr, 0) : nullptr;
#endif
  const int sm_count = sm_count_current();
  static DevOnce once;
  if (once.need()) {
    const char* w_ = "lfsr_conv2d_tc";
    if (opt_in_smem(conv_tc_kernel<false, false, false>, 227 * 1024, w_) || opt_in_smem(conv_tc_kernel<true, false, false>, 227 * 1024, w_) ||
        opt_in_smem(conv_tc_kernel<false, false, true>, 227 * 1024, w_) || opt_in_smem(conv_tc_kernel<true, false, true>, 227 * 1024, w_) ||
        opt_in_smem(conv_tc_kernel<true, false, true, true>, 227 * 1024, w_) || opt_in_smem(conv_tc_kernel<false, false, true, true>, 227 * 1024, w_) ||
        opt_in_smem(conv_tc_kernel<false, false, false, true>, 227 * 1024, w_) || opt_in_smem(conv_tc_kernel<true, false, false, true>, 227 * 1024, w_) ||
#ifdef LFSR_DEBUG_HOOKS
        opt_in_smem(conv_tc_kernel<false, true, false>, 227 * 1024, w_) || opt_in_smem(conv_tc_kernel<true, true, false>, 227 * 1024, w_) ||
        opt_in_smem(conv_tc_kernel<false, true, true>, 227 * 1024, w_) || opt_in_smem(conv_tc_kernel<true, true, true>, 227 * 1024, w_) ||
        opt_in_smem(conv_tc_kernel<true, true, true, true>, 227 * 1024, w_) ||
#endif
        opt_in_smem(conv_tc_halo_kernel<true>, 227 * 1024, w_) || opt_in_smem(conv_tc_halo_kernel<false>, 227 * 1024, w_))
      return LFSR_ERR_CUDA;
    once.done();
  }

  // tile shape TH x TW = 128 minimising padding waste inside a block (prefer wide tiles)
  {
    double best = 1e30;
    for (int tw = 128; tw >= 8; tw >>= 1) {
      const int th = 128 / tw;
      const double waste = (double)(ceil_div(p.bh, th) * th) * (ceil_div(p.bw, tw) * tw) / ((double)p.bh * p.bw);
      if (waste < best - 1e-9) { best = waste; p.TW = tw; p.TH = th; }
    }
    p.tw_shift = 0;
    while ((1 << p.tw_shift) < p.TW) ++p.tw_shift;
  }
  p.tiles_y = ceil_div(p.bh, p.TH); p.tiles_x = ceil_div(p.bw, p.TW);
  const long long tiles = (long long)p.nb_total * p.tiles_y * p.nbx * p.tiles_x * p.nchunks;
  LFSR_REQUIRE(tiles > 0 && tiles < 0x7fffffffLL, "lfsr_conv2d_tc: tile count out of range");
  p.total_tiles = (int)tiles;
  p.m_tiles = (int)(tiles / p.nchunks);
  p.fd_tiles_x = make_fastdiv(p.tiles_x); p.fd_tiles_y = make_fastdiv(p.tiles_y); p.fd_nchunks = make_fastdiv(p.nchunks);
  const int nks = p.kh * p.kw * p.cgs;
  const int tail_bytes = p.tail_rows * 48;
  const int epi16_bytes = 0;
  const int kSmemMax = 227 * 1024 - 1024 - 256 - kEpiWarps * 4096 - tail_bytes - epi16_bytes;  // minus alignment slack, barriers, epilogue staging, tail table
  const long long b_all = (long long)nks * p.b_stage_bytes;
  // Plan = (weights resident?, K-stages per smem stage). Preference: one tap with all its channel groups per stage
  // (short unrolled issue stream, fewer barrier round trips) with enough stages in flight; weights resident when
  // that still fits, else streamed next to the activations.
  static const bool no_resident = dbg_env("LFSR_TC_NO_RESIDENT") != nullptr;   // tuning knobs (profiles/ experiments)
  static const int max_stages_env = dbg_env("LFSR_TC_STAGES") ? atoi(dbg_env("LFSR_TC_STAGES")) : 0;
  static const int kps_env = dbg_env("LFSR_TC_KPS") ? atoi(dbg_env("LFSR_TC_KPS")) : 0;
  auto stages_for = [&](bool res, int kps) -> int {
    if (res) return b_all >= kSmemMax ? 0 : (int)((kSmemMax - b_all) / ((long long)kps * kABytes));
    return (kSmemBudget - kEpiWarps * 4096 - tail_bytes - epi16_bytes) / (kps * (kABytes + p.b_stage_bytes));
  };
  // narrow layers (N <= 64) are bound by the per-stage barrier round trip of the issuing thread: pack up to 4
  // K-stages (whole taps) into one smem stage; wide layers keep one tap per stage so that >= 3 stages fit
  int kps_auto = p.cgs <= 4 ? p.cgs : 1;
  if (p.NC <= 64 && p.cgs <= 2) kps_auto = 4 / p.cgs * p.cgs;
  if (kps_auto > nks) kps_auto = nks;          // 1x1 layers: a stage never holds more than one tile's K-stages
  const int kps_tap = kps_env > 0 ? kps_env : kps_auto;
  const int need = p.NC <= 64 ? 2 : 3;
  struct Cand { bool res; int kps; int min_stages; };
  const Cand cands[4] = {{true, kps_tap, need}, {false, kps_tap, need}, {true, 1, 2}, {false, 1, 2}};
  p.stages = 0;
  const bool per_image_w = d->w_batch_stride > 0;
  for (const Cand& c : cands) {
    if (c.res && (no_resident || per_image_w)) continue;
    const int st = stages_for(c.res, c.kps);
    if (st >= c.min_stages) { p.resident = c.res ? 1 : 0; p.kps = c.kps; p.stages = st; break; }
  }
  if (p.stages > kMaxStages) p.stages = kMaxStages;
  if (max_stages_env >= 2 && p.stages > max_stages_env) p.stages = max_stages_env;
  LFSR_REQUIRE(p.stages >= 2, "lfsr_conv2d_tc: not enough shared memory for two stages");
  // wide layers whose weights are streamed (they do not fit next to the activation stages) are bound by shared-memory
  // traffic: per K=8 MMA the weight slice is written by TMA and read by the tensor core (2 x N x 32 B) next to 2 x 4 KB
  // of activations. CTA pairs with cta_group::2 MMAs (M = 256) halve the weight writes per MMA: each SM stages its own
  // activation tile and HALF of the weight slice, the leader's MMA thread issues for both
  static const bool use_cta2 = dbg_env("LFSR_TC_NO_CTA2") == nullptr;
  p.cta2 = 0;
  static const int cta2_min_nc = dbg_env("LFSR_TC_CTA2_MIN_NC") ? atoi(dbg_env("LFSR_TC_CTA2_MIN_NC")) : 128;
  if (use_cta2 && !p.resident && !per_image_w && p.nchunks == 1 && p.amode == 0 && p.NC >= cta2_min_nc && p.NC % 16 == 0 &&
      p.m_tiles >= 4 && sm_count >= 2) {
    const int per = kABytes + p.b_stage_bytes / 2;
    const int avail = kSmemBudget - kEpiWarps * 4096 - tail_bytes - epi16_bytes;
    const int st = avail / per;
    if (st >= 2) {
      p.cta2 = 1; p.kps = 1; p.stages = st > kMaxStages ? kMaxStages : st;
      // two K-stages per smem stage when three such stages still fit: the issuing lane pays ~290 cycles per stage boundary
      static const int cta2_kps = dbg_env("LFSR_TC_CTA2_KPS") ? atoi(dbg_env("LFSR_TC_CTA2_KPS")) : 2;
      if (cta2_kps > 1 && nks >= cta2_kps && avail / (cta2_kps * per) >= 3) { p.kps = cta2_kps; p.stages = avail / (cta2_kps * per); if (p.stages > kMaxStages) p.stages = kMaxStages; }
    }
  }
  CUtensorMap tmA, tmB;
  {
    const cuuint64_t ld_b = (cuuint64_t)in->ld * (f16 ? 2 : 4);
    const cuuint64_t W_ = in->w, H_ = in->h, N_ = in->n;
    cuuint64_t dims[5] = {(cuuint64_t)p.C, (cuuint64_t)p.bw, (cuuint64_t)p.nbx, (cuuint64_t)p.bh, (cuuint64_t)p.nb_total};
    cuuint64_t strides[4] = {ld_b, ld_b * p.bw, ld_b * in->w, ld_b * in->w * p.bh};
    cuuint32_t box[5] = {(cuuint32_t)(f16 ? 64 : 32), (cuuint32_t)p.TW, 1, (cuuint32_t)p.TH, 1};
    if (p.amode == 1) {          // (c, x%s, x/s, y, image)
      dims[1] = sw; dims[2] = W_ / sw; dims[3] = H_; dims[4] = N_;
      strides[0] = ld_b; strides[1] = ld_b * sw; strides[2] = ld_b * W_; strides[3] = ld_b * W_ * H_;
      box[1] = 1; box[2] = p.TW; box[3] = p.TH; box[4] = 1;
    } else if (p.amode == 2) {   // (c, x, y%s, y/s, image)
      dims[1] = W_; dims[2] = sh; dims[3] = H_ / sh; dims[4] = N_;
      strides[0] = ld_b; strides[1] = ld_b * W_; strides[2] = ld_b * W_ * sh; strides[3] = ld_b * W_ * H_;
      box[1] = p.TW; box[2] = 1; box[3] = p.TH; box[4] = 1;
    } else if (p.amode == 3) {   // (c, x%s, x/s, y%s, image*y/s)
      dims[1] = sw; dims[2] = W_ / sw; dims[3] = sh; dims[4] = N_ * (H_ / sh);
      strides[0] = ld_b; strides[1] = ld_b * sw; strides[2] = ld_b * W_; strides[3] = ld_b * W_ * sh;
      box[1] = 1; box[2] = p.TW; box[3] = 1; box[4] = p.TH;
    }
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&tmA, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, 5, in->ptr, dims,
                        strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("lfsr_conv2d_tc: cuTensorMapEncodeTiled(A) failed with %d", (int)r); return LFSR_ERR_CUDA; }
  }
  {
    cuuint64_t rows = (cuuint64_t)p.nchunks * p.kh * p.kw * p.cgs * p.NC;
    if (per_image_w) {
      LFSR_REQUIRE(d->w_batch_stride == (long long)rows * 32, "lfsr_conv2d_tc: w_batch_stride must equal the packed size");
      p.w_img_rows = (int)rows;
      rows *= (cuuint64_t)in->n;
    }
    cuuint64_t dims[2] = {32, rows};
    cuuint64_t strides[1] = {128};
    cuuint32_t box[2] = {32, (cuuint32_t)p.NC};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(&tmB, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(w_packed_tc), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("lfsr_conv2d_tc: cuTensorMapEncodeTiled(B) failed with %d", (int)r); return LFSR_ERR_CUDA; }
  }
  const size_t smem = 1024 + (size_t)p.stages * p.kps * kABytes +
                      (p.cta2 ? (size_t)p.stages * p.kps * (p.b_stage_bytes / 2) : (size_t)(p.resident ? nks : p.stages * p.kps) * p.b_stage_bytes) +
                      kEpiWarps * 4096 + (size_t)tail_bytes + (size_t)epi16_bytes + (2 * kMaxStages + 5) * 8 + 16;
  LFSR_REQUIRE(smem <= 227 * 1024, "lfsr_conv2d_tc: shared memory plan too large");
  int grid = p.total_tiles < sm_count ? p.total_tiles : sm_count;
  if (p.cta2) { const int clusters = (p.m_tiles + 1) / 2 < sm_count / 2 ? (p.m_tiles + 1) / 2 : sm_count / 2; grid = 2 * clusters; }
  if (p.resident && p.nchunks > 1) {
    grid = grid / p.nchunks * p.nchunks;                   // every CTA owns one cout-chunk for its lifetime
    if (grid < p.nchunks) grid = p.nchunks;
  }
  CUtensorMap tmBh = tmB;
  if (p.cta2) {
    cuuint64_t rows = (cuuint64_t)p.nchunks * p.kh * p.kw * p.cgs * p.NC;
    cuuint64_t dims[2] = {32, rows};
    cuuint64_t strides[1] = {128};
    cuuint32_t box[2] = {32, (cuuint32_t)(p.NC / 2)};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(&tmBh, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(w_packed_tc), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("lfsr_conv2d_tc: cuTensorMapEncodeTiled(B half) failed with %d", (int)r); return LFSR_ERR_CUDA; }
  }
  // output tensor map for the TMA-store epilogue. Without a PixelShuffle: dims (c, x in block, block-x, y in block,
  // image*block-y), exactly the activation map's structure, so partial tiles are clipped at block edges. With one:
  // dims (c, j, x, i, image*OH + y); rows of different images share a dimension there, so tiles must not overhang
  // the image bottom (OH % TH == 0), and residual / multiplier operands stay with the per-row write-out.
  static const bool no_tma_epi = dbg_env("LFSR_TC_NO_TMA_EPI") != nullptr;
  CUtensorMap tmO = tmA;
  {
    const int r2 = ry * rx;
    const int OHc = out->h / ry, OWc = out->w / rx;
    p.OHc = OHc;
    // (the TMA unit clips the channel dimension in 16-byte granules: channel counts that are not multiples of 4 would
    // spill into the pad floats of grouped layouts, so those layers keep the per-row write-out)
    const bool want32 = d->out_mode != 2, want16 = d->out_mode != 0;
    bool ok = !no_tma_epi && (p.cq % 4 == 0) && !(d->res.ptr && d->mul.ptr);
    if (want32) ok = ok && (((uintptr_t)out->ptr & 15) == 0) && (out->ld % 4 == 0);
    if (want16) ok = ok && (p.cq % 8 == 0);
    if (d->res.ptr) ok = ok && (((uintptr_t)d->res.ptr & 15) == 0) && (d->res.ld % 4 == 0);
    if (d->mul.ptr) ok = ok && r2 == 1 && (((uintptr_t)d->mul.ptr & 15) == 0) && (d->mul.ld % 4 == 0);
    // (a short last block reads up to 15 accumulator columns past NC: keep that inside the 256-column stage)
    // (constraints of the output tensor map; the fp16 copy is stored straight from registers and has none of them)
    if (r2 > 1 && want32) ok = ok && p.nbx == 1 && p.nby == 1 && (OHc % p.TH == 0) && (long long)out->n * OHc < 0x7fffffffLL;
    // the epilogue reads a column block with one or two 16-column TMEM loads: replay its block enumeration and keep
    // every load inside the 256-column accumulator stage
    for (int chunk = 0; chunk < p.nchunks && ok; ++chunk) {
      const int lo = chunk * p.NC, hi = lo + p.NC < p.cout ? lo + p.NC : p.cout;
      for (int pc0 = lo, ncols = 0; pc0 < hi && ok; pc0 += ncols) {
        const int c0 = r2 > 1 ? pc0 % p.cq : pc0;
        ncols = p.cq - c0 < 32 ? p.cq - c0 : 32;
        if (hi - pc0 < ncols) ncols = hi - pc0;
        if (pc0 - lo + (ncols > 16 ? 32 : 16) > kAccStride) ok = false;
        if (want16 && want32 && !(ncols == 32 || c0 + ncols == p.cq)) ok = false;   // fp32 + fp16: tensor-store blocks only
        if (want16 && (ncols % 8 || c0 % 8)) ok = false;                             // 16-byte fp16 stores
      }
    }
    if (ok) {
      const cuuint64_t ld_b = (cuuint64_t)out->ld * 4;
      const cuuint32_t box_w = (cuuint32_t)(p.TW < 32 ? p.TW : 32), box_h = 32 / box_w;
      cuuint64_t dims[5], strides[4];
      cuuint32_t box[5], estr[5] = {1, 1, 1, 1, 1};
      if (r2 == 1) {
        dims[0] = (cuuint64_t)p.cq; dims[1] = (cuuint64_t)p.bw; dims[2] = (cuuint64_t)p.nbx; dims[3] = (cuuint64_t)p.bh;
        dims[4] = (cuuint64_t)p.nb_total;
        strides[0] = ld_b; strides[1] = ld_b * p.bw; strides[2] = ld_b * out->w; strides[3] = ld_b * out->w * p.bh;
        box[0] = 32; box[1] = box_w; box[2] = 1; box[3] = box_h; box[4] = 1;
      } else {
        dims[0] = (cuuint64_t)p.cq; dims[1] = (cuuint64_t)rx; dims[2] = (cuuint64_t)OWc; dims[3] = (cuuint64_t)ry;
        dims[4] = (cuuint64_t)out->n * OHc;
        strides[0] = ld_b; strides[1] = ld_b * rx; strides[2] = ld_b * out->w; strides[3] = ld_b * out->w * ry;
        box[0] = 32; box[1] = 1; box[2] = box_w; box[3] = 1; box[4] = box_h;
      }
      if (want32) {
        CUresult r = encode(&tmO, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, out->ptr, dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("lfsr_conv2d_tc: cuTensorMapEncodeTiled(out) failed with %d", (int)r); return LFSR_ERR_CUDA; }
      }
      if (want16) {
        p.out16 = static_cast<__half*>(d->out16.ptr); p.out16_ld = d->out16.ld; p.out16_h = d->out16.h; p.out16_w = d->out16.w;
      }
      p.tma_epi = 1;
    }
    LFSR_REQUIRE(!want16 || p.tma_epi, "lfsr_conv2d_tc: an fp16 output copy needs the tensor-store epilogue (channel counts that are "
                                       "multiples of 8, 16-byte aligned rows, no residual + multiplier pair)");
  }
  static const bool verbose = dbg_env("LFSR_TC_VERBOSE") != nullptr;
  // ---- halo-block CTA pairs (conv_tc_halo_kernel): fp16 3x3 stride-1 dilation-1 "same" convs over whole images (the
  // upsampler convs) with 128 < N <= 256 in one chunk, ending in the tail projection or writing fp16 only ----------------
  {
    static const bool no_halo = dbg_env("LFSR_TC_NO_HALO") != nullptr;     // A/B switch (profiles/ experiments)
    const int r2 = ry * rx;
    const bool tail_ok = p.tail_w && r2 >= 4 && r2 % 4 == 0 && p.cq <= kTailMaxC;
    const bool f16out_ok = !p.tail_w && d->out_mode == 2 && p.tma_epi;      // (tma_epi: every column block is 8-aligned)
    HaloGeom hg;
    const bool halo = !no_halo && f16 && !per_image_w && p.kh == 3 && p.kw == 3 && !strided && p.dil_h == 1 && p.dil_w == 1 &&
                      p.pad_h == 1 && p.pad_w == 1 && p.nby == 1 && p.nbx == 1 && p.cgs == 1 && p.nchunks == 1 && p.NC > 128 &&
                      !d->res.ptr && !d->mul.ptr && (tail_ok || f16out_ok) && !p.dbg && sm_count >= 2 &&
                      plan_halo(p.bh, p.bw, p.NC, hg) &&
                      (long long)in->n * hg.blocks_y * hg.strips_x < 0x7fffffffLL;
    if (halo) {
      p.TWo = hg.TWo; p.Rout = hg.Rout; p.P = hg.P; p.Rin = hg.Rin; p.ntiles = hg.ntiles; p.strips_x = hg.strips_x;
      p.blocks_y = hg.blocks_y; p.a_buf_bytes = hg.a_buf_bytes; p.pdiv_mul = hg.pdiv_mul;
      p.total_blocks = in->n * hg.blocks_y * hg.strips_x;
      p.fd_strips = make_fastdiv(hg.strips_x); p.fd_blocks_y = make_fastdiv(hg.blocks_y);
      CUtensorMap tmH;
      {
        const cuuint64_t ld_b = (cuuint64_t)in->ld * 2;
        cuuint64_t dims[5] = {(cuuint64_t)p.C, (cuuint64_t)in->w, 1, (cuuint64_t)in->h, (cuuint64_t)in->n};
        cuuint64_t strides[4] = {ld_b, ld_b * in->w, ld_b * in->w, ld_b * in->w * in->h};
        cuuint32_t box[5] = {64, (cuuint32_t)p.P, 1, (cuuint32_t)p.Rin, 1};
        cuuint32_t estr[5] = {1, 1, 1, 1, 1};
        CUresult r = encode(&tmH, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, in->ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("lfsr_conv2d_tc: cuTensorMapEncodeTiled(A halo) failed with %d", (int)r); return LFSR_ERR_CUDA; }
      }
      CUtensorMap tmWh;
      {
        cuuint64_t dims[2] = {32, (cuuint64_t)9 * p.NC};
        cuuint64_t strides[1] = {128};
        cuuint32_t box[2] = {32, (cuuint32_t)(p.NC / 2)};
        cuuint32_t estr[2] = {1, 1};
        CUresult r = encode(&tmWh, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(w_packed_tc), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("lfsr_conv2d_tc: cuTensorMapEncodeTiled(B halo) failed with %d", (int)r); return LFSR_ERR_CUDA; }
      }
      const int pairs = (p.total_blocks + 1) / 2;
      const int hgrid = 2 * (pairs < sm_count / 2 ? pairs : sm_count / 2);
      if (verbose)
        fprintf(stderr, "[lfsr tc halo] C=%d cout=%d NC=%d %dx%d block %dx%d P=%d ntiles=%d blocks=%d grid=%d tail=%d smem=%d\n",
                p.C, p.cout, p.NC, p.bh, p.bw, p.Rout, p.TWo, p.P, p.ntiles, p.total_blocks, hgrid, p.tail_w != nullptr, hg.smem);
      cudaLaunchConfig_t cfg;
      memset(&cfg, 0, sizeof(cfg));
      cfg.gridDim = dim3(hgrid); cfg.blockDim = dim3(kHaloThreads); cfg.dynamicSmemBytes = hg.smem; cfg.stream = (cudaStream_t)stream;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr; cfg.numAttrs = 1;
      const cudaError_t le = p.tail_w ? cudaLaunchKernelEx(&cfg, conv_tc_halo_kernel<true>, tmH, tmWh, p, tt)
                                      : cudaLaunchKernelEx(&cfg, conv_tc_halo_kernel<false>, tmH, tmWh, p, NoTailW{});
      if (le != cudaSuccess) { set_error("lfsr_conv2d_tc: launch failed: %s", cudaGetErrorString(le)); return LFSR_ERR_CUDA; }
      g_halo_launches.fetch_add(1);
      return check_launch("conv_tc_halo_kernel");
    }
  }
  // ---- lean path (conv_tc_lean_kernel): narrow fp16 layers run as two independent CTAs per SM -------------------------
  {
    static const bool no_lean = dbg_env("LFSR_TC_NO_LEAN") != nullptr;
    const bool act_ok = p.act == LFSR_ACT_NONE || p.act == LFSR_ACT_RELU || p.act == LFSR_ACT_LRELU;
    // (a short last block is clipped by the output tensor map; the fp16 copy is stored as 16-byte runs of 8 channels)
    const bool cout_ok = d->out_mode == 0 ? p.cout % 4 == 0 : p.cout % 8 == 0;
    bool lean = !no_lean && !p.cta2 && !p.tail_w && p.tma_epi && ry * rx == 1 && !d->mul.ptr && act_ok &&
                p.nchunks == 1 && p.NC <= 64 && cout_ok && !p.dbg && p.m_tiles >= 2 * sm_count;
    if (verbose && !lean)
      fprintf(stderr, "[lfsr tc lean] not eligible: cta2 %d tail %d tma_epi %d r2 %d mul %d act %d nchunks %d NC %d cout_ok %d dbg %d tiles %d\n",
              p.cta2, p.tail_w != nullptr, p.tma_epi, ry * rx, d->mul.ptr != nullptr, p.act, p.nchunks, p.NC, (int)cout_ok,
              p.dbg != nullptr, p.m_tiles);
    int l_kps = 0, l_stages = 0, l_res = 0;
    size_t l_smem = 0;
    if (lean) {
      const int stg = d->out_mode != 2 ? kEpiWarps * 4096 : 0;
      const long long fixed = 1024 + stg + 256 + (2 * kMaxStages + 6) * 8 + 16;
      const long long b_all = (long long)nks * p.b_stage_bytes;
      int kps_hi = kps_env > 0 ? kps_env : (p.cgs <= 2 ? 4 / p.cgs * p.cgs : p.cgs);
      if (kps_hi > nks) kps_hi = nks;
      for (int kps = kps_hi; kps >= 1 && !l_stages; --kps) {
        if (kps_env > 0 && kps != kps_env) break;
        for (int res = (no_resident || per_image_w) ? 0 : 1; res >= 0 && !l_stages; --res) {
          const long long per_stage = (long long)kps * (kABytes + (res ? 0 : p.b_stage_bytes));
          const long long left = kLeanSmem - fixed - (res ? b_all : 0);
          int st = left > 0 ? (int)(left / per_stage) : 0;
          if (st > kMaxStages) st = kMaxStages;
          if (st >= 2) { l_kps = kps; l_stages = st; l_res = res; l_smem = (size_t)(fixed + (res ? b_all : 0) + st * per_stage); }
        }
      }
      lean = l_stages >= 2;
    }
    if (lean) {
      p.kps = l_kps; p.stages = l_stages; p.resident = l_res;
      static DevOnce once_lean;
      if (once_lean.need()) {
        const char* w_ = "lfsr_conv2d_tc (lean)";
#define LFSR_LEAN_OPT(M, R) opt_in_smem(conv_tc_lean_kernel<M, R, true>, kLeanSmem, w_) || opt_in_smem(conv_tc_lean_kernel<M, R, false>, kLeanSmem, w_)
        if (LFSR_LEAN_OPT(0, false) || LFSR_LEAN_OPT(0, true) || LFSR_LEAN_OPT(1, false) || LFSR_LEAN_OPT(1, true) ||
            LFSR_LEAN_OPT(2, false) || LFSR_LEAN_OPT(2, true))
          return LFSR_ERR_CUDA;
#undef LFSR_LEAN_OPT
        once_lean.done();
      }
      const int lgrid = p.m_tiles < 2 * sm_count ? p.m_tiles : 2 * sm_count;
      if (verbose)
        fprintf(stderr, "[lfsr tc lean] C=%d cout=%d NC=%d k=%dx%d tiles=%d grid=%d stages=%d kps=%d resident=%d out_mode=%d res=%d smem=%zu\n",
                p.C, p.cout, p.NC, p.kh, p.kw, p.m_tiles, lgrid, p.stages, p.kps, p.resident, d->out_mode, d->res.ptr ? 1 : 0, l_smem);
      cudaStream_t st_ = (cudaStream_t)stream;
      const bool hr = d->res.ptr != nullptr;
#define LFSR_LEAN_GO(M, R)                                                                            \
  do {                                                                                                \
    if (f16) conv_tc_lean_kernel<M, R, true><<<lgrid, kThreads, l_smem, st_>>>(tmA, tmB, tmO, p);     \
    else conv_tc_lean_kernel<M, R, false><<<lgrid, kThreads, l_smem, st_>>>(tmA, tmB, tmO, p);        \
  } while (0)
      switch (d->out_mode * 2 + (hr ? 1 : 0)) {
        case 0: LFSR_LEAN_GO(0, false); break;
        case 1: LFSR_LEAN_GO(0, true); break;
        case 2: LFSR_LEAN_GO(1, false); break;
        case 3: LFSR_LEAN_GO(1, true); break;
        case 4: LFSR_LEAN_GO(2, false); break;
        default: LFSR_LEAN_GO(2, true); break;
      }
#undef LFSR_LEAN_GO
      g_lean_launches.fetch_add(1);
      return check_launch("conv_tc_lean_kernel");
    }
  }
  if (verbose)
    fprintf(stderr, "[lfsr tc] C=%d cout=%d NC=%d k=%dx%d tiles=%d grid=%d stages=%d kps=%d resident=%d cta2=%d TH=%d TW=%d vec=%d tma_epi=%d smem=%zu\n",
            p.C, p.cout, p.NC, p.kh, p.kw, p.total_tiles, grid, p.stages, p.kps, p.resident, p.cta2, p.TH, p.TW, p.vec, p.tma_epi, smem);
  static const bool no_t16 = dbg_env("LFSR_TC_NO_T16") != nullptr;
  // sub-pixels per cout-chunk (all r2 of them with one chunk): a multiple of 4 keeps the four warp groups balanced
  const int subs_per_chunk = p.nchunks == 1 ? ry * rx : (p.cq > 0 ? p.NC / p.cq : 0);
  const bool t16 = p.tail_w && !no_t16 && subs_per_chunk >= 4 && subs_per_chunk % 4 == 0 && p.cq <= kTailMaxC;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = smem; cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = p.cta2 ? 2 : 1; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaError_t le;
#ifdef LFSR_DEBUG_HOOKS
  if (p.dbg && !f16)
    le = p.cta2 ? cudaLaunchKernelEx(&cfg, conv_tc_kernel<true, true, false>, tmA, tmB, tmBh, tmO, p, NoTailW{})
                : cudaLaunchKernelEx(&cfg, conv_tc_kernel<false, true, false>, tmA, tmB, tmBh, tmO, p, NoTailW{});
  else if (p.dbg && f16 && p.cta2 && t16) {
    cfg.blockDim = dim3(18 * 32);
    le = cudaLaunchKernelEx(&cfg, conv_tc_kernel<true, true, true, true>, tmA, tmB, tmBh, tmO, p, tt);
  } else if (p.dbg)
    le = p.cta2 ? cudaLaunchKernelEx(&cfg, conv_tc_kernel<true, true, true>, tmA, tmB, tmBh, tmO, p, NoTailW{})
                : cudaLaunchKernelEx(&cfg, conv_tc_kernel<false, true, true>, tmA, tmB, tmBh, tmO, p, NoTailW{});
  else
#endif
  if (t16) {     // tail projection with 16 epilogue warps: every warp group owns whole sub-pixels of the chunk
    cfg.blockDim = dim3(18 * 32);
    if (f16) le = p.cta2 ? cudaLaunchKernelEx(&cfg, conv_tc_kernel<true, false, true, true>, tmA, tmB, tmBh, tmO, p, tt)
                         : cudaLaunchKernelEx(&cfg, conv_tc_kernel<false, false, true, true>, tmA, tmB, tmBh, tmO, p, tt);
    else le = p.cta2 ? cudaLaunchKernelEx(&cfg, conv_tc_kernel<true, false, false, true>, tmA, tmB, tmBh, tmO, p, tt)
                     : cudaLaunchKernelEx(&cfg, conv_tc_kernel<false, false, false, true>, tmA, tmB, tmBh, tmO, p, tt);
  } else if (f16)
    le = p.cta2 ? cudaLaunchKernelEx(&cfg, conv_tc_kernel<true, false, true>, tmA, tmB, tmBh, tmO, p, NoTailW{})
                : cudaLaunchKernelEx(&cfg, conv_tc_kernel<false, false, true>, tmA, tmB, tmBh, tmO, p, NoTailW{});
  else
    le = p.cta2 ? cudaLaunchKernelEx(&cfg, conv_tc_kernel<true, false, false>, tmA, tmB, tmBh, tmO, p, NoTailW{})
                : cudaLaunchKernelEx(&cfg, conv_tc_kernel<false, false, false>, tmA, tmB, tmBh, tmO, p, NoTailW{});
  if (le != cudaSuccess) { set_error("lfsr_conv2d_tc: launch failed: %s", cudaGetErrorString(le)); return LFSR_ERR_CUDA; }
  return check_launch("conv_tc_kernel");
}

extern "C" uint64_t lfsr_conv_tc_lean_count(void) { return lfsr::tc::g_lean_launches.load(); }
extern "C" uint64_t lfsr_conv_tc_halo_count(void) { return lfsr::tc::g_halo_launches.load(); }
