// Thin dense convolutions (<= 20 input channels, 20 output channels) of the Track-2 model's spatial branch
// (MyEfficientLFNet.py:134-141: RepConv 3x3 d=A 18->18 + LReLU, conv 3x3 d=A 18->18), fp32 on CUDA cores.
//
// On the tensor-core path these layers are bound by the fixed cost of a K=8 tf32 MMA (128 rows of the A operand are
// fetched whatever N is): 27 MMAs of N=32 per 128-pixel tile, 0.39 ms per layer at batch 64. With 18x18x9 = 2916 MACs
// per pixel they are cheap enough for the FP32 pipe when every instruction is a packed FFMA2 on an output-channel pair
// and weights arrive as broadcast LDS.128:
//   CTA = 32 x 16 output pixels, 256 threads, thread = 2 pixels (same column, 8 rows apart) sharing every weight load;
//   the 20-float pixels (18 channels + the 2 pad floats of the grouped trunk layout) of the tile + dilation halo are
//   fetched by ONE thread with a 4-D TMA box load (out-of-image = zero = the conv's padding); pixel pitch 20 floats
//   makes the per-lane 128-bit tile reads bank-conflict free; weights [tap][cin][20] sit in shared memory.
// Results are fp32-exact (no TF32 rounding), summed tap by tap, input channel by input channel.
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdlib.h>
#include <mutex>
#include "lfsr_common.cuh"

namespace lfsr {

constexpr int TH_W = 32, TH_H = 16, TH_CP = 20, TH_NP = TH_CP / 2;   // tile, pixel pitch (floats), output pairs
constexpr int TH_PPT = 2, TH_NT = 512 / TH_PPT;                       // pixels per thread, threads per CTA

struct ThinArgs {
  TView in, out, mul;    // mul: optional elementwise multiplier of the activated output (20 readable floats per pixel)
  const float* w;        // [kh*kw][cin][20]
  const float* bias;     // [20] or null
  int kh, kw, dh, dw, cin, act;
  float slope;
  int tiles_x, tiles_y;
  CUtensorMap tm;
};

__device__ __forceinline__ uint32_t th_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void th_ld20(const float* src, float* v) {
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const float4 t = reinterpret_cast<const float4*>(src)[i];
    v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
  }
}
__device__ __forceinline__ void th_ldw(const float* row, f32x2* w) {
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const float4 t = reinterpret_cast<const float4*>(row)[i];
    w[2 * i] = pack2(t.x, t.y); w[2 * i + 1] = pack2(t.z, t.w);
  }
}

// TH_PPT = pixels per thread (same column, TH_H / TH_PPT rows apart): every weight row read from shared memory is used for
// TH_PPT pixels. ncu on this version: L1/TEX (shared-memory) pipe 80 % busy, issue slots 49 % - the weight-row broadcasts
// bound it. 4 pixels per thread with 128-thread CTAs has 45 % fewer LDS per FFMA2 but half the warps per SM and measured
// no faster (0.273 vs 0.261 ms per layer).
template <int CIN>
__global__ void __launch_bounds__(TH_NT)
conv_thin_kernel(const __grid_constant__ ThinArgs a) {
  constexpr int PPT = TH_PPT, NT = TH_NT, RSTEP = TH_H / PPT;
  extern __shared__ __align__(16) float th_smem[];
  __shared__ uint64_t bar;
  const int tid = threadIdx.x;
  const int hy = (a.kh / 2) * a.dh, hx = (a.kw / 2) * a.dw;
  const int SH = TH_H + 2 * hy, SW = TH_W + 2 * hx;
  float* tile = th_smem + ((128u - (th_smem_u32(th_smem) & 127u)) & 127u) / 4;      // [SH][SW][20], TMA destination
  float* wsm = tile + SH * SW * TH_CP;                                               // [taps][CIN][20]
  int t_ = blockIdx.x;
  const int tx0 = (t_ % a.tiles_x) * TH_W; t_ /= a.tiles_x;
  const int ty0 = (t_ % a.tiles_y) * TH_H;
  const int img = t_ / a.tiles_y;
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(th_smem_u32(&bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(th_smem_u32(&bar)), "r"(SH * SW * TH_CP * 4) : "memory");
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(th_smem_u32(tile)), "l"(&a.tm), "r"(th_smem_u32(&bar)), "r"(0), "r"(tx0 - hx), "r"(ty0 - hy), "r"(img)
                 : "memory");
  }
  const int taps = a.kh * a.kw;
  for (int i = tid; i < taps * CIN * (TH_CP / 4); i += NT)
    reinterpret_cast<float4*>(wsm)[i] = __ldg(reinterpret_cast<const float4*>(a.w) + i);
  __syncthreads();
  {
    const uint32_t addr = th_smem_u32(&bar);
    uint32_t done = 0;
    for (uint32_t it = 0; it < (1u << 26) && !done; ++it)       // bounded: a protocol bug must fault, not hang the GPU
      asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                   : "=r"(done) : "r"(addr) : "memory");
    if (!done) __trap();
  }
  const int lx = tid & 31, ly = tid >> 5;               // pixels (lx, ly + h * RSTEP), h < PPT
  f32x2 acc[PPT][TH_NP];
#pragma unroll
  for (int i = 0; i < TH_NP; ++i) {
    const f32x2 b = a.bias ? pack2(__ldg(a.bias + 2 * i), __ldg(a.bias + 2 * i + 1)) : pack2(0.f, 0.f);
#pragma unroll
    for (int h = 0; h < PPT; ++h) acc[h][i] = b;
  }
  const int hstep = RSTEP * SW * TH_CP;
  for (int ky = 0; ky < a.kh; ++ky)
    for (int kx = 0; kx < a.kw; ++kx) {
      const float* p0 = tile + ((ly + ky * a.dh) * SW + lx + kx * a.dw) * TH_CP;
      const float* wt = wsm + (ky * a.kw + kx) * CIN * TH_CP;
#pragma unroll
      for (int cq = 0; cq < (CIN + 3) / 4; ++cq) {            // four input channels at a time: one LDS.128 per pixel
        float v[PPT][4];
#pragma unroll
        for (int h = 0; h < PPT; ++h) {
          const float4 t = *reinterpret_cast<const float4*>(p0 + h * hstep + cq * 4);
          v[h][0] = t.x; v[h][1] = t.y; v[h][2] = t.z; v[h][3] = t.w;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int c = cq * 4 + j;
          if (c < CIN) {
            f32x2 w[TH_NP];
            th_ldw(wt + c * TH_CP, w);
#pragma unroll
            for (int h = 0; h < PPT; ++h) {
              const f32x2 bb = pack2(v[h][j], v[h][j]);
#pragma unroll
              for (int i = 0; i < TH_NP; ++i) acc[h][i] = fma2(bb, w[i], acc[h][i]);
            }
          }
        }
      }
    }
  const int ox = tx0 + lx;
  if (ox >= a.out.w) return;
#pragma unroll
  for (int h = 0; h < PPT; ++h) {
    const int oy = ty0 + ly + RSTEP * h;
    if (oy >= a.out.h) continue;
    float o[TH_CP];
#pragma unroll
    for (int i = 0; i < TH_NP; ++i) unpack2(acc[h][i], o[2 * i], o[2 * i + 1]);
    if (a.act) {
#pragma unroll
      for (int i = 0; i < TH_CP; ++i) o[i] = apply_act(o[i], a.act, a.slope);
    }
    if (a.mul.p) {
      const float4* mp = reinterpret_cast<const float4*>(a.mul.p + a.mul.pix(img, oy, ox));
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        const float4 m = mp[i];
        o[4 * i] *= m.x; o[4 * i + 1] *= m.y; o[4 * i + 2] *= m.z; o[4 * i + 3] *= m.w;
      }
    }
    float4* dst = reinterpret_cast<float4*>(a.out.p + a.out.pix(img, oy, ox));
#pragma unroll
    for (int i = 0; i < 5; ++i) dst[i] = make_float4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
  }
}

// ---- stems: ONE input channel (the Y mosaic), <= 64 output channels, <= 9 taps ---------------------------------------
// (MyEfficientLFNet.py:40-43 RepConv(1, C) d=A; MyEfficientLFNetV4_5.py:42.) HBM-bound on the output write: thread = (pixel, output-channel quad), tap weights of the quad in registers,
// the 9 input taps are L1 hits shared by the 16 quads of a pixel.
struct StemArgs {
  TView in, out;
  const float* w;        // [taps][cout]
  const float* bias;
  int kh, kw, dh, dw, ph, pw, act;
  float slope;
  int perm_a;            // > 0: MacPI addressing over SAI storage with dilation == perm_a (see conv_stem_macpi_kernel)
  int bh, bw;            // view blocking (EPIT's per-view Conv3d(1,3,3), EPIT.py:24): taps that leave the bh x bw block of
                         // the output pixel read zero; bh = H, bw = W without blocking
  __half* o16;           // conv_stem_tile_kernel: optional fp16 copy of the output (lfsr_conv_desc.out_mode 1): the operand of
  int o16_ld;            // the first tensor-core layer, so that no separate conversion pass re-reads the fp32 tensor
};

__global__ void __launch_bounds__(256)
conv_stem_kernel(const StemArgs a) {
  const int q = threadIdx.x & 15, lx = threadIdx.x >> 4;
  const int c = q * 4;
  const int ox = blockIdx.x * 16 + lx, oy0 = blockIdx.y * 8, img = blockIdx.z;
  if (c >= a.out.c || ox >= a.out.w) return;
  const int taps = a.kh * a.kw;
  const int H = a.in.h, W = a.in.w;
  float4 wk[9];
  int off[9], dy[9];
  unsigned xmask = 0;                  // taps whose column lies inside the image / the pixel's view (fixed per thread)
  const int bx0 = ox / a.bw * a.bw;    // first column of the block that holds this pixel
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    const int ky = t / a.kw, kx = t - ky * a.kw;
    const int dx = kx * a.dw - a.pw;
    dy[t] = ky * a.dh - a.ph;
    off[t] = dy[t] * W + dx;
    if (t < taps && ox + dx >= bx0 && ox + dx < bx0 + a.bw) xmask |= 1u << t;
    wk[t] = t < taps ? __ldg(reinterpret_cast<const float4*>(a.w + t * a.out.c + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float4 b = a.bias ? __ldg(reinterpret_cast<const float4*>(a.bias + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
  const float* colp = a.in.p + (size_t)img * H * W + ox;          // one input channel: pixel pitch 1
  float* dst = a.out.p + a.out.pix(img, oy0, ox) + c;
  const int orow = a.out.w * a.out.ld;
  const int ymax = min(oy0 + 8, a.out.h);
  for (int oy = oy0; oy < ymax; ++oy, dst += orow) {
    float4 acc = b;
    const float* rowp = colp + oy * W;
    const int by0 = oy / a.bh * a.bh;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const bool ok = ((xmask >> t) & 1u) && (unsigned)(oy + dy[t] - by0) < (unsigned)a.bh;
      const float v = ok ? __ldg(rowp + off[t]) : 0.f;
      acc.x = fmaf(v, wk[t].x, acc.x); acc.y = fmaf(v, wk[t].y, acc.y); acc.z = fmaf(v, wk[t].z, acc.z); acc.w = fmaf(v, wk[t].w, acc.w);
    }
    if (a.act) {
      acc.x = apply_act(acc.x, a.act, a.slope); acc.y = apply_act(acc.y, a.act, a.slope);
      acc.z = apply_act(acc.z, a.act, a.slope); acc.w = apply_act(acc.w, a.act, a.slope);
    }
    *reinterpret_cast<float4*>(dst) = acc;
  }
}

// The same layer with the single-channel input tile (+ dilation halo) staged in shared memory once per CTA: image borders and
// view blocking are resolved while staging (a 16 x 8 tile lies inside one view block when the block size is a multiple of
// 16 x 8), so the row loop is nine unpredicated shared-memory reads (16 lanes share an address) + packed FFMA2 per output
// quad. conv_stem_kernel spends ~260 issued instructions per output row and warp on predicates and address arithmetic
// (ncu: 71 % SM throughput at 17 % of DRAM) for a layer that only has to write its output.
__global__ void __launch_bounds__(256)
conv_stem_tile_kernel(const StemArgs a) {
  extern __shared__ float st_in[];                 // [8 + 2 ph][16 + 2 pw]
  const int q = threadIdx.x & 15, lx = threadIdx.x >> 4;
  const int c = q * 4;
  const int ox0 = blockIdx.x * 16, oy0 = blockIdx.y * 8, img = blockIdx.z;
  const int H = a.in.h, W = a.in.w;
  const int SW = 16 + 2 * a.pw, SH = 8 + 2 * a.ph;
  const int bx0 = ox0 / a.bw * a.bw, by0 = oy0 / a.bh * a.bh;     // the view block of this tile
  const float* src = a.in.p + (size_t)img * H * W;
  if (a.perm_a) {
    // MacPI addressing over SAI storage (DistgSSR.py:21, LF_InterNet.py:24): the tile is staged in MacPI coordinates, a MacPI
    // position (i*A+u, j*A+v) reading pixel (i, j) of view (u, v); outside the MacPI image = outside the view = zero. The layer
    // is then the same dilation-A conv as the SAI stems.
    const int A = a.perm_a, hh = H / A, ww = W / A;
    for (int i = threadIdx.x; i < SH * SW; i += 256) {
      const int ly = i / SW, lxx = i - ly * SW;
      const int Y = oy0 - a.ph + ly, X = ox0 - a.pw + lxx;
      float v = 0.f;
      if (Y >= 0 && Y < H && X >= 0 && X < W) {
        const int ii = Y / A, u = Y - ii * A, jj = X / A, vv = X - jj * A;
        v = __ldg(src + (u * hh + ii) * W + vv * ww + jj);
      }
      st_in[i] = v;
    }
  } else {
    for (int i = threadIdx.x; i < SH * SW; i += 256) {
      const int ly = i / SW, lxx = i - ly * SW;
      const int iy = oy0 - a.ph + ly, ix = ox0 - a.pw + lxx;
      const bool ok = iy >= by0 && iy < by0 + a.bh && iy < H && ix >= bx0 && ix < bx0 + a.bw && ix < W;
      st_in[i] = ok ? __ldg(src + iy * W + ix) : 0.f;
    }
  }
  __syncthreads();
  const int ox = ox0 + lx;
  if (c >= a.out.c || ox >= a.out.w) return;
  const int taps = a.kh * a.kw;
  f32x2 wlo[9], whi[9];
  int toff[9];
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    const int ky = t / a.kw, kx = t - ky * a.kw;
    toff[t] = t < taps ? ky * a.dh * SW + kx * a.dw : 0;
    const float4 w = t < taps ? __ldg(reinterpret_cast<const float4*>(a.w + t * a.out.c + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
    wlo[t] = pack2(w.x, w.y); whi[t] = pack2(w.z, w.w);
  }
  const float4 b = a.bias ? __ldg(reinterpret_cast<const float4*>(a.bias + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
  const f32x2 blo = pack2(b.x, b.y), bhi = pack2(b.z, b.w);
  float* dst = a.out.p + a.out.pix(img, oy0, ox) + c;
  const int orow = a.out.w * a.out.ld;
  const int rows = min(8, a.out.h - oy0);
  const float* tp = st_in + lx;
  for (int r = 0; r < rows; ++r, dst += orow, tp += SW) {
    f32x2 lo = blo, hi = bhi;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const float v = tp[toff[t]];
      const f32x2 vv = pack2(v, v);
      lo = fma2(vv, wlo[t], lo); hi = fma2(vv, whi[t], hi);
    }
    float4 acc;
    unpack2(lo, acc.x, acc.y); unpack2(hi, acc.z, acc.w);
    if (a.act) {
      acc.x = apply_act(acc.x, a.act, a.slope); acc.y = apply_act(acc.y, a.act, a.slope);
      acc.z = apply_act(acc.z, a.act, a.slope); acc.w = apply_act(acc.w, a.act, a.slope);
    }
    *reinterpret_cast<float4*>(dst) = acc;
    if (a.o16) {
      const __half2 h0 = __floats2half2_rn(acc.x, acc.y), h1 = __floats2half2_rn(acc.z, acc.w);
      uint2 v;
      v.x = *reinterpret_cast<const uint32_t*>(&h0); v.y = *reinterpret_cast<const uint32_t*>(&h1);
      *reinterpret_cast<uint2*>(a.o16 + ((size_t)((size_t)img * a.out.h + oy0 + r) * a.out.w + ox) * (size_t)a.o16_ld + c) = v;
    }
  }
}

// MacPI-addressed stems (DistgSSR.py:21, LF_InterNet.py:24: conv d = A over SAI2MacPI(x)): a tap of dilation A moves the
// MacPI coordinate (i*A+u, j*A+v) to (i+k)*A+u - the same view (u, v), neighbouring in-view pixel - so on the SAI
// storage the layer is a dense 3x3 conv inside each view with zero padding at the view border. One coordinate split per
// thread, taps are plain storage offsets; the output is written in the MacPI arrangement the trunk works in.
__global__ void __launch_bounds__(256)
conv_stem_macpi_kernel(const StemArgs a) {
  const int q = threadIdx.x & 15, lx = threadIdx.x >> 4;
  const int c = q * 4;
  const int ox = blockIdx.x * 16 + lx, oy0 = blockIdx.y * 8, img = blockIdx.z;
  if (c >= a.out.c || ox >= a.out.w) return;
  const int A = a.perm_a, H = a.in.h, W = a.in.w, hh = H / A, ww = W / A;
  const int taps = a.kh * a.kw;
  float4 wk[9];
#pragma unroll
  for (int t = 0; t < 9; ++t) wk[t] = t < taps ? __ldg(reinterpret_cast<const float4*>(a.w + t * a.out.c + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
  const float4 b = a.bias ? __ldg(reinterpret_cast<const float4*>(a.bias + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
  const int j = ox / A, v = ox - j * A;                  // MacPI column -> (in-view column j, view v)
  const float* img_p = a.in.p + (size_t)img * H * W;
  const int ymax = min(oy0 + 8, a.out.h);
  for (int oy = oy0; oy < ymax; ++oy) {
    const int i = oy / A, u = oy - i * A;
    const float* vp = img_p + (u * hh) * W + v * ww;     // top-left of view (u, v) in the SAI mosaic
    float4 acc = b;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      if (t >= taps) break;
      const int ky = t / a.kw, kx = t - ky * a.kw;
      const int ii = i + ky - a.kh / 2, jj = j + kx - a.kw / 2;
      const bool ok = (unsigned)ii < (unsigned)hh && (unsigned)jj < (unsigned)ww;
      const float x = ok ? __ldg(vp + ii * W + jj) : 0.f;
      acc.x = fmaf(x, wk[t].x, acc.x); acc.y = fmaf(x, wk[t].y, acc.y); acc.z = fmaf(x, wk[t].z, acc.z); acc.w = fmaf(x, wk[t].w, acc.w);
    }
    if (a.act) {
      acc.x = apply_act(acc.x, a.act, a.slope); acc.y = apply_act(acc.y, a.act, a.slope);
      acc.z = apply_act(acc.z, a.act, a.slope); acc.w = apply_act(acc.w, a.act, a.slope);
    }
    *reinterpret_cast<float4*>(a.out.p + a.out.pix(img, oy, ox) + c) = acc;
  }
}

typedef CUresult (*ThEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static ThEncodeFn th_get_encode() {
  static ThEncodeFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<ThEncodeFn>(p);
  });
  return fn;
}

static size_t thin_smem(const lfsr_tensor* in, const lfsr_conv_desc* d) {
  const int hy = (d->kh / 2) * d->dil_h, hx = (d->kw / 2) * d->dil_w;
  return ((size_t)(TH_H + 2 * hy) * (TH_W + 2 * hx) * TH_CP + (size_t)d->kh * d->kw * in->c * TH_CP) * sizeof(float) + 128;
}

}  // namespace lfsr

using namespace lfsr;

extern "C" int lfsr_conv2d_thin_supported(const lfsr_tensor* in, const lfsr_tensor* out, const lfsr_conv_desc* d) {
  if (!tensor_ok(in) || !tensor_ok(out) || !d) return 0;
  if (in->c != 16 && in->c != 18 && in->c != 20) return 0;
  if (out->c != TH_CP || out->ld % 4 || ((uintptr_t)out->ptr & 15)) return 0;
  // the tile is read as 20-float pixels: the floats behind an 18- or 16-channel view must exist (grouped trunk slices)
  if (in->ld < TH_CP || in->ld % 4 || ((uintptr_t)in->ptr & 15)) return 0;
  if (d->stride_h != 1 || d->stride_w != 1 || d->in_perm || d->out_perm || d->res.ptr || d->in_scale || d->tail_w) return 0;
  if (d->mul.ptr && (d->mul_act || d->mul.c != TH_CP || d->mul.ld % 4 || ((uintptr_t)d->mul.ptr & 15) || d->mul.n != out->n ||
                     d->mul.h != out->h || d->mul.w != out->w)) return 0;
  if (d->shuf_ry > 1 || d->shuf_rx > 1 || d->block_h > 0 || d->block_w > 0 || d->alpha != 1.f) return 0;
  if (!(d->kh & 1) || !(d->kw & 1) || d->kh * d->kw > 9) return 0;
  if (2 * d->pad_h != d->dil_h * (d->kh - 1) || 2 * d->pad_w != d->dil_w * (d->kw - 1)) return 0;
  if (out->n != in->n || out->h != in->h || out->w != in->w) return 0;
  if (TH_W + d->dil_w * (d->kw - 1) > 256 || TH_H + d->dil_h * (d->kh - 1) > 256) return 0;
  if (thin_smem(in, d) > 110 * 1024) return 0;
  return th_get_encode() != nullptr;
}

extern "C" int lfsr_conv2d_thin(const lfsr_tensor* in, const float* w_packed, const lfsr_tensor* out, const lfsr_conv_desc* d,
                                void* stream) {
  LFSR_REQUIRE(w_packed && lfsr_conv2d_thin_supported(in, out, d), "lfsr_conv2d_thin: unsupported problem");
  LFSR_REQUIRE(((uintptr_t)w_packed & 15) == 0, "lfsr_conv2d_thin: weights must be 16-byte aligned");
  ThinArgs a;
  a.in = view_of(in); a.out = view_of(out);
  a.mul = d->mul.ptr ? view_of(&d->mul) : null_view();
  a.w = w_packed; a.bias = d->bias;
  a.kh = d->kh; a.kw = d->kw; a.dh = d->dil_h; a.dw = d->dil_w; a.cin = in->c; a.act = d->act; a.slope = d->act_slope;
  a.tiles_x = ceil_div(out->w, TH_W); a.tiles_y = ceil_div(out->h, TH_H);
  {
    const cuuint64_t ld_b = (cuuint64_t)in->ld * 4;
    cuuint64_t dims[4] = {(cuuint64_t)TH_CP, (cuuint64_t)in->w, (cuuint64_t)in->h, (cuuint64_t)in->n};
    cuuint64_t strides[3] = {ld_b, ld_b * in->w, ld_b * in->w * in->h};
    cuuint32_t box[4] = {(cuuint32_t)TH_CP, (cuuint32_t)(TH_W + d->dil_w * (d->kw - 1)), (cuuint32_t)(TH_H + d->dil_h * (d->kh - 1)), 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = th_get_encode()(&a.tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, in->ptr, dims, strides, box, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("lfsr_conv2d_thin: cuTensorMapEncodeTiled failed with %d", (int)r); return LFSR_ERR_CUDA; }
  }
  const size_t smem = thin_smem(in, d);
  const int blocks = out->n * a.tiles_x * a.tiles_y;
  cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH_THIN(CIN)                                                                                            \
  do {                                                                                                              \
    static DevOnce once;                                                                                            \
    if (once.need()) {                                                                                              \
      if (opt_in_smem(conv_thin_kernel<CIN>, 110 * 1024, "lfsr_conv2d_thin")) return LFSR_ERR_CUDA;                 \
      once.done();                                                                                                  \
    }                                                                                                               \
    conv_thin_kernel<CIN><<<blocks, TH_NT, smem, st>>>(a);                                                          \
  } while (0)
  switch (in->c) {
    case 16: LAUNCH_THIN(16); break;
    case 18: LAUNCH_THIN(18); break;
    default: LAUNCH_THIN(20); break;
  }
#undef LAUNCH_THIN
  return check_launch("conv_thin_kernel");
}

extern "C" int lfsr_conv2d_stem_supported(const lfsr_tensor* in, const lfsr_tensor* out, const lfsr_conv_desc* d) {
  if (!tensor_ok(in) || !tensor_ok(out) || !d) return 0;
  if (in->c != 1 || out->c > 64 || out->c % 4 || out->ld % 4 || ((uintptr_t)out->ptr & 15)) return 0;
  if (d->stride_h != 1 || d->stride_w != 1 || d->out_perm || d->mul.ptr || d->res.ptr || d->in_scale || d->tail_w) return 0;
  if (d->shuf_ry > 1 || d->shuf_rx > 1 || d->alpha != 1.f) return 0;
  if (d->out_mode != 0) {          // fp32 + fp16 copy: the tiled kernel only (same conditions as at launch), never fp16 alone
    const lfsr_tensor* o = &d->out16;
    if (d->out_mode != 1 || d->in_perm || !tensor_ok(o) || o->n != out->n || o->h != out->h || o->w != out->w || o->c != out->c ||
        o->ld % 4 || ((uintptr_t)o->ptr & 7)) return 0;
    const int bh = d->block_h > 0 ? d->block_h : in->h, bw = d->block_w > 0 ? d->block_w : in->w;
    if (!((bw == in->w || bw % 16 == 0) && (bh == in->h || bh % 8 == 0))) return 0;
    if ((size_t)(8 + 2 * d->pad_h) * (16 + 2 * d->pad_w) * sizeof(float) > 40 * 1024) return 0;
  }
  if ((d->block_h > 0 || d->block_w > 0) &&
      (d->in_perm || (d->block_h > 0 && in->h % d->block_h) || (d->block_w > 0 && in->w % d->block_w))) return 0;
  if (d->kh * d->kw > 9 || d->kh < 1 || d->kw < 1) return 0;
  if (2 * d->pad_h != d->dil_h * (d->kh - 1) || 2 * d->pad_w != d->dil_w * (d->kw - 1)) return 0;
  if (out->n != in->n || out->h != in->h || out->w != in->w || out->n > 65535) return 0;
  if (in->ld != 1 || (long long)in->h * in->w >= 0x7fffffffLL) return 0;
  if (d->in_perm) {        // MacPI addressing: only the case that is a per-view dense conv (dilation == angular resolution)
    const int A = d->perm_a;
    if (d->in_perm != LFSR_PERM_MACPI_OVER_SAI || A < 1 || in->h % A || in->w % A || d->dil_h != A || d->dil_w != A) return 0;
  }
  return 1;
}

extern "C" int lfsr_conv2d_stem(const lfsr_tensor* in, const float* w_packed, const lfsr_tensor* out, const lfsr_conv_desc* d,
                                void* stream) {
  LFSR_REQUIRE(w_packed && lfsr_conv2d_stem_supported(in, out, d), "lfsr_conv2d_stem: unsupported problem");
  LFSR_REQUIRE((((uintptr_t)w_packed | (uintptr_t)d->bias) & 15) == 0, "lfsr_conv2d_stem: weights and bias must be 16-byte aligned");
  StemArgs a;
  a.in = view_of(in); a.out = view_of(out);
  a.w = w_packed; a.bias = d->bias;
  a.kh = d->kh; a.kw = d->kw; a.dh = d->dil_h; a.dw = d->dil_w; a.ph = d->pad_h; a.pw = d->pad_w;
  a.act = d->act; a.slope = d->act_slope; a.perm_a = d->in_perm ? d->perm_a : 0;
  a.bh = d->block_h > 0 ? d->block_h : in->h; a.bw = d->block_w > 0 ? d->block_w : in->w;
  a.o16 = d->out_mode == 1 ? (__half*)d->out16.ptr : nullptr;
  a.o16_ld = d->out_mode == 1 ? (int)d->out16.ld : 0;
  dim3 grid(ceil_div(out->w, 16), ceil_div(out->h, 8), out->n);
  if (a.perm_a) {
    const size_t tile_m = (size_t)(8 + 2 * a.ph) * (16 + 2 * a.pw) * sizeof(float);
    if (a.bh == in->h && a.bw == in->w && a.ph == a.dh * (a.kh / 2) && a.pw == a.dw * (a.kw / 2) && tile_m <= 40 * 1024) {
      conv_stem_tile_kernel<<<grid, 256, tile_m, (cudaStream_t)stream>>>(a);
      return check_launch("conv_stem_tile_kernel");
    }
    conv_stem_macpi_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    return check_launch("conv_stem_macpi_kernel");
  }
  const size_t tile_b = (size_t)(8 + 2 * a.ph) * (16 + 2 * a.pw) * sizeof(float);
  if ((a.bw == in->w || a.bw % 16 == 0) && (a.bh == in->h || a.bh % 8 == 0) && tile_b <= 40 * 1024 &&
      (long long)in->h * in->w < 0x7fffffffLL) {
    conv_stem_tile_kernel<<<grid, 256, tile_b, (cudaStream_t)stream>>>(a);
    return check_launch("conv_stem_tile_kernel");
  }
  conv_stem_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a);
  return check_launch("conv_stem_kernel");
}

// ---- angular expand: 1x1 conv cin -> cq*A*A + PixelShuffle(A) + activation * alpha + residual ---------------------------
// (MyEfficientLFNet.py:262-275: AngularAttention.expand, the LReLU, `x + scale * out`.) Per low-resolution pixel this reads
// cin <= 20 values and writes A*A pixels of cq channels: 2916 MACs for 2 KB of output - streaming work. On the tensor-core
// conv it was bound by its epilogue (one residual round trip per 32-pixel block and warp, 0.19 ms at batch 64); here a
// thread owns one (sub-pixel column j, channel quad q) with its cin x 4 weights in registers and walks the low-resolution
// pixels of `yg` rows, every output a coalesced 16-byte store, the residuals of a row loaded together up front.
namespace lfsr {
struct AngExpArgs {
  TView in, res, out;
  const float* w;      // [A][A][cin][cq]  (sub-pixel row i, column j)
  int A, cq4, act, yg, groups;
  float slope, alpha;
};

template <int CIN>
__global__ void __launch_bounds__(256, 2)
ang_expand_kernel(const AngExpArgs a) {
  extern __shared__ __align__(16) float ae_s[];        // [yg][w][20] staged low-resolution rows
  const int tid = threadIdx.x;
  int b = blockIdx.x;
  const int g = b % a.groups; b /= a.groups;
  const int i = b % a.A;
  const int img = b / a.A;
  const int wl = a.in.w, cq = a.cq4 * 4;
  const int y0 = g * a.yg;
  const int rows = min(a.yg, a.in.h - y0);
  // (requesting the CTA's residual rows into L2 up front was tried: 0.170 vs 0.160 ms - the kernel is not latency-bound on them)
  for (int t = tid; t < rows * wl * 5; t += 256) {       // 20 floats per pixel (cin real + zeros)
    const int u = t % 5, px = t / 5;
    const int yy = px / wl, xx = px - yy * wl;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    const float* src = a.in.p + a.in.pix(img, y0 + yy, xx);
    if (4 * u + 3 < CIN) v = __ldg(reinterpret_cast<const float4*>(src + 4 * u));
    else {
      if (4 * u < CIN) v.x = __ldg(src + 4 * u);
      if (4 * u + 1 < CIN) v.y = __ldg(src + 4 * u + 1);
      if (4 * u + 2 < CIN) v.z = __ldg(src + 4 * u + 2);
    }
    reinterpret_cast<float4*>(ae_s)[t] = v;
  }
  const int combos = a.A * a.cq4;
  const int XG = 256 / combos;
  const int xg = tid / combos, r = tid - xg * combos;
  const int j = r / a.cq4, q = r - j * a.cq4;
  float4 w[CIN];
  if (xg < XG) {
    const float* wp = a.w + ((size_t)(i * a.A + j) * CIN) * cq + 4 * q;
#pragma unroll
    for (int k = 0; k < CIN; ++k) w[k] = __ldg(reinterpret_cast<const float4*>(wp + k * cq));
  }
  __syncthreads();
  if (xg >= XG) return;
  constexpr int NX = 4;                                  // low-resolution pixels per thread and pass
  for (int yy = 0; yy < rows; ++yy) {
    const int oy = (y0 + yy) * a.A + i;
    const size_t orow = a.out.pix(img, oy, 0), rrow = a.res.p ? a.res.pix(img, oy, 0) : 0;
    for (int x0 = xg; x0 < wl; x0 += NX * XG) {
      float4 rv[NX];
#pragma unroll
      for (int u = 0; u < NX; ++u) {
        const int X = x0 + u * XG;
        rv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a.res.p && X < wl) rv[u] = *reinterpret_cast<const float4*>(a.res.p + rrow + (size_t)(X * a.A + j) * a.res.ld + 4 * q);
      }
#pragma unroll
      for (int u = 0; u < NX; ++u) {
        const int X = x0 + u * XG;
        if (X >= wl) break;
        const float4* xp = reinterpret_cast<const float4*>(ae_s + (yy * wl + X) * 20);
        float xin[20];
#pragma unroll
        for (int c = 0; c < 5; ++c) { const float4 t4 = xp[c]; xin[4 * c] = t4.x; xin[4 * c + 1] = t4.y; xin[4 * c + 2] = t4.z; xin[4 * c + 3] = t4.w; }
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < CIN; ++k) {
          acc.x = fmaf(xin[k], w[k].x, acc.x); acc.y = fmaf(xin[k], w[k].y, acc.y);
          acc.z = fmaf(xin[k], w[k].z, acc.z); acc.w = fmaf(xin[k], w[k].w, acc.w);
        }
        acc.x = fmaf(apply_act(acc.x, a.act, a.slope), a.alpha, rv[u].x); acc.y = fmaf(apply_act(acc.y, a.act, a.slope), a.alpha, rv[u].y);
        acc.z = fmaf(apply_act(acc.z, a.act, a.slope), a.alpha, rv[u].z); acc.w = fmaf(apply_act(acc.w, a.act, a.slope), a.alpha, rv[u].w);
        *reinterpret_cast<float4*>(a.out.p + orow + (size_t)(X * a.A + j) * a.out.ld + 4 * q) = acc;
      }
    }
  }
}
}  // namespace lfsr

extern "C" int lfsr_ang_expand(const lfsr_tensor* in, const float* w, const lfsr_tensor* res, const lfsr_tensor* out, int A, int act,
                               float slope, float alpha, void* stream) {
  LFSR_REQUIRE(tensor_ok(in) && tensor_ok(out) && w && A >= 1, "lfsr_ang_expand: null/invalid argument");
  LFSR_REQUIRE(out->n == in->n && out->h == in->h * A && out->w == in->w * A, "lfsr_ang_expand: out must be A x the input size");
  LFSR_REQUIRE(out->c % 4 == 0 && out->ld % 4 == 0 && ((uintptr_t)out->ptr & 15) == 0 && ((uintptr_t)w & 15) == 0,
               "lfsr_ang_expand: output channels in 16-byte aligned quads");
  LFSR_REQUIRE(in->ld % 4 == 0 && ((uintptr_t)in->ptr & 15) == 0 && in->ld >= ((in->c + 3) & ~3),
               "lfsr_ang_expand: input pixels must be 16-byte aligned with readable pad floats");
  LFSR_REQUIRE(A * (out->c / 4) <= 256, "lfsr_ang_expand: A x channel quads must fit one CTA");
  const bool has_res = res && res->ptr;
  if (has_res)
    LFSR_REQUIRE(res->n == out->n && res->h == out->h && res->w == out->w && res->c == out->c && res->ld % 4 == 0 &&
                     ((uintptr_t)res->ptr & 15) == 0, "lfsr_ang_expand: res shape / alignment");
  lfsr::AngExpArgs a;
  a.in = view_of(in); a.out = view_of(out); a.res = has_res ? view_of(res) : null_view();
  a.w = w; a.A = A; a.cq4 = out->c / 4; a.act = act; a.slope = slope; a.alpha = alpha;
  a.yg = 8;
  while (a.yg > 1 && (size_t)a.yg * in->w * 20 * 4 > 40 * 1024) a.yg >>= 1;
  LFSR_REQUIRE((size_t)a.yg * in->w * 20 * 4 <= 40 * 1024, "lfsr_ang_expand: input rows too wide");
  a.groups = ceil_div(in->h, a.yg);
  const size_t smem = (size_t)a.yg * in->w * 20 * 4;
  const long long grid = (long long)in->n * A * a.groups;
  LFSR_REQUIRE(grid <= 0x7fffffffLL, "lfsr_ang_expand: grid too large");
  cudaStream_t st = (cudaStream_t)stream;
  switch (in->c) {
    case 16: lfsr::ang_expand_kernel<16><<<(unsigned)grid, 256, smem, st>>>(a); break;
    case 18: lfsr::ang_expand_kernel<18><<<(unsigned)grid, 256, smem, st>>>(a); break;
    case 20: lfsr::ang_expand_kernel<20><<<(unsigned)grid, 256, smem, st>>>(a); break;
    default: LFSR_REQUIRE(false, "lfsr_ang_expand: built for 16 / 18 / 20 input channels, got %d", in->c);
  }
  return check_launch("ang_expand_kernel");
}


// ---- 1x1 conv to 8 / 16 output channels, fp32 --------------------------------------------------------------------------
// DistgSSR's composed reconstruction tail (DistgSSR.py:24-27 folded to one 1x1 64 -> s^2, see lfnets/distgssr.py) produces
// the image itself, so it stays fp32; on the general fp32 implicit GEMM it took 0.6 ms at batch 64 for 1.7 GFLOP. Here a
// thread owns two pixels (one weight read feeds both), weights [cin][cout] are broadcast from shared memory, packed FFMA2.
namespace lfsr {
template <int COUT>
__global__ void __launch_bounds__(256)
conv1x1_few_kernel(TView in, TView out, const float* __restrict__ w, const float* __restrict__ bias, int act, float slope,
                   long long pixels) {
  extern __shared__ __align__(16) float cf_w[];        // [cin][COUT]
  const int C = in.c;
  for (int i = threadIdx.x; i < C * COUT; i += 256) cf_w[i] = __ldg(w + i);
  __syncthreads();
  const long long half = (pixels + 1) / 2;
  for (long long t = (long long)blockIdx.x * 256 + threadIdx.x; t < half; t += (long long)gridDim.x * 256) {
    const long long p0 = t, p1 = t + half;            // two pixels half the tensor apart: both streams stay coalesced
    const bool two = p1 < pixels;
    const float* s0 = in.p + p0 * in.ld;
    const float* s1 = in.p + (two ? p1 : p0) * in.ld;
    f32x2 a0[COUT / 2], a1[COUT / 2];
#pragma unroll
    for (int o = 0; o < COUT / 2; ++o) {
      const f32x2 b = bias ? pack2(__ldg(bias + 2 * o), __ldg(bias + 2 * o + 1)) : pack2(0.f, 0.f);
      a0[o] = b; a1[o] = b;
    }
    for (int c = 0; c < C; c += 4) {
      const float4 x0 = __ldg(reinterpret_cast<const float4*>(s0 + c)), x1 = __ldg(reinterpret_cast<const float4*>(s1 + c));
      const float xs0[4] = {x0.x, x0.y, x0.z, x0.w}, xs1[4] = {x1.x, x1.y, x1.z, x1.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float4* wr = reinterpret_cast<const float4*>(cf_w + (c + k) * COUT);
        const f32x2 v0 = pack2(xs0[k], xs0[k]), v1 = pack2(xs1[k], xs1[k]);
#pragma unroll
        for (int q = 0; q < COUT / 4; ++q) {
          const float4 ww = wr[q];
          const f32x2 wl = pack2(ww.x, ww.y), wh = pack2(ww.z, ww.w);
          a0[2 * q] = fma2(v0, wl, a0[2 * q]); a0[2 * q + 1] = fma2(v0, wh, a0[2 * q + 1]);
          a1[2 * q] = fma2(v1, wl, a1[2 * q]); a1[2 * q + 1] = fma2(v1, wh, a1[2 * q + 1]);
        }
      }
    }
#pragma unroll
    for (int q = 0; q < COUT / 4; ++q) {
      float4 r0, r1;
      unpack2(a0[2 * q], r0.x, r0.y); unpack2(a0[2 * q + 1], r0.z, r0.w);
      unpack2(a1[2 * q], r1.x, r1.y); unpack2(a1[2 * q + 1], r1.z, r1.w);
      if (act) {
        r0.x = apply_act(r0.x, act, slope); r0.y = apply_act(r0.y, act, slope); r0.z = apply_act(r0.z, act, slope); r0.w = apply_act(r0.w, act, slope);
        r1.x = apply_act(r1.x, act, slope); r1.y = apply_act(r1.y, act, slope); r1.z = apply_act(r1.z, act, slope); r1.w = apply_act(r1.w, act, slope);
      }
      *reinterpret_cast<float4*>(out.p + p0 * out.ld + 4 * q) = r0;
      if (two) *reinterpret_cast<float4*>(out.p + p1 * out.ld + 4 * q) = r1;
    }
  }
}
}  // namespace lfsr

extern "C" int lfsr_conv1x1_few_supported(const lfsr_tensor* in, const lfsr_tensor* out, const lfsr_conv_desc* d) {
  if (!tensor_ok(in) || !tensor_ok(out) || !d) return 0;
  if (d->kh != 1 || d->kw != 1 || d->stride_h != 1 || d->stride_w != 1 || d->pad_h || d->pad_w) return 0;
  if (d->in_perm || d->out_perm || d->mul.ptr || d->res.ptr || d->in_scale || d->tail_w || d->out_mode || d->in_f16) return 0;
  if (d->shuf_ry > 1 || d->shuf_rx > 1 || d->block_h > 0 || d->block_w > 0 || d->alpha != 1.f) return 0;
  if (out->n != in->n || out->h != in->h || out->w != in->w) return 0;
  if ((out->c != 8 && out->c != 16) || in->c % 4 || in->c > 256 || in->ld % 4 || out->ld % 4) return 0;
  if (((uintptr_t)in->ptr & 15) || ((uintptr_t)out->ptr & 15)) return 0;
  return 1;
}

extern "C" int lfsr_conv1x1_few(const lfsr_tensor* in, const float* w_packed, const lfsr_tensor* out, const lfsr_conv_desc* d,
                                void* stream) {
  LFSR_REQUIRE(w_packed && lfsr_conv1x1_few_supported(in, out, d), "lfsr_conv1x1_few: unsupported problem");
  const long long pixels = (long long)in->n * in->h * in->w;
  long long blocks = ((pixels + 1) / 2 + 255) / 256;
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  const size_t smem = (size_t)in->c * out->c * sizeof(float);
  cudaStream_t st = (cudaStream_t)stream;
  if (out->c == 16)
    lfsr::conv1x1_few_kernel<16><<<(unsigned)blocks, 256, smem, st>>>(view_of(in), view_of(out), w_packed, d->bias, d->act, d->act_slope, pixels);
  else
    lfsr::conv1x1_few_kernel<8><<<(unsigned)blocks, 256, smem, st>>>(view_of(in), view_of(out), w_packed, d->bias, d->act, d->act_slope, pixels);
  return check_launch("conv1x1_few_kernel");
}
