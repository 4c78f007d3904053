// Reductions, the SA-modulator tail, LayerNorm, band-masked EPI attention and PSNR/SSIM sums.
// All HBM/latency-bound fp32 kernels with warp-shuffle reductions.
#include <stdlib.h>
#include <cuda_fp16.h>
#include "lfsr_common.cuh"

namespace lfsr {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- block mean: one CTA per (n, by, bx); AdaptiveAvgPool2d(1) / (angRes) of
// MyEfficientLFNet.py:159-173,491 when the block tiles the image evenly.
// VEC4 path: 16 lanes x float4 cover up to 64 channels of a pixel (coalesced 256 B), 16 pixel lanes, 4 loads in flight.
template <bool VEC4>
__global__ void __launch_bounds__(256)
block_mean_kernel(TView in, TView out, int bh, int bw) {
  __shared__ float red[16][68];
  // blocks in REVERSE order: the producer of `in` (a persistent conv / a tiled kernel walking the images forward) has just
  // finished with the LAST images, and those are what is still in L2
  int blk = gridDim.x - 1 - blockIdx.x;
  const int nbx = in.w / bw, nby = in.h / bh;
  const int bx = blk % nbx; blk /= nbx;
  const int by = blk % nby;
  const int img = blk / nby;
  const int C = in.c;
  const int npix = bh * bw;
  const float inv = 1.f / (float)npix;
  if (VEC4) {
    const int c4 = threadIdx.x & 15, pl = threadIdx.x >> 4;      // channel chunk, pixel lane
    for (int c0 = 0; c0 < C; c0 += 64) {
      const int c = c0 + c4 * 4;
      float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c < C) {
        const float* base = in.p + in.pix(img, by * bh, bx * bw) + c;
        int p = pl;
        for (; p + 48 < npix; p += 64) {
          float4 v[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int q = p + 16 * u;
            const int y = q / bw, x = q - y * bw;
            v[u] = __ldg(reinterpret_cast<const float4*>(base + ((size_t)y * in.w + x) * in.ld));
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) { s.x += v[u].x; s.y += v[u].y; s.z += v[u].z; s.w += v[u].w; }
        }
        for (; p < npix; p += 16) {
          const int y = p / bw, x = p - y * bw;
          const float4 v = __ldg(reinterpret_cast<const float4*>(base + ((size_t)y * in.w + x) * in.ld));
          s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        }
      }
      red[pl][c4 * 4] = s.x; red[pl][c4 * 4 + 1] = s.y; red[pl][c4 * 4 + 2] = s.z; red[pl][c4 * 4 + 3] = s.w;
      __syncthreads();
      if (threadIdx.x < 64 && c0 + threadIdx.x < C) {
        float t = 0.f;
#pragma unroll
        for (int q = 0; q < 16; ++q) t += red[q][threadIdx.x];
        out.p[out.pix(img, by, bx) + c0 + threadIdx.x] = t * inv;
      }
      __syncthreads();
    }
  } else {
    const int CW = C > 32 ? 64 : (C > 16 ? 32 : 16);
    const int PL = 256 / CW;
    const int cl = threadIdx.x % CW, pl = threadIdx.x / CW;
    float* redf = &red[0][0];
    for (int c0 = 0; c0 < C; c0 += CW) {
      const int c = c0 + cl;
      float s = 0.f;
      if (c < C) {
        for (int p = pl; p < npix; p += PL) {
          const int y = by * bh + p / bw, x = bx * bw + p % bw;
          s += __ldg(in.p + in.pix(img, y, x) + c);
        }
      }
      redf[threadIdx.x] = s;
      __syncthreads();
      if (pl == 0 && c < C) {
        float t = 0.f;
        for (int q = 0; q < PL; ++q) t += redf[q * CW + cl];
        out.p[out.pix(img, by, bx) + c] = t * inv;
      }
      __syncthreads();
    }
  }
}

// ---- SA modulator tail + stage residual (MyEfficientLFNet.py:495-515, 207)
// one thread = one pixel x V consecutive channels (V = 4/2/1 by alignment)
template <int V>
__global__ void __launch_bounds__(256)
sa_modulate_kernel(TView x, const float* __restrict__ dww, const float* __restrict__ bns,
                   const float* __restrict__ bnb, TView amod, float w0, float w1, TView res, TView out, int dil) {
  const int CV = x.c / V;
  const int vh = x.h / amod.h, vw = x.w / amod.w;
  const int img = blockIdx.y;                 // 32-bit index math inside one image
  const int per = x.h * x.w * CV;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < per; t += gridDim.x * blockDim.x) {
    const int c = (t % CV) * V;
    const int r = t / CV;
    const int px = r % x.w;
    const int py = r / x.w;
    float acc[V], xc[V];
#pragma unroll
    for (int e = 0; e < V; ++e) { acc[e] = 0.f; xc[e] = 0.f; }
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int iy = py + (ky - 1) * dil;
      if (iy < 0 || iy >= x.h) continue;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int ix = px + (kx - 1) * dil;
        if (ix < 0 || ix >= x.w) continue;
        const float* src = x.p + x.pix(img, iy, ix) + c;
        const float* wk = dww + (ky * 3 + kx) * x.c + c;
        float v[V];
        if (V == 4) { const float4 q = __ldg(reinterpret_cast<const float4*>(src)); v[0] = q.x; v[1 % V] = q.y; v[2 % V] = q.z; v[3 % V] = q.w; }
        else if (V == 2) { const float2 q = __ldg(reinterpret_cast<const float2*>(src)); v[0] = q.x; v[1 % V] = q.y; }
        else v[0] = __ldg(src);
#pragma unroll
        for (int e = 0; e < V; ++e) acc[e] = fmaf(v[e], __ldg(wk + e), acc[e]);
        if (ky == 1 && kx == 1) {
#pragma unroll
          for (int e = 0; e < V; ++e) xc[e] = v[e];
        }
      }
    }
    const float* am = amod.p + amod.pix(img, py / vh, px / vw) + c;
    float o[V];
#pragma unroll
    for (int e = 0; e < V; ++e) {
      const float s = 1.f / (1.f + expf(-(acc[e] * __ldg(bns + c + e) + __ldg(bnb + c + e))));
      o[e] = xc[e] * (w0 * s + w1 * __ldg(am + e));
    }
    if (res.p) {
      const float* rs = res.p + res.pix(img, py, px) + c;
#pragma unroll
      for (int e = 0; e < V; ++e) o[e] += rs[e];
    }
    float* dst = out.p + out.pix(img, py, px) + c;
    if (V == 4) *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1 % V], o[2 % V], o[3 % V]);
    else if (V == 2) *reinterpret_cast<float2*>(dst) = make_float2(o[0], o[1 % V]);
    else dst[0] = o[0];
  }
}

// Same, for float4-aligned tensors of <= 64 channels (the 60-channel grouped trunk): a CTA owns a 16 x 16 pixel tile,
// thread = (channel quad, pixel column) walking the 16 rows with its 9 tap weights and BN constants in registers; the
// rows a tap needs again 5 and 10 iterations later come out of L1, and there is no index division anywhere.
__global__ void __launch_bounds__(256)
sa_modulate_tile_kernel(TView x, const float* __restrict__ dww, const float* __restrict__ bns,
                        const float* __restrict__ bnb, TView amod, float w0, float w1, TView res, TView out, int dil) {
  const int q = threadIdx.x & 15, lx = threadIdx.x >> 4;
  const int c = q * 4;
  const int px = blockIdx.x * 16 + lx, py0 = blockIdx.y * 16, img = blockIdx.z;
  if (c >= x.c || px >= x.w) return;
  float4 wk[9];
#pragma unroll
  for (int t = 0; t < 9; ++t) wk[t] = __ldg(reinterpret_cast<const float4*>(dww + t * x.c + c));
  const float4 sc = __ldg(reinterpret_cast<const float4*>(bns + c)), sh = __ldg(reinterpret_cast<const float4*>(bnb + c));
  const int vh = x.h / amod.h, vw = x.w / amod.w;
  const int ax = px / vw;
  const int row_f = x.w * x.ld;
  const float* xcol = x.p + x.pix(img, 0, px) + c;
  const bool xl = px - dil >= 0, xr = px + dil < x.w;
  const int ymax = min(py0 + 16, x.h);
  for (int py = py0; py < ymax; ++py) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), xc = acc;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int iy = py + (ky - 1) * dil;
      if (iy < 0 || iy >= x.h) continue;
      const float* rowp = xcol + (size_t)iy * row_f;
      if (xl) { const float4 v = __ldg(reinterpret_cast<const float4*>(rowp - dil * x.ld)); const float4 w = wk[ky * 3];
                acc.x = fmaf(v.x, w.x, acc.x); acc.y = fmaf(v.y, w.y, acc.y); acc.z = fmaf(v.z, w.z, acc.z); acc.w = fmaf(v.w, w.w, acc.w); }
      { const float4 v = __ldg(reinterpret_cast<const float4*>(rowp)); const float4 w = wk[ky * 3 + 1];
        acc.x = fmaf(v.x, w.x, acc.x); acc.y = fmaf(v.y, w.y, acc.y); acc.z = fmaf(v.z, w.z, acc.z); acc.w = fmaf(v.w, w.w, acc.w);
        if (ky == 1) xc = v; }
      if (xr) { const float4 v = __ldg(reinterpret_cast<const float4*>(rowp + dil * x.ld)); const float4 w = wk[ky * 3 + 2];
                acc.x = fmaf(v.x, w.x, acc.x); acc.y = fmaf(v.y, w.y, acc.y); acc.z = fmaf(v.z, w.z, acc.z); acc.w = fmaf(v.w, w.w, acc.w); }
    }
    const float4 am = __ldg(reinterpret_cast<const float4*>(amod.p + amod.pix(img, py / vh, ax) + c));
    float4 o;
    o.x = xc.x * (w0 * __fdividef(1.f, 1.f + __expf(-(acc.x * sc.x + sh.x))) + w1 * am.x);
    o.y = xc.y * (w0 * __fdividef(1.f, 1.f + __expf(-(acc.y * sc.y + sh.y))) + w1 * am.y);
    o.z = xc.z * (w0 * __fdividef(1.f, 1.f + __expf(-(acc.z * sc.z + sh.z))) + w1 * am.z);
    o.w = xc.w * (w0 * __fdividef(1.f, 1.f + __expf(-(acc.w * sc.w + sh.w))) + w1 * am.w);
    if (res.p) {
      const float4 r = *reinterpret_cast<const float4*>(res.p + res.pix(img, py, px) + c);
      o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
    }
    *reinterpret_cast<float4*>(out.p + out.pix(img, py, px) + c) = o;
  }
}

// ---- out = x * scale[n][c] + res : ChannelAttention scaling fused with the block residual
template <int V>
__global__ void __launch_bounds__(256)
scale_add_kernel(TView x, const float* __restrict__ scale, int scale_ld, TView res, TView out) {
  const int CV = x.c / V;
  const int img = blockIdx.y;
  const int per = x.h * x.w * CV;
  const float* sc = scale + (size_t)img * scale_ld;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < per; t += gridDim.x * blockDim.x) {
    const int c = (t % CV) * V;
    const int r = t / CV;
    const int px = r % x.w, py = r / x.w;
    const float* src = x.p + x.pix(img, py, px) + c;
    float v[V];
    if (V == 4) { const float4 q = __ldg(reinterpret_cast<const float4*>(src)); v[0] = q.x; v[1 % V] = q.y; v[2 % V] = q.z; v[3 % V] = q.w; }
    else v[0] = __ldg(src);
#pragma unroll
    for (int e = 0; e < V; ++e) v[e] *= __ldg(sc + c + e);
    if (res.p) {
      const float* rs = res.p + res.pix(img, py, px) + c;
#pragma unroll
      for (int e = 0; e < V; ++e) v[e] += rs[e];
    }
    float* dst = out.p + out.pix(img, py, px) + c;
    if (V == 4) *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1 % V], v[2 % V], v[3 % V]);
    else dst[0] = v[0];
  }
}

// the same with an fp16 result (the tensor only feeds a tensor-core layer): 8 channels per thread, one 16-byte store
__global__ void __launch_bounds__(256)
scale_add16_kernel(TView x, const float* __restrict__ scale, int scale_ld, TView res, __half* __restrict__ out, int out_ld) {
  const int CV = x.c / 8;
  const int img = blockIdx.y;
  const int per = x.h * x.w * CV;
  const float* sc = scale + (size_t)img * scale_ld;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < per; t += gridDim.x * blockDim.x) {
    const int c = (t % CV) * 8;
    const int r = t / CV;
    const int px = r % x.w, py = r / x.w;
    const float* src = x.p + x.pix(img, py, px) + c;
    const float4 a0 = __ldg(reinterpret_cast<const float4*>(src)), a1 = __ldg(reinterpret_cast<const float4*>(src) + 1);
    float v[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] *= __ldg(sc + c + e);
    if (res.p) {
      const float4* rs = reinterpret_cast<const float4*>(res.p + res.pix(img, py, px) + c);
      const float4 r0 = __ldg(rs), r1 = __ldg(rs + 1);
      v[0] += r0.x; v[1] += r0.y; v[2] += r0.z; v[3] += r0.w; v[4] += r1.x; v[5] += r1.y; v[6] += r1.z; v[7] += r1.w;
    }
    const __half2 h0 = __floats2half2_rn(v[0], v[1]), h1 = __floats2half2_rn(v[2], v[3]), h2 = __floats2half2_rn(v[4], v[5]),
                  h3 = __floats2half2_rn(v[6], v[7]);
    uint4 o;
    o.x = *reinterpret_cast<const uint32_t*>(&h0); o.y = *reinterpret_cast<const uint32_t*>(&h1);
    o.z = *reinterpret_cast<const uint32_t*>(&h2); o.w = *reinterpret_cast<const uint32_t*>(&h3);
    *reinterpret_cast<uint4*>(out + ((size_t)((size_t)img * x.h + py) * x.w + px) * (size_t)out_ld + c) = o;
  }
}

// ---- second half of a KxK conv to one channel: sum of the per-tap responses at the shifted positions
__global__ void __launch_bounds__(256)
tap_gather_kernel(TView taps, TView res, TView out, int kh, int kw, const float* __restrict__ bias) {
  const int img = blockIdx.z;
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= out.w || y >= out.h) return;
  float acc = bias ? __ldg(bias) : 0.f;
  for (int ky = 0; ky < kh; ++ky) {
    const int iy = y + ky - kh / 2;
    if (iy < 0 || iy >= taps.h) continue;
    for (int kx = 0; kx < kw; ++kx) {
      const int ix = x + kx - kw / 2;
      if (ix < 0 || ix >= taps.w) continue;
      acc += __ldg(taps.p + taps.pix(img, iy, ix) + ky * kw + kx);
    }
  }
  if (res.p) acc += res.p[res.pix(img, y, x)];
  out.p[out.pix(img, y, x)] = acc;
}

// 3x3 taps stored as 12-float records (what the tail-projection epilogue writes): the 34 x 10 records a 32 x 8 tile
// needs are staged with coalesced 16-byte cp.async (zero fill outside the image = the conv's padding) and every output
// is then nine shared-memory reads - the records are read from HBM once instead of through nine strided 4-byte loads.
__global__ void __launch_bounds__(256)
tap_gather3x3_kernel(TView taps, TView res, TView out, const float* __restrict__ bias) {
  __shared__ __align__(16) float rec[10 * 34 * 12];
  const int img = blockIdx.z;
  const int tx0 = blockIdx.x * 32, ty0 = blockIdx.y * 8;
  for (int i = threadIdx.x; i < 10 * 34 * 3; i += 256) {
    const int q = i % 3, pix = i / 3;
    const int ly = pix / 34, lx = pix - ly * 34;
    const int iy = ty0 - 1 + ly, ix = tx0 - 1 + lx;
    const bool ok = iy >= 0 && iy < taps.h && ix >= 0 && ix < taps.w;
    const float* src = ok ? taps.p + taps.pix(img, iy, ix) + q * 4 : taps.p;
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(rec + pix * 12 + q * 4);
    const int nbytes = ok ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
  }
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;
  const int x = tx0 + lx, y = ty0 + ly;
  if (x >= out.w || y >= out.h) return;
  float acc = bias ? __ldg(bias) : 0.f;
#pragma unroll
  for (int ky = 0; ky < 3; ++ky)
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) acc += rec[((ly + ky) * 34 + lx + kx) * 12 + ky * 3 + kx];
  if (res.p) acc += res.p[res.pix(img, y, x)];
  out.p[out.pix(img, y, x)] = acc;
}

// ---- LayerNorm over channels: one warp per token (EPIT.py:77,84)
__global__ void __launch_bounds__(256)
layernorm_kernel(TView in, TView out, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                 long long tokens) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const int C = in.c;
  for (long long t = warp; t < tokens; t += nwarps) {
    const float* src = in.p + (size_t)t * in.ld;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s += __ldg(src + c);
    const float mean = warp_sum(s) / (float)C;
    float q = 0.f;
    for (int c = lane; c < C; c += 32) { const float d = __ldg(src + c) - mean; q = fmaf(d, d, q); }
    const float rstd = rsqrtf(warp_sum(q) / (float)C + eps);
    float* dst = out.p + (size_t)t * out.ld;
    for (int c = lane; c < C; c += 32) dst[c] = (__ldg(src + c) - mean) * rstd * __ldg(gamma + c) + __ldg(beta + c);
  }
}

// ---- band-masked EPI attention: one CTA per (sequence, head), one thread per query.
// Keys allowed for query (a,s): all a' in [0,A), |s'-s| <= half_window (EPIT.py:93-108 with
// mask_field=[2A,11]); q is pre-scaled by head_dim^-0.5 as nn.MultiheadAttention does.
constexpr int ATT_D = 16;       // head_dim (E=128, 8 heads; EPIT.py:78)
constexpr int ATT_LD = 20;      // padded smem row: conflict-free float4 reads
__global__ void __launch_bounds__(192)
epi_attention_kernel(const float* __restrict__ qk, const float* __restrict__ v, float* __restrict__ out,
                     lfsr_epi_attn_desc d) {
  extern __shared__ float sm[];
  const int L = d.A * d.S;
  float* Ks = sm;                 // [L][ATT_LD]
  float* Vs = sm + L * ATT_LD;    // [L][ATT_LD]
  const int E = d.heads * ATT_D;
  int seq = blockIdx.x;
  const int head = blockIdx.y;
  const int q_ = seq % d.nq; seq /= d.nq;
  const int p_ = seq % d.np;
  const int b_ = seq / d.np;
  const long long base = b_ * d.stride_b + p_ * d.stride_p + q_ * d.stride_q;
  const int tid = threadIdx.x;
  // stage K and V head slices (float4 granules)
  for (int i = tid; i < L * 4; i += blockDim.x) {
    const int tok = i >> 2, part = i & 3;
    const int a = tok / d.S, s = tok - a * d.S;
    const long long g = base + a * d.stride_a + s * d.stride_s;
    const float4 kv = __ldg(reinterpret_cast<const float4*>(qk + (size_t)g * 2 * E + E + head * ATT_D) + part);
    const float4 vv = __ldg(reinterpret_cast<const float4*>(v + (size_t)g * E + head * ATT_D) + part);
    *reinterpret_cast<float4*>(Ks + tok * ATT_LD + part * 4) = kv;
    *reinterpret_cast<float4*>(Vs + tok * ATT_LD + part * 4) = vv;
  }
  __syncthreads();
  if (tid >= L) return;
  const int qa = tid / d.S, qs = tid - qa * d.S;
  const long long gq = base + qa * d.stride_a + qs * d.stride_s;
  float q[ATT_D];
  const float scale = rsqrtf((float)ATT_D);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(qk + (size_t)gq * 2 * E + head * ATT_D) + j);
    q[4 * j] = t.x * scale; q[4 * j + 1] = t.y * scale; q[4 * j + 2] = t.z * scale; q[4 * j + 3] = t.w * scale;
  }
  const int s_lo = max(qs - d.half_window, 0), s_hi = min(qs + d.half_window, d.S - 1);
  float m = -INFINITY, l = 0.f;
  float acc[ATT_D];
#pragma unroll
  for (int j = 0; j < ATT_D; ++j) acc[j] = 0.f;
  for (int a = 0; a < d.A; ++a) {
    for (int s = s_lo; s <= s_hi; ++s) {
      const float* kr = Ks + (a * d.S + s) * ATT_LD;
      float sc = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 t = *reinterpret_cast<const float4*>(kr + 4 * j);
        sc = fmaf(q[4 * j], t.x, sc); sc = fmaf(q[4 * j + 1], t.y, sc);
        sc = fmaf(q[4 * j + 2], t.z, sc); sc = fmaf(q[4 * j + 3], t.w, sc);
      }
      const float mn = fmaxf(m, sc);
      const float corr = __expf(m - mn);   // exp(-inf) = 0 on the first key
      const float pexp = __expf(sc - mn);
      l = l * corr + pexp;
      const float* vr = Vs + (a * d.S + s) * ATT_LD;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 t = *reinterpret_cast<const float4*>(vr + 4 * j);
        acc[4 * j] = fmaf(pexp, t.x, acc[4 * j] * corr);
        acc[4 * j + 1] = fmaf(pexp, t.y, acc[4 * j + 1] * corr);
        acc[4 * j + 2] = fmaf(pexp, t.z, acc[4 * j + 2] * corr);
        acc[4 * j + 3] = fmaf(pexp, t.w, acc[4 * j + 3] * corr);
      }
      m = mn;
    }
  }
  const float inv = 1.f / l;
  float* dst = out + (size_t)gq * E + head * ATT_D;
#pragma unroll
  for (int j = 0; j < 4; ++j)
    reinterpret_cast<float4*>(dst)[j] =
        make_float4(acc[4 * j] * inv, acc[4 * j + 1] * inv, acc[4 * j + 2] * inv, acc[4 * j + 3] * inv);
}

// Same attention for A == 5 views: CTA = one sequence x 4 heads, warp = head, lane = spatial position s, and the lane
// owns ALL FIVE queries (a = 0..4, s): they share one key set (every a', |s' - s| <= half_window), so each K / V row is
// read from shared memory once for five queries instead of once per query (the per-query kernel is bound by exactly
// those reads), dot products and PV updates are packed FFMA2, and the softmax is two-pass (maxima, then exp + PV).
constexpr int ATT_NQ = 5, ATT_HPC = 4;      // queries per lane, heads per CTA
__global__ void __launch_bounds__(32 * ATT_HPC)
epi_attention5_kernel(const float* __restrict__ qk, const float* __restrict__ v, float* __restrict__ out,
                      lfsr_epi_attn_desc d) {
  extern __shared__ float sm[];
  const int L = ATT_NQ * d.S;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* Ks = sm + warp * 2 * L * ATT_LD;      // this head's [L][ATT_LD]
  float* Vs = Ks + L * ATT_LD;
  const int E = d.heads * ATT_D;
  int seq = blockIdx.x;
  const int head = blockIdx.y * ATT_HPC + warp;
  const int q_ = seq % d.nq; seq /= d.nq;
  const int p_ = seq % d.np;
  const int b_ = seq / d.np;
  const long long base = b_ * d.stride_b + p_ * d.stride_p + q_ * d.stride_q;
  if (head >= d.heads) return;
  for (int i = lane; i < L * 4; i += 32) {
    const int tok = i >> 2, part = i & 3;
    const int a = tok / d.S, s = tok - a * d.S;
    const long long g = base + a * d.stride_a + s * d.stride_s;
    *reinterpret_cast<float4*>(Ks + tok * ATT_LD + part * 4) =
        __ldg(reinterpret_cast<const float4*>(qk + (size_t)g * 2 * E + E + head * ATT_D) + part);
    *reinterpret_cast<float4*>(Vs + tok * ATT_LD + part * 4) =
        __ldg(reinterpret_cast<const float4*>(v + (size_t)g * E + head * ATT_D) + part);
  }
  __syncwarp();
  const int qs = lane;
  if (qs >= d.S) return;
  const float scale = rsqrtf((float)ATT_D);
  f32x2 q2[ATT_NQ][ATT_D / 2], acc[ATT_NQ][ATT_D / 2];
  float m[ATT_NQ], l[ATT_NQ];
#pragma unroll
  for (int i = 0; i < ATT_NQ; ++i) {
    const long long gq = base + i * d.stride_a + qs * d.stride_s;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(qk + (size_t)gq * 2 * E + head * ATT_D) + j);
      q2[i][2 * j] = pack2(t.x * scale, t.y * scale);
      q2[i][2 * j + 1] = pack2(t.z * scale, t.w * scale);
    }
#pragma unroll
    for (int j = 0; j < ATT_D / 2; ++j) acc[i][j] = pack2(0.f, 0.f);
    m[i] = -INFINITY; l[i] = 0.f;
  }
  const int s_lo = max(qs - d.half_window, 0), s_hi = min(qs + d.half_window, d.S - 1);
  // pass 1: row maxima (scores only). pass 2: scores again, exp against the final maximum, PV accumulation. Recomputing
  // the 16-wide dot products is cheaper than an online softmax here: no divergent "new maximum" branch (ncu: 39 % branch
  // efficiency with it) and no accumulator rescaling.
  for (int a = 0; a < ATT_NQ; ++a) {
    for (int s = s_lo; s <= s_hi; ++s) {
      const float* kr = Ks + (a * d.S + s) * ATT_LD;
      f32x2 k2[ATT_D / 2];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 t = *reinterpret_cast<const float4*>(kr + 4 * j);
        k2[2 * j] = pack2(t.x, t.y); k2[2 * j + 1] = pack2(t.z, t.w);
      }
#pragma unroll
      for (int i = 0; i < ATT_NQ; ++i) {
        f32x2 da = fma2(q2[i][0], k2[0], pack2(0.f, 0.f)), db = fma2(q2[i][1], k2[1], pack2(0.f, 0.f));
#pragma unroll
        for (int j = 2; j < ATT_D / 2; j += 2) { da = fma2(q2[i][j], k2[j], da); db = fma2(q2[i][j + 1], k2[j + 1], db); }
        float s0, s1, s2, s3;
        unpack2(da, s0, s1); unpack2(db, s2, s3);
        m[i] = fmaxf(m[i], (s0 + s1) + (s2 + s3));
      }
    }
  }
  for (int a = 0; a < ATT_NQ; ++a) {
    for (int s = s_lo; s <= s_hi; ++s) {
      const float* kr = Ks + (a * d.S + s) * ATT_LD;
      const float* vr = Vs + (a * d.S + s) * ATT_LD;
      f32x2 k2[ATT_D / 2], v2[ATT_D / 2];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 t = *reinterpret_cast<const float4*>(kr + 4 * j);
        k2[2 * j] = pack2(t.x, t.y); k2[2 * j + 1] = pack2(t.z, t.w);
        const float4 u = *reinterpret_cast<const float4*>(vr + 4 * j);
        v2[2 * j] = pack2(u.x, u.y); v2[2 * j + 1] = pack2(u.z, u.w);
      }
#pragma unroll
      for (int i = 0; i < ATT_NQ; ++i) {
        f32x2 da = fma2(q2[i][0], k2[0], pack2(0.f, 0.f)), db = fma2(q2[i][1], k2[1], pack2(0.f, 0.f));
#pragma unroll
        for (int j = 2; j < ATT_D / 2; j += 2) { da = fma2(q2[i][j], k2[j], da); db = fma2(q2[i][j + 1], k2[j + 1], db); }
        float s0, s1, s2, s3;
        unpack2(da, s0, s1); unpack2(db, s2, s3);
        const float pexp = __expf(((s0 + s1) + (s2 + s3)) - m[i]);
        l[i] += pexp;
        const f32x2 p2 = pack2(pexp, pexp);
#pragma unroll
        for (int j = 0; j < ATT_D / 2; ++j) acc[i][j] = fma2(p2, v2[j], acc[i][j]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < ATT_NQ; ++i) {
    const long long gq = base + i * d.stride_a + qs * d.stride_s;
    const float inv = 1.f / l[i];
    float* dst = out + (size_t)gq * E + head * ATT_D;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float a0, a1, a2, a3;
      unpack2(acc[i][2 * j], a0, a1);
      unpack2(acc[i][2 * j + 1], a2, a3);
      reinterpret_cast<float4*>(dst)[j] = make_float4(a0 * inv, a1 * inv, a2 * inv, a3 * inv);
    }
  }
}

// ---- PSNR / SSIM partial sums (utils/utils.py:91-134 -> skimage.metrics):
// SSIM: 11x11 Gaussian (sigma 1.5, truncate 3.5), sample covariance (121/120), K1=.01 K2=.03,
// data_range 1, mean over the interior cropped by 5 px -> the filter never touches the border,
// so scipy's 'reflect' mode is never exercised.
constexpr int MT_W = 32, MT_H = 16, MT_R = 5;
struct Gauss11 { float g[11]; };

__global__ void __launch_bounds__(256)
metric_kernel(const float* __restrict__ la, const float* __restrict__ ou, int Av, int h, int w, double* acc,
              int tiles_x, int tiles_y, const Gauss11 gw) {
  __shared__ float sa[MT_H + 2 * MT_R][MT_W + 2 * MT_R];
  __shared__ float sb[MT_H + 2 * MT_R][MT_W + 2 * MT_R];
  __shared__ float hz[5][MT_H + 2 * MT_R][MT_W];
  __shared__ double red[2][8];
  int blk = blockIdx.x;
  const int tx = blk % tiles_x; blk /= tiles_x;
  const int ty = blk % tiles_y;
  const int view = blk / tiles_y;
  const int va = view / Av, vb = view % Av;
  const size_t rs = (size_t)Av * w;
  const float* pa = la + (size_t)va * h * rs + (size_t)vb * w;
  const float* pb = ou + (size_t)va * h * rs + (size_t)vb * w;
  // tile origin in view coordinates; tiles cover the full view, SSIM is only taken on the interior
  const int x0 = tx * MT_W, y0 = ty * MT_H;
  const int tid = threadIdx.x;
  double se = 0.0, ss = 0.0;
  for (int i = tid; i < (MT_H + 2 * MT_R) * (MT_W + 2 * MT_R); i += 256) {
    const int ly = i / (MT_W + 2 * MT_R), lx = i % (MT_W + 2 * MT_R);
    const int y = y0 + ly - MT_R, x = x0 + lx - MT_R;
    float av = 0.f, bv = 0.f;
    if (y >= 0 && y < h && x >= 0 && x < w) { av = __ldg(pa + (size_t)y * rs + x); bv = __ldg(pb + (size_t)y * rs + x); }
    sa[ly][lx] = av; sb[ly][lx] = bv;
    // squared error over the tile's own pixels
    if (ly >= MT_R && ly < MT_R + MT_H && lx >= MT_R && lx < MT_R + MT_W && y < h && x < w) {
      const double dd = (double)av - (double)bv;
      se += dd * dd;
    }
  }
  __syncthreads();
  for (int i = tid; i < (MT_H + 2 * MT_R) * MT_W; i += 256) {
    const int ly = i / MT_W, lx = i % MT_W;
    float f0 = 0.f, f1 = 0.f, f2 = 0.f, f3 = 0.f, f4 = 0.f;
#pragma unroll
    for (int k = 0; k < 11; ++k) {
      const float g = gw.g[k];
      const float av = sa[ly][lx + k], bv = sb[ly][lx + k];
      f0 = fmaf(g, av, f0); f1 = fmaf(g, bv, f1);
      f2 = fmaf(g, av * av, f2); f3 = fmaf(g, bv * bv, f3); f4 = fmaf(g, av * bv, f4);
    }
    hz[0][ly][lx] = f0; hz[1][ly][lx] = f1; hz[2][ly][lx] = f2; hz[3][ly][lx] = f3; hz[4][ly][lx] = f4;
  }
  __syncthreads();
  for (int i = tid; i < MT_H * MT_W; i += 256) {
    const int ly = i / MT_W, lx = i % MT_W;
    const int y = y0 + ly, x = x0 + lx;
    if (y < MT_R || y >= h - MT_R || x < MT_R || x >= w - MT_R) continue;
    float ux = 0.f, uy = 0.f, uxx = 0.f, uyy = 0.f, uxy = 0.f;
#pragma unroll
    for (int k = 0; k < 11; ++k) {
      const float g = gw.g[k];
      ux = fmaf(g, hz[0][ly + k][lx], ux); uy = fmaf(g, hz[1][ly + k][lx], uy);
      uxx = fmaf(g, hz[2][ly + k][lx], uxx); uyy = fmaf(g, hz[3][ly + k][lx], uyy);
      uxy = fmaf(g, hz[4][ly + k][lx], uxy);
    }
    const float cov_norm = 121.f / 120.f;
    const float vx = cov_norm * (uxx - ux * ux), vy = cov_norm * (uyy - uy * uy), vxy = cov_norm * (uxy - ux * uy);
    const float C1 = 0.0001f, C2 = 0.0009f;
    const float A1 = 2.f * ux * uy + C1, A2 = 2.f * vxy + C2;
    const float B1 = ux * ux + uy * uy + C1, B2 = vx + vy + C2;
    ss += (double)((A1 * A2) / (B1 * B2));
  }
  se = warp_sum_d(se); ss = warp_sum_d(ss);
  if ((tid & 31) == 0) { red[0][tid >> 5] = se; red[1][tid >> 5] = ss; }
  __syncthreads();
  if (tid == 0) {
    double e = 0.0, s = 0.0;
    for (int i = 0; i < 8; ++i) { e += red[0][i]; s += red[1][i]; }
    atomicAdd(acc + 2 * view, e);
    atomicAdd(acc + 2 * view + 1, s);
  }
}

}  // namespace lfsr

using namespace lfsr;

static long long capped_blocks(long long total) {
  long long blocks = (total + 255) / 256;
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  return blocks < 1 ? 1 : blocks;
}

extern "C" int lfsr_block_mean(const lfsr_tensor* in, const lfsr_tensor* out, int block_h, int block_w, void* stream) {
  LFSR_REQUIRE(tensor_ok(in) && tensor_ok(out), "lfsr_block_mean: null/invalid tensor");
  LFSR_REQUIRE(block_h > 0 && block_w > 0 && in->h % block_h == 0 && in->w % block_w == 0,
               "lfsr_block_mean: block %dx%d does not tile %dx%d", block_h, block_w, in->h, in->w);
  LFSR_REQUIRE(out->n == in->n && out->h == in->h / block_h && out->w == in->w / block_w && out->c == in->c,
               "lfsr_block_mean: out shape mismatch");
  const int grid = in->n * out->h * out->w;
  const bool vec4 = (in->c % 4 == 0) && (in->ld % 4 == 0) && (((uintptr_t)in->ptr & 15) == 0);
  if (vec4) block_mean_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(view_of(in), view_of(out), block_h, block_w);
  else block_mean_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(view_of(in), view_of(out), block_h, block_w);
  return check_launch("block_mean_kernel");
}

// ---- tiny per-image MLPs of the Track-2 stages ------------------------------------------------------------------
// The channel gates (MyEfficientLFNet.py:159-173: mean over the views -> 1x1 conv + bias -> sigmoid) and the angular part of
// the SA modulator (:505-511: per-view means -> 1x1 -> ReLU -> 1x1 -> sigmoid) are chains of 1x1 convolutions on 1..25
// positions per image. As separate launches of the general conv kernels they cost 17-35 us each - launch- and
// latency-bound, ~0.5 ms per forward; here each chain is one launch with one CTA per image.
//   x[p][c]  = in[img][p][c]                        (pool: x[0][c] = mean over the h*w positions, one position left)
//   h[p][j]  = act1(b1[j] + sum_c x[p][c] w1[c][j])                     w1: [cin][c1]  (lfsr_conv2d_f32 packing of a 1x1)
//   out[p][o] = act2(b2[o] + sum_j h[p][j] w2[j][o])   (w2 == null: out = h)
namespace lfsr {
__global__ void __launch_bounds__(256)
pooled_mlp_kernel(TView in, TView out, int pool, const float* __restrict__ w1, const float* __restrict__ b1, int c1, int act1,
                  const float* __restrict__ w2, const float* __restrict__ b2, int c2, int act2) {
  extern __shared__ float pm_s[];
  const int img = blockIdx.x, tid = threadIdx.x;
  const int P = in.h * in.w, C = in.c;
  const int Pq = pool ? 1 : P;
  float* x = pm_s;                 // [Pq][C]
  float* h = pm_s + Pq * C;        // [Pq][c1]
  float* ws1 = h + Pq * c1;        // [C][c1] and [c1][c2]: staged with coalesced loads (a dependent chain of ~60 global
  float* ws2 = ws1 + C * c1;       // loads per output was most of this kernel's 13 us)
  for (int i = tid; i < C * c1; i += 256) ws1[i] = __ldg(w1 + i);
  if (w2) for (int i = tid; i < c1 * c2; i += 256) ws2[i] = __ldg(w2 + i);
  const float* src = in.p + (size_t)img * P * in.ld;
  float* xs = ws2 + (w2 ? c1 * c2 : 0);        // [P][C] raw positions (pool only)
  if (pool) {
    for (int i = tid; i < P * C; i += 256) { const int q = i / C, c = i - q * C; xs[i] = src[q * in.ld + c]; }
    __syncthreads();
    const float inv = 1.f / (float)P;
    for (int c = tid; c < C; c += 256) {
      float acc = 0.f;
      for (int q = 0; q < P; ++q) acc += xs[q * C + c];
      x[c] = acc * inv;
    }
  } else {
    for (int i = tid; i < P * C; i += 256) { const int q = i / C, c = i - q * C; x[i] = src[q * in.ld + c]; }
  }
  __syncthreads();
  float* dst = out.p + (size_t)img * Pq * out.ld;
  for (int i = tid; i < Pq * c1; i += 256) {
    const int q = i / c1, j = i - q * c1;
    float acc = b1 ? __ldg(b1 + j) : 0.f;
#pragma unroll 4
    for (int c = 0; c < C; ++c) acc = fmaf(x[q * C + c], ws1[c * c1 + j], acc);
    acc = apply_act(acc, act1, 0.f);
    if (w2) h[i] = acc; else dst[q * out.ld + j] = acc;
  }
  if (!w2) return;
  __syncthreads();
  for (int i = tid; i < Pq * c2; i += 256) {
    const int q = i / c2, o = i - q * c2;
    float acc = b2 ? __ldg(b2 + o) : 0.f;
#pragma unroll 4
    for (int j = 0; j < c1; ++j) acc = fmaf(h[q * c1 + j], ws2[j * c2 + o], acc);
    dst[q * out.ld + o] = apply_act(acc, act2, 0.f);
  }
}
}  // namespace lfsr

extern "C" int lfsr_pooled_mlp(const lfsr_tensor* in, int pool, const float* w1, const float* b1, int c1, int act1, const float* w2,
                               const float* b2, int c2, int act2, const lfsr_tensor* out, void* stream) {
  LFSR_REQUIRE(tensor_ok(in) && tensor_ok(out) && w1 && c1 > 0, "lfsr_pooled_mlp: null/invalid argument");
  LFSR_REQUIRE(!w2 || c2 > 0, "lfsr_pooled_mlp: second layer without a width");
  const int P = in->h * in->w, Pq = pool ? 1 : P, cout = w2 ? c2 : c1;
  LFSR_REQUIRE(out->n == in->n && out->h * out->w == Pq && out->c == cout, "lfsr_pooled_mlp: out shape mismatch");
  const size_t smem = ((size_t)Pq * (in->c + c1) + (size_t)in->c * c1 + (w2 ? (size_t)c1 * c2 : 0) + (pool ? (size_t)P * in->c : 0)) *
                      sizeof(float);
  LFSR_REQUIRE(smem <= 48 * 1024 && in->n <= 0x7fffffff, "lfsr_pooled_mlp: positions x channels too large for one CTA");
  pooled_mlp_kernel<<<in->n, 256, smem, (cudaStream_t)stream>>>(view_of(in), view_of(out), pool ? 1 : 0, w1, b1, c1, act1, w2, b2,
                                                               c2, act2);
  return check_launch("pooled_mlp_kernel");
}

int lfsr_sa_modulate_tiled(const lfsr_tensor* x, const float* dw_w, const float* bn_scale, const float* bn_shift,
                           const lfsr_tensor* amod, float w0, float w1, const lfsr_tensor* res, const lfsr_tensor* out, int dil,
                           int* handled, void* stream, const lfsr_tensor* out16 = nullptr, int skip_lo = 0, int skip_hi = 0);     // lfsr_dw.cu

extern "C" int lfsr_sa_modulate(const lfsr_tensor* x, const float* dw_w, const float* bn_scale, const float* bn_shift,
                                const lfsr_tensor* amod, float w0, float w1, const lfsr_tensor* res,
                                const lfsr_tensor* out, int dil, void* stream) {
  LFSR_REQUIRE(tensor_ok(x) && tensor_ok(out) && tensor_ok(amod) && dw_w && bn_scale && bn_shift,
               "lfsr_sa_modulate: null/invalid tensor");
  LFSR_REQUIRE(out->n == x->n && out->h == x->h && out->w == x->w && out->c == x->c, "lfsr_sa_modulate: out shape");
  LFSR_REQUIRE(amod->n == x->n && amod->c == x->c && x->h % amod->h == 0 && x->w % amod->w == 0,
               "lfsr_sa_modulate: amod shape");
  TView r = null_view();
  if (res && res->ptr) {
    LFSR_REQUIRE(res->n == x->n && res->h == x->h && res->w == x->w && res->c == x->c, "lfsr_sa_modulate: res shape");
    r = view_of(res);
  }
  auto al = [](const lfsr_tensor* t, int v) { return t->ld % v == 0 && (((uintptr_t)t->ptr) & (uintptr_t)(4 * v - 1)) == 0; };
  int V = 1;
  for (int v = 2; v <= 4; v *= 2) {
    if (x->c % v == 0 && al(x, v) && al(out, v) && al(amod, v) && (!r.p || al(res, v))) V = v;
    else break;
  }
  LFSR_REQUIRE(x->n <= 65535, "lfsr_sa_modulate: batch too large");
  if (V == 4) {        // shared-memory tiled depthwise kernel with the modulator tail in its epilogue
    int handled = 0;
    int rc = lfsr_sa_modulate_tiled(x, dw_w, bn_scale, bn_shift, amod, w0, w1, res, out, dil, &handled, stream);
    if (rc != LFSR_OK || handled) return rc;
  }
  if (V == 4 && x->c <= 64 && (((uintptr_t)dw_w | (uintptr_t)bn_scale | (uintptr_t)bn_shift) & 15) == 0 &&
      (long long)x->h * x->w * x->ld < 0x7fffffffLL) {
    dim3 grid(ceil_div(x->w, 16), ceil_div(x->h, 16), x->n);
    sa_modulate_tile_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(view_of(x), dw_w, bn_scale, bn_shift, view_of(amod), w0, w1, r,
                                                                    view_of(out), dil);
    return check_launch("sa_modulate_tile_kernel");
  }
  const int per = x->h * x->w * (x->c / V);
  dim3 blocks(ceil_div(per, 256), x->n);
  cudaStream_t st = (cudaStream_t)stream;
  if (V == 4) sa_modulate_kernel<4><<<blocks, 256, 0, st>>>(view_of(x), dw_w, bn_scale, bn_shift, view_of(amod), w0, w1, r, view_of(out), dil);
  else if (V == 2) sa_modulate_kernel<2><<<blocks, 256, 0, st>>>(view_of(x), dw_w, bn_scale, bn_shift, view_of(amod), w0, w1, r, view_of(out), dil);
  else sa_modulate_kernel<1><<<blocks, 256, 0, st>>>(view_of(x), dw_w, bn_scale, bn_shift, view_of(amod), w0, w1, r, view_of(out), dil);
  return check_launch("sa_modulate_kernel");
}

extern "C" int lfsr_sa_modulate16w(const lfsr_tensor* x, const float* dw_w, const float* bn_scale, const float* bn_shift,
                                   const lfsr_tensor* amod, float w0, float w1, const lfsr_tensor* res, const lfsr_tensor* out,
                                   const lfsr_tensor* out16, int skip_lo, int skip_hi, int dil, void* stream);
extern "C" int lfsr_sa_modulate16(const lfsr_tensor* x, const float* dw_w, const float* bn_scale, const float* bn_shift,
                                  const lfsr_tensor* amod, float w0, float w1, const lfsr_tensor* res,
                                  const lfsr_tensor* out, const lfsr_tensor* out16, int dil, void* stream) {
  return lfsr_sa_modulate16w(x, dw_w, bn_scale, bn_shift, amod, w0, w1, res, out, out16, 0, 0, dil, stream);
}

extern "C" int lfsr_sa_modulate16w(const lfsr_tensor* x, const float* dw_w, const float* bn_scale, const float* bn_shift,
                                   const lfsr_tensor* amod, float w0, float w1, const lfsr_tensor* res, const lfsr_tensor* out,
                                   const lfsr_tensor* out16, int skip_lo, int skip_hi, int dil, void* stream) {
  LFSR_REQUIRE(skip_lo >= 0 && skip_hi >= skip_lo && skip_lo % 4 == 0 && skip_hi % 4 == 0, "lfsr_sa_modulate16w: the skipped channel window must be whole quads");
  LFSR_REQUIRE(tensor_ok(x) && tensor_ok(out) && tensor_ok(amod) && dw_w && bn_scale && bn_shift && out16 && out16->ptr,
               "lfsr_sa_modulate16: null/invalid tensor");
  LFSR_REQUIRE(out->n == x->n && out->h == x->h && out->w == x->w && out->c == x->c, "lfsr_sa_modulate16: out shape");
  LFSR_REQUIRE(amod->n == x->n && amod->c == x->c && x->h % amod->h == 0 && x->w % amod->w == 0, "lfsr_sa_modulate16: amod shape");
  LFSR_REQUIRE(out16->n == x->n && out16->h == x->h && out16->w == x->w && out16->c > 0 && out16->c <= x->c && out16->c % 4 == 0 &&
                   out16->ld % 4 == 0 && (((uintptr_t)out16->ptr) & 7) == 0,
               "lfsr_sa_modulate16: the fp16 copy holds the first c16 channels (a multiple of 4, 8-byte aligned pixels)");
  if (res && res->ptr)
    LFSR_REQUIRE(res->n == x->n && res->h == x->h && res->w == x->w && res->c == x->c, "lfsr_sa_modulate16: res shape");
  LFSR_REQUIRE(x->n <= 65535, "lfsr_sa_modulate16: batch too large");
  int handled = 0;
  int rc = lfsr_sa_modulate_tiled(x, dw_w, bn_scale, bn_shift, amod, w0, w1, res, out, dil, &handled, stream, out16, skip_lo, skip_hi);
  if (rc != LFSR_OK) return rc;
  LFSR_REQUIRE(handled, "lfsr_sa_modulate16: these tensors do not qualify for the tiled kernel (16-byte aligned 4-channel groups)");
  return LFSR_OK;
}

extern "C" int lfsr_scale_add(const lfsr_tensor* x, const lfsr_tensor* scale, const lfsr_tensor* res, const lfsr_tensor* out,
                              void* stream) {
  LFSR_REQUIRE(tensor_ok(x) && tensor_ok(scale) && tensor_ok(out), "lfsr_scale_add: null/invalid tensor");
  LFSR_REQUIRE(out->n == x->n && out->h == x->h && out->w == x->w && out->c == x->c, "lfsr_scale_add: out shape");
  LFSR_REQUIRE(scale->n == x->n && scale->h == 1 && scale->w == 1 && scale->c == x->c, "lfsr_scale_add: scale must be [n,1,1,c]");
  LFSR_REQUIRE(x->n <= 65535, "lfsr_scale_add: batch too large");
  TView r = null_view();
  if (res && res->ptr) {
    LFSR_REQUIRE(res->n == x->n && res->h == x->h && res->w == x->w && res->c == x->c, "lfsr_scale_add: res shape");
    r = view_of(res);
  }
  auto al = [](const lfsr_tensor* t) { return t->ld % 4 == 0 && (((uintptr_t)t->ptr) & 15) == 0; };
  const bool v4 = x->c % 4 == 0 && al(x) && al(out) && (!r.p || al(res));
  const int per = x->h * x->w * (x->c / (v4 ? 4 : 1));
  dim3 blocks(ceil_div(per, 256), x->n);
  if (v4) scale_add_kernel<4><<<blocks, 256, 0, (cudaStream_t)stream>>>(view_of(x), (const float*)scale->ptr, scale->ld, r, view_of(out));
  else scale_add_kernel<1><<<blocks, 256, 0, (cudaStream_t)stream>>>(view_of(x), (const float*)scale->ptr, scale->ld, r, view_of(out));
  return check_launch("scale_add_kernel");
}

extern "C" int lfsr_scale_add16(const lfsr_tensor* x, const lfsr_tensor* scale, const lfsr_tensor* res, const lfsr_tensor* out16,
                                void* stream) {
  LFSR_REQUIRE(tensor_ok(x) && tensor_ok(scale) && tensor_ok(out16), "lfsr_scale_add16: null/invalid tensor");
  LFSR_REQUIRE(out16->n == x->n && out16->h == x->h && out16->w == x->w && out16->c == x->c, "lfsr_scale_add16: out shape");
  LFSR_REQUIRE(scale->n == x->n && scale->h == 1 && scale->w == 1 && scale->c == x->c, "lfsr_scale_add16: scale must be [n,1,1,c]");
  LFSR_REQUIRE(x->n <= 65535 && x->c % 8 == 0 && x->ld % 4 == 0 && ((uintptr_t)x->ptr & 15) == 0 && out16->ld % 8 == 0 &&
                   ((uintptr_t)out16->ptr & 15) == 0,
               "lfsr_scale_add16: channels in groups of 8 on 16-byte aligned pixels");
  TView r = null_view();
  if (res && res->ptr) {
    LFSR_REQUIRE(res->n == x->n && res->h == x->h && res->w == x->w && res->c == x->c && res->ld % 4 == 0 &&
                     ((uintptr_t)res->ptr & 15) == 0, "lfsr_scale_add16: res shape / alignment");
    r = view_of(res);
  }
  const int per = x->h * x->w * (x->c / 8);
  dim3 blocks(ceil_div(per, 256), x->n);
  scale_add16_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(view_of(x), (const float*)scale->ptr, scale->ld, r, (__half*)out16->ptr,
                                                              out16->ld);
  return check_launch("scale_add16_kernel");
}

extern "C" int lfsr_tap_gather(const lfsr_tensor* taps, int kh, int kw, const float* bias, const lfsr_tensor* res,
                               const lfsr_tensor* out, void* stream) {
  LFSR_REQUIRE(tensor_ok(taps) && tensor_ok(out), "lfsr_tap_gather: null/invalid tensor");
  LFSR_REQUIRE(kh > 0 && kw > 0 && (kh & 1) && (kw & 1) && taps->c == kh * kw, "lfsr_tap_gather: taps tensor must have kh*kw channels");
  LFSR_REQUIRE(out->c == 1 && out->n == taps->n && out->h == taps->h && out->w == taps->w, "lfsr_tap_gather: out geometry");
  const bool has_res = res && res->ptr;
  if (has_res)
    LFSR_REQUIRE(res->c == 1 && res->n == out->n && res->h == out->h && res->w == out->w, "lfsr_tap_gather: res geometry");
  LFSR_REQUIRE(out->n <= 65535 && (long long)taps->h * taps->w * taps->ld < 0x7fffffffLL, "lfsr_tap_gather: tensor too large");
  dim3 grid(ceil_div(out->w, 32), ceil_div(out->h, 8), out->n);
  if (kh == 3 && kw == 3 && taps->ld == 12 && (((uintptr_t)taps->ptr) & 15) == 0) {
    tap_gather3x3_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(view_of(taps), has_res ? view_of(res) : null_view(), view_of(out), bias);
    return check_launch("tap_gather3x3_kernel");
  }
  tap_gather_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(view_of(taps), has_res ? view_of(res) : null_view(), view_of(out), kh, kw, bias);
  return check_launch("tap_gather_kernel");
}

extern "C" int lfsr_layernorm(const lfsr_tensor* in, const float* gamma, const float* beta, float eps,
                              const lfsr_tensor* out, void* stream) {
  LFSR_REQUIRE(tensor_ok(in) && tensor_ok(out) && gamma && beta, "lfsr_layernorm: null/invalid tensor");
  LFSR_REQUIRE(in->n == out->n && in->h == out->h && in->w == out->w && in->c == out->c, "lfsr_layernorm: shape");
  long long tokens = (long long)in->n * in->h * in->w;
  long long blocks = (tokens + 7) / 8;
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  layernorm_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(view_of(in), view_of(out), gamma, beta, eps, tokens);
  return check_launch("layernorm_kernel");
}

extern "C" int lfsr_epi_attention(const float* qk, const float* v, float* out, const lfsr_epi_attn_desc* d,
                                  void* stream) {
  LFSR_REQUIRE(qk && v && out && d, "lfsr_epi_attention: null pointer");
  LFSR_REQUIRE(d->head_dim == ATT_D, "lfsr_epi_attention: head_dim %d unsupported (16 only)", d->head_dim);
  LFSR_REQUIRE(d->heads > 0 && d->A > 0 && d->S > 0 && d->half_window >= 0 && d->nb > 0 && d->np > 0 && d->nq > 0,
               "lfsr_epi_attention: bad geometry");
  const int L = d->A * d->S;
  LFSR_REQUIRE(L <= 192, "lfsr_epi_attention: sequence length %d > 192", L);
  LFSR_REQUIRE(((uintptr_t)qk % 16 == 0) && ((uintptr_t)v % 16 == 0) && ((uintptr_t)out % 16 == 0),
               "lfsr_epi_attention: pointers must be 16-byte aligned");
  static const bool no_att5 = dbg_env("LFSR_ATT_PER_QUERY") != nullptr;
  if (!no_att5 && d->A == ATT_NQ && d->S <= 32) {       // EPIT's 5 x 5 light fields with 32-pixel patches
    static DevOnce once;
    const size_t smem5 = (size_t)ATT_HPC * 2 * L * ATT_LD * sizeof(float);
    if (once.need()) {
      if (opt_in_smem(epi_attention5_kernel, 110 * 1024, "lfsr_epi_attention")) return LFSR_ERR_CUDA;
      once.done();
    }
    dim3 grid5(d->nb * d->np * d->nq, ceil_div(d->heads, ATT_HPC));
    epi_attention5_kernel<<<grid5, 32 * ATT_HPC, smem5, (cudaStream_t)stream>>>(qk, v, out, *d);
    return check_launch("epi_attention5_kernel");
  }
  dim3 grid(d->nb * d->np * d->nq, d->heads);
  size_t smem = (size_t)2 * L * ATT_LD * sizeof(float);
  epi_attention_kernel<<<grid, 192, smem, (cudaStream_t)stream>>>(qk, v, out, *d);
  return check_launch("epi_attention_kernel");
}

namespace lfsr {
__global__ void __launch_bounds__(256)
to_f16_kernel(const float* __restrict__ in, __half* __restrict__ out, long long pixels, int c, int ld_in, int ld_out) {
  const int c8 = c >> 3;
  const long long total = pixels * c8;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long px = i / c8;
    const int k = (int)(i - px * c8) * 8;
    const float4 a = *reinterpret_cast<const float4*>(in + px * ld_in + k), b = *reinterpret_cast<const float4*>(in + px * ld_in + k + 4);
    __half2 h0 = __floats2half2_rn(a.x, a.y), h1 = __floats2half2_rn(a.z, a.w), h2 = __floats2half2_rn(b.x, b.y), h3 = __floats2half2_rn(b.z, b.w);
    uint4 v;
    v.x = *reinterpret_cast<uint32_t*>(&h0); v.y = *reinterpret_cast<uint32_t*>(&h1);
    v.z = *reinterpret_cast<uint32_t*>(&h2); v.w = *reinterpret_cast<uint32_t*>(&h3);
    *reinterpret_cast<uint4*>(out + px * ld_out + k) = v;
  }
}
}  // namespace lfsr

namespace lfsr {
// thread = one SAI pixel (sy, sx) of the low-resolution mosaic: reads its r*r sub-pixel values from the MacPI-arranged tensor and
// writes the r x r block of the high-resolution SAI image (consecutive threads -> consecutive 4r-byte runs of an output row)
template <int R>
__global__ void __launch_bounds__(256)
macpi_unshuffle_kernel(const float* __restrict__ in, float* __restrict__ out, int H, int W, int A, int ld, int accumulate) {
  const int sx = blockIdx.x * blockDim.x + threadIdx.x, sy = blockIdx.y, img = blockIdx.z;
  if (sx >= W) return;
  const int hh = H / A, ww = W / A;
  const int u = sy / hh, i = sy - u * hh, v = sx / ww, j = sx - v * ww;
  const float* src = in + ((size_t)((size_t)img * H + (i * A + u)) * W + (j * A + v)) * ld;
  float vals[R * R];
  if (R == 4) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float4 t = *reinterpret_cast<const float4*>(src + 4 * k);
      vals[4 * k] = t.x; vals[4 * k + 1] = t.y; vals[4 * k + 2] = t.z; vals[4 * k + 3] = t.w;
    }
  } else {
#pragma unroll
    for (int k = 0; k < R * R; ++k) vals[k] = src[k];
  }
  float* dst = out + ((size_t)((size_t)img * H + sy) * R) * ((size_t)W * R) + (size_t)sx * R;
#pragma unroll
  for (int a = 0; a < R; ++a) {
    float* row = dst + (size_t)a * W * R;
#pragma unroll
    for (int b = 0; b < R; ++b) row[b] = accumulate ? row[b] + vals[a * R + b] : vals[a * R + b];
  }
}
}  // namespace lfsr

namespace lfsr {
__global__ void __launch_bounds__(256)
split_tf32_kernel(const float* __restrict__ in, float* __restrict__ hi, float* __restrict__ lo, long long n4) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 x = reinterpret_cast<const float4*>(in)[i];
    float4 h, l;
    uint32_t t;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.x)); h.x = __uint_as_float(t); l.x = x.x - h.x;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.y)); h.y = __uint_as_float(t); l.y = x.y - h.y;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.z)); h.z = __uint_as_float(t); l.z = x.z - h.z;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(x.w)); h.w = __uint_as_float(t); l.w = x.w - h.w;
    reinterpret_cast<float4*>(hi)[i] = h;
    reinterpret_cast<float4*>(lo)[i] = l;
  }
}
}  // namespace lfsr

extern "C" int lfsr_split_tf32(const float* in, float* hi, float* lo, long long n, void* stream) {
  LFSR_REQUIRE(in && hi && lo && n > 0 && n % 4 == 0 && (((uintptr_t)in | (uintptr_t)hi | (uintptr_t)lo) & 15) == 0,
               "lfsr_split_tf32: 16-byte aligned buffers with a multiple of 4 elements required");
  lfsr::split_tf32_kernel<<<(unsigned)capped_blocks(n / 4), 256, 0, (cudaStream_t)stream>>>(in, hi, lo, n / 4);
  return check_launch("split_tf32_kernel");
}

extern "C" int lfsr_macpi_unshuffle(const lfsr_tensor* in, float* out, int ang, int r, int accumulate, void* stream) {
  LFSR_REQUIRE(tensor_ok(in) && out, "lfsr_macpi_unshuffle: null/invalid tensor");
  LFSR_REQUIRE(ang > 0 && in->h % ang == 0 && in->w % ang == 0 && in->c == r * r && (r == 2 || r == 4) && in->n <= 65535 && in->h <= 65535,
               "lfsr_macpi_unshuffle: needs r in {2, 4}, r*r channels and a mosaic divisible by the angular resolution");
  LFSR_REQUIRE(in->ld % 4 == 0 && ((uintptr_t)in->ptr & 15) == 0, "lfsr_macpi_unshuffle: 16-byte aligned pixels required");
  dim3 grid(ceil_div(in->w, 256), in->h, in->n);
  if (r == 4) lfsr::macpi_unshuffle_kernel<4><<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)in->ptr, out, in->h, in->w, ang, in->ld, accumulate);
  else lfsr::macpi_unshuffle_kernel<2><<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)in->ptr, out, in->h, in->w, ang, in->ld, accumulate);
  return check_launch("macpi_unshuffle_kernel");
}

extern "C" int lfsr_to_f16(const lfsr_tensor* in, const lfsr_tensor* out16, void* stream) {
  LFSR_REQUIRE(tensor_ok(in) && tensor_ok(out16), "lfsr_to_f16: null/invalid tensor");
  LFSR_REQUIRE(in->n == out16->n && in->h == out16->h && in->w == out16->w && in->c == out16->c, "lfsr_to_f16: shape mismatch");
  LFSR_REQUIRE(in->c % 8 == 0 && in->ld % 4 == 0 && out16->ld % 8 == 0 && ((uintptr_t)in->ptr & 15) == 0 && ((uintptr_t)out16->ptr & 15) == 0,
               "lfsr_to_f16: channel count must be a multiple of 8 and rows 16-byte aligned");
  const long long pixels = (long long)in->n * in->h * in->w;
  const long long blocks = capped_blocks(pixels * (in->c / 8));
  lfsr::to_f16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>((const float*)in->ptr, (__half*)out16->ptr, pixels, in->c, in->ld,
                                                                        out16->ld);
  return check_launch("to_f16_kernel");
}

extern "C" int lfsr_metric_sums(const float* label, const float* out, int ang, int h, int w, double* acc,
                                void* stream) {
  return lfsr_metric_sums_uv(label, out, ang, ang, h, w, acc, stream);
}

extern "C" int lfsr_metric_sums_batched(const float* label, const float* out, int n, int ang, int h, int w, double* acc,
                                        void* stream) {
  LFSR_REQUIRE(n > 0, "lfsr_metric_sums: empty batch");
  LFSR_REQUIRE((long long)n * ang < (1LL << 31), "lfsr_metric_sums: too many tiles");
  // n mosaics stacked along y are one mosaic with n * ang view rows: view index = (img * ang + a1) * ang + a2
  return lfsr_metric_sums_uv(label, out, n * ang, ang, h, w, acc, stream);
}

extern "C" int lfsr_metric_sums_uv(const float* label, const float* out, int ang_u, int ang_v, int h, int w, double* acc,
                                   void* stream) {
  LFSR_REQUIRE(label && out && acc, "lfsr_metric_sums: null pointer");
  LFSR_REQUIRE(ang_u > 0 && ang_v > 0 && h >= 11 && w >= 11,
               "lfsr_metric_sums: views must be at least 11x11 (skimage win_size)");
  // scipy.ndimage._gaussian_kernel1d(sigma=1.5, order=0, radius=5): float64 weights, cast to fp32
  Gauss11 gw;
  {
    double g[11], s = 0.0;
    for (int i = -5; i <= 5; ++i) { g[i + 5] = exp(-0.5 / (1.5 * 1.5) * (double)(i * i)); s += g[i + 5]; }
    for (int i = 0; i < 11; ++i) gw.g[i] = (float)(g[i] / s);
  }
  const int tiles_x = ceil_div(w, MT_W), tiles_y = ceil_div(h, MT_H);
  // view index = a1 * ang_v + a2, the row-major order of the views in the [(ang_u h), (ang_v w)] mosaic
  const long long blocks = (long long)ang_u * ang_v * tiles_x * tiles_y;
  LFSR_REQUIRE(blocks < 0x7fffffffLL, "lfsr_metric_sums: too many tiles");
  metric_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(label, out, ang_v, h, w, acc, tiles_x, tiles_y, gw);
  return check_launch("metric_kernel");
}
