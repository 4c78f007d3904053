// LFdivide / LFintegrate gather kernels (reference: utils/utils.py:137-178, train.py:300-319).
// Pure index permutations -> bit-exact by construction. HBM-bound: every output float is written
// once with 128-bit stores; source reads are contiguous (or mirrored-contiguous) 32-float runs.
#include <stdarg.h>
#include "lfsr_common.cuh"

namespace lfsr {

static thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// symmetric (edge-repeating) mirror used by ImageExtend (utils/utils.py:137-149)
__device__ __forceinline__ int mirror(int i, int n) { return i < 0 ? -i - 1 : (i >= n ? 2 * n - 1 - i : i); }

// one thread = 4 consecutive x of one patch row (same view because P % 4 == 0);
// blockIdx.y walks the patches of the shard so all index math is 32-bit
__global__ void __launch_bounds__(256)
divide_kernel(const float* __restrict__ scene, float* __restrict__ patches, int A, int h0, int w0, int P,
              int S, int bdr, int numV, int u_begin, int npatch) {
  const int row = A * P;            // floats per patch row
  const int row4 = row >> 2;
  const int per_patch4 = row * row4;
  const int sw = A * w0;            // scene row stride
  for (int pidx = blockIdx.y; pidx < npatch; pidx += gridDim.y) {
    const int n2 = pidx % numV;
    const int n1 = pidx / numV + u_begin;
    float4* dst = reinterpret_cast<float4*>(patches) + (size_t)pidx * per_patch4;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < per_patch4; t += gridDim.x * blockDim.x) {
      const int x4 = t % row4;
      const int py = t / row4;
      const int a1 = py / P, y = py - a1 * P;
      const int px = x4 << 2;
      const int a2 = px / P, x = px - a2 * P;
      const int sy = mirror(n1 * S + y - bdr, h0);
      const float* src = scene + (size_t)(a1 * h0 + sy) * sw + a2 * w0;
      const int gx = n2 * S + x - bdr;
      float4 v;
      v.x = __ldg(src + mirror(gx, w0));
      v.y = __ldg(src + mirror(gx + 1, w0));
      v.z = __ldg(src + mirror(gx + 2, w0));
      v.w = __ldg(src + mirror(gx + 3, w0));
      dst[t] = v;
    }
  }
}

// blockIdx.y walks (view row a1, output row Y); x covers (a2, X / VEC)
template <int VEC>
__global__ void __launch_bounds__(256)
integrate_kernel(const float* __restrict__ patches, float* __restrict__ out, int A, int pz, int ss, int h,
                 int w, int numV, int u_begin, int y_begin, int y_count) {
  const int wv = w / VEC;           // vectors per view row
  const int bdr = (pz - ss) / 2;
  const size_t prow = (size_t)A * pz;
  for (int ry = blockIdx.y; ry < A * y_count; ry += gridDim.y) {
    const int a1 = ry / y_count;
    const int Y = y_begin + (ry - a1 * y_count);
    const int n1 = Y / ss;
    const float* prow_base = patches + (size_t)(n1 - u_begin) * numV * prow * prow +
                             (size_t)(a1 * pz + bdr + (Y - n1 * ss)) * prow;
    float* orow = out + (size_t)(a1 * h + Y) * ((size_t)A * w);
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < A * wv; t += gridDim.x * blockDim.x) {
      const int a2 = t / wv;
      const int X = (t - a2 * wv) * VEC;
      const int n2 = X / ss;
      const float* src = prow_base + (size_t)n2 * prow * prow + a2 * pz + bdr + (X - n2 * ss);
      float* dst = orow + (size_t)a2 * w + X;
      if (VEC == 4) *reinterpret_cast<float4*>(dst) = __ldg(reinterpret_cast<const float4*>(src));
      else *dst = __ldg(src);
    }
  }
}

// ---- x8 geometric self-ensemble (include/lfsr.h: lfsr_divide_rows_d8 / lfsr_integrate_rows_d8) ----------------------
// Variant t of an L x L patch mosaic M (b0 = t & 1, b1 = t & 2, b2 = t & 4): flip rows, flip columns, transpose, in that
// order. So T_t(M)[y][x] = b2 ? M[f0(x)][f1(y)] : M[f0(y)][f1(x)] with f0 / f1 the row / column flip when b0 / b1 is set,
// and T_t^-1(Z)[r][c] = b2 ? Z[f1(c)][f0(r)] : Z[f0(r)][f1(c)].

// divide_kernel with the variant folded into the source index: blockIdx.y walks (patch, t) pairs in output order, so the
// stores stay dense float4 runs; the scene reads of the transposing variants walk a column of the (L2-resident) LR scene
__global__ void __launch_bounds__(256)
divide_d8_kernel(const float* __restrict__ scene, float* __restrict__ patches, int A, int h0, int w0, int P, int S,
                 int bdr, int numV, int u_begin, int nvar) {
  const int L = A * P;
  const int row4 = L >> 2;
  const int per_patch4 = L * row4;
  const int sw = A * w0;
  for (int vidx = blockIdx.y; vidx < nvar; vidx += gridDim.y) {
    const int pidx = vidx >> 3, t = vidx & 7;
    const bool b0 = t & 1, b1 = t & 2, b2 = t & 4;
    const int n2 = pidx % numV;
    const int n1 = pidx / numV + u_begin;
    // scene offset of patch-mosaic row r / column c (divide_kernel's index math, split by axis)
    auto row_off = [&](int r) {
      if (b0) r = L - 1 - r;
      const int a1 = r / P, y = r - a1 * P;
      return (a1 * h0 + mirror(n1 * S + y - bdr, h0)) * sw;
    };
    auto col_off = [&](int c) {
      if (b1) c = L - 1 - c;
      const int a2 = c / P, x = c - a2 * P;
      return a2 * w0 + mirror(n2 * S + x - bdr, w0);
    };
    float4* dst = reinterpret_cast<float4*>(patches) + (size_t)vidx * per_patch4;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < per_patch4; i += gridDim.x * blockDim.x) {
      const int py = i / row4;
      const int px = (i - py * row4) << 2;
      float4 v;
      if (b2) {
        const int c = col_off(py);
        v.x = __ldg(scene + row_off(px) + c);
        v.y = __ldg(scene + row_off(px + 1) + c);
        v.z = __ldg(scene + row_off(px + 2) + c);
        v.w = __ldg(scene + row_off(px + 3) + c);
      } else {
        const float* src = scene + row_off(py);
        v.x = __ldg(src + col_off(px));
        v.y = __ldg(src + col_off(px + 1));
        v.z = __ldg(src + col_off(px + 2));
        v.w = __ldg(src + col_off(px + 3));
      }
      dst[i] = v;
    }
  }
}

constexpr int D8_TILE = 32;

// One CTA = a 32 x 32 tile of one view (a1, a2) of the stitched mosaic. Each output pixel (Y, X) of the view sits at row
// r(Y), column c(X) of patch (Y / ss, X / ss); the kernel averages T_t^-1(F_t)[r][c] over t. The four non-transposing
// variants are read row-wise straight from global memory (float4 when VEC == 4; reversed quads for b1). The four transposing
// ones read Z_t[f1(c)][f0(r)], a column walk, so each is staged through a padded shared tile: lanes run along Y, which is
// contiguous in Z_t's row, and the tile is read back along X. Sums run in t order with __fadd_rn, then __fmul_rn by 1/8.
template <int VEC>
__global__ void __launch_bounds__(256)
integrate_d8_kernel(const float* __restrict__ patches8, float* __restrict__ out, int A, int pz, int ss, int h, int w,
                    int numV, int u_begin, int y_begin, int y_count, int tiles_x, int tiles_y) {
  __shared__ float tile[4][D8_TILE][D8_TILE + 1];      // [t - 4][Y][X]
  const int L = A * pz;
  const size_t LL = (size_t)L * L;
  const int bdr = (pz - ss) / 2;
  const int a2 = blockIdx.x / tiles_x, X0 = (blockIdx.x - a2 * tiles_x) * D8_TILE;
  const int a1 = blockIdx.y / tiles_y, Y0 = y_begin + (blockIdx.y - a1 * tiles_y) * D8_TILE;
  const int y_end = y_begin + y_count;
  const int lane = threadIdx.x & 31, wy = threadIdx.x >> 5;
  // patch (n1, n2) variant 0 and the in-patch row / column of view pixel (Y, X)
  auto patch_base = [&](int Y, int X) {
    return patches8 + ((size_t)(Y / ss - u_begin) * numV + X / ss) * 8 * LL;
  };
  auto prow = [&](int Y) { return a1 * pz + bdr + Y % ss; };
  auto pcol = [&](int X) { return a2 * pz + bdr + X % ss; };

  // stage the transposing variants: element (Y0 + lane, X0 + wy + 8k) of T_t^-1(Z_t) = Z_t[f1(c)][f0(r)]
  {
    const int Y = Y0 + lane;
    const int r = prow(Y);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int xl = wy + 8 * k, X = X0 + xl;
      if (Y < y_end && X < w) {
        const float* base = patch_base(Y, X);
        const int c = pcol(X);
#pragma unroll
        for (int t = 4; t < 8; ++t) {
          const int zr = (t & 2) ? L - 1 - c : c, zc = (t & 1) ? L - 1 - r : r;
          tile[t - 4][lane][xl] = __ldg(base + t * LL + (size_t)zr * L + zc);
        }
      }
    }
  }
  __syncthreads();

  const size_t ow = (size_t)A * w;
  if (VEC == 4) {
    // thread = one float4 of X in one row: 8 threads per tile row, 32 rows
    const int yl = threadIdx.x >> 3, xl = (threadIdx.x & 7) * 4;
    const int Y = Y0 + yl, X = X0 + xl;
    if (Y < y_end && X < w) {                                    // w % 4 == 0: the whole quad is inside
      const float* base = patch_base(Y, X);
      const int r = prow(Y), c = pcol(X);
      float4 acc;
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        float4 v;
        if (t < 4) {
          const int zr = (t & 1) ? L - 1 - r : r;
          if (t & 2) {                                           // columns L-1-c-3 .. L-1-c, read as one quad, reversed
            const float4 q = __ldg(reinterpret_cast<const float4*>(base + t * LL + (size_t)zr * L + (L - 4 - c)));
            v = make_float4(q.w, q.z, q.y, q.x);
          } else {
            v = __ldg(reinterpret_cast<const float4*>(base + t * LL + (size_t)zr * L + c));
          }
        } else {
          const float* s = tile[t - 4][yl] + xl;
          v = make_float4(s[0], s[1], s[2], s[3]);
        }
        if (t == 0) {
          acc = v;
        } else {
          acc.x = __fadd_rn(acc.x, v.x);
          acc.y = __fadd_rn(acc.y, v.y);
          acc.z = __fadd_rn(acc.z, v.z);
          acc.w = __fadd_rn(acc.w, v.w);
        }
      }
      acc = make_float4(__fmul_rn(acc.x, 0.125f), __fmul_rn(acc.y, 0.125f), __fmul_rn(acc.z, 0.125f),
                        __fmul_rn(acc.w, 0.125f));
      *reinterpret_cast<float4*>(out + (size_t)(a1 * h + Y) * ow + (size_t)a2 * w + X) = acc;
    }
  } else {
    // thread = one X (lane) in rows wy + 8k
    const int X = X0 + lane;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int yl = wy + 8 * k, Y = Y0 + yl;
      if (Y < y_end && X < w) {
        const float* base = patch_base(Y, X);
        const int r = prow(Y), c = pcol(X);
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          float v;
          if (t < 4) {
            const int zr = (t & 1) ? L - 1 - r : r, zc = (t & 2) ? L - 1 - c : c;
            v = __ldg(base + t * LL + (size_t)zr * L + zc);
          } else {
            v = tile[t - 4][yl][lane];
          }
          acc = t == 0 ? v : __fadd_rn(acc, v);
        }
        out[(size_t)(a1 * h + Y) * ow + (size_t)a2 * w + X] = __fmul_rn(acc, 0.125f);
      }
    }
  }
}


}  // namespace lfsr

using namespace lfsr;

extern "C" const char* lfsr_last_error(void) { return g_err; }
extern "C" int lfsr_abi_version(void) { return LFSR_ABI_VERSION; }
extern "C" int lfsr_built_for_sm100a(void) { return 1; }
extern "C" uint64_t lfsr_launch_count(void) { return g_launches.load(); }

// geometry checks + accept / reject rule shared by lfsr_divide_rows and lfsr_divide_rows_d8; sets bdr / numV
static int divide_check(const float* scene, const float* patches, int ang, int h0, int w0, int patch, int stride,
                        int u_begin, int u_end, const char* what, int* bdr_out, int* numv_out) {
  LFSR_REQUIRE(scene && patches, "%s: null pointer", what);
  LFSR_REQUIRE(ang > 0 && h0 > 0 && w0 > 0 && patch > 0 && stride > 0 && patch >= stride,
               "%s: bad geometry A=%d h0=%d w0=%d P=%d S=%d", what, ang, h0, w0, patch, stride);
  LFSR_REQUIRE(patch % 4 == 0, "%s: patch size %d must be a multiple of 4", what, patch);
  const int bdr = (patch - stride) / 2;
  const int numU = (h0 + 2 * bdr - 1) / stride, numV = (w0 + 2 * bdr - 1) / stride;
  // The reference pads bdr above and bdr + stride - 1 below out of ONE mirrored copy of the view (ImageExtend,
  // utils/utils.py:141-147: at most n rows per side) and its unfold must then yield exactly numU x numV windows
  // (utils.py:160-164), else it raises: same accept / reject rule here (oracle/make_golden.py sweeps it against the
  // reference). Accepted geometries never index past one reflection, which is all mirror() implements.
  auto tiles = [&](int n, int want) {
    const int below = bdr + stride - 1 < n ? bdr + stride - 1 : n;
    const int ext = n + bdr + below;
    const int windows = ext >= patch ? (ext - patch) / stride + 1 : 0;
    return n >= bdr && windows >= 1 && windows == want;
  };
  LFSR_REQUIRE(tiles(h0, numU) && tiles(w0, numV),
               "%s: %dx%d views cannot be tiled with patch %d / stride %d (the reference's LFdivide raises too)", what, h0,
               w0, patch, stride);
  LFSR_REQUIRE(0 <= u_begin && u_begin <= u_end && u_end <= numU, "%s: row shard [%d,%d) outside [0,%d)", what,
               u_begin, u_end, numU);
  *bdr_out = bdr;
  *numv_out = numV;
  return LFSR_OK;
}

extern "C" int lfsr_divide_rows(const float* scene, float* patches, int ang, int h0, int w0, int patch,
                                int stride, int u_begin, int u_end, void* stream) {
  int bdr = 0, numV = 0;
  const int st = divide_check(scene, patches, ang, h0, w0, patch, stride, u_begin, u_end, "lfsr_divide", &bdr, &numV);
  if (st != LFSR_OK) return st;
  if (u_begin == u_end) return LFSR_OK;
  const int npatch = (u_end - u_begin) * numV;
  const int per_patch4 = (ang * patch) * (ang * patch / 4);
  dim3 grid(ceil_div(per_patch4, 256 * 4), npatch < 32768 ? npatch : 32768);
  divide_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(scene, patches, ang, h0, w0, patch, stride, bdr, numV, u_begin,
                                                        npatch);
  return check_launch("divide_kernel");
}

extern "C" int lfsr_divide_rows_d8(const float* scene, float* patches, int ang, int h0, int w0, int patch,
                                   int stride, int u_begin, int u_end, void* stream) {
  int bdr = 0, numV = 0;
  const int st = divide_check(scene, patches, ang, h0, w0, patch, stride, u_begin, u_end, "lfsr_divide_rows_d8", &bdr,
                              &numV);
  if (st != LFSR_OK) return st;
  if (u_begin == u_end) return LFSR_OK;
  const int nvar = (u_end - u_begin) * numV * 8;
  const int per_patch4 = (ang * patch) * (ang * patch / 4);
  dim3 grid(ceil_div(per_patch4, 256 * 4), nvar < 32768 ? nvar : 32768);
  divide_d8_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(scene, patches, ang, h0, w0, patch, stride, bdr, numV, u_begin,
                                                           nvar);
  return check_launch("divide_d8_kernel");
}

extern "C" int lfsr_divide(const float* scene, float* patches, int ang, int h0, int w0, int patch, int stride,
                           void* stream) {
  if (patch < stride || stride <= 0) { set_error("lfsr_divide: bad patch/stride"); return LFSR_ERR_INVALID; }
  const int bdr = (patch - stride) / 2;
  const int numU = (h0 + 2 * bdr - 1) / stride;
  return lfsr_divide_rows(scene, patches, ang, h0, w0, patch, stride, 0, numU, stream);
}

// geometry checks shared by lfsr_integrate_rows and lfsr_integrate_rows_d8: the output rows [y_begin, y_begin + y_count)
// of every view that the shard covers (y_count == 0: nothing to do) and whether the float4 path applies
static int integrate_check(const float* patches, const float* out, int ang, int pz, int stride, int h, int w, int num_u,
                           int num_v, int u_begin, int u_end, const char* what, int* y_begin_out, int* y_count_out,
                           bool* vec_out) {
  LFSR_REQUIRE(patches && out, "%s: null pointer", what);
  LFSR_REQUIRE(ang > 0 && pz >= stride && stride > 0 && h > 0 && w > 0, "%s: bad geometry", what);
  LFSR_REQUIRE(h <= num_u * stride && w <= num_v * stride,
               "%s: output %dx%d larger than the stitched grid %dx%d", what, h, w, num_u * stride, num_v * stride);
  LFSR_REQUIRE(0 <= u_begin && u_begin <= u_end && u_end <= num_u, "%s: bad row shard", what);
  const int y_begin = u_begin * stride;
  const int y_end = u_end * stride < h ? u_end * stride : h;
  const int bdr = (pz - stride) / 2;
  *y_begin_out = y_begin;
  *y_count_out = y_end > y_begin ? y_end - y_begin : 0;
  *vec_out = (w % 4 == 0) && (stride % 4 == 0) && (pz % 4 == 0) && (bdr % 4 == 0) &&
             ((uintptr_t)patches % 16 == 0) && ((uintptr_t)out % 16 == 0);
  return LFSR_OK;
}

extern "C" int lfsr_integrate_rows(const float* patches, float* out, int ang, int pz, int stride, int h, int w,
                                   int num_u, int num_v, int u_begin, int u_end, void* stream) {
  int y_begin = 0, y_count = 0;
  bool vec = false;
  const int st = integrate_check(patches, out, ang, pz, stride, h, w, num_u, num_v, u_begin, u_end, "lfsr_integrate",
                                 &y_begin, &y_count, &vec);
  if (st != LFSR_OK) return st;
  if (y_count == 0) return LFSR_OK;
  const int rows = ang * y_count;
  if (vec) {
    dim3 grid(ceil_div(ang * (w / 4), 256), rows < 32768 ? rows : 32768);
    integrate_kernel<4><<<grid, 256, 0, (cudaStream_t)stream>>>(patches, out, ang, pz, stride, h, w, num_v, u_begin,
                                                                y_begin, y_count);
  } else {
    dim3 grid(ceil_div(ang * w, 256), rows < 32768 ? rows : 32768);
    integrate_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(patches, out, ang, pz, stride, h, w, num_v, u_begin,
                                                                y_begin, y_count);
  }
  return check_launch("integrate_kernel");
}

extern "C" int lfsr_integrate_rows_d8(const float* patches8, float* out, int ang, int pz, int stride, int h, int w,
                                      int num_u, int num_v, int u_begin, int u_end, void* stream) {
  int y_begin = 0, y_count = 0;
  bool vec = false;
  const int st = integrate_check(patches8, out, ang, pz, stride, h, w, num_u, num_v, u_begin, u_end,
                                 "lfsr_integrate_rows_d8", &y_begin, &y_count, &vec);
  if (st != LFSR_OK) return st;
  if (y_count == 0) return LFSR_OK;
  const int tiles_x = ceil_div(w, D8_TILE), tiles_y = ceil_div(y_count, D8_TILE);
  LFSR_REQUIRE((long long)ang * tiles_y <= 65535, "lfsr_integrate_rows_d8: %d view rows per shard is too many", y_count);
  dim3 grid(ang * tiles_x, ang * tiles_y);
  if (vec)
    integrate_d8_kernel<4><<<grid, 256, 0, (cudaStream_t)stream>>>(patches8, out, ang, pz, stride, h, w, num_v, u_begin,
                                                                   y_begin, y_count, tiles_x, tiles_y);
  else
    integrate_d8_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(patches8, out, ang, pz, stride, h, w, num_v, u_begin,
                                                                   y_begin, y_count, tiles_x, tiles_y);
  return check_launch("integrate_d8_kernel");
}


// ---- colour tail of test() (train.py:329-341, utils/utils.py:191-204): Y mosaic + CbCr mosaic -> uint8 RGB views -------
// rgb8[u][v][y][x][c] = uint8(clip(M[c][0]*Y + M[c][1]*Cb + M[c][2]*Cr - off[c], 0, 1) * 255), fp64 with separate multiplies and
// adds in the reference's left-to-right order (no FMA contraction) and truncation like numpy's astype('uint8'); the
// (a1 h)(a2 w) -> a1 a2 h w view split (or the mosaic / lenslet image address of the output layout) is folded into the
// store address. 1 byte per channel leaves the GPU, not 4.
namespace lfsr {
struct ColourMat { double m[9]; double off[3]; };
__global__ void __launch_bounds__(256)
ycbcr_rgb8_kernel(const float* __restrict__ y, const float* __restrict__ cb, const float* __restrict__ cr,
                  unsigned char* __restrict__ rgb, int ang_u, int ang_v, int h, int w, int layout, ColourMat cm) {
  const int W = ang_v * w;
  const long long total = (long long)ang_u * h * W;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int X = (int)(t % W), Y = (int)(t / W);
    const int u = Y / h, yy = Y - u * h, v = X / w, xx = X - v * w;
    const double a = (double)y[t], b = (double)cb[t], c = (double)cr[t];
    long long px;                                       // output pixel index in the chosen layout
    if (layout == LFSR_LAYOUT_MOSAIC) px = t;
    else if (layout == LFSR_LAYOUT_LENSLET) px = ((long long)yy * ang_u + u) * W + (long long)xx * ang_v + v;
    else px = (((long long)u * ang_v + v) * h + yy) * w + xx;
    unsigned char* dst = rgb + px * 3;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      double r = __dadd_rn(__dadd_rn(__dmul_rn(cm.m[3 * k], a), __dmul_rn(cm.m[3 * k + 1], b)), __dmul_rn(cm.m[3 * k + 2], c));
      r = __dadd_rn(r, -cm.off[k]);
      r = r < 0.0 ? 0.0 : (r > 1.0 ? 1.0 : r);          // numpy clip (NaN propagates there; inputs here are finite)
      dst[k] = (unsigned char)(int)__dmul_rn(r, 255.0);
    }
  }
}
}  // namespace lfsr

extern "C" int lfsr_ycbcr_to_rgb8(const float* y, const float* cb, const float* cr, unsigned char* rgb, int ang, int h, int w,
                                  const double* mat_inv255, const double* offset, void* stream) {
  return lfsr_ycbcr_to_rgb8_uv(y, cb, cr, rgb, ang, ang, h, w, mat_inv255, offset, stream);
}

extern "C" int lfsr_ycbcr_to_rgb8_uv(const float* y, const float* cb, const float* cr, unsigned char* rgb, int ang_u,
                                     int ang_v, int h, int w, const double* mat_inv255, const double* offset, void* stream) {
  return lfsr_ycbcr_to_rgb8_layout(y, cb, cr, rgb, ang_u, ang_v, h, w, LFSR_LAYOUT_VIEWS, mat_inv255, offset, stream);
}

extern "C" int lfsr_ycbcr_to_rgb8_layout(const float* y, const float* cb, const float* cr, unsigned char* rgb, int ang_u,
                                         int ang_v, int h, int w, int layout, const double* mat_inv255, const double* offset,
                                         void* stream) {
  LFSR_REQUIRE(y && cb && cr && rgb && mat_inv255 && offset, "lfsr_ycbcr_to_rgb8: null pointer");
  LFSR_REQUIRE(ang_u > 0 && ang_v > 0 && h > 0 && w > 0, "lfsr_ycbcr_to_rgb8: bad geometry");
  LFSR_REQUIRE(layout == LFSR_LAYOUT_VIEWS || layout == LFSR_LAYOUT_MOSAIC || layout == LFSR_LAYOUT_LENSLET,
               "lfsr_ycbcr_to_rgb8: unknown output layout %d", layout);
  LFSR_REQUIRE((long long)ang_u * h < (1LL << 31) && (long long)ang_v * w < (1LL << 31),
               "lfsr_ycbcr_to_rgb8: mosaic %lldx%lld too large", (long long)ang_u * h, (long long)ang_v * w);
  lfsr::ColourMat cm;
  for (int i = 0; i < 9; ++i) cm.m[i] = mat_inv255[i];
  for (int i = 0; i < 3; ++i) cm.off[i] = offset[i];
  const long long total = (long long)ang_u * h * ang_v * w;
  long long blocks = (total + 255) / 256;
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  lfsr::ycbcr_rgb8_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(y, cb, cr, rgb, ang_u, ang_v, h, w, layout, cm);
  return lfsr::check_launch("ycbcr_rgb8_kernel");
}


// ---- input side of the light-field preparation (include/lfsr.h, "View preparation"): RGB views -> Y / CbCr mosaics -------
// BasicLFSR's rgb2ycbcr term by term: Y = (((65.481 R + 128.553 G) + 24.966 B) + 16) / 255 and likewise Cb, Cr with the
// signs folded into the constants (exact), every multiply / add / divide rounded on its own (no FMA contraction), cast
// to fp32 round-to-nearest. uint8 views are divided by 255 here in fp64 first. One thread per mosaic pixel in mosaic
// order, so the fp32 stores coalesce; the a1 a2 h w -> (a1 h)(a2 w) rearrange is folded into the load address.
namespace lfsr {
__device__ __forceinline__ double view_value(const unsigned char* p) { return __ddiv_rn((double)*p, 255.0); }
__device__ __forceinline__ double view_value(const double* p) { return *p; }

__device__ __forceinline__ float ycbcr_term(double r, double g, double b, double kr, double kg, double kb, double off) {
  const double s = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(kr, r), __dmul_rn(kg, g)), __dmul_rn(kb, b)), off);
  return __double2float_rn(__ddiv_rn(s, 255.0));
}

template <class T>
__global__ void __launch_bounds__(256)
rgb_ycbcr_mosaic_kernel(const T* __restrict__ views, float* __restrict__ y, float* __restrict__ cb, float* __restrict__ cr,
                        int ang_u, int ang_v, int h, int w) {
  const int W = ang_v * w;
  const long long total = (long long)ang_u * h * W;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int X = (int)(t % W), Y = (int)(t / W);
    const int u = Y / h, yy = Y - u * h, v = X / w, xx = X - v * w;
    const T* src = views + ((((long long)u * ang_v + v) * h + yy) * w + xx) * 3;
    const double r = view_value(src), g = view_value(src + 1), b = view_value(src + 2);
    if (y) y[t] = ycbcr_term(r, g, b, 65.481, 128.553, 24.966, 16.0);
    if (cb) {
      cb[t] = ycbcr_term(r, g, b, -37.797, -74.203, 112.0, 128.0);
      cr[t] = ycbcr_term(r, g, b, 112.0, -93.786, -18.214, 128.0);
    }
  }
}
}  // namespace lfsr

extern "C" int lfsr_rgb_to_ycbcr_mosaic(const void* views, int is_u8, float* y, float* cb, float* cr, int ang, int h, int w,
                                        void* stream) {
  return lfsr_rgb_to_ycbcr_mosaic_uv(views, is_u8, y, cb, cr, ang, ang, h, w, stream);
}

extern "C" int lfsr_rgb_to_ycbcr_mosaic_uv(const void* views, int is_u8, float* y, float* cb, float* cr, int ang_u,
                                           int ang_v, int h, int w, void* stream) {
  LFSR_REQUIRE(views, "lfsr_rgb_to_ycbcr_mosaic: null views");
  LFSR_REQUIRE(y || cb, "lfsr_rgb_to_ycbcr_mosaic: no output (need Y, CbCr or both)");
  LFSR_REQUIRE((cb == nullptr) == (cr == nullptr), "lfsr_rgb_to_ycbcr_mosaic: cb and cr go together");
  LFSR_REQUIRE(ang_u > 0 && ang_v > 0 && h > 0 && w > 0, "lfsr_rgb_to_ycbcr_mosaic: bad geometry ang=%dx%d h=%d w=%d",
               ang_u, ang_v, h, w);
  LFSR_REQUIRE((long long)ang_u * h < (1LL << 31) && (long long)ang_v * w < (1LL << 31),
               "lfsr_rgb_to_ycbcr_mosaic: mosaic %lldx%lld too large", (long long)ang_u * h, (long long)ang_v * w);
  const long long total = (long long)ang_u * h * ang_v * w;
  long long blocks = (total + 255) / 256;
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  if (is_u8) {
    lfsr::rgb_ycbcr_mosaic_kernel<unsigned char><<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(
        (const unsigned char*)views, y, cb, cr, ang_u, ang_v, h, w);
  } else {
    lfsr::rgb_ycbcr_mosaic_kernel<double><<<(int)blocks, 256, 0, (cudaStream_t)stream>>>((const double*)views, y, cb, cr,
                                                                                          ang_u, ang_v, h, w);
  }
  return lfsr::check_launch("rgb_ycbcr_mosaic_kernel");
}

// Image light fields (include/lfsr.h, "View preparation"): the views [u0, u0 + n_u) x [v0, v0 + n_v) of a U x V grid stored
// as one mosaic or lenslet image, each cropped to hc x wc, gathered into view-major uint8 [n_u][n_v][hc][wc][3]. One thread
// per output pixel in output order, so the stores are dense; the layout is folded into the load address.
namespace lfsr {
__global__ void __launch_bounds__(256)
image_to_views_kernel(const unsigned char* __restrict__ img, unsigned char* __restrict__ views, int layout, int U, int V,
                      int H, int W, int u0, int v0, int n_v, int hc, int wc, long long total) {
  const long long row_px = (long long)V * W;            // image pixels per row, both layouts
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(t % wc);
    const long long r = t / wc;
    const int y = (int)(r % hc);
    const int view = (int)(r / hc);
    const int u = u0 + view / n_v, v = v0 + view % n_v;
    const long long px = layout == LFSR_LAYOUT_MOSAIC ? ((long long)u * H + y) * row_px + (long long)v * W + x
                                                      : ((long long)y * U + u) * row_px + (long long)x * V + v;
    const unsigned char* src = img + px * 3;
    unsigned char* dst = views + t * 3;
    dst[0] = __ldg(src);
    dst[1] = __ldg(src + 1);
    dst[2] = __ldg(src + 2);
  }
}
}  // namespace lfsr

extern "C" int lfsr_image_to_views_u8(const unsigned char* img, int layout, int U, int V, int H, int W, int u0, int v0,
                                      int n_u, int n_v, int hc, int wc, unsigned char* views, void* stream) {
  LFSR_REQUIRE(img && views, "lfsr_image_to_views_u8: null pointer");
  LFSR_REQUIRE(layout == LFSR_LAYOUT_MOSAIC || layout == LFSR_LAYOUT_LENSLET,
               "lfsr_image_to_views_u8: unknown image layout %d (1 mosaic, 2 lenslet)", layout);
  LFSR_REQUIRE(U > 0 && V > 0 && H > 0 && W > 0 && n_u > 0 && n_v > 0 && hc > 0 && wc > 0,
               "lfsr_image_to_views_u8: bad geometry grid=%dx%d view=%dx%d sel=%dx%d crop=%dx%d", U, V, H, W, n_u, n_v,
               hc, wc);
  LFSR_REQUIRE(u0 >= 0 && v0 >= 0 && (long long)u0 + n_u <= U && (long long)v0 + n_v <= V,
               "lfsr_image_to_views_u8: views [%d, %d) x [%d, %d) lie outside the %dx%d grid", u0, u0 + n_u, v0, v0 + n_v,
               U, V);
  LFSR_REQUIRE(hc <= H && wc <= W, "lfsr_image_to_views_u8: crop %dx%d larger than the %dx%d views", hc, wc, H, W);
  LFSR_REQUIRE((long long)U * H < (1LL << 31) && (long long)V * W < (1LL << 31),
               "lfsr_image_to_views_u8: image %lldx%lld too large", (long long)U * H, (long long)V * W);
  const long long total = (long long)n_u * n_v * hc * wc;
  long long blocks = (total + 255) / 256;
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  lfsr::image_to_views_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(img, views, layout, U, V, H, W, u0, v0, n_v,
                                                                              hc, wc, total);
  return lfsr::check_launch("image_to_views_kernel");
}


// ---- angular window tiling (include/lfsr.h, "Angular window tiling"): one SR window mosaic [(A h), (A w)] merged into the
// N_u x N_v SR mosaic [(N_u h), (N_v w)] at view offset (o_u, o_v). Per view of the window a mode: 0 = store, 1 = add, c >= 2 = add,
// then divide by c (the last window over that view). Sums with __fadd_rn, the mean with one __fdiv_rn: fp32 `a + b` and
// `a / c` in torch give the same bits. One thread = VEC consecutive x of one view row, in window-mosaic order, so the window
// reads are dense; a window row lands as one contiguous run of the grid row (views o_v .. o_v + A - 1 are adjacent there).
namespace lfsr {
constexpr int WIN_MAX_ANG = 16;
struct WinModes { int m[WIN_MAX_ANG * WIN_MAX_ANG]; };

__device__ __forceinline__ float win_merge(float acc, float v, int mode) {
  const float s = __fadd_rn(acc, v);
  return mode == 1 ? s : __fdiv_rn(s, (float)mode);
}

template <int VEC>
__global__ void __launch_bounds__(256)
window_accumulate_kernel(const float* __restrict__ win, float* __restrict__ grid, int A, int Nv, int h, int w, int o_u,
                         int o_v, WinModes md) {
  const int wv = w / VEC;
  for (int Y = blockIdx.y; Y < A * h; Y += gridDim.y) {
    const int a1 = Y / h, y = Y - a1 * h;
    const float* src = win + (size_t)Y * A * w;
    float* dst = grid + ((size_t)(o_u + a1) * h + y) * ((size_t)Nv * w) + (size_t)o_v * w;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < A * wv; t += gridDim.x * blockDim.x) {
      const int a2 = t / wv;
      const int X = a2 * w + (t - a2 * wv) * VEC;
      const int mode = md.m[a1 * A + a2];
      if (VEC == 4) {
        float4 v = __ldg(reinterpret_cast<const float4*>(src + X));
        float4* o = reinterpret_cast<float4*>(dst + X);
        if (mode != 0) {
          const float4 a = *o;
          v = make_float4(win_merge(a.x, v.x, mode), win_merge(a.y, v.y, mode), win_merge(a.z, v.z, mode),
                          win_merge(a.w, v.w, mode));
        }
        *o = v;
      } else {
        const float v = __ldg(src + X);
        dst[X] = mode == 0 ? v : win_merge(dst[X], v, mode);
      }
    }
  }
}
}  // namespace lfsr

extern "C" int lfsr_window_accumulate(const float* win, float* grid, int ang, int n, int h, int w, int o_u, int o_v,
                                      const int32_t* host_modes, void* stream) {
  return lfsr_window_accumulate_uv(win, grid, ang, n, n, h, w, o_u, o_v, host_modes, stream);
}

extern "C" int lfsr_window_accumulate_uv(const float* win, float* grid, int ang, int n_u, int n_v, int h, int w, int o_u,
                                         int o_v, const int32_t* host_modes, void* stream) {
  using lfsr::WIN_MAX_ANG;
  LFSR_REQUIRE(win && grid && host_modes, "lfsr_window_accumulate: null pointer");
  LFSR_REQUIRE(ang > 0 && ang <= WIN_MAX_ANG && h > 0 && w > 0, "lfsr_window_accumulate: bad geometry A=%d h=%d w=%d "
               "(1 <= A <= %d)", ang, h, w, WIN_MAX_ANG);
  LFSR_REQUIRE(n_u >= ang && n_v >= ang, "lfsr_window_accumulate: a %dx%d grid is smaller than the %dx%d window", n_u, n_v,
               ang, ang);
  LFSR_REQUIRE((long long)n_u * h < (1LL << 31) && (long long)n_v * w < (1LL << 31),
               "lfsr_window_accumulate: mosaic %lldx%lld too large", (long long)n_u * h, (long long)n_v * w);
  LFSR_REQUIRE(0 <= o_u && o_u <= n_u - ang && 0 <= o_v && o_v <= n_v - ang,
               "lfsr_window_accumulate: window at (%d, %d) lies outside the %dx%d grid (A=%d)", o_u, o_v, n_u, n_v, ang);
  const long long win_n = (long long)ang * h * ang * w, grid_n = (long long)n_u * h * n_v * w;
  LFSR_REQUIRE(win + win_n <= grid || grid + grid_n <= win, "lfsr_window_accumulate: window and grid mosaics overlap");
  // a view lies in at most A windows per angular axis (distinct origins in (u - A, u]) and in at most N - A + 1
  const int per_u = ang < n_u - ang + 1 ? ang : n_u - ang + 1, per_v = ang < n_v - ang + 1 ? ang : n_v - ang + 1;
  lfsr::WinModes md;
  for (int i = 0; i < ang * ang; ++i) {
    LFSR_REQUIRE(host_modes[i] >= 0 && host_modes[i] <= per_u * per_v,
                 "lfsr_window_accumulate: bad mode %d for view %d (0 store, 1 add, 2..%d add then divide)", host_modes[i],
                 i, per_u * per_v);
    md.m[i] = host_modes[i];
  }
  const int rows = ang * h;
  const bool vec = w % 4 == 0 && (uintptr_t)win % 16 == 0 && (uintptr_t)grid % 16 == 0;
  const int per_row = vec ? ang * (w / 4) : ang * w;
  dim3 g(ceil_div(per_row, 256), rows < 32768 ? rows : 32768);
  if (vec)
    lfsr::window_accumulate_kernel<4><<<g, 256, 0, (cudaStream_t)stream>>>(win, grid, ang, n_v, h, w, o_u, o_v, md);
  else
    lfsr::window_accumulate_kernel<1><<<g, 256, 0, (cudaStream_t)stream>>>(win, grid, ang, n_v, h, w, o_u, o_v, md);
  return lfsr::check_launch("window_accumulate_kernel");
}
