/*
 * lfsr.h — C ABI of liblfsr_b200.so: the B200 (sm_100a) kernels behind BasicLFSR's
 * patch-wise light-field SR inference path
 *     LFdivide -> get_model(args).forward(lr, data_info) -> LFintegrate -> PSNR/SSIM on Y.
 *
 * The reference (darskkaa/NTIRE-2026-...-Track-2-Efficiency) has NO native/FFI layer: its
 * "plugin ABI" is a Python duck type (model.SR.<name>.get_model / utils.utils.LFdivide ...).
 * Each entry point below therefore cites the reference Python function whose arithmetic it
 * replaces (paths relative to /root/reference). The Python host side (package
 * `..._b200`, re-exported as `lfsr_b200`) binds these with ctypes; INTEGRATION.md shows the
 * stub a reference maintainer would add.
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless named host_*.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing syncs.
 *   - no hidden allocation: workspaces are passed in, sizes come from *_workspace() queries.
 *   - return 0 on success, negative lfsr_status on error; lfsr_last_error() gives the text
 *     (thread-local).
 *   - feature tensors are fp32 NHWC views (`lfsr_tensor`): element (n,y,x,c) lives at
 *     ptr[((n*h + y)*w + x)*ld + c], ld >= c. A channel slice of a wider buffer is the same
 *     struct with ptr advanced and c reduced - this is how torch.cat / torch.split are free.
 *   - single-channel mosaics ([B,1,A*h,A*w] in the reference) are plain dense fp32 images.
 */
#ifndef LFSR_B200_H_
#define LFSR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LFSR_ABI_VERSION 1

typedef enum {
  LFSR_OK = 0,
  LFSR_ERR_INVALID = -1,      /* bad argument / unsupported shape */
  LFSR_ERR_CUDA = -2,         /* CUDA runtime / driver error, see lfsr_last_error() */
  LFSR_ERR_UNSUPPORTED = -3,  /* valid request, not handled by this build */
  LFSR_ERR_WORKSPACE = -4     /* workspace too small */
} lfsr_status;

typedef struct {
  void* ptr;
  int32_t n, h, w, c;
  int32_t ld; /* floats between consecutive pixels */
} lfsr_tensor;

enum { LFSR_ACT_NONE = 0, LFSR_ACT_RELU = 1, LFSR_ACT_LRELU = 2, LFSR_ACT_SIGMOID = 3,
       LFSR_ACT_GELU = 4,      /* nn.GELU() (erf form), MyEfficientLFNetV4_5.py:213,231 */
       LFSR_ACT_SILU = 5       /* F.silu, as `mul_act` on the FastConvSSM gate (:242) */ };
enum { LFSR_PERM_NONE = 0, LFSR_PERM_MACPI_OVER_SAI = 1 };
enum { LFSR_SHUF_CHANNEL_MAJOR = 0, /* nn.PixelShuffle: co = c*ry*rx + i*rx + j   */
       LFSR_SHUF_FACTOR_MAJOR = 1   /* PixelShuffle1D  : co = (i*rx + j)*C + c     */ };
enum { LFSR_INTERP_BICUBIC = 0, LFSR_INTERP_BILINEAR = 1 };

/* Convolution + fused epilogue descriptor.
 *   v = sum_taps W[tap][ci][co] * in_scale[n][ci] * in(n, oy*stride_h - pad_h + ky*dil_h, ..., ci) + bias[co]
 *   v = act(v); v *= mul_act(mul(n,oy,ox,co)); v *= alpha;
 *   (sy,sx,sc) = shuffle(oy,ox,co); v += res(n,sy,sx,sc); out(n,sy,sx,sc) = v
 * in_perm / out_perm = LFSR_PERM_MACPI_OVER_SAI: the logical image the convolution walks is the
 * MacPI arrangement mac[i*A+u][j*A+v] of a tensor stored as SAI sai[u*h+i][v*w+j] (A = perm_a);
 * this folds SAI2MacPI / MacPI2SAI (DistgSSR.py:134-155, LF_InterNet.py:144-165) into addressing. */
typedef struct {
  int32_t kh, kw, stride_h, stride_w, dil_h, dil_w, pad_h, pad_w;
  int32_t in_perm, out_perm, perm_a;
  int32_t shuf_ry, shuf_rx, shuf_mode;
  int32_t block_h, block_w; /* >0: taps leaving the block_h x block_w block of the output pixel read 0
                               (per-view Conv3d(1,3,3) of EPIT.py:24-31 on SAI-mosaic storage); stride 1 only */
  int32_t act;
  float act_slope;
  float alpha;
  int32_t mul_act;       /* activation applied to the `mul` operand before the product (LFSR_ACT_*) */
  const float* bias;     /* [cout] or NULL */
  const float* in_scale; /* [n][in_scale_ld] (first cin used) or NULL */
  int64_t in_scale_ld;   /* floats between samples of in_scale; 0 = cin */
  int64_t w_batch_stride; /* lfsr_conv2d_tc only: >0 = one packed weight set per image, this many floats apart
                             (built by lfsr_scale_pack_tc for per-sample gated convs); 0 = shared weights */
  lfsr_tensor mul;       /* ptr NULL if unused; conv-output geometry */
  lfsr_tensor res;       /* ptr NULL if unused; stored-output geometry */
  /* lfsr_conv2d_tc only, with a PixelShuffle: do not store the tail_c-channel shuffled activation at all but its
   * projection onto tail_taps vectors, out(n, y, x, t) = sum_c tail_w[c][t] * act(shuffle(conv))(n, y, x, c), fp32.
   * With tail_w[c][ky*3+kx] = W_head[0][c][ky][kx] this is the per-tap response of the 3x3 reconstruction conv that
   * follows the last upsampler stage (MyEfficientLFNet.py:70-73,104-109; MyEfficientLFNetV4_5.py:62,98-109), which
   * lfsr_tap_gather then sums over the 9 shifted positions: the widest activation of the network is never written. */
  const float* tail_w;   /* [tail_c][12] (columns >= tail_taps zero) or NULL */
  int32_t tail_taps, tail_c;
  /* lfsr_conv2d_tc only - fp16 activations between tensor-core layers (10-bit mantissa = what the TF32 path keeps of an
   * operand anyway; fp32 accumulation; residual / elementwise consumers keep reading the fp32 tensors):
   *   in_f16   != 0: `in` is an fp16 NHWC view (ld in 2-byte elements, multiple of 8) and the weights were packed by
   *                  lfsr_pack_conv_tc16: kind::f16 MMAs, half the shared-memory bytes and MMA time per MAC
   *   out_mode 0: fp32 output only; 1: fp32 output + an fp16 copy in `out16`; 2: `out16` only (then `out` only carries the
   *              geometry, its pointer is not written). Copies need channel counts that are multiples of 8. */
  int32_t in_f16, out_mode;
  lfsr_tensor out16;     /* fp16 view with out's geometry (ld in 2-byte elements) */
  const float* tail_w_host;   /* host copy of tail_w (required with tail_w): read at launch, passed to the kernel by value */
} lfsr_conv_desc;

const char* lfsr_last_error(void);
int lfsr_abi_version(void);
/* 1 if this build carries sm_100a code for every kernel (always, for this library). */
int lfsr_built_for_sm100a(void);
/* number of kernel launches issued by this library in the calling process since load */
uint64_t lfsr_launch_count(void);
/* how many lfsr_conv2d_tc calls took the two-CTAs-per-SM kernel for narrow fp16 layers (tests assert the path taken) */
uint64_t lfsr_conv_tc_lean_count(void);
/* how many lfsr_conv2d_tc calls took the halo-block CTA-pair kernel (fp16 3x3 convs with 128 < N <= 256: the upsampler) */
uint64_t lfsr_conv_tc_halo_count(void);
/* that kernel's block plan for an h x w image and cout packed output channels: geom[0..7] = output block width, output block rows, padded block width, MMA tiles per block, blocks per image row, block rows
 * per image, bytes of one input buffer, dynamic shared memory bytes. Returns 1 if the kernel can run that geometry, else 0. */
int lfsr_conv_tc_halo_plan(int h, int w, int cout, int* geom);

/* ---- patch pipeline ------------------------------------------------------------------ */
/* LFdivide + ImageExtend (utils/utils.py:137-166): scene [A*h0, A*w0] -> [numU*numV, A*P, A*P],
 * numU = (h0 + 2*((P-S)/2) - 1)/S. Bit-exact gather with symmetric mirror padding. Geometries the reference's
 * unfold / rearrange pair cannot tile (utils.py:160-164 raises: non-overlapping patches, P != 2*S in general, views much
 * smaller than a patch) return LFSR_ERR_INVALID. */
int lfsr_divide(const float* scene, float* patches, int ang, int h0, int w0, int patch, int stride,
                void* stream);
/* same, restricted to patch-grid rows [u_begin, u_end) (multi-GPU row sharding, SURVEY 8e) */
int lfsr_divide_rows(const float* scene, float* patches, int ang, int h0, int w0, int patch,
                     int stride, int u_begin, int u_end, void* stream);
/* LFintegrate (utils/utils.py:169-178) + train.py:314-319: patches [numU*numV, A*pz, A*pz] ->
 * SAI mosaic [A*h, A*w] (the 'a1 a2 h w -> (a1 h) (a2 w)' rearrange is folded in).
 * rows [u_begin,u_end) of the patch grid only; `patches` points at patch (u_begin, 0);
 * out is the full mosaic (rows outside the shard are untouched). */
int lfsr_integrate_rows(const float* patches, float* out, int ang, int pz, int stride, int h, int w,
                        int num_u, int num_v, int u_begin, int u_end, void* stream);

/* ---- x8 geometric self-ensemble (no counterpart in the reference) ---------------------- */
/* The 8 flips / transposes of one patch mosaic M [(a1 P), (a2 P)] of side L; on the SAI mosaic they reverse an angular
 * axis together with its spatial axis, or swap (u, h) with (v, w), so the epipolar geometry is kept. For t in 0..7 with
 * b0 = t & 1, b1 = (t >> 1) & 1, b2 = (t >> 2) & 1:
 *     T_t(M):  m = M;  if b0: m = m[::-1, :];  if b1: m = m[:, ::-1];  if b2: m = m.T
 * and T_t^-1 applies the same steps in reverse order. The ensemble of a patch with network F is, in fp32 without FMA
 * contraction, Y = ((T_0^-1 F(T_0 X) + T_1^-1 F(T_1 X)) + ... + T_7^-1 F(T_7 X)) * 0.125.
 *
 * lfsr_divide_rows_d8: lfsr_divide_rows (same geometry checks and accept / reject rule) that writes the 8 variants of
 * every patch of rows [u_begin, u_end): patches [(u_end - u_begin) * numV][8][A*P][A*P], patch-major, t = T_t(patch).
 * Bit-exact (a pure gather). */
int lfsr_divide_rows_d8(const float* scene, float* patches, int ang, int h0, int w0, int patch, int stride,
                        int u_begin, int u_end, void* stream);
/* lfsr_integrate_rows_d8: patches8 [(u_end - u_begin) * num_v][8][A*pz][A*pz] holds F(T_t X) of each patch (pointing at
 * patch (u_begin, 0), variant 0); writes the LFintegrate of the per-patch ensembles Y into rows [u_begin, u_end) of the
 * mosaic, with the row-shard semantics of lfsr_integrate_rows. Each mosaic pixel is written once (no atomics). */
int lfsr_integrate_rows_d8(const float* patches8, float* out, int ang, int pz, int stride, int h, int w,
                           int num_u, int num_v, int u_begin, int u_end, void* stream);

/* ---- interpolation residual ---------------------------------------------------------- */
/* F.interpolate(mode='bicubic'|'bilinear', align_corners=False) as called at
 * MyEfficientLFNet.py:88-90 (bicubic, whole mosaic), EPIT.py:164-169 (bicubic, per view),
 * DistgSSR.py:30 (bilinear, whole mosaic). in [n, h, w] -> out [n, h*s, w*s];
 * block_h/block_w = size of the independently-clamped block (h,w for whole mosaic; view size
 * for per-view). */
int lfsr_interp(const float* in, float* out, int n, int h, int w, int scale, int mode, int block_h,
                int block_w, void* stream);

/* Colour tail of test() (train.py:332-335 + utils/utils.py:191-204 `ycbcr2rgb`): SR Y mosaic [(a1 h), (a2 w)] and the
 * CbCr mosaics of the same size -> uint8 RGB views [a1][a2][h][w][3]; fp64, uint8 by truncation after clip(0,1)*255.
 * mat_inv255 = inv(M_BT601) * 255 (row-major 3x3) and offset = inv(M) @ [16,128,128] come from the host (host pointers). */
int lfsr_ycbcr_to_rgb8(const float* y, const float* cb, const float* cr, unsigned char* rgb, int ang, int h, int w,
                       const double* mat_inv255, const double* offset, void* stream);
/* the same for an ang_u x ang_v grid of views: mosaics [(ang_u h)][(ang_v w)] -> uint8 views [ang_u][ang_v][h][w][3].
 * lfsr_ycbcr_to_rgb8 is this with ang_u = ang_v = ang. */
int lfsr_ycbcr_to_rgb8_uv(const float* y, const float* cb, const float* cr, unsigned char* rgb, int ang_u, int ang_v, int h,
                          int w, const double* mat_inv255, const double* offset, void* stream);
/* the same with the output in one of the layouts of "Image light fields" below: LFSR_LAYOUT_VIEWS [ang_u][ang_v][h][w][3]
 * (lfsr_ycbcr_to_rgb8_uv is this with layout 0), LFSR_LAYOUT_MOSAIC [(ang_u h)][(ang_v w)][3] or LFSR_LAYOUT_LENSLET
 * [(h ang_u)][(w ang_v)][3]. Only the store address differs between the layouts. LFSR_ERR_INVALID for an unknown layout or
 * a mosaic side of 2^31 or more. */
int lfsr_ycbcr_to_rgb8_layout(const float* y, const float* cb, const float* cr, unsigned char* rgb, int ang_u, int ang_v,
                              int h, int w, int layout, const double* mat_inv255, const double* offset, void* stream);

/* ---- View preparation (input side; BasicLFSR's Generate_Data_for_Test.py / _for_inference.py as recorded in DESIGN.md
 * row f-7: the generator scripts are not in this tree, so parity with them is unpinned). Per scene of U x V RGB views
 * (U, V >= A = angRes), with s = scale_factor:
 *   views   the central A x A: u0 = (U - A) // 2, v0 = (V - A) // 2;
 *   crop    every view top-left to H' = H - H mod s, W' = W - W mod s; x = uint8 / 255.0 in fp64, in [0, 1];
 *   colour  rgb2ycbcr term by term, each operation rounded, no FMA (a term's sign is folded into its constant):
 *             Y  = ((((65.481 R + 128.553 G) + 24.966 B) +  16) / 255
 *             Cb = ((((-37.797 R + -74.203 G) + 112.0 B) + 128) / 255
 *             Cr = ((((112.0 R + -93.786 G) + -18.214 B) + 128) / 255
 *   ground-truth views (test.py): Hr_SAI_y = Y(x); lr_rgb = imresize(x, 1/s) per view (fp64 float path);
 *             Lr_SAI_y = Y(lr_rgb); Sr_SAI_cbcr = CbCr(imresize(lr_rgb, s));
 *   LR views (inference.py): Lr_SAI_y = Y(x); Sr_SAI_cbcr = CbCr(imresize(x, s)); no HR.
 * Outputs are SAI mosaics [(u h), (v w)] cast to fp32 round-to-nearest, Sr_SAI_cbcr as [2][(u h)][(v w)].
 *
 * lfsr_rgb_to_ycbcr_mosaic: views [ang][ang][h][w][3], uint8 (is_u8 = 1; divided by 255.0 in the kernel) or fp64 in
 * [0, 1] (is_u8 = 0) -> the colour step above into fp32 mosaics [(ang h)][(ang w)]. y, or cb and cr together, may be NULL
 * to skip that output; at least one is written. Bit-exact to the numpy statement. */
int lfsr_rgb_to_ycbcr_mosaic(const void* views, int is_u8, float* y, float* cb, float* cr, int ang, int h, int w,
                             void* stream);
/* the same for an ang_u x ang_v grid: views [ang_u][ang_v][h][w][3] -> mosaics [(ang_u h)][(ang_v w)].
 * lfsr_rgb_to_ycbcr_mosaic is this with ang_u = ang_v = ang. */
int lfsr_rgb_to_ycbcr_mosaic_uv(const void* views, int is_u8, float* y, float* cb, float* cr, int ang_u, int ang_v, int h,
                                int w, void* stream);

/* Image light fields: a U x V grid of H x W RGB views stored as ONE 8-bit RGB image instead of U*V view files.
 *   mosaic   (sub-aperture image array) image [(U H)][(V W)][3]: image pixel (u*H + h, v*W + w) is view (u, v) at (h, w);
 *   lenslet  (macro-pixel image, BasicLFSR's MacPI) image [(H U)][(W V)][3]: image pixel (h*U + u, w*V + v) is view (u, v) at
 *            (h, w). For U = V = A this is SAI2MacPI (DistgSSR.py:145-155, oracle/nets.py `sai2macpi`) on each channel.
 * Which views are taken, the crop and the colour / resampling recipe above are exactly those of the same light field
 * stored as View_u_v files, so both give the same Lr_SAI_y / Hr_SAI_y / Sr_SAI_cbcr bit for bit.
 *
 * lfsr_image_to_views_u8: img (uint8, device) in `layout` (LFSR_LAYOUT_MOSAIC or LFSR_LAYOUT_LENSLET) -> the views
 * [u0, u0 + n_u) x [v0, v0 + n_v), each cropped top-left to hc x wc, as view-major uint8 [n_u][n_v][hc][wc][3] (the input
 * of lfsr_rgb_to_ycbcr_mosaic). A pure gather, bit-exact. LFSR_ERR_INVALID for an unknown layout, a selection outside the
 * grid, hc > H or wc > W, or an image side U*H or V*W of 2^31 or more. */
enum { LFSR_LAYOUT_VIEWS = 0, LFSR_LAYOUT_MOSAIC = 1, LFSR_LAYOUT_LENSLET = 2 };
int lfsr_image_to_views_u8(const unsigned char* img, int layout, int U, int V, int H, int W, int u0, int v0, int n_u,
                           int n_v, int hc, int wc, unsigned char* views, void* stream);

/* One separable pass of the reference's MATLAB-style imresize (utils/imresize.py:57-102 `resizeAlongDim`), fp64:
 * out[a][i][b] = sum_p weights[i][p] * in[a][indices[i][p]][b] over a tensor viewed as [outer][in_len][inner]
 * -> [outer][out_len][inner]; weights / border-reflected indices per output sample as imresize.py:32-55 builds them. */
int lfsr_resample_f64(const double* in, double* out, const double* weights, const int32_t* indices, int outer,
                      int in_len, int out_len, int inner, int taps, void* stream);

/* ---- Angular window tiling (no counterpart in the reference; DESIGN.md row f-8): every view of a light field larger than
 * the A x A a network was trained for (A = angRes), off by default (--full_grid 1).
 *   grid     N_u x N_v views of a U x V grid of views, the central ones by the rule of "View preparation"
 *            (u0 = (U - N_u) // 2, v0 = (V - N_v) // 2); A <= N_u <= U and A <= N_v <= V. By default (--grid_views '')
 *            N_u = N_v = N = min(U, V); --grid_views all takes the whole U x V, --grid_views RxC the central R x C.
 *   origins  along each angular axis independently, window_origins(N_u, A, t) and window_origins(N_v, A, t), one stride t
 *            for both, 1 <= t <= A - 1 when the axis is longer than A (default t = A - 1, the fewest windows that cover the
 *            axis): 0, t, 2t, ... while < N - A, then N - A for an axis of N views. N = A: the single origin 0. E.g.
 *            N = 9, A = 5: {0, 4}; N = 13, A = 5: {0, 4, 8}; N = 14, A = 5: {0, 4, 8, 9}.
 *   windows  the pairs (o_u, o_v) in row-major order of (o_u, o_v); that order is the summation order. N_u = N_v gives
 *            exactly the square plan.
 *   window   the LR Y mosaic of views [o_u, o_u + A) x [o_v, o_v + A) through the scene pipeline unchanged (LFdivide ->
 *            forward -> LFintegrate, with the x8 self-ensemble when it is on) -> an SR window mosaic [(A hs), (A ws)].
 *   merge    SR view (u, v) of the N_u x N_v mosaic = (((W_k1 + W_k2) + ...) + W_kc) / c over the windows k1 < k2 < ...
 *            that contain it, c = c_u * c_v their count (c_u origins along u cover u, c_v along v cover v): fp32 sums with __fadd_rn, one __fdiv_rn by (float)c; c = 1 is a plain copy. This is
 *            what torch's fp32 `a + b` then `/ c` (c as a tensor: a Python scalar divisor may become a reciprocal multiply)
 *            computes, bit for bit.
 *
 * lfsr_window_accumulate: merges one SR window mosaic `win` [(ang h)][(ang w)] into the N x N mosaic `grid` [(n h)][(n w)] at
 * view offset (o_u, o_v). host_modes[a1 * ang + a2] (a host array of ang * ang) is the step for window view (a1, a2):
 * 0 = store (the first window over that view), 1 = add, c >= 2 = add then divide by c (the last of its c windows). So the
 * merge needs no zeroing and no normalising pass. float4 loads and stores when w % 4 == 0. LFSR_ERR_INVALID for n < ang,
 * ang > 16, a window outside the grid, overlapping mosaics or a mode outside [0, min(ang, n - ang + 1)^2]. */
int lfsr_window_accumulate(const float* win, float* grid, int ang, int n, int h, int w, int o_u, int o_v,
                           const int32_t* host_modes, void* stream);
/* the same into an n_u x n_v mosaic `grid` [(n_u h)][(n_v w)]: n_u, n_v >= ang, 0 <= o_u <= n_u - ang,
 * 0 <= o_v <= n_v - ang, modes in [0, min(ang, n_u - ang + 1) * min(ang, n_v - ang + 1)]. lfsr_window_accumulate is this
 * with n_u = n_v = n. */
int lfsr_window_accumulate_uv(const float* win, float* grid, int ang, int n_u, int n_v, int h, int w, int o_u, int o_v,
                              const int32_t* host_modes, void* stream);

/* ---- convolutions --------------------------------------------------------------------- */
/* fp32 CUDA-core implicit GEMM; weights packed [kh*kw][cin][cout]. */
int lfsr_conv2d_f32(const lfsr_tensor* in, const float* w_packed, const lfsr_tensor* out,
                    const lfsr_conv_desc* d, void* stream);
/* depthwise conv (groups == channels); weights [kh*kw][c]; optional per-channel affine
 * (folded BatchNorm) then activation. */
int lfsr_dwconv_f32(const lfsr_tensor* in, const float* w_packed, const float* scale,
                    const float* shift, const lfsr_tensor* out, int kh, int kw, int dil_h, int dil_w,
                    int act, float act_slope, void* stream);
/* several depthwise branches of one input in one launch: branch b convolves the channel window
 * in[..., in_c0 : in_c0+c] with its own taps / dilation and writes out[..., out_c0 : out_c0+c]
 * ("same" zero padding, stride 1). Replaces MultiScaleSpatial's conv3/conv5/conv7 on 16-channel slices
 * (MyEfficientLFNetV4_5.py:268-280) and FastConvSSM's conv1/2/4/8 + torch.cat (:218-221, :235-240). */
typedef struct {
  const float* w;      /* [kh*kw][c] */
  const float* scale;  /* [c] folded BatchNorm, or NULL (then shift is NULL too) */
  const float* shift;
  int32_t kh, kw, dil_h, dil_w;
  int32_t in_c0, out_c0, c;
  int32_t act;
  float act_slope;
} lfsr_dw_branch;
int lfsr_dwconv_multi(const lfsr_tensor* in, const lfsr_tensor* out, const lfsr_dw_branch* branches,
                      int n_branches, void* stream);
/* out(n,y,x) = bias + res(n,y,x) + sum_{ky,kx} taps(n, y+ky-kh/2, x+kx-kw/2, ky*kw+kx), zero outside the image: the
 * second half of a kh x kw convolution to ONE channel whose per-tap responses were produced by a `tail_w` epilogue. */
int lfsr_tap_gather(const lfsr_tensor* taps, int kh, int kw, const float* bias, const lfsr_tensor* res,
                    const lfsr_tensor* out, void* stream);
/* thin dense conv on the FP32 pipe (packed FFMA2): 16/18/20 input channels read as 20-float pixels, exactly 20 output
 * channels, stride 1, "same" padding, <= 9 taps, any dilation; bias + activation (+ 20-channel multiplier) fused; weights packed as for
 * lfsr_conv2d_f32. The spatial branch of the Track-2 model (MyEfficientLFNet.py:134-141), where a K=8 tf32 MMA costs
 * the same for N=32 as for N=128 and the CUDA cores win. fp32-exact. */
int lfsr_conv2d_thin_supported(const lfsr_tensor* in, const lfsr_tensor* out, const lfsr_conv_desc* d);
int lfsr_conv2d_thin(const lfsr_tensor* in, const float* w_packed, const lfsr_tensor* out,
                     const lfsr_conv_desc* d, void* stream);
/* stems: 1 input channel -> <= 64 output channels (multiple of 4), <= 9 taps, stride 1, "same" padding; bias +
 * activation fused (MyEfficientLFNet.py:40-43, MyEfficientLFNetV4_5.py:42), optionally view-blocked (block_h / block_w: EPIT.py:24)
 * or MacPI-addressed with dilation ==
 * perm_a (DistgSSR.py:21, LF_InterNet.py:24). Weights packed as for lfsr_conv2d_f32. */
int lfsr_conv2d_stem_supported(const lfsr_tensor* in, const lfsr_tensor* out, const lfsr_conv_desc* d);
int lfsr_conv2d_stem(const lfsr_tensor* in, const float* w_packed, const lfsr_tensor* out,
                     const lfsr_conv_desc* d, void* stream);
/* fp32 1x1 conv to 8 or 16 output channels (DistgSSR's composed reconstruction tail 64 -> s^2, DistgSSR.py:24-27): dense NHWC in / out,
 * weights packed as for lfsr_conv2d_f32 ([cin][cout]); bias and activation fused. */
int lfsr_conv1x1_few_supported(const lfsr_tensor* in, const lfsr_tensor* out, const lfsr_conv_desc* d);
int lfsr_conv1x1_few(const lfsr_tensor* in, const float* w_packed, const lfsr_tensor* out, const lfsr_conv_desc* d, void* stream);
/* direct conv for 1..4 output channels (reconstruction heads 54->1 / 64->1: MyEfficientLFNet.py:70-73,
 * EPIT.py:48): stride 1, "same" padding; weights packed as for lfsr_conv2d_f32; bias/act/alpha/res fused. */
int lfsr_conv2d_small_cout_supported(const lfsr_tensor* in, const lfsr_tensor* out, const lfsr_conv_desc* d);
int lfsr_conv2d_small_cout(const lfsr_tensor* in, const float* w_packed, const lfsr_tensor* out,
                           const lfsr_conv_desc* d, void* stream);
/* MultiScaleEPIBlock (MyEfficientLFNet.py:278-327) in one pass over 18-channel splits:
 *   out = LReLU(fuse . concat_b LReLU(pw_b . dw_b(x))),  b in {1 x klen, klen x 1, 3x3 dilated `dil`}.
 * w_packed = dw_h[klen][18] | dw_v[klen][18] | dw_d[9][18] | pw_h[18 in][18 out] | pw_v | pw_d | fuse[54 in][18 out]. */
int lfsr_mel_epi_branch(const lfsr_tensor* in, const float* w_packed, const lfsr_tensor* out, int klen, int dil,
                        float slope, void* stream);
/* The same block with its four 1x1 contractions on the tensor cores (tcgen05, fp16 operands written by the CTA itself,
 * fp32 accumulation in tensor memory); the depthwise taps stay fp32 on the CUDA cores. Same arguments and weight packing;
 * results differ from lfsr_mel_epi_branch by the fp16 rounding of the contraction operands (~1e-3 relative). */
int lfsr_mel_epi_branch_tc(const lfsr_tensor* in, const float* w_packed, const lfsr_tensor* out, int klen, int dil,
                           float slope, void* stream);
/* The same block with the depthwise taps on the tensor cores as well: dw_b . pw_b is one tcgen05 MMA per tap whose A operand is
 * the fp16 input tile read at a shifted row (channels 0..15; channels 16, 17 go through the CUDA cores and one extra MMA).
 * `in16` is the fp16 copy of `in` (ptr = __half*, the same 18 channels; the 6 halves behind them must be readable inside the pixel,
 * i.e. the slice starts at least 24 halves before the end of a pixel row) that the producer of `in` wrote: the tile is two TMA loads.
 * lfsr_mel_epi_pack (host) turns w_packed into the pre-swizzled operand image the kernel loads with one bulk copy;
 * lfsr_mel_epi_pack_bytes is its size (0: this kernel length is not supported, use lfsr_mel_epi_branch_tc). */
size_t lfsr_mel_epi_pack_bytes(int klen);
int lfsr_mel_epi_pack(const float* w_packed_host, void* image_host, int klen);
int lfsr_mel_epi_branch_mma(const lfsr_tensor* in, const lfsr_tensor* in16, const void* image_dev, const lfsr_tensor* out, int klen,
                            int dil, float slope, void* stream);
/* TF32 tcgen05/TMEM implicit GEMM fed by TMA (sm_100a); weights packed by lfsr_pack_conv_tc.
 * Supports stride 1 (any dilation, "same" zero padding given by pad) and kh*kw <= 25. */
size_t lfsr_conv2d_tc_packed_floats(int kh, int kw, int cin, int cout);
int lfsr_pack_conv_tc(const float* w_oihw_host, float* packed_host, int kh, int kw, int cin, int cout);
/* x = hi + lo with hi = x rounded to TF32 (exactly representable, so the tensor-core path reads it unchanged) and lo the
 * remainder: conv(hi, w_hi) + conv(lo, w_hi) + conv(hi, w_lo) on the TF32 tensor cores equals the fp32 convolution to ~2^-21.
 * Used for the last, image-producing convolution of LF-InterNet, whose rounding error would otherwise reach the output directly.
 * Dense buffers of n floats. */
int lfsr_split_tf32(const float* in, float* hi, float* lo, long long n, void* stream);
/* MacPI2SAI + PixelShuffle(r) of a 1-channel reconstruction (DistgSSR.py:34-35, LF_InterNet.py:137-141 after the algebraic
 * composition of the last two layers, DESIGN.md 5): in [n, H, W, r*r] holds, for the MacPI pixel (i*A+u, j*A+v), the r x r
 * sub-pixel values of SAI pixel (u*H/A + i, v*W/A + j); out [n, H*r, W*r] is the high-resolution SAI image. accumulate != 0
 * adds onto `out` (the interpolation skip already there). Lets the reconstruction conv run on the tensor cores, which do not
 * address MacPI-permuted outputs. r in {2, 4}. */
int lfsr_macpi_unshuffle(const lfsr_tensor* in, float* out, int ang, int r, int accumulate, void* stream);
/* fp32 NHWC tensor -> its fp16 copy (round to nearest even): the operand copy of a tensor that did not come out of a
 * tensor-core epilogue (stems). Channel count a multiple of 8. */
int lfsr_to_f16(const lfsr_tensor* in, const lfsr_tensor* out16, void* stream);
size_t lfsr_conv2d_tc16_packed_bytes(int kh, int kw, int cin, int cout);
int lfsr_pack_conv_tc16(const float* w_oihw_host, void* packed_host, int kh, int kw, int cin, int cout);
int lfsr_conv2d_tc(const lfsr_tensor* in, const float* w_packed_tc, const lfsr_tensor* out,
                   const lfsr_conv_desc* d, void* stream);
/* per-image weight sets for a gated conv: out[img] = packed * gate[img][cin] along the input-channel axis
 * (MyEfficientLFNet.py:193-199: the branch gates multiply the concat before the fusion 1x1). `packed` is the
 * lfsr_pack_conv_tc buffer, `out` holds n copies of it. */
int lfsr_scale_pack_tc(const float* packed, const float* gate, int64_t gate_ld, float* out, int n, int kh, int kw,
                       int cin, int cout, void* stream);
/* 1 if lfsr_conv2d_tc can run this problem (geometry/alignment), else 0 */
int lfsr_conv2d_tc_supported(const lfsr_tensor* in, const lfsr_tensor* out, const lfsr_conv_desc* d);

/* ---- reductions / gates (MyEfficientLFNet.py:159-173, 471-515) ---------------------------- */
/* mean over each (block_h x block_w) block: in [n,h,w,c] -> out [n, h/block_h, w/block_w, c] */
int lfsr_block_mean(const lfsr_tensor* in, const lfsr_tensor* out, int block_h, int block_w,
                    void* stream);
/* Chains of 1x1 convolutions on a handful of positions per image, one launch per chain: the channel gates of a Track-2 stage
 * (MyEfficientLFNet.py:159-173: AdaptiveAvgPool -> 1x1 + bias -> sigmoid; pool = 1) and the angular half of the SA modulator
 * (:505-511: 1x1 -> ReLU -> 1x1 -> sigmoid on the per-view means; pool = 0).
 *   x = pool ? mean over the h*w positions of `in` : in;  h = act1(b1 + x . w1);  out = w2 ? act2(b2 + h . w2) : h
 * w1 is [in->c][c1], w2 [c1][c2] (the lfsr_conv2d_f32 packing of a 1x1 kernel); b1 / b2 / w2 may be null. */
int lfsr_pooled_mlp(const lfsr_tensor* in, int pool, const float* w1, const float* b1, int c1, int act1, const float* w2,
                    const float* b2, int c2, int act2, const lfsr_tensor* out, void* stream);
/* AngularAttention.expand + PixelShuffle(A) + activation, * alpha, + residual (MyEfficientLFNet.py:262-275) as one streaming
 * kernel: out[n, A*Y+i, A*X+j, c] = res[...] + alpha * act(sum_k in[n, Y, X, k] * w[i][j][k][c]).
 * w is [A][A][in->c][out->c] (out->c a multiple of 4: pad channels carry zero weights); in->c is 16, 18 or 20; res may be null. */
int lfsr_ang_expand(const lfsr_tensor* in, const float* w, const lfsr_tensor* res, const lfsr_tensor* out, int A, int act,
                    float slope, float alpha, void* stream);
/* SAModulator tail (MyEfficientLFNet.py:495-515) fused with the stage residual:
 *   s = sigmoid(bn_scale*dw3x3_dil(x) + bn_shift); a = amod[n][y/(h/A)][x/(w/A)][c]
 *   out = x * (w0*s + w1*a) + res */
int lfsr_sa_modulate(const lfsr_tensor* x, const float* dw_w, const float* bn_scale,
                     const float* bn_shift, const lfsr_tensor* amod, float w0, float w1,
                     const lfsr_tensor* res, const lfsr_tensor* out, int dil, void* stream);

/* the same, plus an fp16 copy of output channels [0, out16->c) (fp16 NHWC view, c a multiple of 4): the operand of the
 * tensor-core layers that read this trunk next (Track-2 spatial branch). Tiled kernel only; errors when it does not apply. */
int lfsr_sa_modulate16(const lfsr_tensor* x, const float* dw_w, const float* bn_scale,
                       const float* bn_shift, const lfsr_tensor* amod, float w0, float w1,
                       const lfsr_tensor* res, const lfsr_tensor* out, const lfsr_tensor* out16, int dil, void* stream);
/* the same, leaving channels [skip_lo, skip_hi) (whole quads) out of the fp16 copy: the Track-2 plan keeps ONE fp16 copy of the
 * trunk of which only channels 0..17 (spatial branch) and 40..57 (EPI branch) are ever read */
int lfsr_sa_modulate16w(const lfsr_tensor* x, const float* dw_w, const float* bn_scale, const float* bn_shift,
                        const lfsr_tensor* amod, float w0, float w1, const lfsr_tensor* res, const lfsr_tensor* out,
                        const lfsr_tensor* out16, int skip_lo, int skip_hi, int dil, void* stream);

/* out = x * scale[n][c] + res  (ChannelAttention + block residual, MyEfficientLFNetV4_5.py:148,291-299);
 * scale is an [n,1,1,c] tensor view, res may be NULL. */
int lfsr_scale_add(const lfsr_tensor* x, const lfsr_tensor* scale, const lfsr_tensor* res, const lfsr_tensor* out,
                   void* stream);
/* the same with an fp16 result (a tensor that only a tensor-core layer reads): out16->ptr is __half*, ld in halves, c % 8 == 0 */
int lfsr_scale_add16(const lfsr_tensor* x, const lfsr_tensor* scale, const lfsr_tensor* res, const lfsr_tensor* out16,
                     void* stream);

/* ---- EPIT token ops (EPIT.py:74-128) ------------------------------------------------------ */
/* LayerNorm over c (eps, affine) for every pixel/token */
int lfsr_layernorm(const lfsr_tensor* in, const float* gamma, const float* beta, float eps,
                   const lfsr_tensor* out, void* stream);
/* band-masked multi-head attention over EPI sequences. qk: [T, 2E] (q | k), v: [T, E], out [T,E];
 * tokens are addressed token(seq, a, s) = seq_base(seq) + a*stride_a + s*stride_s with
 * a in [0,A), s in [0,S): key (a',s') allowed iff |s - s'| <= half_window (EPIT.py:93-108 with
 * mask_field [2A, 11]). seq enumerates (b, p, q): seq_base = b*stride_b + p*stride_p + q*stride_q */
typedef struct {
  int32_t heads, head_dim;
  int32_t A, S, half_window;
  int32_t nb, np, nq;
  int64_t stride_a, stride_s, stride_b, stride_p, stride_q; /* in tokens */
} lfsr_epi_attn_desc;
int lfsr_epi_attention(const float* qk, const float* v, float* out, const lfsr_epi_attn_desc* d,
                       void* stream);

/* ---- EPIT BasicTrans, fused (EPIT.py:74-128: linear_in -> LayerNorm -> MultiheadAttention(q = k = norm(x), v = x, 8 heads,
 * additive band mask of :93-108) + x -> LayerNorm -> Linear/ReLU/Linear + x -> linear_out) ----------------------------------
 * ONE tcgen05/TMEM kernel: a CTA owns a run of query positions of one EPI sequence plus the +-half_window positions they
 * attend (all A angular rows), <= 112 token rows; every intermediate stays in TMEM / shared memory, fp16 operands with fp32
 * accumulation, weights streamed by TMA. Sequences and tokens are addressed exactly like
 * lfsr_epi_attention: token(seq, a, s) = seq_base + a*stride_a + s*stride_s, seq_base = b*stride_b + p*stride_p + q*stride_q,
 * in pixels of the [n,h,w,64] NHWC tensors x (in) and y (out, same geometry, must not alias x). BOTH ARE FP16 views (ld in
 * 2-byte elements, multiple of 8): x is the fp16 operand copy of the fp32 feature trunk (lfsr_conv_desc.out_mode / lfsr_to_f16),
 * y only ever feeds the next tensor-core convolution. E = 128, C = 64, 8 heads. */
typedef struct {
  int32_t A, S, half_window, heads, E, C;
  int32_t nb, np, nq;
  int64_t stride_a, stride_s, stride_b, stride_p, stride_q;
  float eps1, eps2;                                           /* of the two LayerNorms (host values) */
  float ln1_g[128], ln1_b[128], ln2_g[128], ln2_b[128];       /* LayerNorm affine parameters (host values) */
} lfsr_basictrans_desc;
size_t lfsr_basictrans_packed_bytes(void);
/* host weights in torch layout [out][in]: linear_in [128][64], attention.in_proj_weight [384][128], attention.out_proj
 * [128][128], feed_forward.1 [256][128], feed_forward.4 [128][256], linear_out [64][128] -> packed_host (then copied to
 * the device by the caller) */
int lfsr_pack_basictrans(const float* w_in, const float* w_qkv, const float* w_o, const float* w_ff1, const float* w_ff2,
                         const float* w_out, void* packed_host);
int lfsr_basictrans_supported(const lfsr_tensor* x, const lfsr_tensor* y, const lfsr_basictrans_desc* d);
int lfsr_epit_basictrans(const lfsr_tensor* x, const void* packed_dev, const lfsr_tensor* y, const lfsr_basictrans_desc* d,
                         void* stream);

/* ---- metrics (utils/utils.py:91-134) ------------------------------------------------------ */
/* per-view sums for PSNR/SSIM on SAI mosaics label/out [A*h, A*w] (row stride = A*w):
 * acc[view] = { sum (a-b)^2 , sum SSIM map over the 5-px-cropped interior } as float64.
 * acc must be zeroed by the caller (cudaMemsetAsync) - 2*A*A doubles. */
int lfsr_metric_sums(const float* label, const float* out, int ang, int h, int w, double* acc,
                     void* stream);
/* the same for n mosaics stored back to back (a [n,1,A*h,A*w] batch of SR patches against their HR patches, BASELINE
 * config 5: on-GPU evaluation of a large batch): acc[(img*A*A + view)] = {sum sq. err, sum SSIM}, 2*n*A*A doubles, zeroed
 * by the caller. */
int lfsr_metric_sums_batched(const float* label, const float* out, int n, int ang, int h, int w, double* acc,
                             void* stream);
/* the same for an ang_u x ang_v mosaic [(ang_u h)][(ang_v w)] (row stride ang_v * w): acc[a1 * ang_v + a2] = {sum sq. err,
 * sum SSIM}, 2 * ang_u * ang_v doubles, zeroed by the caller. lfsr_metric_sums is this with ang_u = ang_v = ang, and
 * lfsr_metric_sums_batched with ang_u = n * ang, ang_v = ang. */
int lfsr_metric_sums_uv(const float* label, const float* out, int ang_u, int ang_v, int h, int w, double* acc,
                        void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LFSR_B200_H_ */
