// image.cu -- the OpenCV image stages of Pipeline.recognize as CUDA kernels, bit-compatible with
// OpenCV 4.x fixed-point arithmetic (models of the arithmetic are pinned against cv2 in
// tests/test_cv_models.py):
//   resize_pad_kernel : cv2.resize INTER_LINEAR on uint8 (tools.py:394-396) + tools.pad(255) (356-375)
//   gray_kernel       : cv2.cvtColor(RGB2GRAY) (recognition.py:510)
//   fit_crops_kernel  : tools.fit(cval=0) (tools.py:402-452) + cvtColor of ragged crops for Recognizer.recognize
//   warp_kernel       : tools.warpBox (tools.py:61-117): get_rotated_box ordering (533-581, rectangle
//                       branch), get_rotated_width_height (41-57), cv2.getPerspectiveTransform (8x8 LU,
//                       fp64), cv2.warpPerspective INTER_LINEAR (1/32-pixel coordinates, 15-bit weights)
#include <math.h>

#include "common.cuh"

namespace {

// ------------------------------------------------------------------------------------ resize + pad
// blockIdx.z = image of a batch of equally sized sources (strides 0 for the one-image entry point); `gray`,
// when given, also receives cv2.cvtColor(RGB2GRAY) of the padded result (recognition.py:510), which saves the
// recognizer a second pass over the batch.
__device__ __forceinline__ uint8_t gray_of(int r, int g, int b) {
  return static_cast<uint8_t>((9798 * r + 19235 * g + 3735 * b + 16384) >> 15);
}

// cv2.resize INTER_LINEAR on uint8 at output pixel (x, y) of an RGB source (hs, ws): OpenCV's scale = 1 / (dsize /
// ssize), source coordinate at pixel centres, float fractions, 11-bit coefficients (INTER_RESIZE_COEF_BITS),
// horizontal pass first.  One row or one column is fine: the clamps keep every read inside the source.
__device__ __forceinline__ void resize_sample(const uint8_t* __restrict__ src, int hs, int ws, int x, int y,
                                              double scale_x, double scale_y, int rgb[3]) {
  float fx = static_cast<float>((x + 0.5) * scale_x - 0.5);
  int sx = static_cast<int>(floorf(fx));
  fx -= sx;
  if (sx < 0) { fx = 0.f; sx = 0; }
  if (sx >= ws - 1) { fx = 0.f; sx = ws - 1; }
  const int sx1 = min(sx + 1, ws - 1);
  const int a0 = __float2int_rn((1.f - fx) * 2048.f), a1 = __float2int_rn(fx * 2048.f);
  float fy = static_cast<float>((y + 0.5) * scale_y - 0.5);
  const int sy = static_cast<int>(floorf(fy));
  fy -= sy;
  const int b0 = __float2int_rn((1.f - fy) * 2048.f), b1 = __float2int_rn(fy * 2048.f);
  const int y0 = min(max(sy, 0), hs - 1), y1 = min(max(sy + 1, 0), hs - 1);
  const uint8_t* r0 = src + static_cast<size_t>(y0) * ws * 3;
  const uint8_t* r1 = src + static_cast<size_t>(y1) * ws * 3;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int s0 = r0[sx * 3 + c] * a0 + r0[sx1 * 3 + c] * a1;
    const int s1 = r1[sx * 3 + c] * a0 + r1[sx1 * 3 + c] * a1;
    const int v = (((b0 * (s0 >> 4)) >> 16) + ((b1 * (s1 >> 4)) >> 16) + 2) >> 2;
    rgb[c] = min(max(v, 0), 255);
  }
}

// scale_x / scale_y = 1 / (dsize / ssize) in fp64, computed once on the host exactly as OpenCV does: two fp64
// divisions per pixel cost more than everything else in this kernel.
__global__ void resize_pad_kernel(const uint8_t* __restrict__ src, int hs, int ws, int hr, int wr,
                                  uint8_t* __restrict__ dst, int hp, int wp, uint8_t* __restrict__ gray,
                                  double scale_x, double scale_y) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  if (x >= wp) return;
  src += static_cast<size_t>(blockIdx.z) * hs * ws * 3;
  const size_t opix = (static_cast<size_t>(blockIdx.z) * hp + y) * wp + x;
  uint8_t* o = dst + opix * 3;
  if (x >= wr || y >= hr) {
    o[0] = 255; o[1] = 255; o[2] = 255;
    if (gray) gray[opix] = gray_of(255, 255, 255);
    return;
  }
  int rgb[3];
  resize_sample(src, hs, ws, x, y, scale_x, scale_y, rgb);
#pragma unroll
  for (int c = 0; c < 3; ++c) o[c] = static_cast<uint8_t>(rgb[c]);
  if (gray) gray[opix] = gray_of(rgb[0], rgb[1], rgb[2]);
}

// ------------------------------------------------------------------------------------ RGB -> gray
__global__ void gray_kernel(const uint8_t* __restrict__ img, long long total, uint8_t* __restrict__ gray) {
  const long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= total) return;
  const uint8_t* q = img + p * 3;
  gray[p] = gray_of(q[0], q[1], q[2]);
}

// ------------------------------------------------------------------------------------ warpBox
struct WarpPlan {
  double m[9];     // inverse homography (destination -> source), fp64 like cv2
  int dw, dh;      // dsize of warpPerspective
  int valid;
};

__device__ double dist2(const float* a, const float* b) {
  const double dx = static_cast<double>(a[0]) - static_cast<double>(b[0]);
  const double dy = static_cast<double>(a[1]) - static_cast<double>(b[1]);
  return sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
}

__device__ void plan_warp(const float* q /*4x2*/, int target_w, int target_h, WarpPlan* plan) {
  plan->valid = 0;
  // --- get_rotated_box on a rectangle: stable sort by x, split, order by y / by distance ---------
  int idx[4] = {0, 1, 2, 3};
  for (int i = 1; i < 4; ++i) {              // insertion sort == numpy's small-array argsort (stable)
    const int v = idx[i];
    int j = i - 1;
    while (j >= 0 && q[2 * idx[j]] > q[2 * v]) { idx[j + 1] = idx[j]; --j; }
    idx[j + 1] = v;
  }
  int l0 = idx[0], l1 = idx[1], r0 = idx[2], r1 = idx[3];
  if (q[2 * l0 + 1] > q[2 * l1 + 1]) { const int t = l0; l0 = l1; l1 = t; }
  const int tl = l0, bl = l1;
  const double d0 = dist2(q + 2 * tl, q + 2 * r0), d1 = dist2(q + 2 * tl, q + 2 * r1);
  // (br, tr) = rightMost[argsort(D)[::-1]]
  int br, tr;
  if (d0 <= d1) { br = r1; tr = r0; } else { br = r0; tr = r1; }
  float box[8] = {q[2 * tl], q[2 * tl + 1], q[2 * tr], q[2 * tr + 1], q[2 * br], q[2 * br + 1], q[2 * bl], q[2 * bl + 1]};
  // --- get_rotated_width_height --------------------------------------------------------------------
  const int w = static_cast<int>((dist2(box + 0, box + 2) + dist2(box + 4, box + 6)) / 2);
  const int h = static_cast<int>((dist2(box + 0, box + 6) + dist2(box + 2, box + 4)) / 2);
  if (w <= 0 || h <= 0) return;              // the reference raises ZeroDivisionError here
  const double sa = static_cast<double>(target_w) / w, sb = static_cast<double>(target_h) / h;
  const double scale = sa < sb ? sa : sb;
  const double sw = scale * w, sh = scale * h;
  const float dst[8] = {0.f, 0.f, static_cast<float>(sw), 0.f, static_cast<float>(sw), static_cast<float>(sh),
                        0.f, static_cast<float>(sh)};
  plan->dw = static_cast<int>(sw);
  plan->dh = static_cast<int>(sh);
  // --- cv2.getPerspectiveTransform: 8x8 system, LU with partial pivoting in fp64 -----------------
  double A[8][8], b[8];
  for (int i = 0; i < 4; ++i) {
    const double sxx = box[2 * i], syy = box[2 * i + 1], dx = dst[2 * i], dy = dst[2 * i + 1];
    for (int k = 0; k < 8; ++k) { A[i][k] = 0.0; A[i + 4][k] = 0.0; }
    A[i][0] = A[i + 4][3] = sxx;
    A[i][1] = A[i + 4][4] = syy;
    A[i][2] = A[i + 4][5] = 1.0;
    A[i][6] = __dmul_rn(-sxx, dx);
    A[i][7] = __dmul_rn(-syy, dx);
    A[i + 4][6] = __dmul_rn(-sxx, dy);
    A[i + 4][7] = __dmul_rn(-syy, dy);
    b[i] = dx;
    b[i + 4] = dy;
  }
  for (int i = 0; i < 8; ++i) {
    int k = i;
    for (int j = i + 1; j < 8; ++j)
      if (fabs(A[j][i]) > fabs(A[k][i])) k = j;
    if (fabs(A[k][i]) < 2.220446049250313e-14) return;     // DBL_EPSILON*100: singular
    if (k != i) {
      for (int j = i; j < 8; ++j) { const double t = A[i][j]; A[i][j] = A[k][j]; A[k][j] = t; }
      const double t = b[i]; b[i] = b[k]; b[k] = t;
    }
    const double d = -1.0 / A[i][i];
    for (int j = i + 1; j < 8; ++j) {
      const double alpha = __dmul_rn(A[j][i], d);
      for (int kk = i + 1; kk < 8; ++kk) A[j][kk] = __dadd_rn(A[j][kk], __dmul_rn(alpha, A[i][kk]));
      b[j] = __dadd_rn(b[j], __dmul_rn(alpha, b[i]));
    }
  }
  for (int i = 7; i >= 0; --i) {
    double s = b[i];
    for (int kk = i + 1; kk < 8; ++kk) s = __dsub_rn(s, __dmul_rn(A[i][kk], b[kk]));
    b[i] = s / A[i][i];
  }
  const double M[9] = {b[0], b[1], b[2], b[3], b[4], b[5], b[6], b[7], 1.0};
  // --- cv::invert of a 3x3 (closed form) -----------------------------------------------------------
#define MM(r, c) M[(r) * 3 + (c)]
#define DET2(a, b, c, d) __dsub_rn(__dmul_rn(a, b), __dmul_rn(c, d))
  const double det = __dadd_rn(
      __dsub_rn(__dmul_rn(MM(0, 0), DET2(MM(1, 1), MM(2, 2), MM(1, 2), MM(2, 1))),
                __dmul_rn(MM(0, 1), DET2(MM(1, 0), MM(2, 2), MM(1, 2), MM(2, 0)))),
      __dmul_rn(MM(0, 2), DET2(MM(1, 0), MM(2, 1), MM(1, 1), MM(2, 0))));
  if (det == 0.0) return;
  const double id = 1.0 / det;
  plan->m[0] = __dmul_rn(DET2(MM(1, 1), MM(2, 2), MM(1, 2), MM(2, 1)), id);
  plan->m[1] = __dmul_rn(DET2(MM(0, 2), MM(2, 1), MM(0, 1), MM(2, 2)), id);
  plan->m[2] = __dmul_rn(DET2(MM(0, 1), MM(1, 2), MM(0, 2), MM(1, 1)), id);
  plan->m[3] = __dmul_rn(DET2(MM(1, 2), MM(2, 0), MM(1, 0), MM(2, 2)), id);
  plan->m[4] = __dmul_rn(DET2(MM(0, 0), MM(2, 2), MM(0, 2), MM(2, 0)), id);
  plan->m[5] = __dmul_rn(DET2(MM(0, 2), MM(1, 0), MM(0, 0), MM(1, 2)), id);
  plan->m[6] = __dmul_rn(DET2(MM(1, 0), MM(2, 1), MM(1, 1), MM(2, 0)), id);
  plan->m[7] = __dmul_rn(DET2(MM(0, 1), MM(2, 0), MM(0, 0), MM(2, 1)), id);
  plan->m[8] = __dmul_rn(DET2(MM(0, 0), MM(1, 1), MM(0, 1), MM(1, 0)), id);
#undef MM
#undef DET2
  plan->valid = 1;
}

// CH = 1: gray image (n,H,W), crops (k,ch,cw), CRNN input (k,cw,ch).  CH = 3 (build_model(color=True),
// recognition.py:214, 508-510: no gray conversion): RGB image (n,H,W,3), crops (k,ch,cw,3), CRNN input (k,cw,ch,3);
// cv2.warpPerspective samples every channel with the same coordinates and weights.  (ch, cw) = the recognizer's crop
// size (31 x 200 by default); the crop is staged in dynamic shared memory (ch * cw * CH bytes).
template <int CH>
__global__ void __launch_bounds__(256)
warp_kernel(const uint8_t* __restrict__ gray, int n, int H, int W, const float* __restrict__ boxes,
            const int* __restrict__ image_index, int crop_h, int crop_w, uint8_t* __restrict__ crops,
            __half* __restrict__ crnn_in) {
  __shared__ WarpPlan plan;
  extern __shared__ uint8_t tile[];
  const int k = blockIdx.x;
  if (threadIdx.x == 0) plan_warp(boxes + static_cast<size_t>(k) * 8, crop_w, crop_h, &plan);
  __syncthreads();
  int img = image_index[k];
  img = min(max(img, 0), n - 1);
  const uint8_t* g = gray + static_cast<size_t>(img) * H * W * CH;
  const int dw = plan.valid ? min(plan.dw, crop_w) : 0, dh = plan.valid ? min(plan.dh, crop_h) : 0;
  // block structure of cv::WarpPerspectiveInvoker (decides where X0/Y0/W0 are re-based)
  int bh0 = min(16, max(dh, 1));
  const int bw0 = min(1024 / bh0, max(dw, 1));
  for (int i = threadIdx.x; i < crop_h * crop_w; i += blockDim.x) {
    const int y = i / crop_w, x = i - y * crop_w;
    int v[CH];
#pragma unroll
    for (int c = 0; c < CH; ++c) v[c] = 0;
    if (x < dw && y < dh) {
      const double* m = plan.m;
      const int bx = (x / bw0) * bw0, x1 = x - bx;
      const double X0 = __dadd_rn(__dadd_rn(__dmul_rn(m[0], bx), __dmul_rn(m[1], y)), m[2]);
      const double Y0 = __dadd_rn(__dadd_rn(__dmul_rn(m[3], bx), __dmul_rn(m[4], y)), m[5]);
      const double W0 = __dadd_rn(__dadd_rn(__dmul_rn(m[6], bx), __dmul_rn(m[7], y)), m[8]);
      double Wv = __dadd_rn(W0, __dmul_rn(m[6], x1));
      Wv = Wv != 0.0 ? 32.0 / Wv : 0.0;
      const double fX = fmax(-2147483648.0, fmin(2147483647.0, __dmul_rn(__dadd_rn(X0, __dmul_rn(m[0], x1)), Wv)));
      const double fY = fmax(-2147483648.0, fmin(2147483647.0, __dmul_rn(__dadd_rn(Y0, __dmul_rn(m[3], x1)), Wv)));
      const int X = __double2int_rn(fX), Y = __double2int_rn(fY);
      const int sx = min(max(X >> 5, -32768), 32767), sy = min(max(Y >> 5, -32768), 32767);
      const int ax = X & 31, ay = Y & 31;
      const bool x0ok = sx >= 0 && sx < W, x1ok = sx + 1 >= 0 && sx + 1 < W;
      const bool y0ok = sy >= 0 && sy < H, y1ok = sy + 1 >= 0 && sy + 1 < H;
      // BilinearTab_i: (1-fx)(1-fy) ... scaled to 2^15; exact for 1/32 steps
      const int w00 = (32 - ax) * (32 - ay) * 32, w01 = ax * (32 - ay) * 32;
      const int w10 = (32 - ax) * ay * 32, w11 = ax * ay * 32;
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        const int p00 = (x0ok && y0ok) ? g[(static_cast<size_t>(sy) * W + sx) * CH + c] : 0;
        const int p01 = (x1ok && y0ok) ? g[(static_cast<size_t>(sy) * W + sx + 1) * CH + c] : 0;
        const int p10 = (x0ok && y1ok) ? g[(static_cast<size_t>(sy + 1) * W + sx) * CH + c] : 0;
        const int p11 = (x1ok && y1ok) ? g[(static_cast<size_t>(sy + 1) * W + sx + 1) * CH + c] : 0;
        v[c] = (p00 * w00 + p01 * w01 + p10 * w10 + p11 * w11 + 16384) >> 15;
      }
    }
#pragma unroll
    for (int c = 0; c < CH; ++c) {
      tile[i * CH + c] = static_cast<uint8_t>(v[c]);
      if (crops) crops[(static_cast<size_t>(k) * crop_h * crop_w + i) * CH + c] = static_cast<uint8_t>(v[c]);
    }
  }
  if (crnn_in == nullptr) return;
  __syncthreads();
  // CRNN input layout (recognition.py:215-216): x[t][j] = crop[ch-1-j][t] / 255
  __half* o = crnn_in + static_cast<size_t>(k) * crop_h * crop_w * CH;
  for (int i = threadIdx.x; i < crop_h * crop_w * CH; i += blockDim.x) {
    const int c = i % CH, q = i / CH;
    const int t = q / crop_h, j = q - t * crop_h;
    o[i] = __float2half_rn(static_cast<float>(tile[((crop_h - 1 - j) * crop_w + t) * CH + c]) / 255.0f);
  }
}

// CRNN input layout (recognition.py:215-216, Permute((2,1,3)) and the axis flip): pixel q = t * crop_h + j of a crop's
// (crop_w, crop_h) input plane reads crop pixel (y, x) = (crop_h - 1 - j, t).
__device__ __forceinline__ int crnn_in_source_pixel(int q, int crop_h, int crop_w) {
  const int t = q / crop_h, j = q - t * crop_h;
  return (crop_h - 1 - j) * crop_w + t;
}

// crops (k,crop_h,crop_w[,ch]) u8 -> CRNN input (k,crop_w,crop_h[,ch]) fp16 = crop / 255 after Permute((2,1,3)) and the
// axis flip
__global__ void crops_to_input_kernel(const uint8_t* __restrict__ crops, long long total, int ch, int crop_h, int crop_w,
                                      __half* __restrict__ out) {
  const long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= total) return;
  const int per = crop_h * crop_w * ch;
  const long long k = p / per;
  const int i = static_cast<int>(p - k * per);
  const int c = i % ch;
  out[p] = __float2half_rn(static_cast<float>(crops[k * per + crnn_in_source_pixel(i / ch, crop_h, crop_w) * ch + c]) / 255.0f);
}

// ------------------------------------------------------------------------------------ tools.fit of ragged crops
// Recognizer.recognize's host preparation (recognition.py:467-489: tools.read_and_fit(cval=0), tools.py:402-452, then
// cvtColor for a gray model) for b RGB crops of any size, one block per crop.  dims[k] = (sh, sw, rh, rw): the
// source size and the cv2.resize dsize tools.fit picks (tools.fit_plan; rh == sh and rw == sw when fit does not
// resize).  Pixels inside rh x rw are resize_pad_kernel's sample, the rest of the crop_h x crop_w crop is 0.  Writes
// the CRNN input (b,crop_w,crop_h[,CH]) in crnn_in_source_pixel order -- CH = 1: gray_of the fitted pixel, CH = 3: RGB
// -- and, when given, the fitted RGB crops (b,crop_h,crop_w,3), i.e. what tools.fit returns.
template <int CH>
__global__ void __launch_bounds__(256)
fit_crops_kernel(const uint8_t* const* __restrict__ srcs, const int32_t* __restrict__ dims, int crop_h, int crop_w,
                 uint8_t* __restrict__ crops, __half* __restrict__ crnn_in) {
  __shared__ double scale[2];
  const int k = blockIdx.x;
  const int sh = dims[4 * k], sw = dims[4 * k + 1], rh = dims[4 * k + 2], rw = dims[4 * k + 3];
  const bool valid = sh > 0 && sw > 0 && rh > 0 && rw > 0;
  const bool copy = rh == sh && rw == sw;            // cv2.resize copies when dsize == ssize
  if (threadIdx.x == 0 && valid) {                   // once per crop: fp64 divisions are slow (see resize_pad_kernel)
    scale[0] = 1.0 / (static_cast<double>(rw) / sw);
    scale[1] = 1.0 / (static_cast<double>(rh) / sh);
  }
  __syncthreads();
  const uint8_t* src = srcs[k];
  const int vh = valid ? min(rh, crop_h) : 0, vw = valid ? min(rw, crop_w) : 0;
  const size_t base = static_cast<size_t>(k) * crop_h * crop_w;
  for (int q = threadIdx.x; q < crop_h * crop_w; q += blockDim.x) {
    const int pix = crnn_in_source_pixel(q, crop_h, crop_w);
    const int y = pix / crop_w, x = pix - y * crop_w;
    int rgb[3] = {0, 0, 0};
    if (y < vh && x < vw) {
      if (copy) {
        const uint8_t* s = src + (static_cast<size_t>(y) * sw + x) * 3;
        rgb[0] = s[0]; rgb[1] = s[1]; rgb[2] = s[2];
      } else {
        resize_sample(src, sh, sw, x, y, scale[0], scale[1], rgb);
      }
    }
    if (crops) {
      uint8_t* o = crops + (base + pix) * 3;
      o[0] = static_cast<uint8_t>(rgb[0]); o[1] = static_cast<uint8_t>(rgb[1]); o[2] = static_cast<uint8_t>(rgb[2]);
    }
    __half* o = crnn_in + (base + q) * CH;
    if (CH == 1) {
      o[0] = __float2half_rn(static_cast<float>(gray_of(rgb[0], rgb[1], rgb[2])) / 255.0f);
    } else {
#pragma unroll
      for (int c = 0; c < CH; ++c) o[c] = __float2half_rn(static_cast<float>(rgb[c]) / 255.0f);
    }
  }
}

}  // namespace

extern "C" int b2o_resize_pad(b2o_ctx* ctx, const uint8_t* src, int hs, int ws, int hr, int wr, uint8_t* dst,
                              int index, int hp, int wp, void* stream) {
  if (!ctx) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  if (!src || !dst || hs <= 0 || ws <= 0 || hr <= 0 || wr <= 0 || hr > hp || wr > wp || index < 0) {
    ctx->set_error("b2o_resize_pad: bad argument (resized image must fit the padded size)");
    return B2O_ERR_ARG;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  resize_pad_kernel<<<dim3((wp + 127) / 128, hp), 128, 0, st>>>(src, hs, ws, hr, wr,
                                                                dst + static_cast<size_t>(index) * hp * wp * 3, hp, wp,
                                                                nullptr, 1.0 / (static_cast<double>(wr) / ws),
                                                                1.0 / (static_cast<double>(hr) / hs));
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}

extern "C" int b2o_resize_pad_batch(b2o_ctx* ctx, const uint8_t* src, int n, int hs, int ws, int hr, int wr,
                                    uint8_t* dst, int hp, int wp, uint8_t* gray, void* stream) {
  if (!ctx) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  if (!src || !dst || n <= 0 || n > 65535 || hs <= 0 || ws <= 0 || hr <= 0 || wr <= 0 || hr > hp || wr > wp || hp > 65535) {
    ctx->set_error("b2o_resize_pad_batch: bad argument (resized image must fit the padded size)");
    return B2O_ERR_ARG;
  }
  resize_pad_kernel<<<dim3((wp + 127) / 128, hp, n), 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      src, hs, ws, hr, wr, dst, hp, wp, gray, 1.0 / (static_cast<double>(wr) / ws), 1.0 / (static_cast<double>(hr) / hs));
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}

extern "C" int b2o_rgb_to_gray(b2o_ctx* ctx, const uint8_t* img, int n, int h, int w, uint8_t* gray, void* stream) {
  if (!ctx) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  if (!img || !gray || n <= 0 || h <= 0 || w <= 0) { ctx->set_error("b2o_rgb_to_gray: bad argument"); return B2O_ERR_ARG; }
  const long long total = static_cast<long long>(n) * h * w;
  gray_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(img, total, gray);
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}

static int warp_boxes_impl(b2o_ctx* ctx, const uint8_t* img, int ch, int n, int h, int w, const float* boxes,
                           const int32_t* image_index, int n_boxes, uint8_t* crops, void* crnn_in, void* stream) {
  if (!ctx) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  if (n_boxes == 0) return B2O_OK;
  if (!img || !boxes || !image_index || n <= 0 || h <= 0 || w <= 0 || n_boxes < 0 || (!crops && !crnn_in)) {
    ctx->set_error("b2o_warp_boxes: bad argument");
    return B2O_ERR_ARG;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int chh = ctx->crnn_geom.height, cw = ctx->crnn_geom.width;
  const size_t smem = static_cast<size_t>(chh) * cw * ch;
  const void* fn = ch == 3 ? reinterpret_cast<const void*>(warp_kernel<3>) : reinterpret_cast<const void*>(warp_kernel<1>);
  if (smem > 48 * 1024 && !ctx->configured.count(fn)) {      // crops past 48 KB (e.g. 64 x 800 RGB): opt in once per device
    B2O_CUDA_CHECK(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             static_cast<int>(static_cast<size_t>(B2O_CRNN_MAX_HEIGHT) * B2O_CRNN_MAX_WIDTH * 3)));
    ctx->configured.insert(fn);
  }
  if (ch == 3) warp_kernel<3><<<n_boxes, 256, smem, st>>>(img, n, h, w, boxes, image_index, chh, cw, crops, reinterpret_cast<__half*>(crnn_in));
  else warp_kernel<1><<<n_boxes, 256, smem, st>>>(img, n, h, w, boxes, image_index, chh, cw, crops, reinterpret_cast<__half*>(crnn_in));
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}

extern "C" int b2o_warp_boxes(b2o_ctx* ctx, const uint8_t* gray, int n, int h, int w, const float* boxes,
                              const int32_t* image_index, int n_boxes, uint8_t* crops, void* crnn_in, void* stream) {
  return warp_boxes_impl(ctx, gray, 1, n, h, w, boxes, image_index, n_boxes, crops, crnn_in, stream);
}

extern "C" int b2o_warp_boxes_color(b2o_ctx* ctx, const uint8_t* rgb, int n, int h, int w, const float* boxes,
                                    const int32_t* image_index, int n_boxes, uint8_t* crops, void* crnn_in, void* stream) {
  return warp_boxes_impl(ctx, rgb, 3, n, h, w, boxes, image_index, n_boxes, crops, crnn_in, stream);
}

static int crops_to_input_impl(b2o_ctx* ctx, const uint8_t* crops, int ch, int b, void* crnn_in, void* stream) {
  if (!ctx) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  if (b == 0) return B2O_OK;
  if (!crops || !crnn_in || b < 0) { ctx->set_error("b2o_crops_to_input: bad argument"); return B2O_ERR_ARG; }
  const int chh = ctx->crnn_geom.height, cw = ctx->crnn_geom.width;
  const long long total = static_cast<long long>(b) * chh * cw * ch;
  crops_to_input_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      crops, total, ch, chh, cw, reinterpret_cast<__half*>(crnn_in));
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}

extern "C" int b2o_crops_to_input(b2o_ctx* ctx, const uint8_t* crops, int b, void* crnn_in, void* stream) {
  return crops_to_input_impl(ctx, crops, 1, b, crnn_in, stream);
}

extern "C" int b2o_crops_to_input_color(b2o_ctx* ctx, const uint8_t* crops, int b, void* crnn_in, void* stream) {
  return crops_to_input_impl(ctx, crops, 3, b, crnn_in, stream);
}

extern "C" int b2o_fit_crops(b2o_ctx* ctx, const uint8_t* const* srcs_dev, const int32_t* dims_dev, int b,
                             uint8_t* crops_dev, void* crnn_in_dev, void* stream) {
  if (!ctx) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  if (b == 0) return B2O_OK;
  if (!srcs_dev || !dims_dev || !crnn_in_dev || b < 0) {
    ctx->set_error("b2o_fit_crops: bad argument (srcs, dims and crnn_in are required, b >= 0)");
    return B2O_ERR_ARG;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int chh = ctx->crnn_geom.height, cw = ctx->crnn_geom.width;
  __half* out = reinterpret_cast<__half*>(crnn_in_dev);
  if (ctx->crnn_in_ch == 3) fit_crops_kernel<3><<<b, 256, 0, st>>>(srcs_dev, dims_dev, chh, cw, crops_dev, out);
  else fit_crops_kernel<1><<<b, 256, 0, st>>>(srcs_dev, dims_dev, chh, cw, crops_dev, out);
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}
