// crnn_tail.cu -- the non-convolutional part of the CRNN (reference keras_ocr/recognition.py):
//   stn_theta_kernel   Dense(64->6) of the localisation net (277)
//   stn_sample_kernel  _transform (73-166): the reference's bilinear sampler *including its quirks*
//                      (coordinates scaled by W/H instead of W-1/H-1, weights from clipped corners)
//   lstm_kernel        keras.layers.LSTM x4 (292-318): gates [i,f,c,o], sigmoid/tanh, go_backwards
//                      outputs kept in processing order; recurrent matrix column-resident in registers
//   add_kernel         keras.layers.Add (305)
//   fc_ctc_kernel      Dense(256->37) (322-327; softmax skipped: argmax-invariant), [:, discard:] (328),
//                      greedy CTC with repeat merge + blank removal, -1 padding (169-184)
#include <math.h>

#include "common.cuh"

namespace {

__global__ void stn_theta_kernel(const __half* __restrict__ d1 /*[B][64]*/, int B, const float* __restrict__ w /*[64][6]*/,
                                 const float* __restrict__ bias, float* __restrict__ theta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * 6) return;
  const int b = i / 6, k = i - b * 6;
  float acc = bias[k];
  for (int c = 0; c < 64; ++c) acc = fmaf(__half2float(d1[b * 64 + c]), w[c * 6 + k], acc);
  theta[i] = acc;
}

__device__ __forceinline__ float linspace_pm1(int i, int n) {
  // torch.linspace(-1, 1, n) in fp32 (symmetric evaluation)
  const float step = 2.0f / static_cast<float>(n - 1);
  return (i < n / 2) ? (-1.0f + step * static_cast<float>(i)) : (1.0f - step * static_cast<float>(n - 1 - i));
}

// feat/out: (B, Hh, Ww, C) fp16 with Hh = T ("height" of the STN, the time axis; 50 at 31 x 200), Ww = Hf (7).
__global__ void stn_sample_kernel(const __half* __restrict__ feat, const float* __restrict__ theta, int B, int Hh,
                                  int Ww, int C, __half* __restrict__ out) {
  // blockIdx.y walks the crops: the index inside one crop is 32-bit (the 64-bit div/mod chain was most of the kernel)
  const unsigned CV = C / 8;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= static_cast<unsigned>(Hh) * Ww * CV) return;
  const unsigned cv = idx % CV, pix = idx / CV;
  const int ix = static_cast<int>(pix % Ww), iy = static_cast<int>(pix / Ww);
  for (int b = blockIdx.y; b < B; b += gridDim.y) {
    const long long pp = static_cast<long long>(b) * Hh * Ww + pix;
    const float* th = theta + b * 6;
    const float gx = linspace_pm1(ix, Ww), gy = linspace_pm1(iy, Hh);
    const float xs = __fadd_rn(__fadd_rn(__fmul_rn(th[0], gx), __fmul_rn(th[1], gy)), th[2]);
    const float ys = __fadd_rn(__fadd_rn(__fmul_rn(th[3], gx), __fmul_rn(th[4], gy)), th[5]);
    const float x = __fmul_rn(__fmul_rn(0.5f, __fadd_rn(xs, 1.0f)), static_cast<float>(Ww));
    const float y = __fmul_rn(__fmul_rn(0.5f, __fadd_rn(ys, 1.0f)), static_cast<float>(Hh));
    // floor -> int32 cast like tf.cast(tf.floor(x), "int32"); clamp the float first so the cast is defined
    int x0 = static_cast<int>(floorf(fminf(fmaxf(x, -1.0e6f), 1.0e6f)));
    int y0 = static_cast<int>(floorf(fminf(fmaxf(y, -1.0e6f), 1.0e6f)));
    int x1 = x0 + 1, y1 = y0 + 1;
    x0 = min(max(x0, 0), Ww - 1); x1 = min(max(x1, 0), Ww - 1);
    y0 = min(max(y0, 0), Hh - 1); y1 = min(max(y1, 0), Hh - 1);
    const float fx0 = static_cast<float>(x0), fx1 = static_cast<float>(x1);
    const float fy0 = static_cast<float>(y0), fy1 = static_cast<float>(y1);
    const float wa = __fmul_rn(fx1 - x, fy1 - y), wb = __fmul_rn(fx1 - x, y - fy0);
    const float wc = __fmul_rn(x - fx0, fy1 - y), wd = __fmul_rn(x - fx0, y - fy0);
    const __half* base = feat + static_cast<size_t>(b) * Hh * Ww * C + cv * 8;
    const uint4 ra = *reinterpret_cast<const uint4*>(base + (static_cast<size_t>(y0) * Ww + x0) * C);
    const uint4 rb = *reinterpret_cast<const uint4*>(base + (static_cast<size_t>(y1) * Ww + x0) * C);
    const uint4 rc = *reinterpret_cast<const uint4*>(base + (static_cast<size_t>(y0) * Ww + x1) * C);
    const uint4 rd = *reinterpret_cast<const uint4*>(base + (static_cast<size_t>(y1) * Ww + x1) * C);
    const __half2* pa = reinterpret_cast<const __half2*>(&ra);
    const __half2* pb = reinterpret_cast<const __half2*>(&rb);
    const __half2* pc = reinterpret_cast<const __half2*>(&rc);
    const __half2* pd = reinterpret_cast<const __half2*>(&rd);
    uint4 r;
    __half2* pr = reinterpret_cast<__half2*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 a = __half22float2(pa[i]), bb = __half22float2(pb[i]);
      const float2 c = __half22float2(pc[i]), d = __half22float2(pd[i]);
      pr[i] = __floats2half2_rn(wa * a.x + wb * bb.x + wc * c.x + wd * d.x, wa * a.y + wb * bb.y + wc * c.y + wd * d.y);
    }
    *reinterpret_cast<uint4*>(out + static_cast<size_t>(pp) * C + cv * 8) = r;
  }
}

// ---------------------------------------------------------------------------------------- STN conv_a tail
// y: (B,H,W,512) fp16 with (H, W) = (T, Hf) of the features, column tap*16 + c = <x[pixel], W[tap][:, c]>;
// out[p][c] = relu(bias[c] + sum over the 25 taps of y[p + offset(tap)][tap*16 + c]) with zero padding ("same",
// recognition.py:268-270).  One thread per output pixel, taps added in (ky, kx) order in fp32.
__global__ void stn_col2im_kernel(const __half* __restrict__ y, const float* __restrict__ bias, int B, int H, int W,
                                  __half* __restrict__ out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= B * H * W) return;
  const int w = p % W, h = (p / W) % H;
  float acc[16];
#pragma unroll
  for (int c = 0; c < 16; ++c) acc[c] = bias[c];
#pragma unroll
  for (int ky = 0; ky < 5; ++ky) {
    const int ih = h + ky - 2;
    if (ih < 0 || ih >= H) continue;
#pragma unroll
    for (int kx = 0; kx < 5; ++kx) {
      const int iw = w + kx - 2;
      if (iw < 0 || iw >= W) continue;
      const uint4* src = reinterpret_cast<const uint4*>(y + (static_cast<size_t>(p) + (ky - 2) * W + (kx - 2)) * 512 +
                                                        (ky * 5 + kx) * 16);
      const uint4 v0 = src[0], v1 = src[1];
      const __half2* h0 = reinterpret_cast<const __half2*>(&v0);
      const __half2* h1 = reinterpret_cast<const __half2*>(&v1);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 a = __half22float2(h0[e]), b = __half22float2(h1[e]);
        acc[2 * e] += a.x; acc[2 * e + 1] += a.y;
        acc[8 + 2 * e] += b.x; acc[8 + 2 * e + 1] += b.y;
      }
    }
  }
  uint4 o0, o1;
  __half2* q0 = reinterpret_cast<__half2*>(&o0);
  __half2* q1 = reinterpret_cast<__half2*>(&o1);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    q0[e] = __floats2half2_rn(fmaxf(acc[2 * e], 0.0f), fmaxf(acc[2 * e + 1], 0.0f));
    q1[e] = __floats2half2_rn(fmaxf(acc[8 + 2 * e], 0.0f), fmaxf(acc[8 + 2 * e + 1], 0.0f));
  }
  uint4* dst = reinterpret_cast<uint4*>(out + static_cast<size_t>(p) * 16);
  dst[0] = o0;
  dst[1] = o1;
}

// ---------------------------------------------------------------------------------------- LSTM
constexpr int kUnits = 128, kGates = 512;
constexpr int kCropsPerCta = 8;
constexpr int kHPitch = kUnits + 8;      // halves per crop row of h: +16 B so the 8 crops hit different banks

__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ void mma_m16n8k16(float* d, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// One CTA = 8 crops, 16 warps, T strictly sequential steps (50 for 31 x 200 crops), so what matters is the latency of
// one step.  The recurrent product z[512 gates x 8 crops] = U^T[512 x 128] . h^T[128 x 8] is exactly the m16n8k16 warp MMA
// shape with the crops as N: warp w owns units 8w..8w+7 and keeps its two 16-row slices of U^T
// ({i,f} gates and {c,o} gates of those units, all 128 k) in registers for the whole sequence; the D fragment
// then hands every thread all four gates of one unit for two crops, so the gate arithmetic needs no exchange
// and the only shared data is the fp16 h vector (double-buffered, one __syncthreads per step).  tcgen05 does
// not apply: M = 128 rows would be 94 % padding and its issue -> commit -> tcgen05.ld round trip is longer
// than this whole step.  h is rounded to fp16 between steps -- the same value that is written to `out`.
// T   : time steps (crop width / 4)
// xw  : (B*T, xw_ld) fp32 input projections x@W + b; this direction's 512 gate columns start at xw_off
// u   : (128, 512) fp16 recurrent kernel (row k = previous-h unit, column g = gate; Keras order i,f,c,o)
// out : (B, T, out_ld) fp16, written at channel offset out_off, indexed by PROCESSING step
__global__ void __launch_bounds__(kGates, 1)
lstm_kernel(const float* __restrict__ xw, int xw_ld, int xw_off, const __half* __restrict__ u, int B, int T,
            int backwards, __half* __restrict__ out, int out_ld, int out_off) {
  __shared__ __align__(16) __half h_s[2][kCropsPerCta][kHPitch];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = lane >> 2, q = lane & 3;
  const int unit = warp * 8 + r;                         // this thread's unit (all four gates)
  const int cA = q * 2;                                  // this thread's crops: cA, cA + 1
  const int b0 = blockIdx.x * kCropsPerCta;
  const int nb = min(kCropsPerCta, B - b0);

  // A fragments of U^T: tile 0 rows = {i[unit], f[unit]}, tile 1 rows = {c[unit], o[unit]}
  uint32_t afrag[2][kUnits / 16][4];
#pragma unroll
  for (int tile = 0; tile < 2; ++tile)
#pragma unroll
    for (int kt = 0; kt < kUnits / 16; ++kt) {
      const int col_lo = (2 * tile) * kUnits + unit, col_hi = (2 * tile + 1) * kUnits + unit;
      const int k0 = kt * 16 + q * 2;
      auto pack = [&](int k, int col) {
        const __half2 v = __halves2half2(u[k * kGates + col], u[(k + 1) * kGates + col]);
        return *reinterpret_cast<const uint32_t*>(&v);
      };
      afrag[tile][kt][0] = pack(k0, col_lo);
      afrag[tile][kt][1] = pack(k0, col_hi);
      afrag[tile][kt][2] = pack(k0 + 8, col_lo);
      afrag[tile][kt][3] = pack(k0 + 8, col_hi);
    }
  for (int i = threadIdx.x; i < 2 * kCropsPerCta * kHPitch; i += blockDim.x) (&h_s[0][0][0])[i] = __float2half_rn(0.0f);

  // input projections of (crop cA / cA+1) x (gates i,f,c,o of `unit`), prefetched one step ahead
  const bool okA = cA < nb, okB = cA + 1 < nb;
  auto load_x = [&](int t, float* z) {
    const float* pa = xw + (static_cast<size_t>(b0 + cA) * T + t) * xw_ld + xw_off + unit;
    const float* pb = pa + static_cast<size_t>(T) * xw_ld;
#pragma unroll
    for (int gidx = 0; gidx < 4; ++gidx) {
      z[2 * gidx] = okA ? pa[gidx * kUnits] : 0.0f;
      z[2 * gidx + 1] = okB ? pb[gidx * kUnits] : 0.0f;
    }
  };
  float xnext[8];
  load_x(backwards ? T - 1 : 0, xnext);
  float c_state[2] = {0.0f, 0.0f};
  __syncthreads();
  for (int step = 0; step < T; ++step) {
    // D fragments: d0 = {i[cA], i[cB], f[cA], f[cB]}, d1 = {c[cA], c[cB], o[cA], o[cB]}
    float d0[4] = {xnext[0], xnext[1], xnext[2], xnext[3]};
    float d1[4] = {xnext[4], xnext[5], xnext[6], xnext[7]};
    if (step + 1 < T) load_x(backwards ? (T - 2 - step) : (step + 1), xnext);
    const __half* hrow = &h_s[step & 1][r][q * 2];     // B fragment: h[crop r][k0 .. k0+1], [k0+8 .. k0+9]
#pragma unroll
    for (int kt = 0; kt < kUnits / 16; ++kt) {
      const uint32_t b0r = *reinterpret_cast<const uint32_t*>(hrow + kt * 16);
      const uint32_t b1r = *reinterpret_cast<const uint32_t*>(hrow + kt * 16 + 8);
      mma_m16n8k16(d0, afrag[0][kt], b0r, b1r);
      mma_m16n8k16(d1, afrag[1][kt], b0r, b1r);
    }
#pragma unroll
    for (int e = 0; e < 2; ++e) {                         // e = 0: crop cA, e = 1: crop cA + 1
      const float zi = d0[e], zf = d0[2 + e], zc = d1[e], zo = d1[2 + e];
      const float c = sigmoidf_acc(zf) * c_state[e] + sigmoidf_acc(zi) * tanhf(zc);
      const __half h = __float2half_rn(sigmoidf_acc(zo) * tanhf(c));
      c_state[e] = c;
      h_s[(step + 1) & 1][cA + e][unit] = h;
      if (cA + e < nb) out[(static_cast<size_t>(b0 + cA + e) * T + step) * out_ld + out_off + unit] = h;
    }
    __syncthreads();
  }
}

__global__ void add_kernel(const __half2* __restrict__ a, const __half2* __restrict__ b, __half2* __restrict__ o, long long n2) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n2) return;
  const float2 x = __half22float2(a[i]), y = __half22float2(b[i]);
  o[i] = __floats2half2_rn(x.x + y.x, x.y + y.y);
}

// ---------------------------------------------------------------------------------------- fc_12 + CTC
constexpr int kFeat = 256, kFcWarps = 8, kStepsPerWarp = 6, kStepsPerPass = kFcWarps * kStepsPerWarp;
constexpr int kMaxKeep = B2O_CRNN_MAX_WIDTH / 4;

// One CTA per crop, one warp per 6 kept time steps of a pass over 48 steps (one pass at the default 48 kept steps);
// lane l owns classes l, l+32, ... (K = len(alphabet)+1 is a run-time value: recognition.py:376-381 sizes the Dense
// layer from the alphabet).  Every logit is the same serial fmaf chain over the 256 features in ascending order
// whatever K and the geometry are; the argmax keeps the first maximum (np.argmax / tf.argmax tie rule).  Each pass
// leaves its per-step argmax in shared memory, and the collapse over all kept steps drops blanks (index K-1) and
// repeats once every pass is done.
__global__ void __launch_bounds__(32 * kFcWarps)
fc_ctc_kernel(const __half* __restrict__ l2 /*[B][T][256]*/, const float* __restrict__ w /*[256][K]*/,
              const float* __restrict__ bias, int B, int K, int T, int discard,
              float* __restrict__ logits /*[B][T-discard][K] or null*/, int* __restrict__ labels /*[B][T-discard]*/) {
  __shared__ int best[kMaxKeep];
  __shared__ __half xs[kStepsPerPass][kFeat];
  const int b = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int keep = T - discard;
  for (int pass = 0; pass < keep; pass += kStepsPerPass) {
    const int rows = min(kStepsPerPass, keep - pass);
    if (pass > 0) __syncthreads();                     // the previous pass is done with xs
    {
      const uint4* src = reinterpret_cast<const uint4*>(l2 + (static_cast<size_t>(b) * T + discard + pass) * kFeat);
      uint4* dst = reinterpret_cast<uint4*>(&xs[0][0]);
      for (int i = threadIdx.x; i < rows * kFeat / 8; i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    const int t0 = warp * kStepsPerWarp;
    if (t0 < rows) {                                   // warp-uniform
      float mx[kStepsPerWarp];
      int arg[kStepsPerWarp];
#pragma unroll
      for (int j = 0; j < kStepsPerWarp; ++j) { mx[j] = -INFINITY; arg[j] = 0x7fffffff; }
      for (int k = lane; k < K; k += 32) {
        float acc[kStepsPerWarp];
        const float bk = bias[k];
#pragma unroll
        for (int j = 0; j < kStepsPerWarp; ++j) acc[j] = bk;
#pragma unroll 4
        for (int c = 0; c < kFeat; ++c) {
          const float wv = __ldg(w + static_cast<size_t>(c) * K + k);
#pragma unroll
          for (int j = 0; j < kStepsPerWarp; ++j) acc[j] = fmaf(__half2float(xs[t0 + j][c]), wv, acc[j]);
        }
#pragma unroll
        for (int j = 0; j < kStepsPerWarp; ++j) {
          if (acc[j] > mx[j]) { mx[j] = acc[j]; arg[j] = k; }            // ascending k: first maximum wins
          if (logits && t0 + j < rows) logits[(static_cast<size_t>(b) * keep + pass + t0 + j) * K + k] = acc[j];
        }
      }
#pragma unroll
      for (int j = 0; j < kStepsPerWarp; ++j) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
          const float om = __shfl_xor_sync(0xffffffffu, mx[j], off);
          const int oa = __shfl_xor_sync(0xffffffffu, arg[j], off);
          if (om > mx[j] || (om == mx[j] && oa < arg[j])) { mx[j] = om; arg[j] = oa; }
        }
        if (lane == 0 && t0 + j < rows) best[pass + t0 + j] = arg[j] == 0x7fffffff ? 0 : arg[j];  // all-NaN row: argmax returns 0
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int* o = labels + static_cast<size_t>(b) * keep;
    int n = 0, prev = -1;
    for (int s = 0; s < keep; ++s) {
      const int c = best[s];
      if (c != K - 1 && c != prev) o[n++] = c;
      prev = c;
    }
    for (; n < keep; ++n) o[n] = -1;
  }
}

inline unsigned nb(long long total, int threads) { return static_cast<unsigned>((total + threads - 1) / threads); }

}  // namespace

int stn_theta_run(b2o_ctx* ctx, const __half* d1, int B, float* theta, cudaStream_t st) {
  stn_theta_kernel<<<nb(B * 6, 128), 128, 0, st>>>(d1, B, ctx->stn_d2_w, ctx->stn_d2_b, theta);
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}

int stn_col2im_run(b2o_ctx* ctx, const __half* y, const float* bias, int B, int H, int W, __half* out, cudaStream_t st) {
  const int total = B * H * W;
  stn_col2im_kernel<<<(total + 127) / 128, 128, 0, st>>>(y, bias, B, H, W, out);
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}

int stn_sample_run(b2o_ctx* ctx, const __half* feat, const float* theta, int B, int Hh, int Ww, __half* out, cudaStream_t st) {
  if (B <= 0) return B2O_OK;
  stn_sample_kernel<<<dim3(nb(Hh * Ww * (512 / 8), 256), B < 65535 ? B : 65535), 256, 0, st>>>(feat, theta, B, Hh, Ww, 512, out);
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}

int lstm_run(b2o_ctx* ctx, const float* xw, int xw_ld, int xw_off, const __half* u, int B, int T, int backwards, __half* out,
             int out_ld, int out_off, cudaStream_t st) {
  lstm_kernel<<<(B + kCropsPerCta - 1) / kCropsPerCta, kGates, 0, st>>>(xw, xw_ld, xw_off, u, B, T, backwards, out, out_ld,
                                                                        out_off);
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}

int add_run(b2o_ctx* ctx, const __half* a, const __half* b, __half* o, long long n, cudaStream_t st) {
  add_kernel<<<nb(n / 2, 256), 256, 0, st>>>(reinterpret_cast<const __half2*>(a), reinterpret_cast<const __half2*>(b),
                                             reinterpret_cast<__half2*>(o), n / 2);
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}

int fc_ctc_run(b2o_ctx* ctx, const __half* l2, int B, int T, int discard, float* logits, int* labels, cudaStream_t st) {
  if (T - discard < 1 || T - discard > kMaxKeep) { ctx->set_error("fc_ctc_run: unsupported step count"); return B2O_ERR_ARG; }
  fc_ctc_kernel<<<B, 32 * kFcWarps, 0, st>>>(l2, ctx->fc12_w, ctx->fc12_b, B, ctx->n_classes, T, discard, logits, labels);
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}
