// Shared declarations for the b2ocr CUDA library (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <map>
#include <set>
#include <string>
#include <vector>

#include "../../include/b2ocr.h"

#define B2O_CUDA_CHECK(ctx, expr)                                                              \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      (ctx)->set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                    \
      return B2O_ERR_CUDA;                                                                     \
    }                                                                                          \
  } while (0)

#define B2O_LAUNCH_CHECK(ctx)                                                                  \
  do {                                                                                         \
    (ctx)->launches++;                                                                         \
    cudaError_t _e = cudaGetLastError();                                                       \
    if (_e != cudaSuccess) {                                                                   \
      (ctx)->set_error(std::string(__FILE__) + ":" + std::to_string(__LINE__) + " launch: " +  \
                       cudaGetErrorString(_e));                                                \
      return B2O_ERR_CUDA;                                                                     \
    }                                                                                          \
  } while (0)

// Every entry point that touches the device runs with the context's device current and puts the caller's device
// back on return (the caller -- torch -- may be driving another GPU of the box in the same process).
struct DeviceGuard {
  int prev = -1;
  bool changed = false;
  explicit DeviceGuard(int device) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != device) changed = cudaSetDevice(device) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (changed) cudaSetDevice(prev);
  }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};

#define B2O_RETURN_IF(expr)                                                                    \
  do {                                                                                         \
    int _s = (expr);                                                                           \
    if (_s != B2O_OK) return _s;                                                               \
  } while (0)

// Epilogue applied by every convolution / dense kernel, per output channel n:
//   y = acc * s1[n] + t1[n];  if (relu) y = max(y, 0);  if (s2) y = y * s2[n] + t2[n]
// CRAFT conv+BN(+ReLU): s1 = gamma/sqrt(var+eps), t1 = (bias-mean)*s1+beta   (detection.py:87-103)
// CRNN  conv+ReLU+BN  : s1 = 1, t1 = bias, relu, s2 = gamma/sqrt(var+eps), t2 = beta-mean*s2
//                       (recognition.py:223-242 -- BN comes AFTER the ReLU there)
struct ConvLayer {
  std::string name;
  int cin = 0, cout = 0, ksize = 1, dil = 1, relu = 0;
  __half* w_kmajor = nullptr;  // [cout][taps*cin] fp16, K index = tap*cin + c   (tcgen05 B operand)
  float* w_simt = nullptr;     // [taps][cin][cout] fp32 holding the fp16-rounded values (SIMT engine)
  float* w_f32 = nullptr;      // [taps][cin][cout] fp32 (only for the 3-channel / 1-channel stems)
  float *s1 = nullptr, *t1 = nullptr, *s2 = nullptr, *t2 = nullptr;
  std::vector<float> h_w_f32;                  // host copy of w_f32 (the 1- / 3-channel CRNN stem: kernel-parameter filter bank)
  std::vector<float> h_w_simt;                 // host copy of w_simt for layers of <= 1024 weights (fused into other kernels' parameters)
  std::vector<float> h_s1, h_t1, h_s2, h_t2;   // host copies: passed to the tensor-core kernel as a kernel parameter (constant bank)
  CUtensorMap wmap;            // TMA map over w_kmajor (box 64 x block_n)
  CUtensorMap wmap_pair;       // the same with box 64 x block_n/2: one CTA's half of a B tile (cta_group::2)
  bool pair_ok = false;        // wmap_pair is valid (64-channel chunks, block_n >= 64)
  int block_n = 0;             // tcgen05 N tile; 0 = layer not eligible for the tensor-core engine
  int kch = 0;                 // tcgen05 K chunk (channels per stage): 64 / 32 / 16
  // channels of the layer the reference defines, where the tensor-core form pads them (3 -> 16 input channels of the
  // CRAFT stem, 400 -> 512 columns of the STN GEMM): what the roofline's algorithmic FLOP count uses.  0 = cin / cout.
  int alg_cin = 0, alg_cout = 0;
};

struct TensorView {            // NHWC fp16 activation living inside a (possibly wider) buffer
  __half* ptr = nullptr;       // address of channel 0 of the slice
  int n = 0, h = 0, w = 0, c = 0;
  int ld = 0;                  // channel stride of the underlying buffer (elements)
};

// Crop geometry of the CRNN (build_model's height / width / rnn_steps_to_discard, recognition.py:13-23, 214, 328).  The
// conv stack sees a (width, height) image (Permute((2,1,3))); both 2x2 max pools floor, so the features are (T, Hf) =
// (width // 4, height // 4) and the LSTMs run T steps, of which the first `discard` are dropped before the CTC decode.
struct CrnnGeometry {
  int height = 31, width = 200, discard = 2;
  int steps() const { return width / 4; }            // T
  int feat_h() const { return height / 4; }          // Hf
  int keep() const { return width / 4 - discard; }   // label row length (CTC input_length)
};

struct b2o_ctx {
  int device = 0;
  int sm_count = 148;
  int conv_engine = B2O_CONV_AUTO;
  int tc_issuers = 0;          // MMA-issuing warps of conv_tc_kernel: 0 = auto (2 for N <= 128 tiles), 1, 2
  bool tc_pair = true;         // CTA pairs (tcgen05 cta_group::2) for the halo-tile layers; B2O_TC_PAIR=0 turns them off
  int tc_box16 = 16;           // width of the single A box per K chunk in MODE 3 layers (B2O_TC_BOX16=0: three 8 x 18 boxes; 10: tile + halo only)
  bool tc_box_forced = false;  // B2O_TC_BOX16 was given: use that width everywhere instead of the per-layer rule
  bool tc_box_all = false;     // B2O_TC_BOX_ALL=1: single-box tiles for every grouped layer (default: N <= 64 with 64-/32-channel chunks)
  bool tc_pair_generic = false;   // B2O_TC_PAIR=2: also pair the generic tiles (1x1 / dilated layers): bit-identical, no gain measured (profiles/r2a_ab_pair2.log)
  // Decoder glue: B2O_UPCONV_COMMUTE=1 commutes the 2x upsampling behind the decoder half of upconvN.conv.0 (low-res GEMM +
  // upsample-add in the full-resolution layer's epilogue).  Numerically validated, but measured SLOWER on B200
  // (profiles/r2e_layers.csv: upconv4.0 1.39 + upsample 0.85 ms -> 0.21 + 2.32 ms): the epilogue's per-pixel 16-byte
  // gathers of the four taps are LSU-wavefront-bound.  Default: explicit UpsampleLike kernels.
  bool tc_aff_const = true;    // epilogue constants as a kernel parameter (constant cache); B2O_TC_AFF=smem: round-1 staging in shared memory / global loads
  bool no_commute = true;
  bool glue_v1 = false;        // B2O_GLUE=v1: the round-1 upsample2x kernel (64-bit index chain, unshared blends) for A/B runs and the bit-identity test
  bool no_fused_tail = false;  // B2O_FUSED_TAIL=0: conv_cls.6/.8 as the separate head_tail_kernel instead of conv_cls.4's epilogue
  std::set<const void*> configured;   // kernels whose per-device launch attributes are set on this device
  int64_t launches = 0;
  std::string error;
  std::map<std::string, ConvLayer> craft, crnn;
  bool craft_loaded = false, crnn_loaded = false;
  int crnn_in_ch = 1;              // 1 = gray crops (default), 3 = RGB crops (build_model(color=True))
  bool crnn_stn = true;            // the loaded CRNN has a spatial transformer (build_model(stn=True), the default)
  CrnnGeometry crnn_geom;          // b2o_set_crnn_geometry (default 31 x 200, 2 steps discarded)
  bool quads_configured = false;   // quads_kernel's dynamic shared-memory opt-in done on this device
  // CRNN tail parameters (device)
  float *stn_d2_w = nullptr, *stn_d2_b = nullptr;              // dense 64 -> 6, fp32
  __half* lstm_u[4] = {nullptr, nullptr, nullptr, nullptr};    // recurrent kernels [128][512] fp16
  float *fc12_w = nullptr, *fc12_b = nullptr;                  // [256][K], [K] fp32, K = len(alphabet) + 1
  int n_classes = 37;                                          // K (last index = CTC blank), <= B2O_MAX_CLASSES
  std::vector<void*> owned;    // device allocations freed in b2o_destroy
  // optional per-launch timing of the tensor-core conv kernel (bench.py's roofline leg)
  bool debug_taps = false;     // b2o_set_debug_taps: the CRNN forward also writes its fp32 logits (tests only)
  bool profile = false;
  std::vector<cudaEvent_t> prof_events;   // (start, stop) pairs
  double prof_flop = 0.0;
  void* jpeg = nullptr;        // nvJPEG handle + state, created on first use (jpeg.cu)
  bool jpeg_failed = false;    // nvJPEG could not be opened on this box: do not try again
  void set_error(const std::string& e) { error = e; }
};
void jpeg_release(b2o_ctx* ctx);

// CRAFT tail fused into the epilogue of a 16-channel tensor-core layer: conv_cls.6 (1x1 16->16, ReLU) and conv_cls.8
// (1x1 16->2) on the 16 channels a thread already holds; fp32 (text, link) scores out (detection.py:404-410).
struct ConvTail {
  const float *w6, *b6, *w8, *b8;   // [cin 16][cout 16] fp32 (fp16-rounded values), [16], [16][2], [2] -- device
  float* scores;                    // (n,h,w,2)
  const float *h_w6 = nullptr, *h_b6 = nullptr, *h_w8 = nullptr, *h_b8 = nullptr;   // the same on the host (kernel-parameter path)
};

// ---- engines (conv_tc.cu, conv_simt.cu) -------------------------------------------------------
int conv_tc_prepare(b2o_ctx* ctx, ConvLayer& L);   // builds wmap / picks block_n (0 if ineligible)
// pool_out != null: also write the 2x2/2 max-pooled output (fused epilogue); write_full = 0 skips `out`
int conv_tc_run(b2o_ctx* ctx, const ConvLayer& L, const TensorView& in, const TensorView& out,
                int out_f32, cudaStream_t st, const TensorView* pool_out = nullptr, int write_full = 1,
                const ConvTail* tail = nullptr, const TensorView* up_add = nullptr);
// up_add (1x1 layers, 64-channel chunks): a (n, h/2, w/2, cout) fp16 tensor whose exact-2x bilinear upsampling is added to
// the accumulator before the affine/ReLU -- the decoder's UpsampleLike + Concatenate + 1x1 conv with the upsampling
// commuted behind the (linear) convolution of the low-resolution half (detection.py:290-309, 380-390)
int conv_simt_run(b2o_ctx* ctx, const ConvLayer& L, const TensorView& in, const TensorView& out,
                  int out_f32, cudaStream_t st);
int conv_run(b2o_ctx* ctx, const ConvLayer& L, const TensorView& in, const TensorView& out,
             int out_f32, cudaStream_t st, const TensorView* pool_out = nullptr, int write_full = 1);
int stem_rgb_run(b2o_ctx* ctx, const ConvLayer& L, const uint8_t* img, int n, int h, int w,
                 const TensorView& out, cudaStream_t st);
int normalize16_run(b2o_ctx* ctx, const uint8_t* img, int n, int h, int w, __half* out, cudaStream_t st);
int stem_crnn_run(b2o_ctx* ctx, const ConvLayer& L, const __half* x, int b, const TensorView& out,
                  cudaStream_t st);
int maxpool2_run(b2o_ctx* ctx, const TensorView& in, const TensorView& out, cudaStream_t st);
int maxpool3s1_run(b2o_ctx* ctx, const TensorView& in, const TensorView& out, cudaStream_t st);
int upsample_run(b2o_ctx* ctx, const TensorView& in, const TensorView& out, cudaStream_t st);
int head_tail_run(b2o_ctx* ctx, const ConvLayer& L6, const ConvLayer& L8, const TensorView& in,
                  float* scores, cudaStream_t st);

static inline TensorView make_view(void* base, int n, int h, int w, int c, int ld = 0, int coff = 0) {
  TensorView v;
  v.ptr = reinterpret_cast<__half*>(base) + coff;
  v.n = n; v.h = h; v.w = w; v.c = c; v.ld = ld ? ld : c;
  return v;
}
