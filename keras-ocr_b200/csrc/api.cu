// api.cu -- C-ABI entry points (include/b2ocr.h): context, weight packing, network orchestration.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <functional>

#include "common.cuh"

int stn_theta_run(b2o_ctx* ctx, const __half* d1, int B, float* theta, cudaStream_t st);
int stn_col2im_run(b2o_ctx* ctx, const __half* y, const float* bias, int B, int H, int W, __half* out, cudaStream_t st);
int stn_sample_run(b2o_ctx* ctx, const __half* feat, const float* theta, int B, int Hh, int Ww, __half* out, cudaStream_t st);
int lstm_run(b2o_ctx* ctx, const float* xw, int xw_ld, int xw_off, const __half* u, int B, int T, int backwards, __half* out,
             int out_ld, int out_off, cudaStream_t st);
int add_run(b2o_ctx* ctx, const __half* a, const __half* b, __half* o, long long n, cudaStream_t st);
int fc_ctc_run(b2o_ctx* ctx, const __half* l2, int B, int T, int discard, float* logits, int* labels, cudaStream_t st);

namespace {

typedef std::map<std::string, const b2o_tensor*> TensorMap;

const b2o_tensor* need(b2o_ctx* ctx, const TensorMap& m, const std::string& name, int ndim, const int64_t* shape) {
  auto it = m.find(name);
  if (it == m.end()) { ctx->set_error("missing weight tensor: " + name); return nullptr; }
  const b2o_tensor* t = it->second;
  if (t->ndim != ndim) { ctx->set_error("bad rank for " + name); return nullptr; }
  for (int i = 0; i < ndim; ++i)
    if (t->shape[i] != shape[i]) { ctx->set_error("bad shape for " + name); return nullptr; }
  return t;
}

template <typename T>
T* dev_alloc(b2o_ctx* ctx, size_t count) {
  void* p = nullptr;
  if (cudaMalloc(&p, count * sizeof(T)) != cudaSuccess) { ctx->set_error("cudaMalloc failed"); return nullptr; }
  ctx->owned.push_back(p);
  return reinterpret_cast<T*>(p);
}

template <typename T>
T* dev_upload(b2o_ctx* ctx, const std::vector<T>& host) {
  T* p = dev_alloc<T>(ctx, host.size());
  if (!p) return nullptr;
  if (cudaMemcpy(p, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) {
    ctx->set_error("cudaMemcpy (weights) failed");
    return nullptr;
  }
  return p;
}

// Build one layer.  wget(o, c, ky, kx) returns the fp32 weight.
int build_layer(b2o_ctx* ctx, ConvLayer& L, const std::string& name, int cin, int cout, int ksize, int dil, int relu,
                const std::function<float(int, int, int, int)>& wget, const std::vector<float>& s1,
                const std::vector<float>& t1, const std::vector<float>* s2, const std::vector<float>* t2,
                bool keep_f32_stem) {
  L = ConvLayer();
  L.name = name; L.cin = cin; L.cout = cout; L.ksize = ksize; L.dil = dil; L.relu = relu;
  const int taps = ksize * ksize;
  if (keep_f32_stem) {
    std::vector<float> wf(static_cast<size_t>(taps) * cin * cout);
    for (int ky = 0; ky < ksize; ++ky)
      for (int kx = 0; kx < ksize; ++kx)
        for (int c = 0; c < cin; ++c)
          for (int o = 0; o < cout; ++o)
            wf[(static_cast<size_t>(ky * ksize + kx) * cin + c) * cout + o] = wget(o, c, ky, kx);
    if (!(L.w_f32 = dev_upload(ctx, wf))) return B2O_ERR_CUDA;
    L.h_w_f32 = wf;
  } else {
    std::vector<__half> wk(static_cast<size_t>(cout) * taps * cin);
    std::vector<float> ws(static_cast<size_t>(taps) * cin * cout);
    for (int o = 0; o < cout; ++o)
      for (int ky = 0; ky < ksize; ++ky)
        for (int kx = 0; kx < ksize; ++kx)
          for (int c = 0; c < cin; ++c) {
            const __half hv = __float2half_rn(wget(o, c, ky, kx));
            const int tap = ky * ksize + kx;
            wk[(static_cast<size_t>(o) * taps + tap) * cin + c] = hv;
            ws[(static_cast<size_t>(tap) * cin + c) * cout + o] = __half2float(hv);
          }
    if (!(L.w_kmajor = dev_upload(ctx, wk))) return B2O_ERR_CUDA;
    if (!(L.w_simt = dev_upload(ctx, ws))) return B2O_ERR_CUDA;
    if (ws.size() <= 1024) L.h_w_simt = ws;
  }
  if (!(L.s1 = dev_upload(ctx, s1))) return B2O_ERR_CUDA;
  if (!(L.t1 = dev_upload(ctx, t1))) return B2O_ERR_CUDA;
  L.h_s1 = s1; L.h_t1 = t1;
  if (s2) { L.h_s2 = *s2; L.h_t2 = *t2; }
  if (s2) {
    if (!(L.s2 = dev_upload(ctx, *s2))) return B2O_ERR_CUDA;
    if (!(L.t2 = dev_upload(ctx, *t2))) return B2O_ERR_CUDA;
  }
  if (!keep_f32_stem) B2O_RETURN_IF(conv_tc_prepare(ctx, L));
  return B2O_OK;
}

struct CraftSpec { const char* name; int cin, cout, k, dil; const char* bn; int relu; };
const CraftSpec kCraft[] = {
    {"basenet.slice1.0", 3, 64, 3, 1, "basenet.slice1.1", 1},     {"basenet.slice1.3", 64, 64, 3, 1, "basenet.slice1.4", 1},
    {"basenet.slice1.7", 64, 128, 3, 1, "basenet.slice1.8", 1},   {"basenet.slice1.10", 128, 128, 3, 1, "basenet.slice1.11", 1},
    {"basenet.slice2.14", 128, 256, 3, 1, "basenet.slice2.15", 1}, {"basenet.slice2.17", 256, 256, 3, 1, "basenet.slice2.18", 1},
    {"basenet.slice3.20", 256, 256, 3, 1, "basenet.slice3.21", 1}, {"basenet.slice3.24", 256, 512, 3, 1, "basenet.slice3.25", 1},
    {"basenet.slice3.27", 512, 512, 3, 1, "basenet.slice3.28", 1}, {"basenet.slice4.30", 512, 512, 3, 1, "basenet.slice4.31", 1},
    {"basenet.slice4.34", 512, 512, 3, 1, "basenet.slice4.35", 1}, {"basenet.slice4.37", 512, 512, 3, 1, "basenet.slice4.38", 0},
    {"basenet.slice5.1", 512, 1024, 3, 6, nullptr, 0},             {"basenet.slice5.2", 1024, 1024, 1, 1, nullptr, 0},
    {"upconv1.conv.0", 1536, 512, 1, 1, "upconv1.conv.1", 1},      {"upconv1.conv.3", 512, 256, 3, 1, "upconv1.conv.4", 1},
    {"upconv2.conv.0", 768, 256, 1, 1, "upconv2.conv.1", 1},       {"upconv2.conv.3", 256, 128, 3, 1, "upconv2.conv.4", 1},
    {"upconv3.conv.0", 384, 128, 1, 1, "upconv3.conv.1", 1},       {"upconv3.conv.3", 128, 64, 3, 1, "upconv3.conv.4", 1},
    {"upconv4.conv.0", 192, 64, 1, 1, "upconv4.conv.1", 1},        {"upconv4.conv.3", 64, 32, 3, 1, "upconv4.conv.4", 1},
    {"conv_cls.0", 32, 32, 3, 1, nullptr, 1},                      {"conv_cls.2", 32, 32, 3, 1, nullptr, 1},
    {"conv_cls.4", 32, 16, 3, 1, nullptr, 1},                      {"conv_cls.6", 16, 16, 1, 1, nullptr, 1},
    {"conv_cls.8", 16, 2, 1, 1, nullptr, 0},
};

// Buffer plan of the CRAFT forward pass (all NHWC fp16 unless noted), carved from one workspace.
struct CraftPlan {
  int n, h1, w1, h2, w2, h4, w4, h8, w8, h16, w16;
  size_t off_a, off_b, off_p1, off_c, off_cat4, off_p2, off_d, off_cat3, off_e, off_p3, off_f, off_cat2, off_g, off_p4,
      off_hh, off_cat1, off_mp, off_s5a, off_u1a, off_u1b, off_u2a, off_u2b, off_u3a, off_u3b, off_u4a, off_u4b, off_h1,
      off_h2, off_h3, off_x16, off_z2, off_z3, off_z4, bytes;
};

// Liveness-based packing: every buffer lives from the launch that first writes it to the launch that last reads it
// (the forward pass is one stream-ordered chain of launches, see b2o_craft_forward: the step numbers below are its
// launch order); buffers whose lifetimes do not overlap share memory.  Greedy by size: largest first, each at the
// lowest offset that is free for its whole lifetime.  32 x 1536 x 1536: 21.8 GB instead of 41 GB with every buffer
// live (the peak is the two full-resolution 64-channel maps around slice1.3), and 73 -> 39 GB at max_size 2048.
CraftPlan plan_craft(int n, int h, int w) {
  CraftPlan p;
  p.n = n; p.h1 = h; p.w1 = w;
  p.h2 = h / 2; p.w2 = w / 2; p.h4 = p.h2 / 2; p.w4 = p.w2 / 2;
  p.h8 = p.h4 / 2; p.w8 = p.w4 / 2; p.h16 = p.h8 / 2; p.w16 = p.w8 / 2;
  struct Buf { size_t* off; size_t bytes; int first, last; };
  std::vector<Buf> bufs;
  auto take = [&](size_t* off, int hh, int ww, int c, int first, int last) {
    bufs.push_back({off, (static_cast<size_t>(n) * hh * ww * c * 2 + 255) / 256 * 256, first, last});
  };
  // step: 0 normalize16, 1 stem, 2 slice1.3, 3 slice1.7, 4 slice1.10, 5 slice2.14, 6 slice2.17, 7 slice3.20, 8 slice3.24,
  // 9 slice3.27, 10 slice4.30, 11 slice4.34, 12 slice4.37, 13 maxpool3, 14 slice5.1, 15 slice5.2, 16 upconv1.0,
  // 17 upconv1.3, 18 upsample, 19 upconv2.0, 20 upconv2.3, 21 upsample, 22 upconv3.0, 23 upconv3.3, 24 upsample,
  // 25 upconv4.0, 26 upconv4.3, 27 conv_cls.0, 28 conv_cls.2, 29 conv_cls.4 (+ fused tail), 30 head_tail
  take(&p.off_x16, p.h1, p.w1, 16, 0, 1);          // normalised input, 3 -> 16 channels, for the tensor-core stem
  take(&p.off_a, p.h1, p.w1, 64, 1, 2);
  take(&p.off_b, p.h1, p.w1, 64, 2, 2);            // full-resolution conv output: only written when the pool is not fused
  take(&p.off_p1, p.h2, p.w2, 64, 2, 3);
  take(&p.off_c, p.h2, p.w2, 128, 3, 4);
  take(&p.off_cat4, p.h2, p.w2, 192, 4, 25);       // [upsampled decoder | tap s1]: written at 4 and 24, read at 25
  take(&p.off_p2, p.h4, p.w4, 128, 4, 5);
  take(&p.off_d, p.h4, p.w4, 256, 5, 6);
  take(&p.off_cat3, p.h4, p.w4, 384, 6, 22);
  take(&p.off_e, p.h4, p.w4, 256, 7, 7);
  take(&p.off_p3, p.h8, p.w8, 256, 7, 8);
  take(&p.off_f, p.h8, p.w8, 512, 8, 9);
  take(&p.off_cat2, p.h8, p.w8, 768, 9, 19);
  take(&p.off_g, p.h8, p.w8, 512, 10, 10);
  take(&p.off_p4, p.h16, p.w16, 512, 10, 11);
  take(&p.off_hh, p.h16, p.w16, 512, 11, 12);
  take(&p.off_cat1, p.h16, p.w16, 1536, 12, 16);
  take(&p.off_mp, p.h16, p.w16, 512, 13, 14);
  take(&p.off_s5a, p.h16, p.w16, 1024, 14, 15);
  take(&p.off_u1a, p.h16, p.w16, 512, 16, 17);
  take(&p.off_u1b, p.h16, p.w16, 256, 17, 18);
  take(&p.off_u2a, p.h8, p.w8, 256, 19, 20);
  take(&p.off_u2b, p.h8, p.w8, 128, 20, 21);
  take(&p.off_u3a, p.h4, p.w4, 128, 22, 23);
  take(&p.off_u3b, p.h4, p.w4, 64, 23, 24);
  take(&p.off_u4a, p.h2, p.w2, 64, 25, 26);
  take(&p.off_u4b, p.h2, p.w2, 32, 26, 27);
  take(&p.off_h1, p.h2, p.w2, 32, 27, 28);
  take(&p.off_h2, p.h2, p.w2, 32, 28, 29);
  take(&p.off_h3, p.h2, p.w2, 16, 29, 30);
  take(&p.off_z2, p.h16, p.w16, 256, 18, 19);      // low-resolution halves of upconv2/3/4.conv.0 (commuted upsampling)
  take(&p.off_z3, p.h8, p.w8, 128, 21, 22);
  take(&p.off_z4, p.h4, p.w4, 64, 24, 25);
  std::vector<int> order(bufs.size());
  for (size_t i = 0; i < order.size(); ++i) order[i] = static_cast<int>(i);
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return bufs[a].bytes > bufs[b].bytes; });
  std::vector<int> placed;
  size_t total = 0;
  for (int i : order) {
    // candidate offsets: 0 and the end of every placed buffer that is live at the same time
    std::vector<std::pair<size_t, size_t>> busy;      // [begin, end) of time-overlapping placed buffers
    for (int j : placed)
      if (bufs[j].first <= bufs[i].last && bufs[i].first <= bufs[j].last) busy.push_back({*bufs[j].off, *bufs[j].off + bufs[j].bytes});
    std::sort(busy.begin(), busy.end());
    size_t at = 0;
    for (const auto& b : busy) {
      if (at + bufs[i].bytes <= b.first) break;
      if (b.second > at) at = b.second;
    }
    *bufs[i].off = at;
    placed.push_back(i);
    if (at + bufs[i].bytes > total) total = at + bufs[i].bytes;
  }
  p.bytes = total;
  return p;
}

struct CrnnPlan {
  int b;
  size_t off_x1, off_x2, off_x3, off_p3, off_x4, off_x5, off_p5, off_x6, off_x7, off_sa, off_sb, off_d1, off_theta,
      off_warp, off_fc9, off_xw1, off_hf, off_hb, off_l1, off_xw2, off_l2, off_logits, bytes;
};

// Buffer plan of the CRNN forward pass at crop geometry g (NHWC fp16 unless noted; the conv stack's "h" axis is the
// crop's width, its "w" axis the crop's height): (W0, H0) = (width, height) -> pooled (W1, H1) -> (T, Hf).
CrnnPlan plan_crnn(int b, const CrnnGeometry& g) {
  CrnnPlan p;
  p.b = b;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t r = off; off += (bytes + 255) / 256 * 256; return r; };
  const size_t B = static_cast<size_t>(b);
  const size_t W0 = g.width, H0 = g.height, W1 = W0 / 2, H1 = H0 / 2, T = g.steps(), Hf = g.feat_h();
  p.off_x1 = take(B * W0 * H0 * 64 * 2); p.off_x2 = take(B * W0 * H0 * 128 * 2); p.off_x3 = take(B * W0 * H0 * 256 * 2);
  p.off_p3 = take(B * W1 * H1 * 256 * 2); p.off_x4 = take(B * W1 * H1 * 256 * 2); p.off_x5 = take(B * W1 * H1 * 512 * 2);
  p.off_p5 = take(B * T * Hf * 512 * 2); p.off_x6 = take(B * T * Hf * 512 * 2); p.off_x7 = take(B * T * Hf * 512 * 2);
  p.off_sa = take(B * T * Hf * 16 * 2); p.off_sb = take(B * T * Hf * 32 * 2); p.off_d1 = take(B * 64 * 2);
  p.off_theta = take(B * 6 * 4); p.off_warp = take(B * T * Hf * 512 * 2); p.off_fc9 = take(B * T * 128 * 2);
  p.off_xw1 = take(B * T * 1024 * 4); p.off_hf = take(B * T * 128 * 2); p.off_hb = take(B * T * 128 * 2);
  p.off_l1 = take(B * T * 128 * 2); p.off_xw2 = take(B * T * 1024 * 4); p.off_l2 = take(B * T * 256 * 2);
  p.off_logits = take(B * g.keep() * B2O_MAX_CLASSES * 4);   // sized for the largest alphabet: independent of the weights
  p.bytes = off;
  return p;
}

std::vector<float> ones(int n) { return std::vector<float>(static_cast<size_t>(n), 1.0f); }
std::vector<float> tovec(const b2o_tensor* t, int n) { return std::vector<float>(t->data, t->data + n); }

}  // namespace

// ------------------------------------------------------------------------------------------------
extern "C" int b2o_version(void) { return 1; }

extern "C" int b2o_create(int device, b2o_ctx** out) {
  if (!out) return B2O_ERR_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return B2O_ERR_CUDA;
  DeviceGuard guard(device);                  // the caller's current device is restored on return
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return B2O_ERR_CUDA;
  if (prop.major != 10) {
    fprintf(stderr, "b2ocr: device %d is sm_%d%d; this library is built for sm_100a only\n", device, prop.major, prop.minor);
    return B2O_ERR_CUDA;
  }
  b2o_ctx* ctx = new b2o_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  if (const char* e = getenv("B2O_TC_ISSUERS")) ctx->tc_issuers = (atoi(e) == 2) ? 2 : (atoi(e) == 1 ? 1 : 0);
  if (const char* e = getenv("B2O_TC_BOX16")) { const int v = atoi(e); ctx->tc_box16 = v == 0 ? 0 : (v == 10 ? 10 : 16); ctx->tc_box_forced = v != 0; }
  if (const char* e = getenv("B2O_TC_BOX_ALL")) ctx->tc_box_all = atoi(e) != 0;
  if (const char* e = getenv("B2O_UPCONV_COMMUTE")) ctx->no_commute = atoi(e) == 0;      // 1: commuted decoder upsampling (opt-in, see common.cuh)
  if (const char* e = getenv("B2O_TC_AFF")) ctx->tc_aff_const = std::string(e) != "smem";
  if (const char* e = getenv("B2O_GLUE")) ctx->glue_v1 = std::string(e) == "v1";
  if (const char* e = getenv("B2O_FUSED_TAIL")) ctx->no_fused_tail = atoi(e) == 0;      // 0: separate head_tail_kernel (A/B, tests)
  if (const char* e = getenv("B2O_TC_PAIR")) {        // default 1; 0 = single-CTA tiles (A/B runs); 2 = generic tiles too
    ctx->tc_pair = atoi(e) != 0;
    ctx->tc_pair_generic = atoi(e) == 2;
  }
  *out = ctx;
  return B2O_OK;
}

extern "C" void b2o_destroy(b2o_ctx* ctx) {
  if (!ctx) return;
  {
    DeviceGuard guard(ctx->device);
    for (void* p : ctx->owned) cudaFree(p);
    for (cudaEvent_t e : ctx->prof_events) cudaEventDestroy(e);
    jpeg_release(ctx);
  }
  delete ctx;
}

extern "C" const char* b2o_last_error(const b2o_ctx* ctx) { return ctx ? ctx->error.c_str() : "null context"; }
extern "C" int64_t b2o_launch_count(const b2o_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" int b2o_profile_enable(b2o_ctx* ctx, int on) {
  if (!ctx) return B2O_ERR_ARG;
  for (cudaEvent_t e : ctx->prof_events) cudaEventDestroy(e);
  ctx->prof_events.clear();
  ctx->prof_flop = 0.0;
  ctx->profile = on != 0;
  return B2O_OK;
}

extern "C" int b2o_profile_read(b2o_ctx* ctx, double* tc_ms, double* tc_flop, int64_t* tc_launches) {
  if (!ctx || !tc_ms || !tc_flop || !tc_launches) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  double ms = 0.0;
  for (size_t i = 0; i + 1 < ctx->prof_events.size(); i += 2) {
    B2O_CUDA_CHECK(ctx, cudaEventSynchronize(ctx->prof_events[i + 1]));
    float t = 0.f;
    B2O_CUDA_CHECK(ctx, cudaEventElapsedTime(&t, ctx->prof_events[i], ctx->prof_events[i + 1]));
    ms += t;
  }
  *tc_ms = ms;
  *tc_flop = ctx->prof_flop;
  *tc_launches = static_cast<int64_t>(ctx->prof_events.size() / 2);
  return B2O_OK;
}

extern "C" int b2o_set_conv_engine(b2o_ctx* ctx, int engine) {
  if (!ctx || (engine != B2O_CONV_AUTO && engine != B2O_CONV_SIMT && engine != B2O_CONV_TC_GENERIC)) return B2O_ERR_ARG;
  ctx->conv_engine = engine;
  return B2O_OK;
}

extern "C" int b2o_load_craft(b2o_ctx* ctx, const b2o_tensor* tensors, int n) {
  if (!ctx || !tensors) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  TensorMap m;
  for (int i = 0; i < n; ++i) m[tensors[i].name] = &tensors[i];
  for (const CraftSpec& s : kCraft) {
    const int64_t wshape[4] = {s.cout, s.cin, s.k, s.k};
    const int64_t vshape[1] = {s.cout};
    const b2o_tensor* w = need(ctx, m, std::string(s.name) + ".weight", 4, wshape);
    const b2o_tensor* b = need(ctx, m, std::string(s.name) + ".bias", 1, vshape);
    if (!w || !b) return B2O_ERR_WEIGHTS;
    std::vector<float> s1 = ones(s.cout), t1 = tovec(b, s.cout);
    if (s.bn) {
      const b2o_tensor* g = need(ctx, m, std::string(s.bn) + ".weight", 1, vshape);
      const b2o_tensor* be = need(ctx, m, std::string(s.bn) + ".bias", 1, vshape);
      const b2o_tensor* mu = need(ctx, m, std::string(s.bn) + ".running_mean", 1, vshape);
      const b2o_tensor* var = need(ctx, m, std::string(s.bn) + ".running_var", 1, vshape);
      if (!g || !be || !mu || !var) return B2O_ERR_WEIGHTS;
      for (int o = 0; o < s.cout; ++o) {      // BN(eps=1e-5) folded around the conv bias (detection.py:95-97)
        const float sc = g->data[o] / sqrtf(var->data[o] + 1e-5f);
        s1[o] = sc;
        t1[o] = (b->data[o] - mu->data[o]) * sc + be->data[o];
      }
    }
    const float* wd = w->data;
    const int cin = s.cin, k = s.k;
    auto wget = [wd, cin, k](int o, int c, int ky, int kx) { return wd[((static_cast<size_t>(o) * cin + c) * k + ky) * k + kx]; };
    ConvLayer& L = ctx->craft[s.name];
    B2O_RETURN_IF(build_layer(ctx, L, s.name, s.cin, s.cout, s.k, s.dil, s.relu, wget, s1, t1, nullptr, nullptr, s.cin == 3));
    // decoder glue: upconvN.conv.0 reads Concatenate([upsampled decoder (cy channels), encoder tap]); the upsampling
    // commutes with this 1x1 convolution, so the layer is also kept as two halves -- ".y": the decoder columns, applied
    // at LOW resolution without bias / BN / ReLU; ".s": the tap columns at full resolution, whose epilogue adds the
    // upsampled ".y" result before the folded BN + ReLU (detection.py:65-84, 380-390)
    int cy = 0;
    if (std::string(s.name) == "upconv2.conv.0") cy = 256;
    if (std::string(s.name) == "upconv3.conv.0") cy = 128;
    if (std::string(s.name) == "upconv4.conv.0") cy = 64;
    if (cy) {
      auto wy = [wd, cin](int o, int c, int, int) { return wd[static_cast<size_t>(o) * cin + c]; };
      auto wsk = [wd, cin, cy](int o, int c, int, int) { return wd[static_cast<size_t>(o) * cin + cy + c]; };
      ConvLayer& Ly = ctx->craft[std::string(s.name) + ".y"];
      B2O_RETURN_IF(build_layer(ctx, Ly, std::string(s.name) + ".y", cy, s.cout, 1, 1, 0, wy, ones(s.cout),
                                std::vector<float>(s.cout, 0.0f), nullptr, nullptr, false));
      ConvLayer& Ls = ctx->craft[std::string(s.name) + ".s"];
      B2O_RETURN_IF(build_layer(ctx, Ls, std::string(s.name) + ".s", s.cin - cy, s.cout, 1, 1, s.relu, wsk, s1, t1, nullptr, nullptr, false));
    }
    if (s.cin == 3) {      // tensor-core stem: same filters over a 16-channel (zero-padded) input
      auto wget16 = [wd, cin, k](int o, int c, int ky, int kx) {
        return c < 3 ? wd[((static_cast<size_t>(o) * cin + c) * k + ky) * k + kx] : 0.0f;
      };
      ConvLayer& L16 = ctx->craft["stem16"];
      B2O_RETURN_IF(build_layer(ctx, L16, "stem16", 16, s.cout, s.k, 1, s.relu, wget16, s1, t1, nullptr, nullptr, false));
      L16.alg_cin = 3;
    }
  }
  ctx->craft_loaded = true;
  return B2O_OK;
}

extern "C" int b2o_load_crnn(b2o_ctx* ctx, const b2o_tensor* tensors, int n) {
  if (!ctx || !tensors) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  TensorMap m;
  for (int i = 0; i < n; ++i) m[tensors[i].name] = &tensors[i];
  struct Spec { const char* name; int cin, cout, k; const char* bn; };
  const Spec convs[] = {{"conv_1", 1, 64, 3, nullptr},    {"conv_2", 64, 128, 3, nullptr}, {"conv_3", 128, 256, 3, "bn_3"},
                        {"conv_4", 256, 256, 3, nullptr}, {"conv_5", 256, 512, 3, "bn_5"}, {"conv_6", 512, 512, 3, nullptr},
                        {"conv_7", 512, 512, 3, "bn_7"},  {"stn.conv_a", 512, 16, 5, nullptr}, {"stn.conv_b", 16, 32, 5, nullptr}};
  // build_model(stn=False) (recognition.py:196, 243): a checkpoint without the localisation net's tensors is the
  // recognizer without the spatial transformer -- the conv features go straight to the reshape + fc_9
  const bool has_stn = m.count("stn.conv_a.kernel") != 0;
  ctx->crnn_stn = has_stn;
  // build_model(color=True) (recognition.py:214): conv_1 takes 3 input channels (RGB crops, no gray conversion)
  auto c1 = m.find("conv_1.kernel");
  const int in_ch = (c1 != m.end() && c1->second->ndim == 4 && c1->second->shape[2] == 3) ? 3 : 1;
  ctx->crnn_in_ch = in_ch;
  for (const Spec& s0 : convs) {
    Spec s = s0;
    if (std::string(s.name) == "conv_1") s.cin = in_ch;
    if (!has_stn && std::string(s.name).rfind("stn.", 0) == 0) continue;
    const int64_t wshape[4] = {s.k, s.k, s.cin, s.cout};
    const int64_t vshape[1] = {s.cout};
    const b2o_tensor* w = need(ctx, m, std::string(s.name) + ".kernel", 4, wshape);
    const b2o_tensor* b = need(ctx, m, std::string(s.name) + ".bias", 1, vshape);
    if (!w || !b) return B2O_ERR_WEIGHTS;
    std::vector<float> s1 = ones(s.cout), t1 = tovec(b, s.cout), s2, t2;
    if (s.bn) {                                // BatchNormalization AFTER the ReLU, Keras eps = 1e-3
      const b2o_tensor* g = need(ctx, m, std::string(s.bn) + ".gamma", 1, vshape);
      const b2o_tensor* be = need(ctx, m, std::string(s.bn) + ".beta", 1, vshape);
      const b2o_tensor* mu = need(ctx, m, std::string(s.bn) + ".moving_mean", 1, vshape);
      const b2o_tensor* var = need(ctx, m, std::string(s.bn) + ".moving_variance", 1, vshape);
      if (!g || !be || !mu || !var) return B2O_ERR_WEIGHTS;
      s2.resize(s.cout); t2.resize(s.cout);
      for (int o = 0; o < s.cout; ++o) {
        const float sc = g->data[o] / sqrtf(var->data[o] + 1e-3f);
        s2[o] = sc;
        t2[o] = be->data[o] - mu->data[o] * sc;
      }
    }
    const float* wd = w->data;
    const int cin = s.cin, cout = s.cout, k = s.k;
    auto wget = [wd, cin, cout, k](int o, int c, int ky, int kx) {
      return wd[((static_cast<size_t>(ky) * k + kx) * cin + c) * cout + o];
    };
    ConvLayer& L = ctx->crnn[s.name];
    B2O_RETURN_IF(build_layer(ctx, L, s.name, s.cin, s.cout, s.k, 1, 1, wget, s1, t1, s.bn ? &s2 : nullptr,
                              s.bn ? &t2 : nullptr, std::string(s.name) == "conv_1"));
    if (std::string(s.name) == "stn.conv_a") {
      // The 5x5, 512 -> 16 convolution as ONE 1x1 GEMM with N = 25 taps x 16 channels (400, padded to 512)
      // followed by a shift-and-add of the 25 column groups (stn_col2im): 16-column MMAs cost as much tensor
      // pipe time as 64-column ones, 256-column ones are ~5x cheaper per output.
      auto wgemm = [wd, cin, cout, k](int o, int c, int, int) {
        return o < k * k * cout ? wd[(static_cast<size_t>(o / cout) * cin + c) * cout + (o % cout)] : 0.0f;
      };
      ConvLayer& G = ctx->crnn["stn.conv_a_gemm"];
      B2O_RETURN_IF(build_layer(ctx, G, "stn.conv_a_gemm", s.cin, 512, 1, 1, 0, wgemm, ones(512),
                                std::vector<float>(512, 0.0f), nullptr, nullptr, false));
      G.alg_cout = k * k * cout;                 // 400 of the 512 columns are real
    }
  }
  // dense layers as 1x1 "convolutions" over a (1,1,rows,K) view; their input widths follow the crop geometry:
  // Flatten of the (T, Hf, 32) localisation features, Reshape to (T, Hf*512) (recognition.py:275, 282)
  struct Dense { const char* name; int k, n, relu; };
  const CrnnGeometry& g = ctx->crnn_geom;
  const Dense dense[] = {{"stn.dense_a", g.steps() * g.feat_h() * 32, 64, 1}, {"fc_9", g.feat_h() * 512, 128, 1}};
  for (const Dense& d : dense) {
    if (!has_stn && std::string(d.name).rfind("stn.", 0) == 0) continue;
    const int64_t wshape[2] = {d.k, d.n};
    const int64_t vshape[1] = {d.n};
    const b2o_tensor* w = need(ctx, m, std::string(d.name) + ".kernel", 2, wshape);
    const b2o_tensor* b = need(ctx, m, std::string(d.name) + ".bias", 1, vshape);
    if (!w || !b) {
      ctx->set_error(ctx->error + " (expected (" + std::to_string(d.k) + ", " + std::to_string(d.n) + ") for crops of " +
                     std::to_string(g.height) + " x " + std::to_string(g.width) + ", see b2o_set_crnn_geometry)");
      return B2O_ERR_WEIGHTS;
    }
    const float* wd = w->data;
    const int nn = d.n;
    auto wget = [wd, nn](int o, int c, int, int) { return wd[static_cast<size_t>(c) * nn + o]; };
    ConvLayer& L = ctx->crnn[d.name];
    B2O_RETURN_IF(build_layer(ctx, L, d.name, d.k, d.n, 1, 1, d.relu, wget, ones(d.n), tovec(b, d.n), nullptr, nullptr, false));
  }
  if (has_stn) {
    const int64_t wshape[2] = {64, 6};
    const int64_t vshape[1] = {6};
    const b2o_tensor* w = need(ctx, m, "stn.dense_b.kernel", 2, wshape);
    const b2o_tensor* b = need(ctx, m, "stn.dense_b.bias", 1, vshape);
    if (!w || !b) return B2O_ERR_WEIGHTS;
    if (!(ctx->stn_d2_w = dev_upload(ctx, tovec(w, 64 * 6)))) return B2O_ERR_CUDA;
    if (!(ctx->stn_d2_b = dev_upload(ctx, tovec(b, 6)))) return B2O_ERR_CUDA;
  }
  // LSTM input projections: forward and go_backwards kernels side by side -> one GEMM per layer
  const char* lstm_names[4] = {"lstm_10", "lstm_10_back", "lstm_11", "lstm_11_back"};
  for (int layer = 0; layer < 2; ++layer) {
    const int64_t wshape[2] = {128, 512};
    const int64_t vshape[1] = {512};
    const b2o_tensor* wf = need(ctx, m, std::string(lstm_names[2 * layer]) + ".kernel", 2, wshape);
    const b2o_tensor* wb = need(ctx, m, std::string(lstm_names[2 * layer + 1]) + ".kernel", 2, wshape);
    const b2o_tensor* bf = need(ctx, m, std::string(lstm_names[2 * layer]) + ".bias", 1, vshape);
    const b2o_tensor* bb = need(ctx, m, std::string(lstm_names[2 * layer + 1]) + ".bias", 1, vshape);
    if (!wf || !wb || !bf || !bb) return B2O_ERR_WEIGHTS;
    const float* f = wf->data;
    const float* bk = wb->data;
    auto wget = [f, bk](int o, int c, int, int) { return o < 512 ? f[c * 512 + o] : bk[c * 512 + (o - 512)]; };
    std::vector<float> bias(1024);
    for (int i = 0; i < 512; ++i) { bias[i] = bf->data[i]; bias[512 + i] = bb->data[i]; }
    const std::string lname = layer == 0 ? "lstm_in_1" : "lstm_in_2";
    ConvLayer& L = ctx->crnn[lname];
    B2O_RETURN_IF(build_layer(ctx, L, lname, 128, 1024, 1, 1, 0, wget, ones(1024), bias, nullptr, nullptr, false));
    for (int dir = 0; dir < 2; ++dir) {
      const b2o_tensor* u = need(ctx, m, std::string(lstm_names[2 * layer + dir]) + ".recurrent_kernel", 2, wshape);
      if (!u) return B2O_ERR_WEIGHTS;
      std::vector<__half> uh(128 * 512);
      for (int i = 0; i < 128 * 512; ++i) uh[i] = __float2half_rn(u->data[i]);
      if (!(ctx->lstm_u[2 * layer + dir] = dev_upload(ctx, uh))) return B2O_ERR_CUDA;
    }
  }
  {
    // Dense(len(alphabet)+1) (recognition.py:322-327, 376-381): the class count comes from the tensor itself
    auto fc = m.find("fc_12.kernel");
    const int64_t K = fc != m.end() && fc->second->ndim == 2 ? fc->second->shape[1] : 0;
    if (K < 2 || K > B2O_MAX_CLASSES) { ctx->set_error("fc_12.kernel must be (256, K) with 2 <= K <= 1024"); return B2O_ERR_WEIGHTS; }
    const int64_t wshape[2] = {256, K};
    const int64_t vshape[1] = {K};
    const b2o_tensor* w = need(ctx, m, "fc_12.kernel", 2, wshape);
    const b2o_tensor* b = need(ctx, m, "fc_12.bias", 1, vshape);
    if (!w || !b) return B2O_ERR_WEIGHTS;
    if (!(ctx->fc12_w = dev_upload(ctx, tovec(w, 256 * K)))) return B2O_ERR_CUDA;
    if (!(ctx->fc12_b = dev_upload(ctx, tovec(b, K)))) return B2O_ERR_CUDA;
    ctx->n_classes = static_cast<int>(K);
  }
  ctx->crnn_loaded = true;
  return B2O_OK;
}

extern "C" int b2o_set_crnn_geometry(b2o_ctx* ctx, int height, int width, int rnn_steps_to_discard) {
  if (!ctx) return B2O_ERR_ARG;
  if (height < B2O_CRNN_MIN_HEIGHT || height > B2O_CRNN_MAX_HEIGHT || width < B2O_CRNN_MIN_WIDTH || width > B2O_CRNN_MAX_WIDTH ||
      rnn_steps_to_discard < 0 || rnn_steps_to_discard >= width / 4) {
    ctx->set_error("b2o_set_crnn_geometry: unsupported geometry " + std::to_string(height) + " x " + std::to_string(width) +
                   ", " + std::to_string(rnn_steps_to_discard) + " steps discarded");
    return B2O_ERR_ARG;
  }
  if (ctx->crnn_loaded) { ctx->set_error("b2o_set_crnn_geometry: call it before b2o_load_crnn"); return B2O_ERR_STATE; }
  ctx->crnn_geom.height = height;
  ctx->crnn_geom.width = width;
  ctx->crnn_geom.discard = rnn_steps_to_discard;
  return B2O_OK;
}

// ------------------------------------------------------------------------------------------------
extern "C" size_t b2o_craft_workspace_bytes(int n, int h, int w) {
  if (n <= 0 || h < 32 || w < 32) return 0;
  return plan_craft(n, h, w).bytes;
}

extern "C" int b2o_craft_forward(b2o_ctx* ctx, const uint8_t* img, int n, int h, int w, float* scores, void* ws,
                                 size_t ws_bytes, void* stream) {
  if (!ctx) return B2O_ERR_ARG;
  if (!ctx->craft_loaded) { ctx->set_error("b2o_craft_forward: CRAFT weights not loaded"); return B2O_ERR_STATE; }
  DeviceGuard guard(ctx->device);
  if (!img || !scores || !ws || n <= 0 || h < 32 || w < 32) { ctx->set_error("b2o_craft_forward: bad argument"); return B2O_ERR_ARG; }
  const CraftPlan p = plan_craft(n, h, w);
  if (ws_bytes < p.bytes) { ctx->set_error("b2o_craft_forward: workspace too small"); return B2O_ERR_WORKSPACE; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* base = reinterpret_cast<uint8_t*>(ws);
  auto V = [&](size_t off, int hh, int ww, int c, int ld = 0, int coff = 0) { return make_view(base + off, n, hh, ww, c, ld, coff); };
  auto L = [&](const char* name) -> const ConvLayer& { return ctx->craft[name]; };

  const TensorView a = V(p.off_a, p.h1, p.w1, 64), b = V(p.off_b, p.h1, p.w1, 64), p1 = V(p.off_p1, p.h2, p.w2, 64);
  const TensorView c = V(p.off_c, p.h2, p.w2, 128);
  const TensorView cat4 = V(p.off_cat4, p.h2, p.w2, 192), cat4_y = V(p.off_cat4, p.h2, p.w2, 64, 192, 0),
                   s1 = V(p.off_cat4, p.h2, p.w2, 128, 192, 64);
  const TensorView p2 = V(p.off_p2, p.h4, p.w4, 128), d = V(p.off_d, p.h4, p.w4, 256);
  const TensorView cat3 = V(p.off_cat3, p.h4, p.w4, 384), cat3_y = V(p.off_cat3, p.h4, p.w4, 128, 384, 0),
                   s2 = V(p.off_cat3, p.h4, p.w4, 256, 384, 128);
  const TensorView e = V(p.off_e, p.h4, p.w4, 256), p3 = V(p.off_p3, p.h8, p.w8, 256), f = V(p.off_f, p.h8, p.w8, 512);
  const TensorView cat2 = V(p.off_cat2, p.h8, p.w8, 768), cat2_y = V(p.off_cat2, p.h8, p.w8, 256, 768, 0),
                   s3 = V(p.off_cat2, p.h8, p.w8, 512, 768, 256);
  const TensorView g = V(p.off_g, p.h8, p.w8, 512), p4 = V(p.off_p4, p.h16, p.w16, 512), hh = V(p.off_hh, p.h16, p.w16, 512);
  const TensorView cat1 = V(p.off_cat1, p.h16, p.w16, 1536), s5 = V(p.off_cat1, p.h16, p.w16, 1024, 1536, 0),
                   s4 = V(p.off_cat1, p.h16, p.w16, 512, 1536, 1024);
  const TensorView mp = V(p.off_mp, p.h16, p.w16, 512), s5a = V(p.off_s5a, p.h16, p.w16, 1024);
  const TensorView u1a = V(p.off_u1a, p.h16, p.w16, 512), u1b = V(p.off_u1b, p.h16, p.w16, 256);
  const TensorView u2a = V(p.off_u2a, p.h8, p.w8, 256), u2b = V(p.off_u2b, p.h8, p.w8, 128);
  const TensorView u3a = V(p.off_u3a, p.h4, p.w4, 128), u3b = V(p.off_u3b, p.h4, p.w4, 64);
  const TensorView u4a = V(p.off_u4a, p.h2, p.w2, 64), u4b = V(p.off_u4b, p.h2, p.w2, 32);
  const TensorView h1 = V(p.off_h1, p.h2, p.w2, 32), h2 = V(p.off_h2, p.h2, p.w2, 32), h3 = V(p.off_h3, p.h2, p.w2, 16);

  // encoder (detection.py:312-324); taps s1..s4 are written straight into the concat buffers
  if (ctx->conv_engine == B2O_CONV_SIMT || L("stem16").block_n == 0) {
    B2O_RETURN_IF(stem_rgb_run(ctx, L("basenet.slice1.0"), img, n, h, w, a, st));          // fp32 CUDA-core stem
  } else {
    const TensorView x16 = V(p.off_x16, p.h1, p.w1, 16);
    B2O_RETURN_IF(normalize16_run(ctx, img, n, h, w, x16.ptr, st));
    B2O_RETURN_IF(conv_run(ctx, L("stem16"), x16, a, 0, st));
  }
  B2O_RETURN_IF(conv_run(ctx, L("basenet.slice1.3"), a, b, 0, st, &p1, 0));     // conv + fused 2x2 max pool
  B2O_RETURN_IF(conv_run(ctx, L("basenet.slice1.7"), p1, c, 0, st));
  B2O_RETURN_IF(conv_run(ctx, L("basenet.slice1.10"), c, s1, 0, st, &p2, 1));   // tap s1 (full) + pooled
  B2O_RETURN_IF(conv_run(ctx, L("basenet.slice2.14"), p2, d, 0, st));
  B2O_RETURN_IF(conv_run(ctx, L("basenet.slice2.17"), d, s2, 0, st));
  B2O_RETURN_IF(conv_run(ctx, L("basenet.slice3.20"), s2, e, 0, st, &p3, 0));
  B2O_RETURN_IF(conv_run(ctx, L("basenet.slice3.24"), p3, f, 0, st));
  B2O_RETURN_IF(conv_run(ctx, L("basenet.slice3.27"), f, s3, 0, st));
  B2O_RETURN_IF(conv_run(ctx, L("basenet.slice4.30"), s3, g, 0, st, &p4, 0));
  B2O_RETURN_IF(conv_run(ctx, L("basenet.slice4.34"), p4, hh, 0, st));
  B2O_RETURN_IF(conv_run(ctx, L("basenet.slice4.37"), hh, s4, 0, st));          // BN only, no ReLU (333)
  // slice5 (365-378)
  B2O_RETURN_IF(maxpool3s1_run(ctx, s4, mp, st));
  B2O_RETURN_IF(conv_run(ctx, L("basenet.slice5.1"), mp, s5a, 0, st));
  B2O_RETURN_IF(conv_run(ctx, L("basenet.slice5.2"), s5a, s5, 0, st));
  // decoder (380-390)
  B2O_RETURN_IF(conv_run(ctx, L("upconv1.conv.0"), cat1, u1a, 0, st));
  B2O_RETURN_IF(conv_run(ctx, L("upconv1.conv.3"), u1a, u1b, 0, st));
  // UpsampleLike + Concatenate + 1x1 conv (380-390).  Opt-in (B2O_UPCONV_COMMUTE=1): where the skip tensor is exactly
  // twice the decoder tensor the upsampling is commuted behind the convolution -- the decoder half of the 1x1 conv runs
  // at LOW resolution and the full-resolution half adds its bilinear upsampling in the epilogue, so no upsampled tensor
  // is written or read back.  Correct (tests) but slower than the explicit UpsampleLike on B200, hence not the default.
  auto level = [&](const char* name, const TensorView& y, const TensorView& cat_y, const TensorView& cat, const TensorView& skip,
                   size_t off_z, const TensorView& out) -> int {
    const std::string base(name);
    const bool commute = ctx->conv_engine == B2O_CONV_AUTO && !ctx->no_commute && skip.h == 2 * y.h && skip.w == 2 * y.w &&
                         ctx->craft[base + ".y"].block_n != 0 && ctx->craft[base + ".s"].kch == 64 && ctx->craft[base + ".s"].block_n >= 64;
    if (!commute) {
      B2O_RETURN_IF(upsample_run(ctx, y, cat_y, st));
      return conv_run(ctx, ctx->craft[base], cat, out, 0, st);
    }
    const TensorView z = V(off_z, y.h, y.w, out.c);
    B2O_RETURN_IF(conv_run(ctx, ctx->craft[base + ".y"], y, z, 0, st));
    return conv_tc_run(ctx, ctx->craft[base + ".s"], skip, out, 0, st, nullptr, 1, nullptr, &z);
  };
  B2O_RETURN_IF(level("upconv2.conv.0", u1b, cat2_y, cat2, s3, p.off_z2, u2a));
  B2O_RETURN_IF(conv_run(ctx, L("upconv2.conv.3"), u2a, u2b, 0, st));
  B2O_RETURN_IF(level("upconv3.conv.0", u2b, cat3_y, cat3, s2, p.off_z3, u3a));
  B2O_RETURN_IF(conv_run(ctx, L("upconv3.conv.3"), u3a, u3b, 0, st));
  B2O_RETURN_IF(level("upconv4.conv.0", u3b, cat4_y, cat4, s1, p.off_z4, u4a));
  B2O_RETURN_IF(conv_run(ctx, L("upconv4.conv.3"), u4a, u4b, 0, st));
  // head (392-410)
  B2O_RETURN_IF(conv_run(ctx, L("conv_cls.0"), u4b, h1, 0, st));
  B2O_RETURN_IF(conv_run(ctx, L("conv_cls.2"), h1, h2, 0, st));
  if (ctx->conv_engine == B2O_CONV_AUTO && L("conv_cls.4").block_n == 16 && !ctx->no_fused_tail) {
    // conv_cls.6 + conv_cls.8 ride in conv_cls.4's epilogue (same arithmetic as head_tail_kernel, bit for bit):
    // one launch and the 16-channel map's round trip through HBM less
    const ConvLayer &L6 = L("conv_cls.6"), &L8 = L("conv_cls.8");
    ConvTail tail = {L6.w_simt, L6.t1, L8.w_simt, L8.t1, scores};
    if (L6.h_w_simt.size() == 256 && L8.h_w_simt.size() == 32) {
      tail.h_w6 = L6.h_w_simt.data(); tail.h_b6 = L6.h_t1.data(); tail.h_w8 = L8.h_w_simt.data(); tail.h_b8 = L8.h_t1.data();
    }
    B2O_RETURN_IF(conv_tc_run(ctx, L("conv_cls.4"), h2, h3, 0, st, nullptr, 1, &tail));
  } else {
    B2O_RETURN_IF(conv_run(ctx, L("conv_cls.4"), h2, h3, 0, st));
    B2O_RETURN_IF(head_tail_run(ctx, L("conv_cls.6"), L("conv_cls.8"), h3, scores, st));
  }
  return B2O_OK;
}

// ------------------------------------------------------------------------------------------------
extern "C" size_t b2o_crnn_workspace_bytes(int b) { return b > 0 ? plan_crnn(b, CrnnGeometry()).bytes : 0; }

extern "C" size_t b2o_crnn_workspace_bytes_for(const b2o_ctx* ctx, int b) {
  return ctx && b > 0 ? plan_crnn(b, ctx->crnn_geom).bytes : 0;
}

extern "C" int b2o_crnn_forward(b2o_ctx* ctx, const void* crnn_in, int b, int32_t* labels, void* ws, size_t ws_bytes,
                                void* stream) {
  if (!ctx) return B2O_ERR_ARG;
  if (!ctx->crnn_loaded) { ctx->set_error("b2o_crnn_forward: CRNN weights not loaded"); return B2O_ERR_STATE; }
  DeviceGuard guard(ctx->device);
  if (b == 0) return B2O_OK;
  if (!crnn_in || !labels || !ws || b < 0) { ctx->set_error("b2o_crnn_forward: bad argument"); return B2O_ERR_ARG; }
  const CrnnGeometry& g = ctx->crnn_geom;
  const CrnnPlan p = plan_crnn(b, g);
  if (ws_bytes < p.bytes) { ctx->set_error("b2o_crnn_forward: workspace too small"); return B2O_ERR_WORKSPACE; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* base = reinterpret_cast<uint8_t*>(ws);
  auto V = [&](size_t off, int nn, int hh, int ww, int c) { return make_view(base + off, nn, hh, ww, c); };
  auto L = [&](const char* name) -> const ConvLayer& { return ctx->crnn[name]; };
  const int W0 = g.width, H0 = g.height, W1 = W0 / 2, H1 = H0 / 2, T = g.steps(), Hf = g.feat_h();
  const TensorView x1 = V(p.off_x1, b, W0, H0, 64), x2 = V(p.off_x2, b, W0, H0, 128), x3 = V(p.off_x3, b, W0, H0, 256);
  const TensorView p3 = V(p.off_p3, b, W1, H1, 256), x4 = V(p.off_x4, b, W1, H1, 256), x5 = V(p.off_x5, b, W1, H1, 512);
  const TensorView p5 = V(p.off_p5, b, T, Hf, 512), x6 = V(p.off_x6, b, T, Hf, 512), x7 = V(p.off_x7, b, T, Hf, 512);
  const TensorView sa = V(p.off_sa, b, T, Hf, 16), sb = V(p.off_sb, b, T, Hf, 32);
  // conv stack (recognition.py:217-242)
  B2O_RETURN_IF(stem_crnn_run(ctx, L("conv_1"), reinterpret_cast<const __half*>(crnn_in), b, x1, st));
  B2O_RETURN_IF(conv_run(ctx, L("conv_2"), x1, x2, 0, st));
  B2O_RETURN_IF(conv_run(ctx, L("conv_3"), x2, x3, 0, st, &p3, 0));
  B2O_RETURN_IF(conv_run(ctx, L("conv_4"), p3, x4, 0, st));
  B2O_RETURN_IF(conv_run(ctx, L("conv_5"), x4, x5, 0, st, &p5, 0));
  B2O_RETURN_IF(conv_run(ctx, L("conv_6"), p5, x6, 0, st));
  B2O_RETURN_IF(conv_run(ctx, L("conv_7"), x6, x7, 0, st));
  __half* warped = reinterpret_cast<__half*>(base + p.off_warp);
  if (!ctx->crnn_stn) {
    warped = x7.ptr;                                      // stn=False: Reshape consumes bn_7's output directly (282)
  } else {
  // spatial transformer (263-281)
  if (ctx->conv_engine == B2O_CONV_AUTO && L("stn.conv_a_gemm").block_n != 0) {
    const TensorView y = V(p.off_warp, b, T, Hf, 512);   // the warp buffer is free until stn_sample
    B2O_RETURN_IF(conv_run(ctx, L("stn.conv_a_gemm"), x7, y, 0, st));
    B2O_RETURN_IF(stn_col2im_run(ctx, y.ptr, L("stn.conv_a").t1, b, T, Hf, sa.ptr, st));
  } else {
    B2O_RETURN_IF(conv_run(ctx, L("stn.conv_a"), x7, sa, 0, st));
  }
  B2O_RETURN_IF(conv_run(ctx, L("stn.conv_b"), sa, sb, 0, st));
  const TensorView sb_flat = make_view(base + p.off_sb, 1, 1, b, T * Hf * 32), d1 = make_view(base + p.off_d1, 1, 1, b, 64);
  B2O_RETURN_IF(conv_run(ctx, L("stn.dense_a"), sb_flat, d1, 0, st));
  float* theta = reinterpret_cast<float*>(base + p.off_theta);
  B2O_RETURN_IF(stn_theta_run(ctx, d1.ptr, b, theta, st));
  B2O_RETURN_IF(stn_sample_run(ctx, x7.ptr, theta, b, T, Hf, warped, st));
  }
  // reshape + fc_9 (282-290)
  const TensorView seq_in = make_view(warped, 1, 1, b * T, Hf * 512), fc9 = make_view(base + p.off_fc9, 1, 1, b * T, 128);
  B2O_RETURN_IF(conv_run(ctx, L("fc_9"), seq_in, fc9, 0, st));
  // BiLSTM (292-319)
  const TensorView xw1 = make_view(base + p.off_xw1, 1, 1, b * T, 1024);
  TensorView xw1v = xw1;      // fp32 output: the view's pointer arithmetic is done by the engine in floats
  B2O_RETURN_IF(conv_run(ctx, L("lstm_in_1"), fc9, xw1v, 1, st));
  __half* hf = reinterpret_cast<__half*>(base + p.off_hf);
  __half* hb = reinterpret_cast<__half*>(base + p.off_hb);
  __half* l1 = reinterpret_cast<__half*>(base + p.off_l1);
  const float* xw1f = reinterpret_cast<const float*>(base + p.off_xw1);
  B2O_RETURN_IF(lstm_run(ctx, xw1f, 1024, 0, ctx->lstm_u[0], b, T, 0, hf, 128, 0, st));
  B2O_RETURN_IF(lstm_run(ctx, xw1f, 1024, 512, ctx->lstm_u[1], b, T, 1, hb, 128, 0, st));
  B2O_RETURN_IF(add_run(ctx, hf, hb, l1, static_cast<long long>(b) * T * 128, st));
  const TensorView l1v = make_view(l1, 1, 1, b * T, 128), xw2 = make_view(base + p.off_xw2, 1, 1, b * T, 1024);
  B2O_RETURN_IF(conv_run(ctx, L("lstm_in_2"), l1v, xw2, 1, st));
  const float* xw2f = reinterpret_cast<const float*>(base + p.off_xw2);
  __half* l2 = reinterpret_cast<__half*>(base + p.off_l2);
  B2O_RETURN_IF(lstm_run(ctx, xw2f, 1024, 0, ctx->lstm_u[2], b, T, 0, l2, 256, 0, st));
  B2O_RETURN_IF(lstm_run(ctx, xw2f, 1024, 512, ctx->lstm_u[3], b, T, 1, l2, 256, 128, st));
  // fc_12 + discard + greedy CTC (321-333)
  B2O_RETURN_IF(fc_ctc_run(ctx, l2, b, T, g.discard, ctx->debug_taps ? reinterpret_cast<float*>(base + p.off_logits) : nullptr, labels, st));
  return B2O_OK;
}

extern "C" int b2o_set_debug_taps(b2o_ctx* ctx, int on) {
  if (!ctx) return B2O_ERR_ARG;
  ctx->debug_taps = on != 0;
  return B2O_OK;
}

extern "C" int b2o_crnn_tap(b2o_ctx* ctx, const char* name, const void* ws, int b, void* out, size_t out_bytes, void* stream) {
  if (!ctx || !name || !ws || !out || b <= 0) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  const CrnnGeometry& g = ctx->crnn_geom;
  const CrnnPlan p = plan_crnn(b, g);
  const size_t B = static_cast<size_t>(b), T = g.steps(), Hf = g.feat_h();
  size_t off = 0, bytes = 0;
  const std::string s(name);
  if (s == "features") { off = p.off_x7; bytes = B * T * Hf * 512 * 2; }
  else if ((s == "theta" || s == "warped") && !ctx->crnn_stn) { ctx->set_error("b2o_crnn_tap: this recognizer has no spatial transformer"); return B2O_ERR_STATE; }
  else if (s == "theta") { off = p.off_theta; bytes = B * 6 * 4; }
  else if (s == "warped") { off = p.off_warp; bytes = B * T * Hf * 512 * 2; }
  else if (s == "fc_9") { off = p.off_fc9; bytes = B * T * 128 * 2; }
  else if (s == "l1") { off = p.off_l1; bytes = B * T * 128 * 2; }
  else if (s == "l2") { off = p.off_l2; bytes = B * T * 256 * 2; }
  else if (s == "logits") {
    if (!ctx->debug_taps) { ctx->set_error("b2o_crnn_tap: logits are only kept after b2o_set_debug_taps(ctx, 1)"); return B2O_ERR_STATE; }
    off = p.off_logits; bytes = B * g.keep() * ctx->n_classes * 4;
  }
  else { ctx->set_error("b2o_crnn_tap: unknown tap " + s); return B2O_ERR_ARG; }
  if (out_bytes < bytes) { ctx->set_error("b2o_crnn_tap: output too small"); return B2O_ERR_ARG; }
  B2O_CUDA_CHECK(ctx, cudaMemcpyAsync(out, reinterpret_cast<const uint8_t*>(ws) + off, bytes, cudaMemcpyDeviceToDevice,
                                      reinterpret_cast<cudaStream_t>(stream)));
  return B2O_OK;
}

extern "C" int b2o_conv2d_test(b2o_ctx* ctx, const void* x, int n, int h, int w, int cin, const float* wgt, int cout,
                               int ksize, int dilation, const float* s1, const float* t1, int relu, const float* s2,
                               const float* t2, void* out, int engine, void* stream) {
  if (!ctx || !x || !wgt || !s1 || !t1 || !out) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  const size_t owned_before = ctx->owned.size();
  ConvLayer L;
  auto wget = [wgt, cin, ksize](int o, int c, int ky, int kx) {
    return wgt[((static_cast<size_t>(o) * ksize + ky) * ksize + kx) * cin + c];
  };
  std::vector<float> vs1(s1, s1 + cout), vt1(t1, t1 + cout), vs2, vt2;
  if (s2 && t2) { vs2.assign(s2, s2 + cout); vt2.assign(t2, t2 + cout); }
  int rc = build_layer(ctx, L, "test", cin, cout, ksize, dilation, relu, wget, vs1, vt1, s2 ? &vs2 : nullptr,
                       s2 ? &vt2 : nullptr, false);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (rc == B2O_OK) {
    const TensorView in = make_view(const_cast<void*>(x), n, h, w, cin), o = make_view(out, n, h, w, cout);
    const int saved = ctx->conv_engine;
    ctx->conv_engine = engine;
    if (engine == B2O_CONV_SIMT) rc = conv_simt_run(ctx, L, in, o, 0, st);
    else rc = conv_tc_run(ctx, L, in, o, 0, st);
    ctx->conv_engine = saved;
  }
  cudaError_t e = cudaStreamSynchronize(st);
  if (rc == B2O_OK && e != cudaSuccess) { ctx->set_error(std::string("conv2d_test: ") + cudaGetErrorString(e)); rc = B2O_ERR_CUDA; }
  while (ctx->owned.size() > owned_before) { cudaFree(ctx->owned.back()); ctx->owned.pop_back(); }
  return rc;
}
