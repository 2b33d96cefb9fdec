// boxes.cu -- getBoxes (reference keras_ocr/detection.py:207-287) on the GPU.
//
//   binarize_kernel   cv2.threshold x2 (strict >, 221-226) + union mask (228) + label init
//   merge/flatten     cv2.connectedComponentsWithStats(connectivity=4) (227-229): union-find whose
//                     root is the smallest pixel index of the component, i.e. its first pixel in
//                     raster order -- OpenCV numbers labels in exactly that order
//   stats_kernel      area / bbox (stats[...]) and np.max(textmap[labels == id]) (233-241)
//   select_kernel     size + detection-threshold filters, order-preserving compaction
//   quads_kernel      per kept component: segmap minus (text & link) (244-246), rectangular dilation
//                     in the ROI (258-264), last 8-connected blob == contours[0] of findContours
//                     (267-272), convex hull + rotating calipers == cv2.minAreaRect + boxPoints (273),
//                     diamond test (276-281), clockwise roll (284), x2 (285)
//
// All score-map traffic is coalesced; the per-component work lives in shared-memory bit planes.
#include <math.h>

#include "common.cuh"

namespace {

constexpr int kMaxHullRows = 2048;      // score maps are at most 1024 rows (max_size 2048 / 2)

struct Component {                       // one kept connected component
  int root, x, y, w, h, area;
};

// cv2.threshold x2 + union mask + label init.  A pixel's initial label is the start of its horizontal run
// inside the warp's 32-pixel segment (ballot + clz), so row runs need no union at all except across
// segment boundaries -- this removes >90 % of the atomics of the merge pass.
__global__ void binarize_kernel(const float* __restrict__ scores, long long total, int hw, int ws, float text_thr,
                                float link_thr, uint8_t* __restrict__ mask, int* __restrict__ label) {
  const long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  bool fg = false, both = false;
  int q = 0, row = -1;
  if (p < total) {
    const float2 s = reinterpret_cast<const float2*>(scores)[p];
    const bool t = s.x > text_thr, l = s.y > link_thr;
    fg = t || l; both = t && l;
    q = static_cast<int>(p % hw);
    row = static_cast<int>(p / ws);                       // global row id (image * hs + y)
  }
  const uint32_t same_row = __match_any_sync(0xffffffffu, row);
  const uint32_t m = __ballot_sync(0xffffffffu, fg) & same_row;
  if (p >= total) return;
  int lab = -1, run = 0;
  if (fg) {
    const uint32_t below = (lane == 0) ? 0u : (m << (32 - lane));   // bit (lane-1) -> bit 31
    run = __clz(~below);                                           // consecutive foreground pixels to the left
    if (run > lane) run = lane;
    lab = q - run;
  }
  // mask bits: 1 = foreground, 2 = text & link, 4 = first pixel of its run inside this 32-pixel segment
  mask[p] = static_cast<uint8_t>(fg ? (1 | (both ? 2 : 0) | (run == 0 ? 4 : 0)) : 0);
  label[p] = lab;
}

__device__ __forceinline__ int uf_find(const int* L, int a) {
  while (true) {
    const int p = *reinterpret_cast<const volatile int*>(L + a);
    if (p == a) return a;
    a = p;
  }
}
__device__ __forceinline__ void uf_unite(int* L, int a, int b) {
  while (true) {
    a = uf_find(L, a);
    b = uf_find(L, b);
    if (a == b) return;
    if (a < b) { const int t = a; a = b; b = t; }
    const int old = atomicMin(L + a, b);     // hang the larger root under the smaller one
    if (old == a) return;
    a = old;
  }
}

__global__ void merge_kernel(const uint8_t* __restrict__ mask, int* __restrict__ label, long long total, int hs,
                             int ws) {
  const long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= total) return;
  if (!(mask[p] & 1)) return;
  const int hw = hs * ws;
  const int img = static_cast<int>(p / hw);
  const int q = static_cast<int>(p % hw);
  const int x = q % ws, y = q / ws;
  int* L = label + static_cast<size_t>(img) * hw;
  const bool left = x > 0 && (mask[p - 1] & 1);
  // horizontal: only where the warp-segment run labelling of binarize_kernel could not see the neighbour
  if (left && (mask[p] & 4)) uf_unite(L, q, q - 1);
  // vertical: once per pair of overlapping runs (if left and up-left are foreground, `left` already did it)
  if (y > 0 && (mask[p - ws] & 1)) {
    const bool upleft = x > 0 && (mask[p - ws - 1] & 1);
    if (!(left && upleft)) uf_unite(L, q, q - ws);
  }
}

__global__ void flatten_kernel(int* __restrict__ label, long long total, int hw) {
  const long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= total) return;
  if (label[p] < 0) return;
  int* L = label + (p / hw) * hw;
  label[p] = uf_find(L, static_cast<int>(p % hw));
}

// order-preserving int key for atomicMax over floats
__device__ __forceinline__ int float_key(float f) {
  const int b = __float_as_int(f);
  return b >= 0 ? b : b ^ 0x7fffffff;
}

struct Stats {        // indexed by root pixel
  int* area; int* minx; int* maxx; int* miny; int* maxy; int* maxtext;
};

// Warp-aggregated: the lanes of a warp that belong to the same component (usually one run of a word blob)
// reduce their contribution with __reduce_*_sync over their __match_any group and the group's first lane
// issues the six atomics -- one set per run instead of one per pixel on the same ~32 hot addresses per image.
__global__ void stats_kernel(const float* __restrict__ scores, const int* __restrict__ label, long long total,
                             int hw, int ws, Stats st) {
  const long long p = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int r = p < total ? label[p] : -1;
  const uint32_t active = __ballot_sync(0xffffffffu, r >= 0);
  if (r < 0) return;
  const long long base = (p / hw) * hw;
  const int q = static_cast<int>(p - base);
  const int x = q % ws, y = q / ws;
  const long long ri = base + r;
  const uint32_t grp = __match_any_sync(active, ri);
  const int minx = __reduce_min_sync(grp, x), maxx = __reduce_max_sync(grp, x);
  const int miny = __reduce_min_sync(grp, y), maxy = __reduce_max_sync(grp, y);
  const int mt = __reduce_max_sync(grp, float_key(scores[2 * p]));
  if ((threadIdx.x & 31) == __ffs(grp) - 1) {
    atomicAdd(st.area + ri, __popc(grp));
    atomicMin(st.minx + ri, minx);
    atomicMax(st.maxx + ri, maxx);
    atomicMin(st.miny + ri, miny);
    atomicMax(st.maxy + ri, maxy);
    atomicMax(st.maxtext + ri, mt);
  }
}

// One CTA per image: walk the pixels in raster order, keep roots that pass the filters
// (detection.py:233-241) and compact them -- the slot order is the reference's label order.
// Each thread looks at 4 consecutive pixels per round; rounds without any kept root (almost all of them:
// a page has tens of components in 590k pixels) cost one __syncthreads_or.
__global__ void __launch_bounds__(1024)
select_kernel(const int* __restrict__ label, int hw, Stats st, int size_thr, float det_thr, Component* __restrict__ comps,
              int max_boxes, int* __restrict__ counts) {
  __shared__ int warp_sums[32];
  __shared__ int carry;
  const int img = blockIdx.x;
  const long long base = static_cast<long long>(img) * hw;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int det_key = float_key(det_thr);
  const bool vec = (hw % 4 == 0);                          // rows of int4 stay aligned for every image
  for (int start = 0; start < hw; start += 4 * blockDim.x) {
    const int q0 = start + 4 * threadIdx.x;
    int lab[4] = {-1, -1, -1, -1};
    if (vec && q0 + 3 < hw) {
      const int4 v4 = *reinterpret_cast<const int4*>(label + base + q0);
      lab[0] = v4.x; lab[1] = v4.y; lab[2] = v4.z; lab[3] = v4.w;
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (q0 + e < hw) lab[e] = label[base + q0 + e];
    }
    int keepmask = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (lab[e] == q0 + e) {
        // "size < size_threshold -> skip" and "max < detection_threshold -> skip"
        if ((st.area[base + q0 + e] >= size_thr) && (st.maxtext[base + q0 + e] >= det_key)) keepmask |= 1 << e;
      }
    if (!__syncthreads_or(keepmask)) continue;             // block-uniform
    const int cnt = __popc(keepmask);
    int v = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += t;
    }
    if (lane == 31) warp_sums[wid] = v;
    __syncthreads();
    if (wid == 0) {
      int sacc = warp_sums[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, sacc, o);
        if (lane >= o) sacc += t;
      }
      warp_sums[lane] = sacc;
    }
    __syncthreads();
    int slot = carry + (wid ? warp_sums[wid - 1] : 0) + v - cnt;
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (keepmask & (1 << e)) {
        if (slot < max_boxes) {
          const int q = q0 + e;
          Component c;
          c.root = q;
          c.x = st.minx[base + q];
          c.y = st.miny[base + q];
          c.w = st.maxx[base + q] - c.x + 1;
          c.h = st.maxy[base + q] - c.y + 1;
          c.area = st.area[base + q];
          comps[static_cast<size_t>(img) * max_boxes + slot] = c;
        }
        ++slot;
      }
    __syncthreads();
    if (threadIdx.x == 0) carry += warp_sums[31];
    __syncthreads();
  }
  if (threadIdx.x == 0) counts[img] = carry;
}

// --------------------------------------------------------------------------- geometry (one thread)
struct P2 { float x, y; };

// cv2.minAreaRect's rotating calipers on a convex polygon, fp32 like OpenCV (no fma contraction).
__device__ void rotating_calipers(const P2* pts, int n, float* vect_x, float* vect_y, float* inv_len, float* out) {
  int left = 0, bottom = 0, right = 0, top = 0;
  P2 pt0 = pts[0];
  float left_x = pt0.x, right_x = pt0.x, top_y = pt0.y, bottom_y = pt0.y;
  for (int i = 0; i < n; ++i) {
    if (pt0.x < left_x) { left_x = pt0.x; left = i; }
    if (pt0.x > right_x) { right_x = pt0.x; right = i; }
    if (pt0.y > top_y) { top_y = pt0.y; top = i; }
    if (pt0.y < bottom_y) { bottom_y = pt0.y; bottom = i; }
    const P2 pt = pts[(i + 1 == n) ? 0 : i + 1];
    const double dx = static_cast<double>(pt.x) - static_cast<double>(pt0.x);
    const double dy = static_cast<double>(pt.y) - static_cast<double>(pt0.y);
    vect_x[i] = static_cast<float>(dx);
    vect_y[i] = static_cast<float>(dy);
    inv_len[i] = static_cast<float>(1.0 / sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy))));
    pt0 = pt;
  }
  float orientation = 0.f;
  {
    double ax = vect_x[n - 1], ay = vect_y[n - 1];
    for (int i = 0; i < n; ++i) {
      const double bx = vect_x[i], by = vect_y[i];
      const double convexity = __dsub_rn(__dmul_rn(ax, by), __dmul_rn(ay, bx));
      if (convexity != 0) { orientation = convexity > 0 ? 1.f : -1.f; break; }
      ax = bx; ay = by;
    }
  }
  float base_a = orientation, base_b = 0.f;
  int seq[4] = {bottom, right, top, left};
  float minarea = 3.402823466e+38f;
  int best_left = 0, best_bottom = 0;
  float best_a = 1.f, best_b = 0.f, best_w = 0.f, best_h = 0.f;
  for (int k = 0; k < n; ++k) {
    float dp[4];
    dp[0] = __fadd_rn(__fmul_rn(+base_a, vect_x[seq[0]]), __fmul_rn(base_b, vect_y[seq[0]]));
    dp[1] = __fadd_rn(__fmul_rn(-base_b, vect_x[seq[1]]), __fmul_rn(base_a, vect_y[seq[1]]));
    dp[2] = __fsub_rn(__fmul_rn(-base_a, vect_x[seq[2]]), __fmul_rn(base_b, vect_y[seq[2]]));
    dp[3] = __fsub_rn(__fmul_rn(+base_b, vect_x[seq[3]]), __fmul_rn(base_a, vect_y[seq[3]]));
    float maxcos = __fmul_rn(dp[0], inv_len[seq[0]]);
    int main_element = 0;
    for (int i = 1; i < 4; ++i) {
      const float cosalpha = __fmul_rn(dp[i], inv_len[seq[i]]);
      if (cosalpha > maxcos) { main_element = i; maxcos = cosalpha; }
    }
    {
      const int pindex = seq[main_element];
      const float lead_x = __fmul_rn(vect_x[pindex], inv_len[pindex]);
      const float lead_y = __fmul_rn(vect_y[pindex], inv_len[pindex]);
      switch (main_element) {
        case 0: base_a = lead_x; base_b = lead_y; break;
        case 1: base_a = lead_y; base_b = -lead_x; break;
        case 2: base_a = -lead_x; base_b = -lead_y; break;
        default: base_a = -lead_y; base_b = lead_x; break;
      }
    }
    seq[main_element] += 1;
    if (seq[main_element] == n) seq[main_element] = 0;
    float dx = __fsub_rn(pts[seq[1]].x, pts[seq[3]].x);
    float dy = __fsub_rn(pts[seq[1]].y, pts[seq[3]].y);
    const float width = __fadd_rn(__fmul_rn(dx, base_a), __fmul_rn(dy, base_b));
    dx = __fsub_rn(pts[seq[2]].x, pts[seq[0]].x);
    dy = __fsub_rn(pts[seq[2]].y, pts[seq[0]].y);
    const float height = __fadd_rn(__fmul_rn(-dx, base_b), __fmul_rn(dy, base_a));
    const float area = __fmul_rn(width, height);
    if (area <= minarea) {
      minarea = area;
      best_left = seq[3]; best_bottom = seq[0];
      best_a = base_a; best_b = base_b; best_w = width; best_h = height;
    }
  }
  const float A1 = best_a, B1 = best_b, A2 = -best_b, B2 = best_a;
  const float C1 = __fadd_rn(__fmul_rn(A1, pts[best_left].x), __fmul_rn(pts[best_left].y, B1));
  const float C2 = __fadd_rn(__fmul_rn(A2, pts[best_bottom].x), __fmul_rn(pts[best_bottom].y, B2));
  const float idet = __fdiv_rn(1.f, __fsub_rn(__fmul_rn(A1, B2), __fmul_rn(A2, B1)));
  out[0] = __fmul_rn(__fsub_rn(__fmul_rn(C1, B2), __fmul_rn(C2, B1)), idet);
  out[1] = __fmul_rn(__fsub_rn(__fmul_rn(A1, C2), __fmul_rn(A2, C1)), idet);
  out[2] = __fmul_rn(A1, best_w);
  out[3] = __fmul_rn(B1, best_w);
  out[4] = __fmul_rn(A2, best_h);
  out[5] = __fmul_rn(B2, best_h);
}

// cv2.boxPoints(cv2.minAreaRect(hull)) for n >= 3 hull points.
__device__ void min_area_box(const P2* hull, int n, float* vx, float* vy, float* il, P2* box) {
  float cx, cy, w, h, ang;
  if (n > 2) {
    float out[6];
    rotating_calipers(hull, n, vx, vy, il, out);
    cx = __fadd_rn(out[0], __fmul_rn(__fadd_rn(out[2], out[4]), 0.5f));
    cy = __fadd_rn(out[1], __fmul_rn(__fadd_rn(out[3], out[5]), 0.5f));
    w = static_cast<float>(sqrt(__dadd_rn(__dmul_rn((double)out[2], (double)out[2]), __dmul_rn((double)out[3], (double)out[3]))));
    h = static_cast<float>(sqrt(__dadd_rn(__dmul_rn((double)out[4], (double)out[4]), __dmul_rn((double)out[5], (double)out[5]))));
    ang = static_cast<float>(atan2(static_cast<double>(out[3]), static_cast<double>(out[2])));
  } else if (n == 2) {
    cx = __fmul_rn(__fadd_rn(hull[0].x, hull[1].x), 0.5f);
    cy = __fmul_rn(__fadd_rn(hull[0].y, hull[1].y), 0.5f);
    const double dx = static_cast<double>(hull[1].x) - hull[0].x, dy = static_cast<double>(hull[1].y) - hull[0].y;
    w = static_cast<float>(sqrt(dx * dx + dy * dy));
    h = 0.f;
    ang = static_cast<float>(atan2(dy, dx));
  } else {
    cx = hull[0].x; cy = hull[0].y; w = 0.f; h = 0.f; ang = 0.f;
  }
  ang = static_cast<float>(static_cast<double>(ang) * 180.0 / 3.1415926535897932384626433832795);
  const double rad = static_cast<double>(ang) * 3.1415926535897932384626433832795 / 180.0;
  const float b = __fmul_rn(static_cast<float>(cos(rad)), 0.5f);
  const float a = __fmul_rn(static_cast<float>(sin(rad)), 0.5f);
  box[0].x = __fsub_rn(__fsub_rn(cx, __fmul_rn(a, h)), __fmul_rn(b, w));
  box[0].y = __fsub_rn(__fadd_rn(cy, __fmul_rn(b, h)), __fmul_rn(a, w));
  box[1].x = __fsub_rn(__fadd_rn(cx, __fmul_rn(a, h)), __fmul_rn(b, w));
  box[1].y = __fsub_rn(__fsub_rn(cy, __fmul_rn(b, h)), __fmul_rn(a, w));
  box[2].x = __fsub_rn(__fmul_rn(2.f, cx), box[0].x);
  box[2].y = __fsub_rn(__fmul_rn(2.f, cy), box[0].y);
  box[3].x = __fsub_rn(__fmul_rn(2.f, cx), box[1].x);
  box[3].y = __fsub_rn(__fmul_rn(2.f, cy), box[1].y);
}

__device__ __forceinline__ long long cross_i(int ox, int oy, int ax, int ay, int bx, int by) {
  return static_cast<long long>(ax - ox) * (by - oy) - static_cast<long long>(ay - oy) * (bx - ox);
}

// --------------------------------------------------------------------------- quads kernel
// Bit planes are rh rows of `stride` 32-bit words; bit b of word k is ROI column 32*k + b.
__device__ __forceinline__ uint32_t funnel_left(const uint32_t* row, int k, int stride, int s) {
  // bits shifted towards higher columns by s (0 <= s < 32): out bit c = in bit c - s
  const uint32_t cur = row[k];
  const uint32_t prev = k > 0 ? row[k - 1] : 0u;
  return s == 0 ? cur : ((cur << s) | (prev >> (32 - s)));
}
__device__ __forceinline__ uint32_t funnel_right(const uint32_t* row, int k, int stride, int s) {
  // out bit c = in bit c + s
  const uint32_t cur = row[k];
  const uint32_t next = (k + 1 < stride) ? row[k + 1] : 0u;
  return s == 0 ? cur : ((cur >> s) | (next << (32 - s)));
}

// The dilation ROI of a component (detection.py:258-265) as a bit plane.
struct Roi { int niter, sx, sy, rw, rh, stride, plane_words; };

__device__ __forceinline__ Roi roi_of(const Component& c, int hs, int ws) {
  Roi r;
  // detection.py:258-260
  const int mn = c.w < c.h ? c.w : c.h;
  r.niter = static_cast<int>(sqrt(static_cast<double>(static_cast<long long>(c.area) * mn) /
                                  static_cast<double>(static_cast<long long>(c.w) * c.h)) * 2.0);
  r.sx = max(c.x - r.niter, 0); r.sy = max(c.y - r.niter, 0);
  const int ex = min(c.x + c.w + r.niter + 1, ws), ey = min(c.y + c.h + r.niter + 1, hs);
  r.rw = ex - r.sx; r.rh = ey - r.sy;
  r.stride = (r.rw + 31) >> 5;
  r.plane_words = r.stride * r.rh;
  return r;
}

// Whether a component can be handled by the small-tile launch: both bit planes and the hull scratch that later
// reuses plane B (worst case 2*rh hull points: 56 bytes per row + the padding of the index arrays) fit `words` words.
__device__ __forceinline__ bool fits_words(const Roi& r, int words) {
  return r.plane_words <= words && 56 * r.rh + 64 <= 4 * words;
}

// One component -> one quad.  `dyn_smem` holds two planes of `smem_plane_words` words; a component whose planes
// do not fit works on the per-image global scratch planes instead (serialised by a per-image lock).
__device__ void quad_of_component(const uint8_t* __restrict__ mask, const int* __restrict__ label, int hs, int ws,
                                  const Component c, int img, float* __restrict__ out,
                                  uint32_t* __restrict__ big_planes, int* __restrict__ big_locks,
                                  uint32_t* dyn_smem, int smem_plane_words) {
  __shared__ int row_min[kMaxHullRows / 2], row_max[kMaxHullRows / 2];   // per blob row (<= 1024 rows)
  __shared__ int first_word;
  const int hw = hs * ws;
  const uint8_t* M = mask + static_cast<size_t>(img) * hw;
  const int* L = label + static_cast<size_t>(img) * hw;

  const Roi roi = roi_of(c, hs, ws);
  const int niter = roi.niter, sx = roi.sx, sy = roi.sy, rw = roi.rw, rh = roi.rh;
  const int stride = roi.stride, plane_words = roi.plane_words;
  // cv2.dilate with a (1+niter)^2 rectangle, anchor k/2: a source pixel at j sets [j-(k-1-a), j+a]
  const int ksz = 1 + niter, grow_hi = ksz / 2, grow_lo = ksz - 1 - grow_hi;

  uint32_t *A, *B;
  bool big = plane_words > smem_plane_words;
  if (!big) {
    A = dyn_smem; B = dyn_smem + smem_plane_words;
  } else {
    // oversized component: serialise on the per-image global scratch planes
    if (threadIdx.x == 0) { while (atomicCAS(big_locks + img, 0, 1) != 0) { __nanosleep(200); } }
    __syncthreads();
    const size_t full = static_cast<size_t>((ws + 31) / 32) * hs;
    A = big_planes + static_cast<size_t>(img) * 2 * full; B = A + full;
  }

  // plane B <- source mask S (component pixels minus text&link) ------------------------------
  // one warp per ROI row, lane b tests column 32k + b of the row's word k (coalesced label / mask reads), the ballot
  // is the word; four words per round so that their eight loads are in flight together
  {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    for (int ry = warp; ry < rh; ry += nwarps) {
      const int y = sy + ry;
      const bool row_in = y >= c.y && y < c.y + c.h;
      for (int k0 = 0; k0 < stride; k0 += 4) {
        bool bit[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int x = sx + 32 * (k0 + u) + lane;
          bit[u] = false;
          if (row_in && k0 + u < stride && x >= c.x && x < c.x + c.w) {
            const int q = y * ws + x;
            bit[u] = L[q] == c.root && !(M[q] & 2);
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint32_t bits = __ballot_sync(0xffffffffu, bit[u]);
          if (lane == 0 && k0 + u < stride) B[ry * stride + k0 + u] = bits;
        }
      }
    }
  }
  __syncthreads();
  // plane A <- horizontal dilation of B ------------------------------------------------------
  for (int i = threadIdx.x; i < plane_words; i += blockDim.x) {
    const int ry = i / stride, k = i - ry * stride;
    const uint32_t* row = B + ry * stride;
    uint32_t acc = 0;
    // out(c) = OR_{j = c - grow_hi}^{c + grow_lo} src(j)
    for (int s = 0; s <= grow_hi; ++s) {
      const int wsh = s >> 5, bs = s & 31;
      if (k - wsh >= 0) acc |= funnel_left(row, k - wsh, stride, bs);
    }
    for (int s = 1; s <= grow_lo; ++s) {
      const int wsh = s >> 5, bs = s & 31;
      if (k + wsh < stride) acc |= funnel_right(row, k + wsh, stride, bs);
    }
    if (k == stride - 1 && (rw & 31)) acc &= (1u << (rw & 31)) - 1u;   // clip to the ROI
    A[i] = acc;
  }
  __syncthreads();
  // plane B <- vertical dilation of A  (= the dilated segmap D inside the ROI) ---------------
  for (int i = threadIdx.x; i < plane_words; i += blockDim.x) {
    const int ry = i / stride, k = i - ry * stride;
    uint32_t acc = 0;
    const int lo = max(ry - grow_hi, 0), hi = min(ry + grow_lo, rh - 1);
    for (int r = lo; r <= hi; ++r) acc |= A[r * stride + k];
    B[i] = acc;
  }
  __syncthreads();

  // findContours(...)[0]: the 8-connected blob whose first raster pixel comes last ------------
  // Flood-fill blobs one at a time in raster order of their first pixel; the last one survives in A.
  bool have_blob = false;
  while (true) {
    if (threadIdx.x == 0) first_word = 0x7fffffff;
    __syncthreads();
    for (int i = threadIdx.x; i < plane_words; i += blockDim.x)
      if (B[i]) { atomicMin(&first_word, i); break; }
    __syncthreads();
    const int fw = first_word;
    if (fw == 0x7fffffff) break;
    have_blob = true;
    for (int i = threadIdx.x; i < plane_words; i += blockDim.x) A[i] = 0;
    __syncthreads();
    if (threadIdx.x == 0) A[fw] = B[fw] & (0u - B[fw]);           // lowest set bit = first pixel
    __syncthreads();
    // Close A under "8-neighbour inside B" with ONE warp sweeping the rows, alternately downwards and upwards, lane =
    // word of the row: a sweep carries the fill through every row it passes, so a blob takes about three sweeps
    // (down, up, one that changes nothing) where the all-words-at-once iteration took one round per row of the blob
    // -- 64 rounds over ~480 words on the bench pages, half of this kernel's instructions (profiles/r2o_quads_source.txt).
    // The result is the same set: the smallest one that contains the seed and is closed under that neighbourhood.
    if (threadIdx.x < 32) {
      const int lane = threadIdx.x;
      bool down = true;
      while (true) {
        bool changed = false;
        for (int rr = 0; rr < rh; ++rr) {
          const int r = down ? rr : rh - 1 - rr;
          for (int k0 = 0; k0 < stride; k0 += 32) {
            const int k = k0 + lane;
            uint32_t cur = 0, grown = 0;
            if (k < stride) {
              const uint32_t d = B[r * stride + k];
              if (d) {
                uint32_t nb = 0;
                for (int dr = -1; dr <= 1; ++dr) {
                  const int r2 = r + dr;
                  if (r2 < 0 || r2 >= rh) continue;
                  const uint32_t* row = A + r2 * stride;
                  const uint32_t mid = row[k];
                  const uint32_t prev = k > 0 ? row[k - 1] : 0u;
                  const uint32_t next = (k + 1 < stride) ? row[k + 1] : 0u;
                  if (dr == 0) cur = mid;
                  nb |= mid | (mid << 1) | (mid >> 1) | (prev >> 31) | (next << 31);
                }
                grown = nb & d;
                // finish the fill along the row inside this word (runs of d reachable from grown)
                uint32_t prevg;
                do { prevg = grown; grown |= ((grown << 1) | (grown >> 1)) & d; } while (grown != prevg);
                grown &= ~cur;
              }
            }
            __syncwarp();                                   // every lane has read row r before any lane writes it
            if (grown) { A[r * stride + k] = cur | grown; changed = true; }
            __syncwarp();
          }
        }
        if (!__any_sync(0xffffffffu, changed)) break;       // a whole sweep without a change: closed
        down = !down;
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < plane_words; i += blockDim.x) B[i] &= ~A[i];
    __syncthreads();
  }

  if (!have_blob) {
    // The reference raises IndexError here (contours[0] of an empty list); we emit a NaN box.
    if (threadIdx.x < 8) out[threadIdx.x] = nanf("");
    if (big) { __syncthreads(); if (threadIdx.x == 0) atomicExch(big_locks + img, 0); }
    return;
  }
  // per-row extents of the blob (ROI coordinates) ---------------------------------------------
  for (int r = threadIdx.x; r < rh; r += blockDim.x) {
    int lo = -1, hi = -1;
    for (int k = 0; k < stride; ++k) {
      const uint32_t v = A[r * stride + k];
      if (v) {
        if (lo < 0) lo = 32 * k + __ffs(v) - 1;
        hi = 32 * k + 31 - __clz(v);
      }
    }
    row_min[r] = lo; row_max[r] = hi;
  }
  __syncthreads();
  if (big) { if (threadIdx.x == 0) atomicExch(big_locks + img, 0); }

  if (threadIdx.x == 0) {
    // hull stack lives in the (now free) plane B / dynamic smem: 2*rh points + 3*2*rh floats
    // Convex hull in cv2.convexHull(clockwise=False) order of the contour: right side top->bottom,
    // then left side bottom->top, ending at the blob's first raster pixel.
    int* hx = reinterpret_cast<int*>(big ? reinterpret_cast<uint32_t*>(dyn_smem) : B);
    int* hy = hx + 2 * rh + 4;
    int n = 0, r_first = -1, r_last = -1;
    for (int r = 0; r < rh; ++r) if (row_min[r] >= 0) { if (r_first < 0) r_first = r; r_last = r; }
    int base = 0;
    for (int r = r_first; r <= r_last; ++r) {               // right chain
      if (row_max[r] < 0) continue;
      const int px = row_max[r], py = r;
      while (n - base >= 2 && cross_i(hx[n - 2], hy[n - 2], hx[n - 1], hy[n - 1], px, py) <= 0) --n;
      hx[n] = px; hy[n] = py; ++n;
    }
    const int n_right = n;
    base = n_right;
    for (int r = r_last; r >= r_first; --r) {               // left chain
      if (row_min[r] < 0) continue;
      const int px = row_min[r], py = r;
      while (n - base >= 2 && cross_i(hx[n - 2], hy[n - 2], hx[n - 1], hy[n - 1], px, py) <= 0) --n;
      hx[n] = px; hy[n] = py; ++n;
    }
    // drop duplicated joints, then clean concave / collinear joints
    int m = 0;
    for (int i = 0; i < n; ++i)
      if (m == 0 || hx[i] != hx[m - 1] || hy[i] != hy[m - 1]) { hx[m] = hx[i]; hy[m] = hy[i]; ++m; }
    if (m > 1 && hx[0] == hx[m - 1] && hy[0] == hy[m - 1]) --m;
    bool changed = true;
    while (changed && m > 2) {
      changed = false;
      for (int i = 0; i < m; ++i) {
        const int ip = (i + m - 1) % m, in = (i + 1) % m;
        if (cross_i(hx[ip], hy[ip], hx[i], hy[i], hx[in], hy[in]) <= 0) {
          for (int j = i; j + 1 < m; ++j) { hx[j] = hx[j + 1]; hy[j] = hy[j + 1]; }
          --m; changed = true; break;
        }
      }
    }
    // rotate so that the first raster pixel (row r_first, its leftmost column) comes last
    int kfirst = 0;
    for (int i = 0; i < m; ++i) if (hx[i] == row_min[r_first] && hy[i] == r_first) { kfirst = i; break; }
    P2* hull = reinterpret_cast<P2*>(hy + 2 * rh + 4);
    for (int i = 0; i < m; ++i) {
      const int j = (kfirst + 1 + i) % m;
      hull[i].x = static_cast<float>(hx[j] + sx);
      hull[i].y = static_cast<float>(hy[j] + sy);
    }
    float* vx = reinterpret_cast<float*>(hull + m + 1);
    float* vy = vx + m + 1;
    float* il = vy + m + 1;
    P2 box[4];
    min_area_box(hull, m, vx, vy, il, box);
    // diamond test, detection.py:276-281
    const float w = sqrtf(__fadd_rn(__fmul_rn(box[0].x - box[1].x, box[0].x - box[1].x),
                                    __fmul_rn(box[0].y - box[1].y, box[0].y - box[1].y)));
    const float h = sqrtf(__fadd_rn(__fmul_rn(box[1].x - box[2].x, box[1].x - box[2].x),
                                    __fmul_rn(box[1].y - box[2].y, box[1].y - box[2].y)));
    const float ratio = __fdiv_rn(fmaxf(w, h), __fadd_rn(fminf(w, h), 1e-5f));
    P2 res[4];
    if (fabsf(1.f - ratio) <= 0.1f) {
      int l = 0x7fffffff, rr = -1;
      for (int r = r_first; r <= r_last; ++r)
        if (row_min[r] >= 0) { l = min(l, row_min[r]); rr = max(rr, row_max[r]); }
      const float fl = static_cast<float>(l + sx), fr = static_cast<float>(rr + sx);
      const float ft = static_cast<float>(r_first + sy), fb = static_cast<float>(r_last + sy);
      res[0] = {fl, ft}; res[1] = {fr, ft}; res[2] = {fr, fb}; res[3] = {fl, fb};
    } else {
      int first = 0;
      float best = __fadd_rn(box[0].x, box[0].y);
      for (int i = 1; i < 4; ++i) {
        const float s = __fadd_rn(box[i].x, box[i].y);
        if (s < best) { best = s; first = i; }
      }
      for (int i = 0; i < 4; ++i) res[i] = box[(first + i) & 3];
    }
    for (int i = 0; i < 4; ++i) { out[2 * i] = 2.f * res[i].x; out[2 * i + 1] = 2.f * res[i].y; }
  }
}

// Pass 1, one block of 128 threads per (box slot, image) with SMALL planes: eight blocks per SM instead of the two
// that 96 KB planes allow (the work is a chain of short latency-bound phases, profiles/r2n_glue_full.csv: 17 % of
// the warp slots active with the large planes).  Components that do not fit are queued for pass 2.
__global__ void __launch_bounds__(256)
quads_kernel(const uint8_t* __restrict__ mask, const int* __restrict__ label, int hs, int ws,
             const Component* __restrict__ comps, const int* __restrict__ counts, int max_boxes,
             float* __restrict__ boxes, uint32_t* __restrict__ big_planes, int* __restrict__ big_locks,
             int smem_plane_words, int* __restrict__ queue, int* __restrict__ queue_len) {
  extern __shared__ uint32_t dyn_smem[];
  const int img = blockIdx.y, slot = blockIdx.x;
  int cnt = counts[img];
  if (cnt > max_boxes) cnt = max_boxes;
  if (slot >= cnt) return;
  const size_t id = static_cast<size_t>(img) * max_boxes + slot;
  const Component c = comps[id];
  if (!fits_words(roi_of(c, hs, ws), smem_plane_words)) {
    if (threadIdx.x == 0) queue[atomicAdd(queue_len, 1)] = static_cast<int>(id);
    return;
  }
  quad_of_component(mask, label, hs, ws, c, img, boxes + id * 8, big_planes, big_locks, dyn_smem, smem_plane_words);
}

// Pass 2, a few blocks with the large planes walking the queue of pass 1 (normally empty).
__global__ void __launch_bounds__(256)
quads_queue_kernel(const uint8_t* __restrict__ mask, const int* __restrict__ label, int hs, int ws,
                   const Component* __restrict__ comps, int max_boxes, float* __restrict__ boxes,
                   uint32_t* __restrict__ big_planes, int* __restrict__ big_locks, int smem_plane_words,
                   const int* __restrict__ queue, const int* __restrict__ queue_len) {
  extern __shared__ uint32_t dyn_smem[];
  const int len = *queue_len;
  for (int i = blockIdx.x; i < len; i += gridDim.x) {
    const int id = queue[i];
    quad_of_component(mask, label, hs, ws, comps[id], id / max_boxes, boxes + static_cast<size_t>(id) * 8, big_planes,
                      big_locks, dyn_smem, smem_plane_words);
    __syncthreads();       // thread 0 builds the hull in the planes' shared memory after the others have left
  }
}

inline unsigned nblocks(long long total, int threads) { return static_cast<unsigned>((total + threads - 1) / threads); }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

constexpr int kQuadSmemPlaneWords = 12 * 1024;     // pass 2: 2 planes x 48 KB, ROIs up to ~390k pixels stay in smem
constexpr int kQuadSmallPlaneWords = 2 * 1024;     // pass 1: 2 planes x 8 KB, ROIs up to 65k pixels and 145 rows

struct BoxWorkspace {
  uint8_t* mask; int* label; Stats st; Component* comps; uint32_t* big_planes; int* big_locks;
  int* queue; int* queue_len;       // components that pass 1 of the quads leaves to pass 2
  size_t bytes;
};

BoxWorkspace carve(void* ws, int n, int hs, int ws_w, int max_boxes) {
  BoxWorkspace w;
  const size_t px = static_cast<size_t>(n) * hs * ws_w;
  uint8_t* p = reinterpret_cast<uint8_t*>(ws);
  size_t off = 0;
  auto take = [&](size_t bytes) { void* r = p ? p + off : nullptr; off += align_up(bytes, 256); return r; };
  w.label = reinterpret_cast<int*>(take(px * 4));
  w.st.area = reinterpret_cast<int*>(take(px * 4));
  w.st.minx = reinterpret_cast<int*>(take(px * 4));
  w.st.maxx = reinterpret_cast<int*>(take(px * 4));
  w.st.miny = reinterpret_cast<int*>(take(px * 4));
  w.st.maxy = reinterpret_cast<int*>(take(px * 4));
  w.st.maxtext = reinterpret_cast<int*>(take(px * 4));
  w.mask = reinterpret_cast<uint8_t*>(take(px));
  w.comps = reinterpret_cast<Component*>(take(static_cast<size_t>(n) * max_boxes * sizeof(Component)));
  w.big_planes = reinterpret_cast<uint32_t*>(take(static_cast<size_t>(n) * 2 * ((ws_w + 31) / 32) * hs * 4));
  w.big_locks = reinterpret_cast<int*>(take(static_cast<size_t>(n) * 4));
  w.queue = reinterpret_cast<int*>(take(static_cast<size_t>(n) * max_boxes * 4));
  w.queue_len = reinterpret_cast<int*>(take(4));
  w.bytes = off;
  return w;
}

}  // namespace

extern "C" size_t b2o_boxes_workspace_bytes(int n, int hs, int ws, int max_boxes) {
  return carve(nullptr, n, hs, ws, max_boxes).bytes;
}

extern "C" int b2o_get_boxes(b2o_ctx* ctx, const float* scores, int n, int hs, int ws, float detection_threshold,
                             float text_threshold, float link_threshold, int size_threshold, float* boxes,
                             int32_t* counts, int max_boxes, void* ws_dev, size_t ws_bytes, void* stream) {
  if (!ctx) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  if (!scores || !boxes || !counts || !ws_dev || n <= 0 || hs <= 0 || ws <= 0 || max_boxes <= 0) {
    ctx->set_error("b2o_get_boxes: bad argument");
    return B2O_ERR_ARG;
  }
  if (hs > kMaxHullRows / 2 || static_cast<long long>(hs) * ws >= (1LL << 30)) {
    ctx->set_error("b2o_get_boxes: score map larger than 1024 rows is not supported");
    return B2O_ERR_ARG;
  }
  BoxWorkspace w = carve(ws_dev, n, hs, ws, max_boxes);
  if (w.bytes > ws_bytes) { ctx->set_error("b2o_get_boxes: workspace too small"); return B2O_ERR_WORKSPACE; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const long long total = static_cast<long long>(n) * hs * ws;
  const size_t px = static_cast<size_t>(total);
  B2O_CUDA_CHECK(ctx, cudaMemsetAsync(w.st.area, 0, px * 4, st));
  B2O_CUDA_CHECK(ctx, cudaMemsetAsync(w.st.minx, 0x7f, px * 4, st));
  B2O_CUDA_CHECK(ctx, cudaMemsetAsync(w.st.miny, 0x7f, px * 4, st));
  B2O_CUDA_CHECK(ctx, cudaMemsetAsync(w.st.maxx, 0xff, px * 4, st));     // -1
  B2O_CUDA_CHECK(ctx, cudaMemsetAsync(w.st.maxy, 0xff, px * 4, st));
  B2O_CUDA_CHECK(ctx, cudaMemsetAsync(w.st.maxtext, 0x80, px * 4, st));  // very negative key
  B2O_CUDA_CHECK(ctx, cudaMemsetAsync(w.big_locks, 0, static_cast<size_t>(n) * 4, st));
  B2O_CUDA_CHECK(ctx, cudaMemsetAsync(w.queue_len, 0, 4, st));
  binarize_kernel<<<nblocks(total, 256), 256, 0, st>>>(scores, total, hs * ws, ws, text_threshold, link_threshold,
                                                      w.mask, w.label);
  B2O_LAUNCH_CHECK(ctx);
  merge_kernel<<<nblocks(total, 256), 256, 0, st>>>(w.mask, w.label, total, hs, ws);
  B2O_LAUNCH_CHECK(ctx);
  flatten_kernel<<<nblocks(total, 256), 256, 0, st>>>(w.label, total, hs * ws);
  B2O_LAUNCH_CHECK(ctx);
  stats_kernel<<<nblocks(total, 256), 256, 0, st>>>(scores, w.label, total, hs * ws, ws, w.st);
  B2O_LAUNCH_CHECK(ctx);
  select_kernel<<<n, 1024, 0, st>>>(w.label, hs * ws, w.st, size_threshold, detection_threshold, w.comps, max_boxes,
                                    counts);
  B2O_LAUNCH_CHECK(ctx);
  const int dyn = 2 * kQuadSmemPlaneWords * 4, dyn_small = 2 * kQuadSmallPlaneWords * 4;
  if (!ctx->quads_configured) {        // a per-device attribute, hence per context (one context per device)
    B2O_CUDA_CHECK(ctx, cudaFuncSetAttribute(quads_queue_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn));
    ctx->quads_configured = true;
  }
  quads_kernel<<<dim3(max_boxes, n), 128, dyn_small, st>>>(w.mask, w.label, hs, ws, w.comps, counts, max_boxes, boxes,
                                                           w.big_planes, w.big_locks, kQuadSmallPlaneWords, w.queue,
                                                           w.queue_len);
  B2O_LAUNCH_CHECK(ctx);
  const long long slots = static_cast<long long>(n) * max_boxes;
  quads_queue_kernel<<<static_cast<unsigned>(std::min<long long>(slots, 2 * ctx->sm_count)), 256, dyn, st>>>(
      w.mask, w.label, hs, ws, w.comps, max_boxes, boxes, w.big_planes, w.big_locks, kQuadSmemPlaneWords, w.queue,
      w.queue_len);
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}

// ------------------------------------------------------------------------------------------------
// Box bookkeeping of recognize_from_boxes (recognition.py:511-521: crops appended image after image,
// `start_end` = running offsets) and the result records of Pipeline.recognize (pipeline.py:66-75), done on
// the device so that the host needs nothing but the per-image counts it already reads.
namespace {

// sum over images j < i of min(max(counts[j], 0), cap); every thread of the block gets the result
__device__ int boxes_before(const int32_t* __restrict__ counts, int i, int cap) {
  __shared__ int warp_sums[32];
  __shared__ int total;
  int s = 0;
  for (int j = threadIdx.x; j < i; j += blockDim.x) s += min(max(counts[j], 0), cap);
  for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    int v = threadIdx.x < (blockDim.x + 31) / 32 ? warp_sums[threadIdx.x] : 0;
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    if (threadIdx.x == 0) total = v;
  }
  __syncthreads();
  return total;
}

__global__ void __launch_bounds__(128)
compact_boxes_kernel(const float* __restrict__ boxes, const int32_t* __restrict__ counts, int max_boxes,
                     float* __restrict__ flat, int32_t* __restrict__ image_index) {
  const int i = blockIdx.x;
  const int off = boxes_before(counts, i, max_boxes);
  const int c = min(max(counts[i], 0), max_boxes);
  const float4* src = reinterpret_cast<const float4*>(boxes + static_cast<size_t>(i) * max_boxes * 8);
  float4* dst = reinterpret_cast<float4*>(flat + static_cast<size_t>(off) * 8);
  for (int t = threadIdx.x; t < 2 * c; t += blockDim.x) dst[t] = src[t];
  for (int t = threadIdx.x; t < c; t += blockDim.x) image_index[off + t] = i;
}

constexpr int kDefaultSteps = 48;                  // label steps per word at the default geometry (recognition.py:20: 50 - 2)

// label int8 slots of one word: `steps` bytes, the label area rounded up to whole floats per word
__host__ __device__ inline size_t label_floats(int steps) { return (static_cast<size_t>(steps) + 3) / 4; }

// steps = label row length (T - rnn_steps_to_discard of the recognizer); the words' labels lie back to back as int8
// in the record's rec_boxes * ceil(steps / 4) label floats, every byte past the last stored word -1
__global__ void __launch_bounds__(128)
pack_records_kernel(const float* __restrict__ boxes, const int32_t* __restrict__ counts,
                    const int32_t* __restrict__ labels, const float* __restrict__ inv_scale, int n, int max_boxes,
                    int rec_boxes, int steps, float* __restrict__ rec) {
  const int row = blockIdx.x;
  const int lab_bytes = rec_boxes * static_cast<int>(label_floats(steps)) * 4;
  const int rec_len = 1 + rec_boxes * 8 + lab_bytes / 4;
  float* r = rec + static_cast<size_t>(row) * rec_len;
  int8_t* lab = reinterpret_cast<int8_t*>(r + 1 + rec_boxes * 8);
  int c = 0, off = 0, held = 0;
  float inv = 1.f;
  if (row < n) {                                   // uniform per block
    off = boxes_before(counts, row, max_boxes);
    held = min(max(counts[row], 0), max_boxes);      // boxes of this image in the table
    c = min(held, rec_boxes);                        // ... of which the record has room for c
    inv = inv_scale[row];
  }
  // count field: what the image HAS (the reader refuses a record whose count exceeds rec_boxes instead of silently
  // dropping words); -1 marks the padding rows of a short shard
  if (threadIdx.x == 0) r[0] = row < n ? static_cast<float>(held) : -1.f;
  const float* src = boxes + static_cast<size_t>(min(row, n - 1)) * max_boxes * 8;
  for (int t = threadIdx.x; t < rec_boxes * 8; t += blockDim.x)
    r[1 + t] = t < c * 8 ? __fmul_rn(src[t], inv) : 0.f;                  // tools.adjust_boxes (tools.py:232-260)
  for (int t = threadIdx.x; t < lab_bytes; t += blockDim.x) {
    const int k = t / steps;
    lab[t] = (k < c && labels) ? static_cast<int8_t>(labels[static_cast<size_t>(off + k) * steps + (t - k * steps)])
                   : static_cast<int8_t>(-1);
  }
}

}  // namespace

extern "C" int b2o_compact_boxes(b2o_ctx* ctx, const float* boxes, const int32_t* counts, int n, int max_boxes,
                                 float* flat, int32_t* image_index, void* stream) {
  if (!ctx) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  if (!boxes || !counts || !flat || !image_index || n <= 0 || max_boxes <= 0) {
    ctx->set_error("b2o_compact_boxes: bad argument");
    return B2O_ERR_ARG;
  }
  compact_boxes_kernel<<<n, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(boxes, counts, max_boxes, flat,
                                                                            image_index);
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}

extern "C" size_t b2o_record_floats_steps(int rec_boxes, int steps) {
  return rec_boxes > 0 && steps > 0 ? 1 + static_cast<size_t>(rec_boxes) * 8 + static_cast<size_t>(rec_boxes) * label_floats(steps) : 0;
}

extern "C" size_t b2o_record_floats(int rec_boxes) { return b2o_record_floats_steps(rec_boxes, kDefaultSteps); }

extern "C" int b2o_pack_records_steps(b2o_ctx* ctx, const float* boxes, const int32_t* counts, const int32_t* labels,
                                      const float* inv_scale, int n, int max_boxes, int rows, int rec_boxes, int steps,
                                      float* records, void* stream) {
  if (!ctx) return B2O_ERR_ARG;
  DeviceGuard guard(ctx->device);
  if (!boxes || !counts || !inv_scale || !records || n <= 0 || rows < n || max_boxes <= 0 || rec_boxes <= 0 || steps <= 0) {
    ctx->set_error("b2o_pack_records: bad argument");      // labels may be NULL when no image has a box
    return B2O_ERR_ARG;
  }
  pack_records_kernel<<<rows, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(boxes, counts, labels, inv_scale, n,
                                                                              max_boxes, rec_boxes, steps, records);
  B2O_LAUNCH_CHECK(ctx);
  return B2O_OK;
}

extern "C" int b2o_pack_records(b2o_ctx* ctx, const float* boxes, const int32_t* counts, const int32_t* labels,
                                const float* inv_scale, int n, int max_boxes, int rows, int rec_boxes, float* records,
                                void* stream) {
  return b2o_pack_records_steps(ctx, boxes, counts, labels, inv_scale, n, max_boxes, rows, rec_boxes, kDefaultSteps,
                                records, stream);
}
