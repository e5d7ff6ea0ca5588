// Light bars -> armors on the GPU: the B200 form of IrmDetector::extract_armors
// (reference src/irm_detector.cpp:292-355) and the Light / Armor constructors
// (reference include/irmv_detection/armor.hpp:11-77).  Oracle: oracle/armor_ref.py (pinned against
// cv2.cvtColor / findContours / minAreaRect).
//
// The reference walks the detections on the CPU: ROI of the rotated frame -> cvtColor(BGR2GRAY) ->
// threshold -> findContours(RETR_EXTERNAL, CHAIN_APPROX_SIMPLE) -> per contour with >= 5 points
// minAreaRect -> Light -> is_light -> the first two lights make the armor.  Here one CTA owns one
// detection and never materialises the rotated frame, the gray ROI or a contour:
//   1. the ROI is thresholded straight from the camera frame (rot180 and, for Bayer sources, the
//      demosaic folded into the fetch) into a 1-bit-per-pixel bitmap in shared memory, one
//      __ballot per 32 pixels;
//   2. the exterior background (4-connected to the ROI frame) is flood-filled on the bitmap with
//      carry-propagation word fills: a component is top level (RETR_EXTERNAL) iff the background
//      left of its first pixel is exterior;
//   3. every start candidate (foreground pixel, exterior background to the W, background to the NW,
//      N, NE) is followed with the Suzuki-Abe border walk by one lane; the walk is dropped as soon
//      as it meets a pixel that precedes the candidate in raster order (then it is not the
//      component's first pixel, or it is a hole border), and it counts the CHAIN_APPROX_SIMPLE
//      vertices (direction changes) instead of storing them;
//   4. for a kept border the per-row extreme columns give the convex hull (monotone chain), the
//      hull edges are scanned in parallel for the minimum-area rectangle (same rectangle as
//      rotating calipers), and lane 0 applies the Light constructor and the light filter;
//   5. OpenCV returns contours in reverse raster order of their first pixel, so "the first two
//      lights" are the two valid lights with the largest start index.
// Bitmaps of ROIs larger than the shared-memory budget live in a per-CTA global scratch slot.
#include <math_constants.h>

#include "common.cuh"

namespace irmv {
namespace {

constexpr int kThreads = 256, kWarps = kThreads / 32;
constexpr int kSmemWords = 2048;       // per bitmap: ROIs up to 64 K padded pixels keep their bitmaps in shared memory
constexpr int kRows = 256;             // ... and up to this many rows (per-warp row-extreme arrays, hull)
constexpr int kHullSmem = 2 * kRows + 2;   // a row adds at most two hull vertices (global scratch: slot_hull_cap)
// Coordinates are packed into 16 bits (x | y << 16 in the hull and the candidate list, short row extremes), and
// cross3's products of ROI coordinate differences stay below 2^31 for sides up to kMaxSide; the border walk's step
// cap 8 * (w + 2) * (h + 2) is an int
constexpr int kMaxSide = 32766;
constexpr int kCandCap = 64;         // ROIs with at most this many start candidates spread them over the warps
// (large ROIs use a global scratch slot per CTA: with 64 shared slots behind locks the slots, not the SMs,
// limited the stage when most boxes are large -- 15 ms per 6400 random-init boxes)
constexpr unsigned kFull = 0xffffffffu;

struct LightRec {
  float cx, cy, tx, ty, bx, by;        // centre, top, bottom (source pixels, already offset by the ROI origin)
  double length;
  unsigned key;                        // raster index of the contour's first pixel inside the padded ROI
};

struct WarpBuf {                       // per warp: row extremes of the border being examined and its hull
  short *rmin, *rmax;
  int *hull;                           // x | y << 16, ROI coordinates
  int hull_cap;
};

struct Shared {
  uint32_t fg[kSmemWords];
  uint32_t ext[kSmemWords];
  short rmin[kWarps][kRows], rmax[kWarps][kRows];
  int hull[kWarps][kHullSmem];
  LightRec best[2];
  int nbest;
  int lock;
  int slot;
  int ncand;                           // start candidates of the ROI (may exceed kCandCap)
  int cand[kCandCap];                  // x | y << 16, padded ROI coordinates
};

// words of one global scratch slot: two whole-frame bitmaps + the per-warp arrays, sized by the source height
// (an ROI has at most src_h rows; its border walk indexes rows 0 .. rh of the row-extreme arrays)
__host__ __device__ inline size_t slot_bitmap_words(int src_w, int src_h) {
  return (((size_t)src_w + 2 + 31) / 32) * ((size_t)src_h + 2);
}
__host__ __device__ inline int slot_rows(int src_h) { return src_h + 2; }
__host__ __device__ inline int slot_hull_cap(int src_h) { return 2 * slot_rows(src_h) + 2; }
__host__ __device__ inline size_t slot_warp_words(int src_h) {     // rmin, rmax (shorts: one word per row) + hull
  return (size_t)slot_rows(src_h) + slot_hull_cap(src_h);
}
__host__ __device__ inline size_t slot_words(int src_w, int src_h) {
  return 2 * slot_bitmap_words(src_w, src_h) + kWarps * slot_warp_words(src_h) + 16;
}

__device__ __forceinline__ int reflect101(int i, int n) {
  if (i < 0) i = -i;
  if (i >= n) i = 2 * n - 2 - i;
  return i;
}

// Gray value of pixel (X, Y) of the rotated frame as cv::cvtColor(COLOR_BGR2GRAY) computes it on the
// buffer the reference holds (memory channel 0 takes the blue weight, whatever the channel really
// is: src/irm_detector.cpp:310; a Bayer source is demosaiced to RGB like the vendor ISP does).
// Branch-free, so that the loads of several pixels can be in flight together.
// LUT (Bayer only): every raw sample first goes through the raw-domain colour table lut[y & 1][x & 1][s]
// (ArmorParams::raw_lut, staged in shared memory); reflect-101 keeps a mirrored neighbour on its colour site, so
// the neighbours of (sx, sy) use the tables of parity (sx ^ 1) and (sy ^ 1).
// CCM (Bayer only): the demosaiced pixel then goes through the colour-correction block `ccm` (ArmorParams::ccm, staged
// in shared memory) before the gray sum; memory channel 0 still takes the blue weight.
template <bool BAYER, bool LUT, bool CCM>
__device__ __forceinline__ int gray_at(const uint8_t *__restrict__ frame, const uint8_t *lut, const uint8_t *ccm, int W, int H,
                                       int red_y, int red_x, int rot, int X, int Y) {
  const int sx = rot ? W - 1 - X : X, sy = rot ? H - 1 - Y : Y;
  int c0, c1, c2;
  if (BAYER) {
    const int ym = reflect101(sy - 1, H), yp = reflect101(sy + 1, H);
    const int xm = reflect101(sx - 1, W), xp = reflect101(sx + 1, W);
    const uint8_t *r0 = frame + (size_t)ym * W, *r1 = frame + (size_t)sy * W, *r2 = frame + (size_t)yp * W;
    int nw = r0[xm], n = r0[sx], ne = r0[xp], w = r1[xm], c = r1[sx], e = r1[xp], sw = r2[xm], s = r2[sx], se = r2[xp];
    if (LUT) {
      const uint8_t *tc = lut + (((sy & 1) << 9) | ((sx & 1) << 8));                       // own site
      const uint8_t *th = tc + ((sx & 1) ? -256 : 256), *tv = tc + ((sy & 1) ? -512 : 512), *td = th + ((sy & 1) ? -512 : 512);
      c = tc[c]; w = th[w]; e = th[e]; n = tv[n]; s = tv[s];
      nw = td[nw]; ne = td[ne]; sw = td[sw]; se = td[se];
    }
    const int cross = (n + s + w + e + 2) >> 2, diag = (nw + ne + sw + se + 2) >> 2;
    const int horiz = (w + e + 1) >> 1, vert = (n + s + 1) >> 1;
    const bool red_row = ((sy & 1) == red_y), red_col = ((sx & 1) == red_x);
    const bool is_r = red_row && red_col, is_b = !red_row && !red_col;
    c1 = (is_r || is_b) ? cross : c;
    c0 = is_r ? c : (is_b ? diag : (red_row ? horiz : vert));
    c2 = is_b ? c : (is_r ? diag : (red_row ? vert : horiz));
    if (CCM) apply_ccm(ccm, c0, c1, c2);
  } else {
    const uint8_t *s = frame + ((size_t)sy * W + sx) * 3;
    c0 = s[0]; c1 = s[1]; c2 = s[2];
  }
  return (c0 * 3735 + c1 * 19235 + c2 * 9798 + (1 << 14)) >> 15;     // OpenCV BY15, GY15, RY15
}

// ROI -> 1-bit-per-pixel threshold bitmap, padded by one background pixel all round: a warp builds one
// word per ballot, eight words per round with their loads issued together (clamped coordinates keep
// the fetch branch-free).
template <bool BAYER, bool LUT, bool CCM>
__device__ __forceinline__ void build_bitmap(uint32_t *fg, const uint8_t *__restrict__ frame, const uint8_t *lut, const uint8_t *ccm, int W, int H, int chan, int rot,
                                             int rx, int ry, int rw, int rh, int wpr, int words, int thr, int warp, int lane) {
  int red_y = 0, red_x = 0;
  if (chan == 3) { red_y = 1; red_x = 1; }
  else if (chan == 4) { red_y = 0; red_x = 1; }
  else if (chan == 5) { red_y = 1; red_x = 0; }
  constexpr int U = BAYER ? 4 : 8;       // a demosaiced pixel is nine loads, a packed one three
  for (int w0 = warp * U; w0 < words; w0 += kWarps * U) {
    int g[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int w = min(w0 + u, words - 1);
      const int row = w / wpr, wi = w - row * wpr;
      const int x = wi * 32 + lane - 1, y = row - 1;
      const bool in = x >= 0 && x < rw && y >= 0 && y < rh;
      g[u] = gray_at<BAYER, LUT, CCM>(frame, lut, ccm, W, H, red_y, red_x, rot, rx + min(max(x, 0), rw - 1), ry + min(max(y, 0), rh - 1));
      if (!in) g[u] = -1;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint32_t m = __ballot_sync(kFull, g[u] > thr);
      if (lane == 0 && w0 + u < words) fg[w0 + u] = m;
    }
  }
}

// Seeds `s` (subset of mask `m`) spread along the runs of ones of `m` inside one word.
__device__ __forceinline__ uint32_t fill_runs(uint32_t s, uint32_t m) {
  const uint32_t up = (m & ~(m + s)) | s;
  const uint32_t mr = __brev(m), sr = __brev(s);
  const uint32_t dn = __brev((mr & ~(mr + sr)) | sr);
  return up | dn;
}

// chain code of OpenCV: 0 E, 1 NE, 2 N, 3 NW, 4 W, 5 SW, 6 S, 7 SE (y down)
// (one byte-permute each: byte s of an 8-byte table of signed offsets)
__device__ __forceinline__ int dir_dx(int s) { return (int)(signed char)__byte_perm(0xFF000101u, 0x0100FFFFu, s); }
__device__ __forceinline__ int dir_dy(int s) { return (int)(signed char)__byte_perm(0xFFFFFF00u, 0x01010100u, s); }

// 8-neighbour mask of padded pixel (x, y): bit s = neighbour in chain-code direction s is foreground.
// One word per row covers x-1..x+1 unless x sits on a word boundary.
__device__ __forceinline__ uint32_t nbr8(const uint32_t *fg, int wpr, int x, int y) {
  const int b = x & 31;
  const uint32_t *q = fg + y * wpr + (x >> 5);
  uint32_t r0, r1, r2;                   // bits 0..2 = x-1, x, x+1 of rows y-1, y, y+1
  if (b >= 1 && b <= 30) {
    r0 = (q[-wpr] >> (b - 1)) & 7u; r1 = (q[0] >> (b - 1)) & 7u; r2 = (q[wpr] >> (b - 1)) & 7u;
  } else if (b == 0) {
    r0 = ((q[-wpr] & 3u) << 1) | (q[-wpr - 1] >> 31);
    r1 = ((q[0] & 3u) << 1) | (q[-1] >> 31);
    r2 = ((q[wpr] & 3u) << 1) | (q[wpr - 1] >> 31);
  } else {
    r0 = (q[-wpr] >> 30) | ((q[-wpr + 1] & 1u) << 2);
    r1 = (q[0] >> 30) | ((q[1] & 1u) << 2);
    r2 = (q[wpr] >> 30) | ((q[wpr + 1] & 1u) << 2);
  }
  return (r1 >> 2) | ((r0 >> 2) << 1) | (((r0 >> 1) & 1u) << 2) | ((r0 & 1u) << 3) | ((r1 & 1u) << 4) | ((r2 & 1u) << 5) |
         (((r2 >> 1) & 1u) << 6) | ((r2 >> 2) << 7);
}

// Suzuki-Abe outer-border walk from (x0, y0) (padded ROI coordinates).  Returns false when the
// border holds a pixel that precedes (x0, y0) in raster order.  npts = CHAIN_APPROX_SIMPLE vertex
// count, ymax = last row of the border.  RECORD: per-row extreme columns into rmin / rmax (rows
// relative to y0, which is the component's first row when the walk is the owner's).
template <bool RECORD>
__device__ __forceinline__ bool walk_border(const uint32_t *fg, int wpr, int x0, int y0, int step_cap, int &npts, int &ymax,
                                            short *rmin, short *rmax) {
  uint32_t nb = nbr8(fg, wpr, x0, y0);
  ymax = y0;
  if (nb == 0) {                         // isolated pixel
    npts = 1;
    if (RECORD) { rmin[0] = (short)x0; rmax[0] = (short)x0; }
    return true;
  }
  // first neighbour clockwise from W: directions 3, 2, 1, 0, 7, 6, 5 (4 = W itself is background)
  int s = 3;
  while (!((nb >> s) & 1u)) s = (s - 1) & 7;
  const int x1 = x0 + dir_dx(s), y1 = y0 + dir_dy(s);
  int x3 = x0, y3 = y0, prev_s = s ^ 4, n = 0;
  for (int it = 0; it < step_cap; ++it) {
    // next neighbour counter-clockwise after s: rotate the mask so that direction s + 1 is bit 0
    const uint32_t rot = ((nb | (nb << 8)) >> ((s + 1) & 7)) & 0xffu;
    s = (s + __ffs(rot)) & 7;
    const int x4 = x3 + dir_dx(s), y4 = y3 + dir_dy(s);
    if (y4 < y0 || (y4 == y0 && x4 < x0)) return false;
    if (s != prev_s) ++n;
    if (RECORD) {
      const int r = y3 - y0;
      if (x3 < rmin[r]) rmin[r] = (short)x3;
      if (x3 > rmax[r]) rmax[r] = (short)x3;
    }
    ymax = max(ymax, y3);
    prev_s = s;
    if (x4 == x0 && y4 == y0 && x3 == x1 && y3 == y1) { npts = n; return true; }
    x3 = x4; y3 = y4; s = (s + 4) & 7;
    nb = nbr8(fg, wpr, x3, y3);
  }
  return false;                          // safety net: never reached on a consistent bitmap
}

__device__ __forceinline__ int cross3(int a, int b, int cx, int cy) {
  const int ax = a & 0xffff, ay = a >> 16, bx = b & 0xffff, by = b >> 16;
  return (bx - ax) * (cy - ay) - (by - ay) * (cx - ax);
}

// Kept border -> Light (armor.hpp:15-29) -> filter (armor.hpp:31-38) -> best-two list.
// Warp-cooperative; (x0, y0) padded ROI coordinates of the first pixel, ymax its last row.
// need_walk: the row extremes are not in wb yet (the ownership walk ran without recording).
__device__ __forceinline__ void process_border(Shared &sh, const WarpBuf &wb, const uint32_t *fg, int wpr, int x0, int y0,
                                               int ymax, bool need_walk, int step_cap, float min_x, float min_y,
                                               const ArmorParams &p, int lane) {
  const int rows = ymax - y0 + 1;
  if (need_walk) {
    for (int r = lane; r < rows; r += 32) { wb.rmin[r] = 32767; wb.rmax[r] = -1; }
    __syncwarp();
  }
  int nh = 0;
  if (lane == 0) {
    if (need_walk) {
      int npts, ym;
      walk_border<true>(fg, wpr, x0, y0, step_cap, npts, ym, wb.rmin, wb.rmax);
    }
    // convex hull from the row extremes: right side downwards, then left side upwards; both chains
    // turn the same way, end points are hull vertices (extreme rows)
    int n = 0;
    bool overflow = false;
    for (int r = 0; r < rows && !overflow; ++r) {
      const int px = wb.rmax[r] - 1, py = y0 + r - 1;
      while (n >= 2 && cross3(wb.hull[n - 2], wb.hull[n - 1], px, py) <= 0) --n;
      if (n >= wb.hull_cap) { overflow = true; break; }
      wb.hull[n++] = px | (py << 16);
    }
    const int base = n;
    for (int r = rows - 1; r >= 0 && !overflow; --r) {
      const int px = wb.rmin[r] - 1, py = y0 + r - 1;
      while (n - base >= 2 && cross3(wb.hull[n - 2], wb.hull[n - 1], px, py) <= 0) --n;
      if (n >= wb.hull_cap) { overflow = true; break; }
      wb.hull[n++] = px | (py << 16);
    }
    if (!overflow) {
      // junction duplicates: bottom (single-pixel last row) and top (single-pixel first row)
      if (n > base && base > 0 && wb.hull[base] == wb.hull[base - 1]) {
        for (int i = base; i + 1 < n; ++i) wb.hull[i] = wb.hull[i + 1];
        --n;
      }
      if (n > 1 && wb.hull[n - 1] == wb.hull[0]) --n;
      nh = n;
    }
  }
  nh = __shfl_sync(kFull, nh, 0);
  __syncwarp();
  if (nh < 2) return;
  // minimum-area enclosing rectangle: one hull edge per lane; projections relative to hull[0]
  // (small integers: the FP32 products are exact or nearly so whatever the ROI size)
  const int org_x = wb.hull[0] & 0xffff, org_y = wb.hull[0] >> 16;
  float best_area = CUDART_INF_F;
  int best_i = 0x7fffffff;
  for (int i = lane; i < nh; i += 32) {
    const int a = wb.hull[i], b = wb.hull[i + 1 == nh ? 0 : i + 1];
    const int ex = (b & 0xffff) - (a & 0xffff), ey = (b >> 16) - (a >> 16);
    const float ln = __fsqrt_rn((float)(ex * ex + ey * ey));
    const float ux = __fdiv_rn((float)ex, ln), uy = __fdiv_rn((float)ey, ln), vx = -uy, vy = ux;
    float u0 = CUDART_INF_F, u1 = -CUDART_INF_F, v0 = CUDART_INF_F, v1 = -CUDART_INF_F;
    for (int j = 0; j < nh; ++j) {
      const int h = wb.hull[j];
      const float hx = (float)((h & 0xffff) - org_x), hy = (float)((h >> 16) - org_y);
      const float pu = __fadd_rn(__fmul_rn(hx, ux), __fmul_rn(hy, uy));
      const float pv = __fadd_rn(__fmul_rn(hx, vx), __fmul_rn(hy, vy));
      u0 = fminf(u0, pu); u1 = fmaxf(u1, pu); v0 = fminf(v0, pv); v1 = fmaxf(v1, pv);
    }
    const float area = __fmul_rn(__fsub_rn(u1, u0), __fsub_rn(v1, v0));
    if (area < best_area) { best_area = area; best_i = i; }
  }
#pragma unroll
  for (int off = 16; off; off >>= 1) {
    const float oa = __shfl_xor_sync(kFull, best_area, off);
    const int oi = __shfl_xor_sync(kFull, best_i, off);
    if (oa < best_area || (oa == best_area && oi < best_i)) { best_area = oa; best_i = oi; }
  }
  if (lane != 0 || best_i == 0x7fffffff) return;
  // corners of the chosen rectangle
  float cxs[4], cys[4];
  {
    const int i = best_i;
    const int a = wb.hull[i], b = wb.hull[i + 1 == nh ? 0 : i + 1];
    const int ex = (b & 0xffff) - (a & 0xffff), ey = (b >> 16) - (a >> 16);
    const float ln = __fsqrt_rn((float)(ex * ex + ey * ey));
    const float ux = __fdiv_rn((float)ex, ln), uy = __fdiv_rn((float)ey, ln), vx = -uy, vy = ux;
    float u0 = CUDART_INF_F, u1 = -CUDART_INF_F, v0 = CUDART_INF_F, v1 = -CUDART_INF_F;
    for (int j = 0; j < nh; ++j) {
      const int h = wb.hull[j];
      const float hx = (float)((h & 0xffff) - org_x), hy = (float)((h >> 16) - org_y);
      const float pu = __fadd_rn(__fmul_rn(hx, ux), __fmul_rn(hy, uy));
      const float pv = __fadd_rn(__fmul_rn(hx, vx), __fmul_rn(hy, vy));
      u0 = fminf(u0, pu); u1 = fmaxf(u1, pu); v0 = fminf(v0, pv); v1 = fmaxf(v1, pv);
    }
    const float us[4] = {u0, u1, u1, u0}, vs[4] = {v0, v0, v1, v1};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      cxs[k] = __fadd_rn(__fadd_rn(__fmul_rn(ux, us[k]), __fmul_rn(vx, vs[k])), (float)org_x);
      cys[k] = __fadd_rn(__fadd_rn(__fmul_rn(uy, us[k]), __fmul_rn(vy, vs[k])), (float)org_y);
    }
  }
  const float cen_x = __fmul_rn(__fadd_rn(cxs[0], cxs[2]), 0.5f), cen_y = __fmul_rn(__fadd_rn(cys[0], cys[2]), 0.5f);
  // Light::Light: corners by ascending y (stable), top / bottom = midpoints of the upper / lower pair
  int o0 = 0, o1 = 1, o2 = 2, o3 = 3;
  auto cswap = [&](int &a, int &b) { if (cys[b] < cys[a]) { const int t = a; a = b; b = t; } };
  cswap(o0, o1); cswap(o2, o3); cswap(o0, o2); cswap(o1, o3); cswap(o1, o2);
  // (the 5-comparator network is not stable by itself; equal y only happens for axis-parallel
  // rectangles, where either order gives the same midpoints and the same width)
  const float tx = __fdiv_rn(__fadd_rn(cxs[o0], cxs[o1]), 2.f), ty = __fdiv_rn(__fadd_rn(cys[o0], cys[o1]), 2.f);
  const float bx = __fdiv_rn(__fadd_rn(cxs[o2], cxs[o3]), 2.f), by = __fdiv_rn(__fadd_rn(cys[o2], cys[o3]), 2.f);
  const float dx = __fsub_rn(tx, bx), dy = __fsub_rn(ty, by);
  const double length = sqrt((double)dx * dx + (double)dy * dy);
  const float wx = __fsub_rn(cxs[o0], cxs[o1]), wy = __fsub_rn(cys[o0], cys[o1]);
  const double width = sqrt((double)wx * wx + (double)wy * wy);
  const double tilt = (double)atan2f(fabsf(dx), fabsf(dy)) / 3.1415926535897932384626433832795 * 180.0;
  const double ratio = width / length;                 // 0/0 = NaN compares false like the reference
  if (!((double)p.min_ratio < ratio && ratio < (double)p.max_ratio && tilt < (double)p.max_angle)) return;
  LightRec rec;
  rec.cx = __fadd_rn(cen_x, min_x); rec.cy = __fadd_rn(cen_y, min_y);     // Light::offset_bbox
  rec.tx = __fadd_rn(tx, min_x); rec.ty = __fadd_rn(ty, min_y);
  rec.bx = __fadd_rn(bx, min_x); rec.by = __fadd_rn(by, min_y);
  rec.length = length;
  rec.key = (unsigned)(y0 * wpr * 32 + x0);
  while (atomicCAS(&sh.lock, 0, 1) != 0) {}
  __threadfence_block();
  {
    volatile int *nb = &sh.nbest;
    const int n = *nb;
    LightRec b0 = sh.best[0], b1 = sh.best[1];
    if (n == 0 || rec.key > b0.key) { sh.best[1] = b0; sh.best[0] = rec; }
    else if (n == 1 || rec.key > b1.key) sh.best[1] = rec;
    *nb = n < 2 ? n + 1 : 2;
  }
  __threadfence_block();
  atomicExch(&sh.lock, 0);
}

// One detection: bitmap -> exterior flood -> border walks -> lights -> armor.  LARGE selects where
// the per-ROI state lives, so that the small path compiles to shared-memory instructions.
// LUT: Bayer frames go through the raw-domain colour table `lut` (shared memory); CCM: and through the
// colour-correction block `ccm` (shared memory)
template <bool LARGE, bool LUT, bool CCM>
__device__ __forceinline__ void roi_body(Shared &sh, const ArmorParams &p, uint32_t *slot, const uint8_t *frame, const uint8_t *lut,
                                         const uint8_t *ccm, int W, int H,
                                         bool bayer, int rx, int ry, int rw, int rh, float min_x, float min_y, int item,
                                         ArmorOut *out, int tid, int lane, int warp) {
  const int PW = rw + 2, PH = rh + 2, wpr = (PW + 31) >> 5, words = PH * wpr;
  // small ROI: bitmaps, row extremes and hull in shared memory (LDS/STS with 32-bit addresses);
  // large ROI: everything in the global scratch slot this CTA holds for the duration of the ROI
  uint32_t *fg, *ext;
  WarpBuf wb;
  if (LARGE) {
    const size_t bw = slot_bitmap_words(W, H);
    fg = slot; ext = slot + bw;
    uint32_t *wbase = slot + 2 * bw + (size_t)warp * slot_warp_words(H);
    wb.rmin = reinterpret_cast<short *>(wbase);
    wb.rmax = wb.rmin + slot_rows(H);
    wb.hull = reinterpret_cast<int *>(wbase + slot_rows(H));
    wb.hull_cap = slot_hull_cap(H);
  } else {
    fg = sh.fg; ext = sh.ext;
    wb.rmin = sh.rmin[warp]; wb.rmax = sh.rmax[warp]; wb.hull = sh.hull[warp]; wb.hull_cap = kHullSmem;
  }
  long long t0 = 0, t1 = 0, t2 = 0, t3 = 0;
  int rounds = 0;
  if (p.prof && tid == 0) t0 = clock64();
  // 1. threshold bitmap
  if (bayer) build_bitmap<true, LUT, CCM>(fg, frame, lut, ccm, W, H, p.chan_order, p.rotate180, rx, ry, rw, rh, wpr, words, p.binary_threshold, warp, lane);
  else build_bitmap<false, false, false>(fg, frame, nullptr, nullptr, W, H, p.chan_order, p.rotate180, rx, ry, rw, rh, wpr, words, p.binary_threshold, warp, lane);
  __syncthreads();
  if (p.prof && tid == 0) t1 = clock64();
  // 2. exterior background.  Seeds on the padding, spread along runs inside each word; then rounds of
  //    (a) a vertical pass: a warp owns a word column, 32 rows per step, and propagates "exterior"
  //        down and up the column with a warp scan over (generate = exterior, propagate = background)
  //        pairs -- all 32 bit lanes at once, any distance in one pass (the space between two light
  //        bars is open only at its top and bottom);
  //    (b) a relaxation pass by all threads: a word takes the exterior bits of its four neighbours
  //        and spreads them along its runs (one word per round horizontally)
  //    until nothing changes.
  for (int w = tid; w < words; w += kThreads) {
    const int row = w / wpr, wi = w - row * wpr;
    const uint32_t m = ~fg[w];
    uint32_t sd = (row == 0 || row == PH - 1) ? kFull : 0u;
    if (wi == 0) sd |= 1u;
    if (wi == wpr - 1) sd |= kFull << ((PW - 1) & 31);
    ext[w] = fill_runs(sd & m, m);
  }
  __syncthreads();
  {
    const int d_row = kThreads / wpr, d_wi = kThreads - d_row * wpr;
    const int inner = PH - 2;                              // rows 1 .. PH-2
    for (;;) {
      bool changed = false;
      for (int wi = warp; wi < wpr; wi += kWarps) {
#pragma unroll 1
        for (int dirn = 0; dirn < 2; ++dirn) {
          uint32_t carry = ext[(dirn ? PH - 1 : 0) * wpr + wi];
          for (int c0 = 0; c0 < inner; c0 += 32) {
            const int i = c0 + lane;
            const bool valid = i < inner;
            const int r = dirn ? PH - 2 - i : 1 + i;
            const uint32_t e_old = valid ? ext[r * wpr + wi] : 0u;
            const uint32_t m0 = valid ? ~fg[r * wpr + wi] : 0u;
            uint32_t g = e_old, pm = m0;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
              const uint32_t g2 = __shfl_up_sync(kFull, g, d), p2 = __shfl_up_sync(kFull, pm, d);
              if (lane >= d) { g |= pm & g2; pm &= p2; }
            }
            const uint32_t o = g | (pm & carry);
            carry = __shfl_sync(kFull, o, 31);
            // (written run-closed: the relaxation pass only spreads bits that arrive from a neighbour)
            if (valid && o != e_old) { ext[r * wpr + wi] = fill_runs(o, m0); changed = true; }
          }
        }
      }
      __syncthreads();
      int row = tid / wpr, wi = tid - row * wpr;
      for (int w = tid; w < words; w += kThreads) {
        if (row >= 1 && row <= PH - 2) {
          const uint32_t m = ~fg[w], e = ext[w];
          if (m & ~e) {                                    // background bits not yet exterior
            const uint32_t lft = wi > 0 ? ext[w - 1] >> 31 : 0u, rgt = wi + 1 < wpr ? ext[w + 1] & 1u : 0u;
            const uint32_t sd = e | (m & (ext[w - wpr] | ext[w + wpr] | lft | (rgt << 31)));
            if (sd != e) { ext[w] = fill_runs(sd, m); changed = true; }
          }
        }
        row += d_row; wi += d_wi;
        if (wi >= wpr) { wi -= wpr; ++row; }
      }
      ++rounds;
      if (!__syncthreads_or(changed)) break;
    }
  }
  if (p.prof && tid == 0) t2 = clock64();
  // 3. border walks from the start candidates, 4. lights
  const int step_cap = 8 * PW * PH;
  // start candidates: foreground, exterior background to the W, background to the NW, N, NE
  auto candidates_of = [&](int w, int row, int wi) -> uint32_t {
    if (row < 1 || row > PH - 2) return 0u;
    const uint32_t f0 = fg[w], e0 = ext[w];
    if (!f0) return 0u;
    const uint32_t ep = wi > 0 ? ext[w - 1] >> 31 : 0u;
    const uint32_t un = fg[w - wpr];
    const uint32_t up = wi > 0 ? fg[w - wpr - 1] >> 31 : 0u, ux = wi + 1 < wpr ? fg[w - wpr + 1] << 31 : 0u;
    const uint32_t ext_w = (e0 << 1) | ep;
    const uint32_t above = un | (un << 1) | up | (un >> 1) | ux;
    return f0 & ext_w & ~above;
  };
  {
    const int d_row = kThreads / wpr, d_wi = kThreads - d_row * wpr;
    int row = tid / wpr, wi = tid - row * wpr;
    for (int w = tid; w < words; w += kThreads) {
      uint32_t cand = candidates_of(w, row, wi);
      while (cand) {
        const int b = __ffs(cand) - 1;
        cand &= cand - 1;
        const int idx = atomicAdd(&sh.ncand, 1);
        if (idx < kCandCap) sh.cand[idx] = (wi * 32 + b) | (row << 16);
      }
      row += d_row; wi += d_wi;
      if (wi >= wpr) { wi -= wpr; ++row; }
    }
  }
  __syncthreads();
  const int ncand_roi = sh.ncand;
  if (ncand_roi <= kCandCap) {
    // few candidates (the usual case: a light bar has one, a number sticker a handful): the warps
    // take them round-robin, one walk each, recording the row extremes as it goes, so a kept border
    // is walked once and the borders of one ROI are walked side by side
    for (int c = warp; c < ncand_roi; c += kWarps) {
      const int X0 = sh.cand[c] & 0xffff, Y0 = sh.cand[c] >> 16;
      const int span = PH - 1 - Y0;                        // rows the border can reach
      for (int r = lane; r < span; r += 32) { wb.rmin[r] = 32767; wb.rmax[r] = -1; }
      __syncwarp();
      int ok = 0, ymax = 0;
      long long c0 = 0, c1 = 0;
      if (lane == 0) {
        int npts = 0;
        if (p.prof) c0 = clock64();
        ok = walk_border<true>(fg, wpr, X0, Y0, step_cap, npts, ymax, wb.rmin, wb.rmax) && npts >= 5;
        if (p.prof) c1 = clock64();
      }
      ok = __shfl_sync(kFull, ok, 0);
      const int YM = __shfl_sync(kFull, ymax, 0);
      if (ok) process_border(sh, wb, fg, wpr, X0, Y0, YM, false, step_cap, min_x, min_y, p, lane);
      __syncwarp();
      if (p.prof && lane == 0) {
        atomicAdd(p.prof + 6, (unsigned long long)(c1 - c0));
        atomicAdd(p.prof + 7, (unsigned long long)(clock64() - c1));
      }
    }
  } else {
    // many candidates (speckle): a warp takes 32 words at a time, every lane walks its own
    // candidate for ownership and vertex count; the few that pass are walked again, recording
    const int nchunks = (words + 31) >> 5;
    for (int chunk = warp; chunk < nchunks; chunk += kWarps) {
      const int w = chunk * 32 + lane;
      uint32_t cand = 0;
      int row = 0, wi = 0;
      if (w < words) {
        row = w / wpr; wi = w - row * wpr;
        cand = candidates_of(w, row, wi);
      }
      while (__any_sync(kFull, cand != 0)) {
        bool acc = false;
        int x0 = 0, y0 = 0, ymax = 0;
        if (cand) {
          const int bpos = __ffs(cand) - 1;
          cand &= cand - 1;
          x0 = wi * 32 + bpos; y0 = row;
          int npts = 0;
          acc = walk_border<false>(fg, wpr, x0, y0, step_cap, npts, ymax, nullptr, nullptr) && npts >= 5;
        }
        uint32_t m = __ballot_sync(kFull, acc);
        while (m) {
          const int src = __ffs(m) - 1;
          m &= m - 1;
          const int X0 = __shfl_sync(kFull, x0, src), Y0 = __shfl_sync(kFull, y0, src), YM = __shfl_sync(kFull, ymax, src);
          process_border(sh, wb, fg, wpr, X0, Y0, YM, true, step_cap, min_x, min_y, p, lane);
          __syncwarp();
        }
      }
    }
  }
  __syncthreads();
  if (p.prof && tid == 0) t3 = clock64();
  // 5. Armor::Armor (armor.hpp:58-68) and the centre-distance filter (src/irm_detector.cpp:333-350)
  if (tid == 0) {
    int valid = 0;
    if (sh.nbest >= 2) {
      const LightRec l0 = sh.best[0], l1 = sh.best[1];
      const bool first_left = l0.cx < l1.cx;
      const LightRec L = first_left ? l0 : l1, R = first_left ? l1 : l0;
      const double avg_len = (l0.length + l1.length) / 2;
      const float ddx = __fsub_rn(L.cx, R.cx), ddy = __fsub_rn(L.cy, R.cy);
      const double cd = sqrt((double)ddx * ddx + (double)ddy * ddy) / avg_len;
      const int size = cd > p.min_large ? 1 : 0;
      bool ok = true;
      if (size == 0 && (p.min_small > cd || p.max_small < cd)) ok = false;
      if (size == 1 && (p.min_large > cd || p.max_large < cd)) ok = false;
      if (ok) {
        out->pts[0] = L.bx; out->pts[1] = L.by; out->pts[2] = L.tx; out->pts[3] = L.ty;
        out->pts[4] = R.tx; out->pts[5] = R.ty; out->pts[6] = R.bx; out->pts[7] = R.by;
        out->center[0] = __fdiv_rn(__fadd_rn(L.cx, R.cx), 2.f);
        out->center[1] = __fdiv_rn(__fadd_rn(L.cy, R.cy), 2.f);
        out->score = p.scores[item];
        const int c = p.classes[item];
        out->class_id = (c >= 0 && c < 14) ? c : 14;
        out->size = size;
        valid = 1;
      }
    }
    out->valid = valid;
    if (p.prof) {
      const long long t4 = clock64();
      atomicAdd(p.prof + 0, (unsigned long long)(t1 - t0)); atomicAdd(p.prof + 1, (unsigned long long)(t2 - t1));
      atomicAdd(p.prof + 2, (unsigned long long)(t3 - t2)); atomicAdd(p.prof + 3, (unsigned long long)(t4 - t3));
      atomicAdd(p.prof + 4, 1ull); atomicAdd(p.prof + 5, (unsigned long long)rounds);
    }
  }
}

// LUT: Bayer frames with a raw-domain colour table; the table (1 KB) follows Shared in dynamic shared memory
// and is visible after the barrier that precedes the first ROI.  CCM: Bayer frames with a colour-correction block
// (kCcmBytes), staged behind the raw table's place the same way.  FRAME_CCM (with CCM): one block per frame
// (p.ccm_stride, auto white balance), staged again before every ROI -- a separate instantiation, so that the
// engine-wide one keeps its registers and spills.
template <bool LUT, bool CCM, bool FRAME_CCM = false>
__global__ void __launch_bounds__(kThreads, 3) extract_armors_kernel(ArmorParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  Shared &sh = *reinterpret_cast<Shared *>(smem_raw);
  uint8_t *lut = smem_raw + sizeof(Shared);
  uint8_t *ccm = lut + (LUT ? 1024 : 0);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (LUT) reinterpret_cast<uint32_t *>(lut)[tid] = reinterpret_cast<const uint32_t *>(p.raw_lut)[tid];   // kThreads == 256 words
  if (CCM && !FRAME_CCM) stage_ccm(ccm, p.ccm, tid);
  const int W = p.src_w, H = p.src_h;
  const bool bayer = p.chan_order >= 2;
  const size_t frame_bytes = (size_t)W * H * (bayer ? 1 : 3);
  const uint8_t *base = p.src_indirect ? *p.src_indirect : p.src;
  const int total = p.n * p.max_det;
  // detection-major work order: the real detections (k < num[f]) come first and spread evenly over
  // the CTAs; the empty slots that follow only clear their flag
  for (int it = blockIdx.x; it < total; it += gridDim.x) {
    const int k = it / p.n, f = it - k * p.n;
    const int item = f * p.max_det + k;
    ArmorOut *out = p.out + item;
    if (k >= p.num[f]) {
      if (tid == 0) out->valid = 0;
      continue;
    }
    // ROI (src/irm_detector.cpp:299-304): float clamp, cv::Rect truncation
    const float4 b = reinterpret_cast<const float4 *>(p.boxes)[item];
    const float x1 = __fmul_rn(__fsub_rn(b.x, p.box_px), p.box_sx), y1 = __fmul_rn(__fsub_rn(b.y, p.box_py), p.box_sy);
    const float x2 = __fmul_rn(__fsub_rn(b.z, p.box_px), p.box_sx), y2 = __fmul_rn(__fsub_rn(b.w, p.box_py), p.box_sy);
    const float min_x = x1 > 0.f ? x1 : 0.f, min_y = y1 > 0.f ? y1 : 0.f;
    const float max_x = x2 < (float)W ? x2 : (float)W, max_y = y2 < (float)H ? y2 : (float)H;
    const int rx = (int)min_x, ry = (int)min_y;
    const int rw = (int)__fsub_rn(max_x, min_x), rh = (int)__fsub_rn(max_y, min_y);
    if (!(min_x < max_x && min_y < max_y) || rw <= 0 || rh <= 0) {
      if (tid == 0) out->valid = 0;
      continue;
    }
    const int words_roi = (rh + 2) * ((rw + 2 + 31) >> 5);
    const bool large = words_roi > kSmemWords || rh > kRows;
    // the previous ROI is done with the block (barrier at the end of the loop), the barrier below publishes this one
    if (FRAME_CCM) stage_ccm(ccm, p.ccm + (size_t)f * p.ccm_stride, tid);
    if (tid == 0) {
      sh.nbest = 0; sh.lock = 0; sh.slot = -1; sh.ncand = 0;
      if (large) sh.slot = blockIdx.x;   // this CTA's own global scratch slot
    }
    __syncthreads();
    const uint8_t *frame = base + (size_t)f * frame_bytes;
    if (large) {
      roi_body<true, LUT, CCM>(sh, p, p.scratch + (size_t)sh.slot * p.scratch_words_per_cta, frame, lut, ccm, W, H, bayer, rx, ry, rw, rh, min_x,
                     min_y, item, out, tid, lane, warp);
    } else {
      roi_body<false, LUT, CCM>(sh, p, nullptr, frame, lut, ccm, W, H, bayer, rx, ry, rw, rh, min_x, min_y, item, out, tid, lane, warp);
    }
    __syncthreads();
  }
}

// Armor corners {left.bottom, left.top, right.top, right.bottom} -> PnP quads in the calibration
// frame (src/pnp_solver.cpp:41-44); slots without an armor get a fixed valid quad and are masked after.
__global__ void quads_from_armors_kernel(const ArmorOut *armors, int total, float sx, float sy, float *pts, float *centers) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const ArmorOut &a = armors[i];
  float q[8] = {150.f, 160.f, 150.f, 140.f, 200.f, 140.f, 200.f, 160.f};
  if (a.valid) {
#pragma unroll
    for (int k = 0; k < 4; ++k) { q[2 * k] = a.pts[2 * k] * sx; q[2 * k + 1] = a.pts[2 * k + 1] * sy; }
  }
  float4 *o = reinterpret_cast<float4 *>(pts + (size_t)i * 8);
  o[0] = make_float4(q[0], q[1], q[2], q[3]);
  o[1] = make_float4(q[4], q[5], q[6], q[7]);
  // Armor::center in the calibration frame (argument of calculateDistanceToCenter, reference src/irm_detector.cpp:229)
  if (centers) reinterpret_cast<float2 *>(centers)[i] = a.valid ? make_float2(a.center[0] * sx, a.center[1] * sy) : make_float2(175.f, 150.f);
}

__global__ void mask_pose_ok_kernel(const ArmorOut *armors, int total, uint8_t *ok) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total && !armors[i].valid) ok[i] = 0;
}

}  // namespace

int armors_grid(int num_sms) { return num_sms * 3; }

// scratch layout: [64 words, unused][one slot per CTA of the grid]
size_t armors_scratch_words_per_cta(int src_w, int src_h) { return slot_words(src_w, src_h); }
size_t armors_scratch_total_words(int src_w, int src_h, int grid) { return 64 + (size_t)grid * slot_words(src_w, src_h); }

// armors_grid() runs 3 CTAs per SM: the tables must leave room for them (228 KB per SM, 1 KB reserved per CTA)
static_assert(3 * (sizeof(Shared) + 1024 + kCcmBytes + 1024) <= 228 * 1024, "colour tables cost the armor stage a CTA per SM");

const char *armors_geometry_error(int src_w, int src_h) {
  if (src_w < 1 || src_h < 1) return "extract_armors: the source must have at least one row and one column";
  if (src_w > kMaxSide || src_h > kMaxSide)
    return "extract_armors: source width and height must be at most 32766 (coordinates are packed into 16 bits)";
  if (8 * ((long long)src_w + 2) * ((long long)src_h + 2) > 0x7fffffffLL)
    return "extract_armors: 8 * (width + 2) * (height + 2) must stay below 2^31 (the border walk's step cap is an int)";
  return nullptr;
}

cudaError_t launch_extract_armors(const ArmorParams &p, cudaStream_t s) {
  if ((p.raw_lut || p.ccm) && p.chan_order < 2) return cudaErrorInvalidValue;   // the tables are defined for Bayer sources only
  auto kernel = p.ccm && p.ccm_stride ? (p.raw_lut ? extract_armors_kernel<true, true, true> : extract_armors_kernel<false, true, true>)
              : p.ccm ? (p.raw_lut ? extract_armors_kernel<true, true> : extract_armors_kernel<false, true>)
                      : (p.raw_lut ? extract_armors_kernel<true, false> : extract_armors_kernel<false, false>);
  const size_t smem = sizeof(Shared) + (p.raw_lut ? 1024 : 0) + (p.ccm ? kCcmBytes : 0);
  {   // per device and cheap: no process-wide "already configured" flag (several engines / devices per process)
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  const int total = p.n * p.max_det;
  if (total <= 0) return cudaSuccess;
  const int grid = total < p.grid ? total : p.grid;
  kernel<<<grid, kThreads, smem, s>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_quads_from_armors(const ArmorOut *armors, int total, float sx, float sy, float *pts, float *centers, cudaStream_t s) {
  if (total <= 0) return cudaSuccess;
  quads_from_armors_kernel<<<(total + 127) / 128, 128, 0, s>>>(armors, total, sx, sy, pts, centers);
  return cudaGetLastError();
}

cudaError_t launch_mask_pose_ok(const ArmorOut *armors, int total, uint8_t *ok, cudaStream_t s) {
  if (total <= 0) return cudaSuccess;
  mask_pose_ok_kernel<<<(total + 127) / 128, 128, 0, s>>>(armors, total, ok);
  return cudaGetLastError();
}

}  // namespace irmv
