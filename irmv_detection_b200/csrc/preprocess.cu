// Fused preprocess for sm_100a: one kernel replaces the reference's four NPP calls
// (nppiMirror -> nppiResize LINEAR -> nppiScale /255 -> nppiCopy HWC->CHW,
// reference src/yolo_engine.cpp:179-200) and the camera ISP's Bayer->RGB step
// (reference src/mv_camera.cpp:96).  HBM-bound: each source byte is read once with 128-bit
// loads into shared memory, each output pixel is written once as one 16-byte NHWC8 FP16 store.
//
// Arithmetic is written with explicitly rounded FP32 intrinsics so it is bit-identical to
// oracle/preprocess_ref.py (no FMA contraction).
#include <cstdlib>

#include "common.cuh"

namespace irmv {
namespace {

constexpr int TH = 8;     // output rows per CTA
constexpr int TW = 64;    // output cols per CTA
constexpr int NT = 256;

struct Taps { int i0, i1; float f; int ok; };   // ok = 0: letterbox padding (value 114)

// half_pixel = 0: NPP's measured convention (corner-aligned, src = dst * scale), reference-exact;
// half_pixel = 1: OpenCV-style pixel centres.
__device__ __forceinline__ Taps axis_taps(int d, float scale, int n_src, int half_pixel) {
  float s = half_pixel ? __fsub_rn(__fmul_rn(__fadd_rn((float)d, 0.5f), scale), 0.5f)
                       : __fmul_rn((float)d, scale);
  float fl = floorf(s);
  Taps t;
  t.ok = 1;
  t.f = __fsub_rn(s, fl);
  int i0 = (int)fl;
  t.i0 = min(max(i0, 0), n_src - 1);
  t.i1 = min(max(i0 + 1, 0), n_src - 1);
  return t;
}

// Network-input coordinate d of a letterboxed axis: the resized image occupies [pad, pad + n_new).
__device__ __forceinline__ Taps axis_taps_lb(int d, int pad, int n_new, float scale, int n_src, int half_pixel) {
  const int dr = d - pad;
  Taps t = axis_taps(min(max(dr, 0), n_new - 1), scale, n_src, half_pixel);
  t.ok = dr >= 0 && dr < n_new;
  return t;
}

__device__ __forceinline__ int reflect101(int i, int n) {
  if (i < 0) i = -i;
  if (i >= n) i = 2 * n - 2 - i;
  return i;
}

struct Region {
  const uint8_t *frame;   // frame base (global)
  const uint8_t *smem;    // staged rows
  int row_lo;             // first staged source row
  int pitch_s;            // bytes per staged row
  int col_byte_lo;        // first needed byte inside a source row
  int src_pitch;          // bytes per source row
  int shift0, dshift;     // (address of staged row 0) & 15, and src_pitch & 15: row r starts at
                          // smem offset r*pitch_s + ((shift0 + r*dshift) & 15)
  int nrows, nbytes;      // staged rows, needed bytes per row
};

// byte of source row `sy`, byte column `bx` (already inside the staged window)
__device__ __forceinline__ int rd(const Region &r, int sy, int bx) {
  const int rr = sy - r.row_lo;
  return r.smem[rr * r.pitch_s + ((r.shift0 + rr * r.dshift) & 15) + (bx - r.col_byte_lo)];
}

// pointer such that rowp(r, sy)[bx] is byte column bx of source row sy
__device__ __forceinline__ const uint8_t *rowp(const Region &r, int sy) {
  const int rr = sy - r.row_lo;
  return r.smem + rr * r.pitch_s + ((r.shift0 + rr * r.dshift) & 15) - r.col_byte_lo;
}

// RGB at source pixel (sy,sx) of a Bayer mosaic, bilinear demosaic (oracle demosaic_bilinear)
__device__ __forceinline__ void bayer_rgb(const Region &r, int sy, int sx, int H, int W, int red_y,
                                          int red_x, int &R, int &G, int &B) {
  int ym = sy - 1, yp = sy + 1, xm = sx - 1, xp = sx + 1;
  if (sy == 0 || sx == 0 || sy == H - 1 || sx == W - 1) {       // image border: mirror (reflect-101)
    ym = reflect101(ym, H); yp = reflect101(yp, H);
    xm = reflect101(xm, W); xp = reflect101(xp, W);
  }
  // branch-free: neighbouring samples sit on different colour sites, so a site-dependent branch
  // would run both arms for most warps anyway
  const uint8_t *r0 = rowp(r, ym), *r1 = rowp(r, sy), *r2 = rowp(r, yp);
  const int nw = r0[xm], n = r0[sx], ne = r0[xp];
  const int w = r1[xm], c = r1[sx], e = r1[xp];
  const int sw = r2[xm], s = r2[sx], se = r2[xp];
  const int cross = (n + s + w + e + 2) >> 2, diag = (nw + ne + sw + se + 2) >> 2;
  const int horiz = (w + e + 1) >> 1, vert = (n + s + 1) >> 1;
  const bool red_row = ((sy & 1) == red_y), red_col = ((sx & 1) == red_x);
  const bool is_r = red_row && red_col, is_b = !red_row && !red_col;
  G = (is_r || is_b) ? cross : c;
  R = is_r ? c : (is_b ? diag : (red_row ? horiz : vert));
  B = is_b ? c : (is_r ? diag : (red_row ? vert : horiz));
}

// Same demosaic with the column part hoisted: oxm / ox0 / oxp are the byte offsets of columns
// sx-1 / sx / sx+1 (already mirrored at the image border) inside a staged row, red_col is the
// column's colour-site parity.  Used by the stem's fast path, where one thread walks down a column.
__device__ __forceinline__ void bayer_rgb_col(const Region &r, int sy, int H, int oxm, int ox0, int oxp,
                                              bool red_col, int red_y, int &R, int &G, int &B) {
  int ym = sy - 1, yp = sy + 1;
  if (sy == 0 || sy == H - 1) { ym = reflect101(ym, H); yp = reflect101(yp, H); }
  const uint8_t *r0 = rowp(r, ym) + r.col_byte_lo, *r1 = rowp(r, sy) + r.col_byte_lo, *r2 = rowp(r, yp) + r.col_byte_lo;
  const int nw = r0[oxm], n = r0[ox0], ne = r0[oxp];
  const int w = r1[oxm], c = r1[ox0], e = r1[oxp];
  const int sw = r2[oxm], s = r2[ox0], se = r2[oxp];
  const int cross = (n + s + w + e + 2) >> 2, diag = (nw + ne + sw + se + 2) >> 2;
  const int horiz = (w + e + 1) >> 1, vert = (n + s + 1) >> 1;
  const bool red_row = ((sy & 1) == red_y);
  const bool is_r = red_row && red_col, is_b = !red_row && !red_col;
  G = (is_r || is_b) ? cross : c;
  R = is_r ? c : (is_b ? diag : (red_row ? horiz : vert));
  B = is_b ? c : (is_r ? diag : (red_row ? vert : horiz));
}

__device__ __forceinline__ float lerp4(float p00, float p01, float p10, float p11, float fx,
                                       float fy) {
  float ofx = __fsub_rn(1.0f, fx), ofy = __fsub_rn(1.0f, fy);
  float top = __fadd_rn(__fmul_rn(p00, ofx), __fmul_rn(p01, fx));
  float bot = __fadd_rn(__fmul_rn(p10, ofx), __fmul_rn(p11, fx));
  return __fadd_rn(__fmul_rn(top, ofy), __fmul_rn(bot, fy));
}

// lut[k] = k/255 (FP32, exactly rounded): the 8-bit intermediate makes the final division a lookup
__device__ __forceinline__ float finish(float v, int quantize, const float *lut) {
  if (quantize) return lut[(int)fminf(fmaxf(floorf(__fadd_rn(v, 0.5f)), 0.0f), 255.0f)];
  return __fdiv_rn(v, 255.0f);
}

// One network-input pixel (oy, ox): rot180 + resize taps + (demosaic | channel swap) + lerp +
// 8-bit quantisation + /255, from the staged source window.  v = {R, G, B} as fed to the net.
// CCM: every demosaiced pixel goes through the colour-correction block `ccm` (shared memory) before the lerp.
template <bool CCM>
__device__ __forceinline__ void sample_pixel(const Region &reg, const PreprocessParams &p, const Taps &ty,
                                             const Taps &tx, int red_y, int red_x, const float *lut,
                                             const uint8_t *ccm, float (&v)[3]) {
  const int H = p.src_h, W = p.src_w;
  const bool bayer = p.chan_order >= 2;
  const bool swap = (p.chan_order == 1);
  int ys[2] = {ty.i0, ty.i1}, xs[2] = {tx.i0, tx.i1};
  float pix[2][2][3];
  // a tap with weight exactly 0 contributes p*0 = +0 to an exactly rounded sum: skipping it is
  // bit-identical and halves the work when the scale is an integer (1280 -> 640: fx == 0)
  const bool need_x1 = tx.f != 0.0f, need_y1 = ty.f != 0.0f;
#pragma unroll
  for (int a = 0; a < 2; ++a) {
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      if ((a == 1 && !need_y1) || (b == 1 && !need_x1)) {
        pix[a][b][0] = pix[a][b][1] = pix[a][b][2] = 0.0f;
        continue;
      }
      int sy = p.rotate180 ? H - 1 - ys[a] : ys[a];
      int sx = p.rotate180 ? W - 1 - xs[b] : xs[b];
      int R, G, B;
      if (bayer) {
        bayer_rgb(reg, sy, sx, H, W, red_y, red_x, R, G, B);
        if (CCM) apply_ccm(ccm, R, G, B);
      } else {
        R = rd(reg, sy, sx * 3 + 0);
        G = rd(reg, sy, sx * 3 + 1);
        B = rd(reg, sy, sx * 3 + 2);
        if (swap) { int t = R; R = B; B = t; }
      }
      pix[a][b][0] = (float)R; pix[a][b][1] = (float)G; pix[a][b][2] = (float)B;
    }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c)
    v[c] = finish(lerp4(pix[0][0][c], pix[0][1][c], pix[1][0][c], pix[1][1][c], tx.f, ty.f), p.quantize_u8, lut);
}

// Stage the source window needed by network-input rows [iy_lo, iy_hi] x cols [ix_lo, ix_hi] into
// shared memory with 16-byte loads aligned on absolute addresses; returns the Region describing it.
__device__ __forceinline__ Region stage_window(const PreprocessParams &p, const uint8_t *base, const uint8_t *frame,
                                               uint8_t *smem, int pitch_s, int iy_lo, int iy_hi, int ix_lo, int ix_hi,
                                               float scale_x, float scale_y, int hp, int nthreads) {
  const bool bayer = p.chan_order >= 2;
  const int bpp = bayer ? 1 : 3;
  const int H = p.src_h, W = p.src_w;
  const int src_pitch = W * bpp;
  const size_t frame_bytes = (size_t)H * src_pitch;
  Taps ty0 = axis_taps_lb(iy_lo, p.pad_y, p.new_h, scale_y, H, hp), ty1 = axis_taps_lb(iy_hi, p.pad_y, p.new_h, scale_y, H, hp);
  Taps tx0 = axis_taps_lb(ix_lo, p.pad_x, p.new_w, scale_x, W, hp), tx1 = axis_taps_lb(ix_hi, p.pad_x, p.new_w, scale_x, W, hp);
  int ry_lo = ty0.i0, ry_hi = ty1.i1, rx_lo = tx0.i0, rx_hi = tx1.i1;
  int sy_lo = p.rotate180 ? H - 1 - ry_hi : ry_lo, sy_hi = p.rotate180 ? H - 1 - ry_lo : ry_hi;
  int sx_lo = p.rotate180 ? W - 1 - rx_hi : rx_lo, sx_hi = p.rotate180 ? W - 1 - rx_lo : rx_hi;
  if (bayer) {
    sy_lo = max(sy_lo - 2, 0); sy_hi = min(sy_hi + 2, H - 1);
    sx_lo = max(sx_lo - 2, 0); sx_hi = min(sx_hi + 2, W - 1);
  }
  const int nrows = sy_hi - sy_lo + 1;
  const int col_byte_lo = sx_lo * bpp;
  const int nbytes = (sx_hi - sx_lo + 1) * bpp;
  const int chunks_per_row = pitch_s >> 4;
  const uint8_t *alloc_end = base + (size_t)(p.frame0 + p.n) * frame_bytes;
  auto stage_chunk = [&](int r, int c) {
    const uint8_t *row = frame + (size_t)(sy_lo + r) * src_pitch + col_byte_lo;
    const uint8_t *a = (const uint8_t *)((size_t)row & ~(size_t)15) + (size_t)c * 16;
    // asynchronous copy (zero fill outside the window): the caller overlaps it with its table set-up
    // and waits with stage_wait()
    const bool in = a < row + nbytes && a < alloc_end;
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem + (size_t)r * pitch_s + c * 16);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(in ? a : frame), "r"(in ? 16u : 0u) : "memory");
  };
  if (chunks_per_row <= 8) {                    // 8 threads per staged row, no division
    const int c = threadIdx.x & 7;
    if (c < chunks_per_row)
      for (int r = threadIdx.x >> 3; r < nrows; r += nthreads >> 3) stage_chunk(r, c);
  } else {
    for (int i = threadIdx.x; i < nrows * chunks_per_row; i += nthreads) {
      const int r = i / chunks_per_row;
      stage_chunk(r, i - r * chunks_per_row);
    }
  }
  const int shift0 = (int)((size_t)(frame + (size_t)sy_lo * src_pitch + col_byte_lo) & 15);
  return Region{frame, smem, sy_lo, pitch_s, col_byte_lo, src_pitch, shift0, src_pitch & 15, nrows, nbytes};
}

__device__ __forceinline__ void stage_wait() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Raw-domain colour stage of a Bayer source (PreprocessParams::raw_lut), in place on the staged window after
// stage_wait() + a barrier: the sample of source row sy, column sx becomes lut[sy & 1][sx & 1][sample].  The caller
// adds a barrier before the window is read.
__device__ __forceinline__ void apply_raw_lut(const Region &r, const uint8_t *__restrict__ lut, int nthreads) {
  uint8_t *smem = const_cast<uint8_t *>(r.smem);
  for (int i = threadIdx.x; i < r.nrows * r.nbytes; i += nthreads) {
    const int rr = i / r.nbytes, k = i - rr * r.nbytes;
    const int sy = r.row_lo + rr, sx = r.col_byte_lo + k;
    uint8_t &b = smem[rr * r.pitch_s + ((r.shift0 + rr * r.dshift) & 15) + k];
    b = __ldg(lut + ((sy & 1) * 2 + (sx & 1)) * 256 + b);
  }
}

// LUT: Bayer source with a raw-domain colour table (p.raw_lut).  CCM: Bayer source with a colour-correction block
// (p.ccm; the frame's own block when p.ccm_stride is set), staged behind the source window (rows_cap * pitch_s bytes)
template <bool LUT, bool CCM>
__global__ void __launch_bounds__(NT)
preprocess_kernel(PreprocessParams p, int rows_cap, int pitch_s) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint8_t *ccm = smem + (size_t)rows_cap * pitch_s;
  const int n = blockIdx.z;
  if (CCM) stage_ccm(ccm, p.ccm + (size_t)(p.frame0 + n) * p.ccm_stride, threadIdx.x);
  const int oy0 = blockIdx.y * TH, ox0 = blockIdx.x * TW;
  const bool bayer = p.chan_order >= 2;
  const int bpp = bayer ? 1 : 3;
  const int H = p.src_h, W = p.src_w;
  const int src_pitch = W * bpp;
  const size_t frame_bytes = (size_t)H * src_pitch;
  const uint8_t *base = p.src_indirect ? *p.src_indirect : p.src;
  const uint8_t *frame = base + (size_t)(p.frame0 + n) * frame_bytes;
  const float scale_x = __fdiv_rn((float)W, (float)p.new_w);
  const float scale_y = __fdiv_rn((float)H, (float)p.new_h);
  const int hp = (p.resize_mode != 0);

  __shared__ float lut[256];
  __shared__ Taps ytap[TH], xtap[TW];
  lut[threadIdx.x & 255] = __fdiv_rn((float)(threadIdx.x & 255), 255.0f);
  if (threadIdx.x < TH) ytap[threadIdx.x] = axis_taps_lb(min(oy0 + (int)threadIdx.x, kNet - 1), p.pad_y, p.new_h, scale_y, H, hp);
  else if (threadIdx.x < TH + TW) xtap[threadIdx.x - TH] = axis_taps_lb(min(ox0 + (int)threadIdx.x - TH, kNet - 1), p.pad_x, p.new_w, scale_x, W, hp);
  Region reg = stage_window(p, base, frame, smem, pitch_s, oy0, min(oy0 + TH, kNet) - 1, ox0, min(ox0 + TW, kNet) - 1,
                            scale_x, scale_y, hp, NT);
  stage_wait();
  __syncthreads();
  if (LUT) {
    apply_raw_lut(reg, p.raw_lut, NT);
    __syncthreads();
  }

  int red_y = 0, red_x = 0;
  if (p.chan_order == 3) { red_y = 1; red_x = 1; }       // BGGR
  else if (p.chan_order == 4) { red_y = 0; red_x = 1; }  // GRBG
  else if (p.chan_order == 5) { red_y = 1; red_x = 0; }  // GBRG

  for (int q = threadIdx.x; q < TH * TW; q += NT) {
    int oy = oy0 + q / TW, ox = ox0 + q % TW;
    if (oy >= kNet || ox >= kNet) continue;
    float v[3];
    if (ytap[q / TW].ok && xtap[q % TW].ok) sample_pixel<CCM>(reg, p, ytap[q / TW], xtap[q % TW], red_y, red_x, lut, ccm, v);
    else v[0] = v[1] = v[2] = lut[114];                 // letterbox padding: 114 / 255
    __half2 h01 = __halves2half2(__float2half_rn(v[0]), __float2half_rn(v[1]));
    __half2 h23 = __halves2half2(__float2half_rn(v[2]), __float2half_rn(0.0f));
    uint4 o;
    o.x = *reinterpret_cast<uint32_t *>(&h01);
    o.y = *reinterpret_cast<uint32_t *>(&h23);
    o.z = 0u; o.w = 0u;
    size_t pix_idx = (size_t)pr_index(n, oy, ox, kNet, kNet);
    *reinterpret_cast<uint4 *>(p.dst + pix_idx * kInC) = o;
  }
}

// ------------------------------------------------------------------------------------ fused stem
// preprocess + conv0 (3x3, stride 2, 3->16, bias, SiLU) in one kernel: the 640x640x3 network input
// is produced tile by tile in shared memory and consumed there, so it never touches HBM (it would
// be 6.5 MB written + read per frame as NHWC8).  conv0 is 88 MFLOP per frame with K = 27: CUDA-core
// FP32 FMAs from shared memory; the input values are rounded to FP16 first so the result matches
// the unfused (tensor-core) path's operands.
constexpr int ST = 16;                 // output tile side
constexpr int SI = 2 * ST + 1;         // input tile side (33)

__device__ __forceinline__ float silu_fast(float x) {
  const float h = 0.5f * x;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

// LUT / CCM: as preprocess_kernel; the colour-correction block follows the source window (smem_win bytes)
template <bool LUT, bool CCM>
__global__ void __launch_bounds__(ST * ST)
stem_kernel(PreprocessParams p, const float *__restrict__ w, const float *__restrict__ bias, __half *out,
            long long out_pstride, __half *out2, long long out2_pstride, int pitch_s, int fast_x, int smem_win) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint8_t *ccm = smem + smem_win;
  if (CCM) stage_ccm(ccm, p.ccm + (size_t)(p.frame0 + blockIdx.z) * p.ccm_stride, threadIdx.x);
  __shared__ __half tile[3][SI][SI + 1];             // network-input tile, already rounded to FP16
  __shared__ uint32_t sbf[16][16];                   // conv0 weights as half2 {w[n][2j], w[n][2j+1]}, K padded to 32
  __shared__ float sbias[16];
  __shared__ short skoff[32];                        // tile offset (halfs) of GEMM column k = tap*3 + c
  const int n = blockIdx.z, oy0 = blockIdx.y * ST, ox0 = blockIdx.x * ST;
  const bool bayer = p.chan_order >= 2;
  const int H = p.src_h, W = p.src_w;
  const size_t frame_bytes = (size_t)H * W * (bayer ? 1 : 3);
  const uint8_t *base = p.src_indirect ? *p.src_indirect : p.src;
  const uint8_t *frame = base + (size_t)(p.frame0 + n) * frame_bytes;
  const float scale_x = __fdiv_rn((float)W, (float)p.new_w), scale_y = __fdiv_rn((float)H, (float)p.new_h);
  const int hp = (p.resize_mode != 0);
  __shared__ float lut[256];
  __shared__ __half lut_h[256];
  __shared__ Taps ytap[SI], xtap[SI];
  // network-input window of this tile: rows 2*oy0-1 .. 2*oy0+2*ST-1 (clipped: outside is conv padding).
  // The source window is fetched with cp.async first; the tables below are built while it lands.
  const int iy_lo = 2 * oy0 - 1, ix_lo = 2 * ox0 - 1;
  Region reg = stage_window(p, base, frame, smem, pitch_s, max(iy_lo, 0), min(iy_lo + SI - 1, kNet - 1), max(ix_lo, 0),
                            min(ix_lo + SI - 1, kNet - 1), scale_x, scale_y, hp, ST * ST);
  {
    const int nn = threadIdx.x >> 4, k0 = 2 * (threadIdx.x & 15);
    const __half2 hw = __floats2half2_rn(k0 < 27 ? w[nn * 27 + k0] : 0.f, k0 + 1 < 27 ? w[nn * 27 + k0 + 1] : 0.f);
    sbf[nn][threadIdx.x & 15] = *reinterpret_cast<const uint32_t *>(&hw);
    if (threadIdx.x < 16) sbias[threadIdx.x] = bias[threadIdx.x];
    if (threadIdx.x < 32) {
      const int k = threadIdx.x, tap = k / 3, cc = k - tap * 3, ky = tap / 3, kx = tap - ky * 3;
      skoff[k] = k < 27 ? (short)((cc * SI + ky) * (SI + 1) + kx) : (short)0;   // pad columns: any finite value
    }
  }
  lut[threadIdx.x] = __fdiv_rn((float)threadIdx.x, 255.0f);                       // ST*ST == 256 threads
  lut_h[threadIdx.x] = __float2half_rn(__fdiv_rn((float)threadIdx.x, 255.0f));
  if (threadIdx.x < SI) ytap[threadIdx.x] = axis_taps_lb(min(max(2 * oy0 - 1 + (int)threadIdx.x, 0), kNet - 1), p.pad_y, p.new_h, scale_y, H, hp);
  else if (threadIdx.x < 2 * SI) xtap[threadIdx.x - SI] = axis_taps_lb(min(max(2 * ox0 - 1 + (int)threadIdx.x - SI, 0), kNet - 1), p.pad_x, p.new_w, scale_x, W, hp);
  stage_wait();
  __syncthreads();
  if (LUT) {
    apply_raw_lut(reg, p.raw_lut, ST * ST);
    __syncthreads();
  }
  int red_y = 0, red_x = 0;
  if (p.chan_order == 3) { red_y = 1; red_x = 1; }
  else if (p.chan_order == 4) { red_y = 0; red_x = 1; }
  else if (p.chan_order == 5) { red_y = 1; red_x = 0; }
  if (fast_x && bayer) {
    // Fast path (Bayer source, integer horizontal scale: every x tap has weight 0 on its second
    // sample, so a network-input pixel is a vertical lerp of two demosaiced source pixels of ONE
    // column).  7 x 33 threads: a thread owns a column and five consecutive input rows and walks
    // down its source column with a 3x3 window of raw samples in registers (three byte loads per
    // source row); column addressing and colour-site parity are loop invariants.  The source rows
    // an input row needs are monotone in the input row, so the window only ever slides forward.
    // Bit-identical to sample_pixel().
    constexpr int RG = 5, NG = (SI + RG - 1) / RG;
    if (threadIdx.x < NG * SI) {
      const int grp = threadIdx.x / SI, c = threadIdx.x - grp * SI;
      const int ix = ix_lo + c;
      const bool xin = ix >= 0 && ix < kNet;
      const int sx = p.rotate180 ? W - 1 - xtap[c].i0 : xtap[c].i0;
      int xm = sx - 1, xp = sx + 1;
      if (sx == 0 || sx == W - 1) { xm = reflect101(xm, W); xp = reflect101(xp, W); }
      const bool red_col = ((sx & 1) == red_x);
      const int dir = p.rotate180 ? -1 : 1;          // source rows move this way as the input row grows
      // window rows: wa = row cur - dir, wb = row cur, wc = row cur + dir (mirrored at the border);
      // the demosaic is symmetric in north/south, so the orientation does not matter
      int cur = -1 << 20;
      int a0 = 0, a1 = 0, a2 = 0, b0 = 0, b1 = 0, b2 = 0, c0 = 0, c1 = 0, c2 = 0;
      auto load_row = [&](int y, int &v0, int &v1, int &v2) {
        const uint8_t *rp = rowp(reg, reflect101(y, H));
        v0 = rp[xm]; v1 = rp[sx]; v2 = rp[xp];
      };
      auto seek = [&](int sy) {                       // make `sy` the window centre
        if (sy == cur) return;
        if (sy == cur + dir) {                        // slide by one row
          a0 = b0; a1 = b1; a2 = b2; b0 = c0; b1 = c1; b2 = c2;
        } else if (sy == cur + 2 * dir) {             // slide by two rows
          a0 = c0; a1 = c1; a2 = c2;
          load_row(sy, b0, b1, b2);
        } else {                                      // first use (or a vertical scale above 2)
          load_row(sy - dir, a0, a1, a2);
          load_row(sy, b0, b1, b2);
        }
        load_row(sy + dir, c0, c1, c2);
        cur = sy;
      };
      // colour-site cases: with an even integer scale the column parity is the same for every
      // thread, so both branches below are warp-uniform (a warp works on one input row)
      auto demosaic = [&](int sy, int &R, int &G, int &B) {
        const bool red_row = ((sy & 1) == red_y);
        if (red_row == red_col) {            // red or blue site: own colour, green cross, other colour diagonal
          const int cross = (a1 + c1 + b0 + b2 + 2) >> 2, diag = (a0 + a2 + c0 + c2 + 2) >> 2;
          G = cross;
          R = red_row ? b1 : diag;
          B = red_row ? diag : b1;
        } else {                             // green site
          const int horiz = (b0 + b2 + 1) >> 1, vert = (a1 + c1 + 1) >> 1;
          G = b1;
          R = red_row ? horiz : vert;
          B = red_row ? vert : horiz;
        }
        if (CCM) apply_ccm(ccm, R, G, B);
      };
      // v is a convex combination of 8-bit values: no clamp needed, floor(v + 0.5) is one F2I
      auto finish_h = [&](float v) -> __half {
        if (p.quantize_u8) return lut_h[__float2int_rd(__fadd_rn(v, 0.5f))];
        return __float2half_rn(__fdiv_rn(v, 255.0f));
      };
#pragma unroll
      for (int k = 0; k < RG; ++k) {
        const int r = grp * RG + k;
        if (r >= SI) break;
        const int iy = iy_lo + r;
        __half h0 = __float2half_rn(0.f), h1 = h0, h2 = h0;
        if (xin && iy >= 0 && iy < kNet) {
          const Taps ty = ytap[r];
          const int sy0 = p.rotate180 ? H - 1 - ty.i0 : ty.i0, sy1 = p.rotate180 ? H - 1 - ty.i1 : ty.i1;
          int R0, G0, B0, R1, G1, B1;
          seek(sy0);
          demosaic(sy0, R0, G0, B0);
          seek(sy1);
          demosaic(sy1, R1, G1, B1);
          const float fy = ty.f, ofy = __fsub_rn(1.0f, fy);
          h0 = finish_h(__fadd_rn(__fmul_rn((float)R0, ofy), __fmul_rn((float)R1, fy)));
          h1 = finish_h(__fadd_rn(__fmul_rn((float)G0, ofy), __fmul_rn((float)G1, fy)));
          h2 = finish_h(__fadd_rn(__fmul_rn((float)B0, ofy), __fmul_rn((float)B1, fy)));
        }
        tile[0][r][c] = h0; tile[1][r][c] = h1; tile[2][r][c] = h2;
      }
    }
  } else {
    for (int q = threadIdx.x; q < SI * SI; q += ST * ST) {
      const int r = q / SI, c = q - r * SI;
      const int iy = iy_lo + r, ix = ix_lo + c;
      float v[3] = {0.f, 0.f, 0.f};
      if (iy >= 0 && iy < kNet && ix >= 0 && ix < kNet) {
        if (ytap[r].ok && xtap[c].ok) sample_pixel<CCM>(reg, p, ytap[r], xtap[c], red_y, red_x, lut, ccm, v);
        else v[0] = v[1] = v[2] = lut[114];             // letterbox padding: 114 / 255
      }
      tile[0][r][c] = __float2half_rn(v[0]); tile[1][r][c] = __float2half_rn(v[1]); tile[2][r][c] = __float2half_rn(v[2]);
    }
  }
  // conv0 as an implicit GEMM on mma.sync m16n8k16 (FP16 operands, FP32 accumulate): an m-tile is
  // one output row of the CTA's 16x16 tile (16 pixels), N = 16 = two n-tiles, K = 27 padded to 32.
  // (K = 27 and N = 16 are too small for a tcgen05 tile to pay for its TMEM round trip; the warp
  // MMA replaces 432 FP32 FMAs per pixel.)  Fragment layout: PTX ISA, mma.m16n8k16 .f16.
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  __syncthreads();
  int koff[2][4];          // tile offset (halfs) of k = 16*s + {2t, 2t+1, 2t+8, 2t+9}
  uint32_t bfrag[2][2][2];  // [n-tile][k-step][2]
#pragma unroll
  for (int s2 = 0; s2 < 2; ++s2)
#pragma unroll
    for (int j = 0; j < 4; ++j) koff[s2][j] = skoff[16 * s2 + 2 * t + (j & 1) + (j >> 1) * 8];
#pragma unroll
  for (int nt = 0; nt < 2; ++nt)
#pragma unroll
    for (int s2 = 0; s2 < 2; ++s2)
#pragma unroll
      for (int h = 0; h < 2; ++h) bfrag[nt][s2][h] = sbf[nt * 8 + g][8 * s2 + t + 4 * h];
  const __half *tl = &tile[0][0][0];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
    const int ty = 2 * warp + mt;
    float acc[2][4];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      acc[nt][0] = acc[nt][2] = sbias[nt * 8 + 2 * t];
      acc[nt][1] = acc[nt][3] = sbias[nt * 8 + 2 * t + 1];
    }
    const int base0 = (2 * ty) * (SI + 1) + 2 * g;          // pixel tx = g; pixel g + 8 is 16 halfs further
#pragma unroll
    for (int s2 = 0; s2 < 2; ++s2) {
      uint32_t afrag[4];
#pragma unroll
      for (int hk = 0; hk < 2; ++hk)        // k pair {2t, 2t+1} / {2t+8, 2t+9}
#pragma unroll
        for (int hr = 0; hr < 2; ++hr) {    // row g / g + 8
          const int b0 = base0 + hr * 16;
          const __half2 v = __halves2half2(tl[b0 + koff[s2][2 * hk]], tl[b0 + koff[s2][2 * hk + 1]]);
          afrag[hk * 2 + hr] = *reinterpret_cast<const uint32_t *>(&v);
        }
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(acc[nt][0]), "+f"(acc[nt][1]), "+f"(acc[nt][2]), "+f"(acc[nt][3])
                     : "r"(afrag[0]), "r"(afrag[1]), "r"(afrag[2]), "r"(afrag[3]), "r"(bfrag[nt][s2][0]), "r"(bfrag[nt][s2][1]));
    }
    // thread holds channels {2t, 2t+1} of n-tile 0 (plane 0) and of n-tile 1 (plane 1) for pixels
    // tx = g and g + 8: 4-byte stores, the four lanes of a quad complete one 16-byte pixel
#pragma unroll
    for (int hr = 0; hr < 2; ++hr) {
      const int y = oy0 + ty, x = ox0 + g + 8 * hr;
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        const __half2 hv = __floats2half2_rn(silu_fast(acc[nt][2 * hr]), silu_fast(acc[nt][2 * hr + 1]));
        if (out) {
          const size_t pix = (size_t)pr_index(n, y, x, kNet / 2, kNet / 2);
          *reinterpret_cast<__half2 *>(out + (long long)nt * out_pstride + pix * 8 + 2 * t) = hv;
        }
        if (out2) {   // parity-split twin for the stride-2 consumer (common.cuh, ConvParams)
          const size_t pix2 = (size_t)pr_index(n, y >> 1, x >> 1, kNet / 4, kNet / 4);
          *reinterpret_cast<__half2 *>(out2 + (long long)(((y & 1) * 2 + (x & 1)) * 2 + nt) * out2_pstride + pix2 * 8 + 2 * t) = hv;
        }
      }
    }
  }
}

// Optional: materialise the rotated RGB frame (what get_rotated_image() exposes in the reference,
// include/irmv_detection/yolo_engine.hpp:34) for consumers of the rotated source image.
// LUT: Bayer source with a raw-domain colour table (p.raw_lut), applied to each of the nine raw reads.
// CCM: Bayer source with a colour-correction block (p.ccm), applied to the demosaiced pixel (read through L1).
template <bool LUT, bool CCM>
__global__ void rotate_kernel(PreprocessParams p) {
  const bool bayer = p.chan_order >= 2;
  const int H = p.src_h, W = p.src_w, bpp = bayer ? 1 : 3;
  const size_t frame_bytes = (size_t)H * W * bpp;
  const uint8_t *base = p.src_indirect ? *p.src_indirect : p.src;
  size_t total = (size_t)p.n * H * W;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total;
       i += (size_t)gridDim.x * blockDim.x) {
    int n = (int)(i / ((size_t)H * W));
    int rem = (int)(i - (size_t)n * H * W);
    int y = rem / W, x = rem - y * W;
    int sy = p.rotate180 ? H - 1 - y : y, sx = p.rotate180 ? W - 1 - x : x;
    const uint8_t *frame = base + (size_t)(p.frame0 + n) * frame_bytes;
    int R, G, B;
    if (bayer) {
      Region reg{frame, frame, 0, W, 0, W, 0, 0};
      // direct global reads: shift term must vanish, so index manually
      auto g = [&](int yy, int xx) {
        const int v = frame[(size_t)yy * W + xx];
        return LUT ? (int)__ldg(p.raw_lut + ((yy & 1) * 2 + (xx & 1)) * 256 + v) : v;
      };
      int red_y = 0, red_x = 0;
      if (p.chan_order == 3) { red_y = 1; red_x = 1; }
      else if (p.chan_order == 4) { red_y = 0; red_x = 1; }
      else if (p.chan_order == 5) { red_y = 1; red_x = 0; }
      int ym = reflect101(sy - 1, H), yp = reflect101(sy + 1, H);
      int xm = reflect101(sx - 1, W), xp = reflect101(sx + 1, W);
      int c = g(sy, sx), py = sy & 1, px = sx & 1;
      bool is_r = (py == red_y) && (px == red_x), is_b = (py != red_y) && (px != red_x);
      if (is_r || is_b) {
        int cross = (g(ym, sx) + g(yp, sx) + g(sy, xm) + g(sy, xp) + 2) >> 2;
        int diag = (g(ym, xm) + g(ym, xp) + g(yp, xm) + g(yp, xp) + 2) >> 2;
        G = cross;
        if (is_r) { R = c; B = diag; } else { B = c; R = diag; }
      } else {
        int horiz = (g(sy, xm) + g(sy, xp) + 1) >> 1, vert = (g(ym, sx) + g(yp, sx) + 1) >> 1;
        G = c;
        bool on_red_row = (py == red_y);
        R = on_red_row ? horiz : vert;
        B = on_red_row ? vert : horiz;
      }
      if (CCM) apply_ccm(p.ccm + (size_t)(p.frame0 + n) * p.ccm_stride, R, G, B);
      (void)reg;
    } else {
      const uint8_t *s = frame + ((size_t)sy * W + sx) * 3;
      R = s[0]; G = s[1]; B = s[2];
      if (p.chan_order == 1) { int t = R; R = B; B = t; }
    }
    uint8_t *d = p.rotated + i * 3;
    d[0] = (uint8_t)R; d[1] = (uint8_t)G; d[2] = (uint8_t)B;
  }
}

}  // namespace

cudaError_t launch_rotate(const PreprocessParams &p, cudaStream_t s) {
  if (p.n <= 0 || !p.rotated) return cudaSuccess;
  size_t total = (size_t)p.n * p.src_h * p.src_w;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (p.ccm) {
    if (p.raw_lut) rotate_kernel<true, true><<<blocks, 256, 0, s>>>(p);
    else rotate_kernel<false, true><<<blocks, 256, 0, s>>>(p);
  } else {
    if (p.raw_lut) rotate_kernel<true, false><<<blocks, 256, 0, s>>>(p);
    else rotate_kernel<false, false><<<blocks, 256, 0, s>>>(p);
  }
  return cudaGetLastError();
}

cudaError_t launch_preprocess(const PreprocessParams &p_in, cudaStream_t s) {
  PreprocessParams p = p_in;
  letterbox_geometry(p.src_w, p.src_h, p.resize_mode, &p.pad_x, &p.pad_y, &p.new_w, &p.new_h);
  if (p.n <= 0) return cudaSuccess;
  const bool bayer = p.chan_order >= 2;
  const int bpp = bayer ? 1 : 3;
  const float sx = (float)p.src_w / p.new_w, sy = (float)p.src_h / p.new_h;
  int rows_cap = (int)(TH * sy) + 4 + (bayer ? 4 : 0);
  int cols_cap = (int)(TW * sx) + 4 + (bayer ? 4 : 0);
  int pitch_s = ((cols_cap * bpp + 15) / 16 + 2) * 16;   // +1 chunk for the alignment shift
  size_t smem = (size_t)rows_cap * pitch_s;
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
  if ((p.raw_lut || p.ccm) && !bayer) return cudaErrorInvalidValue;   // the tables are defined for Bayer sources only
  auto kernel = p.ccm ? (p.raw_lut ? preprocess_kernel<true, true> : preprocess_kernel<false, true>)
                      : (p.raw_lut ? preprocess_kernel<true, false> : preprocess_kernel<false, false>);
  if (p.ccm) smem += kCcmBytes;
  if (smem > 48 * 1024) {                 // per device, cheap: no process-wide flag
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  dim3 grid((kNet + TW - 1) / TW, (kNet + TH - 1) / TH, p.n);
  kernel<<<grid, NT, smem, s>>>(p, rows_cap, pitch_s);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  return launch_rotate(p, s);
}


cudaError_t launch_stem(const PreprocessParams &p_in, const float *w, const float *bias, const uint32_t *fast_tab, __half *out,
                        long long out_pstride, __half *out2, long long out2_pstride, cudaStream_t s) {
  PreprocessParams p = p_in;
  letterbox_geometry(p.src_w, p.src_h, p.resize_mode, &p.pad_x, &p.pad_y, &p.new_w, &p.new_h);
  if (p.n <= 0) return cudaSuccess;
  if (fast_tab && stem_bayer2x_applies(p)) {
    cudaError_t e = launch_stem_bayer2x(p, p.frame0, fast_tab, out, out_pstride, out2, out2_pstride, s);
    return e == cudaSuccess ? launch_rotate(p, s) : e;
  }
  const bool bayer = p.chan_order >= 2;
  if ((p.raw_lut || p.ccm) && !bayer) return cudaErrorInvalidValue;
  const int bpp = bayer ? 1 : 3;
  const float sx = (float)p.src_w / p.new_w, sy = (float)p.src_h / p.new_h;
  int rows_cap = (int)(SI * sy) + 4 + (bayer ? 4 : 0);
  int cols_cap = (int)(SI * sx) + 4 + (bayer ? 4 : 0);
  int pitch_s = ((cols_cap * bpp + 15) / 16 + 2) * 16;
  const int smem_win = rows_cap * pitch_s;
  size_t smem = (size_t)smem_win;
  if (smem > 160 * 1024) return cudaErrorInvalidValue;
  auto kernel = p.ccm ? (p.raw_lut ? stem_kernel<true, true> : stem_kernel<false, true>)
                      : (p.raw_lut ? stem_kernel<true, false> : stem_kernel<false, false>);
  if (p.ccm) smem += kCcmBytes;
  if (smem > 30 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  dim3 grid(kNet / 2 / ST, kNet / 2 / ST, p.n);
  // integer horizontal scale without half-pixel centres: every second x tap has weight exactly 0
  const int fast_x = (p.src_w % kNet == 0) && p.resize_mode == 0;
  kernel<<<grid, ST * ST, smem, s>>>(p, w, bias, out, out_pstride, out2, out2_pstride, pitch_s, fast_x, smem_win);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? launch_rotate(p, s) : e;
}

}  // namespace irmv
