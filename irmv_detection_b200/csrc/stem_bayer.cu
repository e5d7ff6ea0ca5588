// Fused stem for the camera case: 8-bit Bayer mosaic, source width exactly 2 x 640, corner-aligned
// stretch (the reference's NPP map, src/yolo_engine.cpp:186-190), 8-bit intermediate.
//   demosaic (camera ISP step, reference src/mv_camera.cpp:96) -> rot180 (nppiMirror :182-184) ->
//   bilinear resize to 640 x 640, u8 (nppiResize :186-190) -> /255 (nppiScale :192-194) ->
//   conv0 3x3 s2 3->16 + bias + SiLU (first layer of the TensorRT engine, :105)
// in one kernel; the 640 x 640 x 3 network input only ever exists as a shared-memory tile.
//
// Why a second stem kernel: the generic one (preprocess.cu) is instruction-issue bound
// (profiles/r1_summary.md section 4: 630 M warp instructions per 128 frames, 12 % of the HBM
// roofline).  Three properties of the camera case remove most of that work:
//   * x scale is exactly 2 and the map is corner-aligned, so the second x tap has weight 0 and a
//     network-input pixel needs ONE source column; every needed column has the same Bayer column
//     parity, so the colour-site case is uniform per source row.
//   * two neighbouring needed columns live in one 32-bit word of the raw row: the demosaic runs on
//     2 x 16-bit lanes packed in a register (sums of <= 4 bytes + rounding never carry between
//     lanes), one thread produces two network-input pixels.
//   * y scale = P/Q (1024/640 = 8/5): the vertical weight is k/Q, k integer, so
//     floor(a*(1-f) + b*f + 0.5) == (2(Q-k)*a + 2k*b + Q) / 2Q exactly (checked exhaustively over
//     all rows and byte pairs against the oracle's FP32 arithmetic: tests/test_oracle_cpu.py
//     test_stem_integer_lerp_equals_float_oracle).  The numerator (< 2Q*255 + Q + 1) indexes a
//     shared-memory table of the FP16 values of q/255: lerp + quantise + scale = 2 IMAD + 1 LDS.
// A CTA owns a full-width strip of OROWS conv0 output rows: staging is whole 1280-byte rows
// (16-byte cp.async, always aligned), the tile is [2*OROWS+1][641 px][3] halves, conv0 runs as
// mma.sync m16n8k16 with K ordered (ky, 3 px x 3 ch + 1 pad) so that every A fragment register is one
// aligned, bank-conflict-free 32-bit shared-memory load.
#include <cstdio>
#include <cstring>
#include <vector>

#include "common.cuh"

namespace irmv {
namespace {

constexpr int SW = 1280;                 // source width handled by this kernel (2 * kNet)
constexpr int FMT_BAYER = 0, FMT_BAYER_REDCOL = 1, FMT_RGB = 2, FMT_BGR = 3;
constexpr int row_pitch(int fmt) { return 16 + (fmt >= FMT_RGB ? 3 * SW : SW) + 16; }   // staged raw row: [16 B apron | row | 16 B apron]
constexpr int PITCHW = 965;              // tile row pitch in 32-bit words (641 px * 6 B = 3846 B -> 962 words + skew)
constexpr int OWID = kNet / 2;           // conv0 output side, 320
constexpr int NWARPS = OWID / 16;        // 20: one warp per 16-pixel column block of the conv0 output
constexpr int NTHREADS = NWARPS * 32;    // 640
// conv0 output rows per CTA (template parameter OROWS): 8 for Bayer sources (2 CTAs per SM), 4 for packed
// 3-byte sources (their staged rows are three times as long); network-input rows of a strip = 2*OROWS + 1
// (one halo row on top).
// FMT: 0 / 1 = Bayer with the needed columns on non-red / red columns, 2 = packed u8x3 passed through (the
// reference: whatever byte order is in the buffer goes to the net, src/yolo_engine.cpp:186-199), 3 = packed with R and B swapped.
constexpr int orows_for(int fmt) { return fmt >= FMT_RGB ? 4 : 8; }

struct RowTab { int off; uint32_t w_lo, w_hi; int flags; };   // flags: 1 = lo is a site row, 2 = conv padding row

struct StemBayerArgs {
  const uint8_t *src;                    // frames [..][H][1280]; used when src_indirect == null
  const uint8_t *const *src_indirect;
  int n, H, frame0;                      // frame0: first source frame of this launch
  int rev;                               // walk frames and strips from the last to the first
  int Q, lut_n;                          // H / 640 = P / Q; entries of the lerp table: 2*Q*255 + Q + 1
  int tab_strip;                         // word offset of the per-strip tables inside tab
  const uint32_t *tab;                   // device tables built by stem_bayer2x_tables()
  __half *out; long long out_ps;         // normal layout (may be null)
  __half *out2; long long out2_ps;       // parity-split twin (may be null)
  const uint8_t *raw_lut;                // [2][2][256] raw-domain colour stage (PreprocessParams::raw_lut), LUT instantiations only
  const uint8_t *ccm;                    // colour-correction block (PreprocessParams::ccm), LUT == LUT_COLOUR only
  int ccm_stride;                        // PreprocessParams::ccm_stride
};

// Table modes of the Bayer instantiations (template parameter LUT): no table, the raw table, the raw table (when one
// is set) and the colour-correction stage.  Dynamic shared memory each mode adds behind the lerp table:
constexpr int LUT_NONE = 0, LUT_RAW = 1, LUT_COLOUR = 2;
constexpr size_t lut_bytes(int lut) { return lut == LUT_NONE ? 0 : lut == LUT_RAW ? 1024 : 1024 + kCcmBytes; }
int lut_mode(const PreprocessParams &p) { return p.ccm ? LUT_COLOUR : p.raw_lut ? LUT_RAW : LUT_NONE; }

// Device table block (built once per engine, stem_bayer2x_tables):
//   TAB_BFRAG  conv0 B fragments per lane [32][8]: weights * 0.5 as FP16 pairs, K ordered (ky, 3 px x 3 ch + pad)
//   TAB_BIAS   bias * 0.5 [16] FP32   (SiLU(v) = h + h * tanh(h), h = v / 2: the 0.5 is folded into weights
//              and bias, exact since it is a power of two)
//   TAB_LUT    lerp table: entry x (the lerp numerator, < lut_n) = FP16(floor(x / 2Q) / 255)
//   tab_strip  per strip of OROWS output rows: {vlo, nr, 0, 0} + RowTab[NIR] (sampling parameters per
//              network-input row: byte offset of source row lo-1 (Bayer) / lo (packed) in the staged window, the
//              two vertical weights (doubled, so the numerator is the byte offset into the FP16 table), flags)
constexpr int TAB_BFRAG = 0, TAB_BIAS = 256, TAB_LUT = 272;   // offsets in 32-bit words
constexpr int strip_words(int orows) { return 4 + 4 * (2 * orows + 1); }

__host__ __device__ inline int reflect101(int i, int n) {
  if (i < 0) i = -i;
  if (i >= n) i = 2 * n - 2 - i;
  return i;
}

struct Px3 { uint32_t w, c, e; };        // west / centre / east neighbours of the two needed columns, 2 x 16-bit lanes

// Needed columns of unit j.  ROT (needed columns are odd): 4j+1 (low lane), 4j+3 (high lane);
// otherwise (even): 4j (low), 4j+2 (high).  rowj = the row's word j.
template <bool ROT>
__device__ __forceinline__ Px3 unpack(const uint32_t *rowj) {
  constexpr uint32_t M = 0x00ff00ffu;
  const uint32_t C = rowj[0];
  Px3 o;
  if (ROT) {
    const uint32_t N = rowj[1];
    o.c = (C >> 8) & M;
    o.w = C & M;
    o.e = __funnelshift_r(C, N, 16) & M;
  } else {
    const uint32_t P = rowj[-1];
    o.c = C & M;
    o.e = (C >> 8) & M;
    o.w = __funnelshift_r(P, C, 24) & M;
  }
  return o;
}

// OUT1 / OUT2: write the normal layout / the parity-split twin (exactly one of them).
// LUT (Bayer formats only): LUT_RAW: the staged rows go through the raw-domain colour table before the demosaic; the
// [2][2][256]-byte table sits in shared memory between the lerp table and the staged rows.  LUT_COLOUR: the same
// (when a.raw_lut is set), and every demosaiced pixel goes through the colour-correction stage before the vertical
// lerp; its block (kCcmBytes) sits behind the raw table.
template <bool ROT, int FMT, bool OUT1, bool OUT2, int LUT>
__global__ void __launch_bounds__(NTHREADS, 2) stem_bayer2x_kernel(const __grid_constant__ StemBayerArgs a) {
  constexpr int OROWS = orows_for(FMT), NIR = 2 * OROWS + 1, RP = row_pitch(FMT), STRIP_WORDS = strip_words(OROWS);
  constexpr bool PACKED = FMT >= FMT_RGB, RED_COL = FMT == FMT_BAYER_REDCOL;
  constexpr int SROW = PACKED ? 3 * SW : SW;          // bytes of a source row
  extern __shared__ __align__(16) uint8_t smem[];
  uint32_t *tile_w = reinterpret_cast<uint32_t *>(smem);                       // [NIR][PITCHW]
  uint8_t *lut = smem + (size_t)NIR * PITCHW * 4;                              // [lut_n] halves
  uint8_t *rlut = smem + (((size_t)NIR * PITCHW * 4 + (size_t)a.lut_n * 2 + 15) & ~(size_t)15);  // [2][2][256] (LUT)
  uint8_t *ccm = rlut + 1024;                                                                    // (LUT_COLOUR)
  uint8_t *raw = rlut + lut_bytes(LUT);                                                          // [nr][RP]
  __shared__ __align__(16) RowTab rowtab[NIR];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int H = a.H;
  // blockIdx.x walks the strips of a frame, blockIdx.y the frames: the launch order follows memory order
  const int sidx = a.rev ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x;
  const int n = a.rev ? (int)(gridDim.y - 1 - blockIdx.y) : (int)blockIdx.y, oy0 = sidx * OROWS;
  const uint8_t *base = a.src_indirect ? *a.src_indirect : a.src;
  const uint8_t *frame = base + (size_t)(a.frame0 + n) * ((size_t)H * SROW);
  const uint32_t *strip = a.tab + a.tab_strip + sidx * STRIP_WORDS;

  // ---- source rows of the strip: virtual rows [vlo, vlo + nr), slot = v - vlo, content = row reflect101(v)
  const int vlo = (int)strip[0], nr = (int)strip[1];
  const bool aligned = ((size_t)frame & 15) == 0;
  for (int r = warp; r < nr; r += NWARPS) {        // a warp stages whole rows in 16-byte chunks
    const uint8_t *g = frame + (size_t)min(reflect101(vlo + r, H), H - 1) * SROW;
    uint8_t *d = raw + (size_t)r * RP + 16;
    if (aligned) {
      const uint32_t dst = (uint32_t)__cvta_generic_to_shared(d);
#pragma unroll
      for (int c = 0; c < (SROW / 16 + 31) / 32; ++c)
        if ((c + 1) * 32 <= SROW / 16 || c * 32 + lane < SROW / 16)
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + (uint32_t)(c * 32 + lane) * 16u), "l"(g + (c * 32 + lane) * 16) : "memory");
    } else {                                        // caller's frames are not 16-byte aligned: plain byte copies
      for (int c = lane; c < SROW; c += 32) d[c] = g[c];
    }
    if (!PACKED && lane == 0) { d[-1] = g[1]; d[SW] = g[SW - 2]; }   // mirrored columns -1 and W (reflect-101) for the demosaic
  }
  {
    const uint32_t *gl = a.tab + TAB_LUT;
    uint32_t *sl = reinterpret_cast<uint32_t *>(lut);
    for (int i = tid; i < (a.lut_n + 1) / 2; i += NTHREADS) sl[i] = gl[i];
  }
  const bool raw_lut = LUT == LUT_RAW || (LUT == LUT_COLOUR && a.raw_lut);
  if (raw_lut && tid < 256) reinterpret_cast<uint32_t *>(rlut)[tid] = reinterpret_cast<const uint32_t *>(a.raw_lut)[tid];
  if (LUT == LUT_COLOUR) stage_ccm(ccm, a.ccm + (size_t)(a.frame0 + n) * a.ccm_stride, tid);
  if (tid < NIR) {
    reinterpret_cast<uint4 *>(rowtab)[tid] = reinterpret_cast<const uint4 *>(strip + 4)[tid];
    // conv padding of the tile: column 0 (ix = -1) and the pad half behind the last pixel
    uint16_t *row16 = reinterpret_cast<uint16_t *>(tile_w + (size_t)tid * PITCHW);
    row16[0] = row16[1] = row16[2] = 0;
    row16[3 * 641] = 0; row16[3 * 641 + 1] = 0;
  }
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncthreads();
  if (raw_lut) {
    // raw-domain colour stage, in place: a sample of sensor row y, column x becomes rlut[y & 1][x & 1][s].  The
    // parity is that of the row and column actually read; reflect-101 keeps a mirrored sample on its colour site
    // (column -1 holds column 1, column SW holds column SW - 2).
    for (int r = warp; r < nr; r += NWARPS) {
      const uint8_t *te = rlut + (min(reflect101(vlo + r, H), H - 1) & 1) * 512, *to = te + 256;   // even / odd columns
      uint8_t *d = raw + (size_t)r * RP + 16;
      uint32_t *dw = reinterpret_cast<uint32_t *>(d);
      for (int c = lane; c < SW / 4; c += 32) {
        const uint32_t v = dw[c];
        dw[c] = (uint32_t)te[v & 0xffu] | ((uint32_t)to[(v >> 8) & 0xffu] << 8) | ((uint32_t)te[(v >> 16) & 0xffu] << 16) |
                ((uint32_t)to[v >> 24] << 24);
      }
      if (lane == 0) { d[-1] = to[d[-1]]; d[SW] = te[d[SW]]; }
    }
    __syncthreads();
  }

  // ---- sampling: a warp owns 32 units (= 64 network-input columns) and every second input row
  {
    constexpr uint32_t M = 0x00ff00ffu;
    const uint32_t K1 = 0x00010001u, K2 = 0x00020002u;
    const uint32_t QQ = 2u * (uint32_t)a.Q * 0x00010001u;   // rounding term in both lanes (doubled like the weights)
    const uint32_t lut_s = (uint32_t)__cvta_generic_to_shared(lut);
    auto lut_ld = [&](uint32_t byte_off) -> uint32_t {
      uint16_t v;
      asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(lut_s + byte_off));
      return (uint32_t)v;
    };
    const int chunk = warp % 10, j = chunk * 32 + lane;
    // first / second pixel of the unit in ascending ix; tile column = ix + 1
    uint8_t *dst = reinterpret_cast<uint8_t *>(tile_w) + (ROT ? 6 * 639 - 12 * j : 6 + 12 * j) + (size_t)(warp / 10) * (PITCHW * 4);
    const uint32_t *rawj = reinterpret_cast<const uint32_t *>(raw) + j;
    for (int r = warp / 10; r < NIR; r += 2, dst += 2 * PITCHW * 4) {
      const RowTab rt = rowtab[r];
      if (rt.flags & 2) {                   // conv padding row above the image
        *reinterpret_cast<uint16_t *>(dst) = 0;
        *reinterpret_cast<uint32_t *>(dst + 2) = 0;
        *reinterpret_cast<uint32_t *>(dst + 6) = 0;
        *reinterpret_cast<uint16_t *>(dst + 10) = 0;
        continue;
      }
      uint32_t xr, xg, xb;
      if (PACKED) {
        // packed u8x3: the two needed pixels of unit j sit in the 12-byte group [12j, 12j + 12) of the row:
        // ROT pixels 4j+1 (low lane) and 4j+3 (high lane), otherwise 4j and 4j+2.  No demosaic: a
        // network-input value is the vertical lerp of the two source rows lo and lo + 1.
        const uint32_t *ra = reinterpret_cast<const uint32_t *>(raw + rt.off) + 3 * j;
        uint32_t v[2][3];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const uint32_t W0 = ra[q * (RP / 4)], W1 = ra[q * (RP / 4) + 1], W2 = ra[q * (RP / 4) + 2];
          if (ROT) {
            v[q][0] = (W0 >> 24) | ((W2 << 8) & 0x00ff0000u);
            v[q][1] = (W1 & 0xffu) | (W2 & 0x00ff0000u);
            v[q][2] = ((W1 >> 8) & 0xffu) | ((W2 >> 8) & 0x00ff0000u);
          } else {
            v[q][0] = (W0 & 0xffu) | (W1 & 0x00ff0000u);
            v[q][1] = ((W0 >> 8) & 0xffu) | ((W1 >> 8) & 0x00ff0000u);
            v[q][2] = ((W0 >> 16) & 0xffu) | ((W2 << 16) & 0x00ff0000u);
          }
        }
        const uint32_t x0 = v[0][0] * rt.w_lo + v[1][0] * rt.w_hi + QQ;
        const uint32_t x1 = v[0][1] * rt.w_lo + v[1][1] * rt.w_hi + QQ;
        const uint32_t x2 = v[0][2] * rt.w_lo + v[1][2] * rt.w_hi + QQ;
        xr = FMT == FMT_BGR ? x2 : x0; xg = x1; xb = FMT == FMT_BGR ? x0 : x2;
      } else {
      const uint32_t *rp = rawj + (rt.off >> 2);
      const Px3 r0 = unpack<ROT>(rp), r1 = unpack<ROT>(rp + RP / 4), r2 = unpack<ROT>(rp + 2 * (RP / 4)),
                r3 = unpack<ROT>(rp + 3 * (RP / 4));
      uint32_t cross, diag, cS, horiz, vert, cG, wS, wG;
      if (rt.flags & 1) {                   // site row = lo (r0 r1 r2), green row = lo + 1 (r1 r2 r3)
        cross = ((r0.c + r2.c + r1.w + r1.e + K2) >> 2) & M;
        diag = ((r0.w + r0.e + r2.w + r2.e + K2) >> 2) & M;
        cS = r1.c;
        horiz = ((r2.w + r2.e + K1) >> 1) & M;
        vert = ((r1.c + r3.c + K1) >> 1) & M;
        cG = r2.c;
        wS = rt.w_lo; wG = rt.w_hi;
      } else {                              // green row = lo, site row = lo + 1
        horiz = ((r1.w + r1.e + K1) >> 1) & M;
        vert = ((r0.c + r2.c + K1) >> 1) & M;
        cG = r1.c;
        cross = ((r1.c + r3.c + r2.w + r2.e + K2) >> 2) & M;
        diag = ((r1.w + r1.e + r3.w + r3.e + K2) >> 2) & M;
        cS = r2.c;
        wG = rt.w_lo; wS = rt.w_hi;
      }
      // site row: own colour at the centre, green = cross, the other colour = diagonal; green row on a
      // red row (RED_COL == false): R horizontal, B vertical; on a blue row: R vertical, B horizontal
      uint32_t RS = RED_COL ? cS : diag, BS = RED_COL ? diag : cS;
      uint32_t RG = RED_COL ? vert : horiz, BG = RED_COL ? horiz : vert;
      if (LUT == LUT_COLOUR) {
        // colour-correction stage on the four demosaiced pixels (two lanes of the site row and of the green row)
        auto cc = [&](uint32_t &r, uint32_t &g, uint32_t &b) {
          int r0 = (int)(r & 0xffffu), g0 = (int)(g & 0xffffu), b0 = (int)(b & 0xffffu);
          int r1 = (int)(r >> 16), g1 = (int)(g >> 16), b1 = (int)(b >> 16);
          apply_ccm(ccm, r0, g0, b0);
          apply_ccm(ccm, r1, g1, b1);
          r = (uint32_t)r0 | ((uint32_t)r1 << 16); g = (uint32_t)g0 | ((uint32_t)g1 << 16); b = (uint32_t)b0 | ((uint32_t)b1 << 16);
        };
        cc(RS, cross, BS);
        cc(RG, cG, BG);
      }
      xr = RS * wS + RG * wG + QQ;
      xg = cross * wS + cG * wG + QQ;
      xb = BS * wS + BG * wG + QQ;
      }
      const uint32_t r_l = lut_ld(xr & 0xffffu), r_h = lut_ld(xr >> 16);
      const uint32_t g_l = lut_ld(xg & 0xffffu), g_h = lut_ld(xg >> 16);
      const uint32_t b_l = lut_ld(xb & 0xffffu), b_h = lut_ld(xb >> 16);
      // ROT: the high lane (column 4j+3) is the smaller ix
      const uint32_t R1 = ROT ? r_h : r_l, G1 = ROT ? g_h : g_l, B1 = ROT ? b_h : b_l;
      const uint32_t R2 = ROT ? r_l : r_h, G2 = ROT ? g_l : g_h, B2 = ROT ? b_l : b_h;
      *reinterpret_cast<uint16_t *>(dst) = (uint16_t)R1;
      *reinterpret_cast<uint32_t *>(dst + 2) = G1 | (B1 << 16);
      *reinterpret_cast<uint32_t *>(dst + 6) = R2 | (G2 << 16);
      *reinterpret_cast<uint16_t *>(dst + 10) = (uint16_t)B2;
    }
  }
  __syncthreads();

  // ---- conv0: implicit GEMM on mma.sync m16n8k16 (FP16 operands, FP32 accumulate).  An m-tile is 16
  // consecutive pixels of one output row; A[px][k] = tile[2*orow + ky][2*px + kx][c] = the 10 halves
  // starting at word 3*px of tile row 2*orow + ky.  A warp owns one 16-pixel column block and walks
  // down the OROWS output rows, so every address below advances by a constant.
  const int g = lane >> 2, t = lane & 3;
  uint32_t bfrag[2][2][2];                 // [n-tile][k-step][2], constants from the table block
  {
    const uint4 b0 = reinterpret_cast<const uint4 *>(a.tab + TAB_BFRAG)[lane * 2];
    const uint4 b1 = reinterpret_cast<const uint4 *>(a.tab + TAB_BFRAG)[lane * 2 + 1];
    bfrag[0][0][0] = b0.x; bfrag[0][0][1] = b0.y; bfrag[0][1][0] = b0.z; bfrag[0][1][1] = b0.w;
    bfrag[1][0][0] = b1.x; bfrag[1][0][1] = b1.y; bfrag[1][1][0] = b1.z; bfrag[1][1][1] = b1.w;
  }
  int off[2][2];
#pragma unroll
  for (int s2 = 0; s2 < 2; ++s2)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      // K slot (s2, h, t) -> tile word: the four lanes t of one load read ONE tile row (a load that mixes rows
      // ky and ky+1 is a 2-way bank conflict for any row pitch): slots (0,0) (0,1) (1,0) = words 0..3 of rows
      // ky = 0, 1, 2; slot (1,1) = word 4 of rows 0, 1, 2 (banks of different residues mod 3) + one pad lane
      const int ky = (s2 == 1 && h == 1) ? (t < 3 ? t : 0) : 2 * s2 + h, tp = (s2 == 1 && h == 1) ? 4 : t;
      off[s2][h] = ky * PITCHW + tp;
    }
  float hbias[2][2];                       // bias / 2
  {
    const float *hb = reinterpret_cast<const float *>(a.tab + TAB_BIAS);
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) { hbias[nt][0] = hb[nt * 8 + 2 * t]; hbias[nt][1] = hb[nt * 8 + 2 * t + 1]; }
  }
  const int xb = warp * 16;
  const uint32_t *tw = tile_w + 3 * (xb + g);
  // output pointers for row oy0 (even): normal layout, and the twin's plane group of (y & 1 = 0, x & 1 = g & 1);
  // lane holds channels {2t, 2t+1} of plane 0 (nt = 0) and plane 1 for pixels xb + g and xb + g + 8
  __half *o1 = a.out + ((long long)(n * (OWID + 1) + 1 + oy0) * (OWID + 1) + xb + g) * 8 + 2 * t;
  __half *o2 = a.out2 + (long long)((g & 1) * 2) * a.out2_ps +
               ((long long)(n * (OWID / 2 + 1) + 1 + (oy0 >> 1)) * (OWID / 2 + 1) + ((xb + g) >> 1)) * 8 + 2 * t;
  const long long ps1 = a.out_ps, ps2 = a.out2_ps;
#pragma unroll 1
  for (int orow = 0; orow < OROWS; ++orow, tw += 2 * PITCHW) {
    float acc[2][4];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      acc[nt][0] = acc[nt][2] = hbias[nt][0];
      acc[nt][1] = acc[nt][3] = hbias[nt][1];
    }
#pragma unroll
    for (int s2 = 0; s2 < 2; ++s2) {
      const uint32_t a0 = tw[off[s2][0]], a1 = tw[24 + off[s2][0]], a2 = tw[off[s2][1]], a3 = tw[24 + off[s2][1]];
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(acc[nt][0]), "+f"(acc[nt][1]), "+f"(acc[nt][2]), "+f"(acc[nt][3])
                     : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(bfrag[nt][s2][0]), "r"(bfrag[nt][s2][1]));
    }
    // acc = v / 2 (folded 0.5): SiLU(v) = h + h * tanh(h)
    __half2 hv[2][2];
#pragma unroll
    for (int hr = 0; hr < 2; ++hr)
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        float t0, t1;
        const float h0 = acc[nt][2 * hr], h1 = acc[nt][2 * hr + 1];
        asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(h0));
        asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(h1));
        hv[hr][nt] = __floats2half2_rn(fmaf(h0, t0, h0), fmaf(h1, t1, h1));
      }
    if (OUT1) {
#pragma unroll
      for (int hr = 0; hr < 2; ++hr)
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) *reinterpret_cast<__half2 *>(o1 + nt * ps1 + hr * 64) = hv[hr][nt];
      o1 += (OWID + 1) * 8;
    }
    if (OUT2) {                            // parity-split twin for the stride-2 consumer (common.cuh, ConvParams)
      __half *o = o2 + ((orow & 1) ? 4 * ps2 : 0);     // plane group of row parity y & 1 (oy0 is even)
#pragma unroll
      for (int hr = 0; hr < 2; ++hr)
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) *reinterpret_cast<__half2 *>(o + nt * ps2 + hr * 32) = hv[hr][nt];
      if (orow & 1) o2 += (OWID / 2 + 1) * 8;
    }
  }
}


template <bool ROT, int FMT, bool OUT1, bool OUT2, int LUT>
cudaError_t launch_o(const StemBayerArgs &a, size_t smem, cudaStream_t s) {
  cudaError_t e = cudaFuncSetAttribute(stem_bayer2x_kernel<ROT, FMT, OUT1, OUT2, LUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  dim3 grid(OWID / orows_for(FMT), a.n);
  stem_bayer2x_kernel<ROT, FMT, OUT1, OUT2, LUT><<<grid, NTHREADS, smem, s>>>(a);
  return cudaGetLastError();
}

template <bool ROT, int FMT>
cudaError_t launch_t(const StemBayerArgs &a, size_t smem, cudaStream_t s) {
  if (!a.out == !a.out2) return cudaErrorInvalidValue;   // exactly one layout
  if constexpr (FMT < FMT_RGB) {
    if (a.ccm) {                                       // raw table (if any) and colour block behind the lerp table
      if (a.out2) return launch_o<ROT, FMT, false, true, LUT_COLOUR>(a, smem + lut_bytes(LUT_COLOUR), s);
      return launch_o<ROT, FMT, true, false, LUT_COLOUR>(a, smem + lut_bytes(LUT_COLOUR), s);
    }
    if (a.raw_lut) {                                   // the table's 1 KB sits behind the lerp table
      if (a.out2) return launch_o<ROT, FMT, false, true, LUT_RAW>(a, smem + 1024, s);
      return launch_o<ROT, FMT, true, false, LUT_RAW>(a, smem + 1024, s);
    }
  } else {
    if (a.raw_lut || a.ccm) return cudaErrorInvalidValue;   // the tables are defined for Bayer sources only
  }
  if (a.out2) return launch_o<ROT, FMT, false, true, LUT_NONE>(a, smem, s);
  return launch_o<ROT, FMT, true, false, LUT_NONE>(a, smem, s);
}

template <bool ROT>
cudaError_t launch_f(int fmt, const StemBayerArgs &a, size_t smem, cudaStream_t s) {
  switch (fmt) {
    case FMT_BAYER: return launch_t<ROT, FMT_BAYER>(a, smem, s);
    case FMT_BAYER_REDCOL: return launch_t<ROT, FMT_BAYER_REDCOL>(a, smem, s);
    case FMT_RGB: return launch_t<ROT, FMT_RGB>(a, smem, s);
    default: return launch_t<ROT, FMT_BGR>(a, smem, s);
  }
}

int gcd_i(int a, int b) { while (b) { int t = a % b; a = b; b = t; } return a; }

// kernel format of a source (chan_order: IRMV_CH_*; needed columns are odd with rot180, even without)
int format_of(int chan_order, int rotate180) {
  if (chan_order == 0) return FMT_RGB;
  if (chan_order == 1) return FMT_BGR;
  const int red_x = (chan_order == 3 || chan_order == 4) ? 1 : 0;       // BGGR, GRBG: red on odd columns
  return ((rotate180 ? 1 : 0) == red_x) ? FMT_BAYER_REDCOL : FMT_BAYER;
}

// staged-row capacity of a strip for a source of height H (H / 640 = P / Q)
int nr_max_for(int P, int Q, int fmt) { return (2 * orows_for(fmt) * P + Q - 1) / Q + (fmt >= FMT_RGB ? 4 : 6); }

constexpr size_t kMaxSmem = 227 * 1024;  // dynamic shared memory a block may have on sm_100

// dynamic shared memory of a launch without the tables: tile + lerp table, then the staged rows
size_t smem_for(int H, int fmt) {
  const int g = gcd_i(H, kNet), P = H / g, Q = kNet / g;
  const size_t lut_n = 2 * Q * 255 + Q + 1;
  return (((size_t)(2 * orows_for(fmt) + 1) * PITCHW * 4 + lut_n * 2 + 15) & ~(size_t)15) +
         (size_t)nr_max_for(P, Q, fmt) * row_pitch(fmt);
}

// CTAs per SM with `smem` bytes of dynamic shared memory.  Every instantiation of a format has the same static
// shared memory, and __launch_bounds__(NTHREADS, 2) keeps the registers of two CTAs within an SM's file, so the
// answer depends on the format, the table mode and smem only.
template <int FMT, int LUT>
int ctas_per_sm(size_t smem) {
  auto k = stem_bayer2x_kernel<false, FMT, true, false, LUT>;
  int n = 0;
  if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k, NTHREADS, smem) != cudaSuccess) {
    (void)cudaGetLastError();            // a refused query must not surface as the next launch's error
    return 0;
  }
  return n;
}

// CTAs per SM in table mode `lut`; smem is the dynamic shared memory without the tables
template <int FMT>
int ctas_bayer(int lut, size_t smem) {
  switch (lut) {
    case LUT_NONE: return ctas_per_sm<FMT, LUT_NONE>(smem);
    case LUT_RAW: return ctas_per_sm<FMT, LUT_RAW>(smem + lut_bytes(LUT_RAW));
    default: return ctas_per_sm<FMT, LUT_COLOUR>(smem + lut_bytes(LUT_COLOUR));
  }
}

int ctas_for(int fmt, int lut, size_t smem) {
  switch (fmt) {
    case FMT_BAYER: return ctas_bayer<FMT_BAYER>(lut, smem);
    case FMT_BAYER_REDCOL: return ctas_bayer<FMT_BAYER_REDCOL>(lut, smem);
    case FMT_RGB: return lut ? 0 : ctas_per_sm<FMT_RGB, LUT_NONE>(smem);
    default: return lut ? 0 : ctas_per_sm<FMT_BGR, LUT_NONE>(smem);
  }
}

}  // namespace

// The fast path applies to: 8-bit Bayer or packed u8x3 source of width 1280, height >= 640 with
// H/640 = P/Q, Q <= 16, reference resize (corner-aligned stretch) and the 8-bit intermediate, when its shared
// memory fits a block: packed sources of 3400 rows and more stage rows three times as long and do not.  With a raw
// table (p.raw_lut, 1 KB) or the colour-correction stage (p.ccm, 1 KB + kCcmBytes) the tables must also keep the
// CTAs per SM of the launch without them (the kernel is sized for two at the camera's 1024 rows, where about 2.5 KB
// per CTA are left); where they would cost one, stem_kernel runs instead, at its full occupancy.  Called without
// tables at engine creation (no device query) and with them at every launch.
bool stem_bayer2x_applies(const PreprocessParams &p) {
  if (p.chan_order < 0 || p.chan_order > 5 || p.src_w != SW || p.resize_mode != 0 || !p.quantize_u8 || p.src_h < kNet || p.src_h > 4096) return false;
  const int g = gcd_i(p.src_h, kNet);
  if (kNet / g > 16) return false;
  const int fmt = format_of(p.chan_order, p.rotate180);
  const size_t smem = smem_for(p.src_h, fmt);
  const int lut = lut_mode(p);
  if (lut == LUT_NONE) return smem <= kMaxSmem;
  if (fmt >= FMT_RGB || smem + lut_bytes(lut) > kMaxSmem) return false;
  return ctas_for(fmt, lut, smem) >= ctas_for(fmt, LUT_NONE, smem);
}

int stem_bayer2x_ctas(const PreprocessParams &p) {
  if (!stem_bayer2x_applies(p)) return 0;
  const int fmt = format_of(p.chan_order, p.rotate180);
  return ctas_for(fmt, lut_mode(p), smem_for(p.src_h, fmt));
}

// Host side of the table block (layout above): conv0 weights w[16][9 taps][3] and bias[16] as the engine
// keeps them (FP32 values that are FP16-exact), for a source of height src_h in the given format and rotation.
std::vector<uint32_t> stem_bayer2x_tables(const float *w, const float *bias, int src_h, int chan_order, int rotate180) {
  const int g0 = gcd_i(src_h, kNet), P = src_h / g0, Q = kNet / g0, H = src_h;
  const int fmt = format_of(chan_order, rotate180);
  const bool packed = fmt >= FMT_RGB;
  const int OROWS = orows_for(fmt), NIR = 2 * OROWS + 1, RP = row_pitch(fmt), STRIP_WORDS = strip_words(OROWS);
  const int lut_n = 2 * Q * 255 + Q + 1;
  const int tab_strip = TAB_LUT + (lut_n + 7) / 8 * 4;
  const int nstrips = OWID / OROWS;
  std::vector<uint32_t> tab(tab_strip + nstrips * STRIP_WORDS, 0u);
  for (int lane = 0; lane < 32; ++lane) {
    const int g = lane >> 2, t = lane & 3;
    for (int nt = 0; nt < 2; ++nt)
      for (int s2 = 0; s2 < 2; ++s2)
        for (int h = 0; h < 2; ++h) {
          uint16_t v[2];
          for (int e = 0; e < 2; ++e) {
            // same K slot -> (ky, j) map as the kernel's `off` table; j = 9 and the pad lane carry zero weights
            const bool last = s2 == 1 && h == 1;
            const int ky = last ? t : 2 * s2 + h, j = last ? 8 + e : 2 * t + e;
            const float wv = (ky < 3 && j < 9) ? 0.5f * w[(nt * 8 + g) * 27 + ky * 9 + j] : 0.f;
            const __half hv = __float2half_rn(wv);
            memcpy(&v[e], &hv, 2);
          }
          tab[TAB_BFRAG + lane * 8 + nt * 4 + s2 * 2 + h] = (uint32_t)v[0] | ((uint32_t)v[1] << 16);
        }
  }
  for (int i = 0; i < 16; ++i) {
    const float hb = 0.5f * bias[i];
    memcpy(&tab[TAB_BIAS + i], &hb, 4);
  }
  uint16_t *lut = reinterpret_cast<uint16_t *>(tab.data() + TAB_LUT);
  for (int x = 0; x < lut_n; ++x) {
    const __half hv = __float2half_rn((float)(x / (2 * Q)) / 255.0f);
    memcpy(&lut[x], &hv, 2);
  }
  const bool rot = rotate180 != 0;
  const int red_y = (chan_order == 3 || chan_order == 5) ? 1 : 0;       // BGGR, GBRG: red on odd rows
  const bool red_col = fmt == FMT_BAYER_REDCOL;
  const int halo = packed ? 0 : 1;                                      // demosaic reads one row above / below
  for (int sidx = 0; sidx < nstrips; ++sidx) {
    uint32_t *st = tab.data() + tab_strip + sidx * STRIP_WORDS;
    const int iy0 = 2 * sidx * OROWS - 1;
    const int ry_min = ((iy0 > 0 ? iy0 : 0) * P) / Q;
    int ry_max = ((iy0 + NIR - 1) * P) / Q + 1;
    if (ry_max > H - 1) ry_max = H - 1;
    const int vlo = (rot ? H - 1 - ry_max : ry_min) - halo;
    st[0] = (uint32_t)vlo;
    st[1] = (uint32_t)(ry_max - ry_min + 2 + 2 * halo);             // rows lo - halo .. lo + 1 + halo of every input row
    for (int r = 0; r < NIR; ++r) {
      RowTab rt{0, 0u, 0u, 2};
      const int iy = iy0 + r;
      if (iy >= 0) {
        const int tt = iy * P, i0 = tt / Q, k = tt - i0 * Q, i1 = (i0 + 1 < H - 1) ? i0 + 1 : H - 1;
        int wA = 2 * (Q - k), wB = 2 * k;
        if (i1 == i0) { wA += wB; wB = 0; }
        const int sy0 = rot ? H - 1 - i0 : i0, sy1 = rot ? H - 1 - i1 : i1;
        const int lo = sy0 < sy1 ? sy0 : sy1;
        // weights doubled: the lerp numerator then is the BYTE offset into the FP16 table
        rt.w_lo = 2u * (uint32_t)(sy0 <= sy1 ? wA : wB);
        rt.w_hi = 2u * (uint32_t)(sy0 <= sy1 ? wB : wA);
        // a "site" row holds the red or blue sample at the needed columns, a "green" row the green one
        rt.flags = (!packed && (((lo & 1) == red_y) == red_col)) ? 1 : 0;
        rt.off = (lo - halo - vlo) * RP + 16;
      }
      memcpy(st + 4 + 4 * r, &rt, 16);
    }
  }
  return tab;
}

cudaError_t launch_stem_bayer2x(const PreprocessParams &p, int frame0, const uint32_t *tab, __half *out,
                                long long out_ps, __half *out2, long long out2_ps, cudaStream_t s) {
  StemBayerArgs a{};
  a.src = p.src; a.src_indirect = p.src_indirect; a.n = p.n; a.H = p.src_h; a.frame0 = frame0; a.rev = p.rev_order;
  const int Q = kNet / gcd_i(p.src_h, kNet);
  const int fmt = format_of(p.chan_order, p.rotate180);
  a.Q = Q; a.lut_n = 2 * Q * 255 + Q + 1;
  a.tab_strip = TAB_LUT + (a.lut_n + 7) / 8 * 4;
  a.tab = tab; a.out = out; a.out_ps = out_ps; a.out2 = out2; a.out2_ps = out2_ps;
  a.raw_lut = p.raw_lut; a.ccm = p.ccm; a.ccm_stride = p.ccm_stride;
  const size_t smem = smem_for(p.src_h, fmt);
  if (smem + lut_bytes(lut_mode(p)) > kMaxSmem) return cudaErrorInvalidValue;
  return p.rotate180 ? launch_f<true>(fmt, a, smem, s) : launch_f<false>(fmt, a, smem, s);
}

}  // namespace irmv
