// Auto white balance (AwbParams, common.cuh): per frame, statistics over the 2x2 quads of the 8-bit mosaic, grey-world
// gains, and the colour-correction block the frame is then demosaiced with.  raw_lut.awb_statistics / awb_gains /
// awb_matrix are the definition; everything is integer arithmetic, so the result does not depend on the order in which
// CTAs add their sums.
//
// Grid (CTAs per frame, frames).  A thread classifies a few items of its frame -- an item is a 16-byte chunk of a row
// pair (8 quads) when W is a multiple of 16, else one quad read byte by byte -- and keeps 32-bit sums;
// the CTA reduces them and adds them to the frame's 64-bit accumulators.  The last CTA of a frame to finish turns the
// sums into gains, writes the frame's colour block and record, and zeroes the accumulators for the next launch (a
// captured graph replays this kernel with the same accumulators).
#include "common.cuh"

namespace irmv {
namespace {

constexpr int kAwbThreads = 256;
constexpr int kWideItems = 4;       // 16-byte chunk pairs per thread: 128 bytes in flight
constexpr int kByteItems = 32;      // quads per thread on the byte path

struct QuadSums { unsigned r, g, b, counted, dark, clipped; };

// One quad: samples s[py][px] at row parity py, column parity px; red at (ry, rx), blue at (1 - ry, 1 - rx)
__device__ __forceinline__ void add_quad(QuadSums &q, unsigned s00, unsigned s01, unsigned s10, unsigned s11, int ry, int rx,
                                         unsigned dark_level, unsigned clip_level) {
  const unsigned hi = max(max(s00, s01), max(s10, s11)), lo = min(min(s00, s01), min(s10, s11));
  if (hi > clip_level) { ++q.clipped; return; }
  if (lo < dark_level) { ++q.dark; return; }
  const unsigned r = ry ? (rx ? s11 : s10) : (rx ? s01 : s00);
  const unsigned b = ry ? (rx ? s00 : s01) : (rx ? s10 : s11);
  q.r += r;
  q.b += b;
  q.g += s00 + s01 + s10 + s11 - r - b;
  ++q.counted;
}

// 16 bytes at any alignment
__device__ __forceinline__ uint4 bytes16(const uint8_t *p) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) w[i] = (uint32_t)p[4 * i] | (uint32_t)p[4 * i + 1] << 8 | (uint32_t)p[4 * i + 2] << 16 | (uint32_t)p[4 * i + 3] << 24;
  return make_uint4(w[0], w[1], w[2], w[3]);
}

// WIDE (W % 16 == 0): an item is a 16-byte chunk of a row pair, loaded as one vector per row when the frame is 16-byte
// aligned and byte by byte otherwise (a caller's device batch may start anywhere); else an item is one quad.
template <bool WIDE, bool LUT>
__global__ void __launch_bounds__(kAwbThreads) awb_kernel(AwbParams p) {
  __shared__ __align__(16) uint8_t lut[LUT ? 1024 : 16];
  __shared__ unsigned red[kAwbThreads / 32][6];
  __shared__ int last;
  __shared__ int mf[9];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (LUT) reinterpret_cast<uint32_t *>(lut)[tid] = reinterpret_cast<const uint32_t *>(p.raw_lut)[tid];   // 256 words
  const int f = blockIdx.y;
  const int W = p.src_w, H = p.src_h;
  const uint8_t *base = p.src_indirect ? *p.src_indirect : p.src;
  const uint8_t *frame = base + (size_t)f * W * H;
  const unsigned dark_level = (unsigned)p.cfg[0], clip_level = (unsigned)p.cfg[1];
  int ry = 0, rx = 0;
  if (p.chan_order == 3) { ry = 1; rx = 1; }        // BGGR
  else if (p.chan_order == 4) { rx = 1; }           // GRBG
  else if (p.chan_order == 5) { ry = 1; }           // GBRG
  if (LUT) __syncthreads();
  // sample value at row parity py, column parity px
  auto map = [&](unsigned v, int py, int px) -> unsigned { return LUT ? lut[(py * 2 + px) * 256 + v] : v; };

  QuadSums q{0, 0, 0, 0, 0, 0};
  const int H2 = H >> 1;
  if (WIDE) {
    const int cpr = W >> 4;                           // 16-byte chunks per row
    const long long items = (long long)H2 * cpr;
    const long long it0 = (long long)blockIdx.x * (kAwbThreads * kWideItems) + tid;
    const bool aligned = ((uintptr_t)frame & 15) == 0;   // W % 16 == 0: every row then is aligned too
    uint4 a[kWideItems], b[kWideItems];
#pragma unroll
    for (int k = 0; k < kWideItems; ++k) {            // all loads first
      const long long it = it0 + (long long)k * kAwbThreads;
      if (it < items) {
        const int i = (int)(it / cpr), c = (int)(it - (long long)i * cpr);
        const uint8_t *row = frame + (size_t)(2 * i) * W + 16 * c;
        if (aligned) {
          a[k] = __ldg(reinterpret_cast<const uint4 *>(row));
          b[k] = __ldg(reinterpret_cast<const uint4 *>(row + W));
        } else {
          a[k] = bytes16(row);
          b[k] = bytes16(row + W);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < kWideItems; ++k) {
      if (it0 + (long long)k * kAwbThreads >= items) break;
      const uint32_t wa[4] = {a[k].x, a[k].y, a[k].z, a[k].w}, wb[4] = {b[k].x, b[k].y, b[k].z, b[k].w};
#pragma unroll
      for (int j = 0; j < 8; ++j) {                   // quad j: bytes 2j, 2j + 1 of both rows (columns even, odd)
        const uint32_t ua = wa[j >> 1] >> ((j & 1) * 16), ub = wb[j >> 1] >> ((j & 1) * 16);
        add_quad(q, map(ua & 255u, 0, 0), map((ua >> 8) & 255u, 0, 1), map(ub & 255u, 1, 0), map((ub >> 8) & 255u, 1, 1),
                 ry, rx, dark_level, clip_level);
      }
    }
  } else {
    const int qpr = W >> 1;
    const long long items = (long long)H2 * qpr;
    const long long it0 = (long long)blockIdx.x * (kAwbThreads * kByteItems) + tid;
    for (int k = 0; k < kByteItems; ++k) {
      const long long it = it0 + (long long)k * kAwbThreads;
      if (it >= items) break;
      const int i = (int)(it / qpr), j = (int)(it - (long long)i * qpr);
      const uint8_t *s = frame + (size_t)(2 * i) * W + 2 * j;
      add_quad(q, map(s[0], 0, 0), map(s[1], 0, 1), map(s[W], 1, 0), map(s[W + 1], 1, 1), ry, rx, dark_level, clip_level);
    }
  }

  // CTA sums (at most kAwbThreads * 32 quads * 510: 32 bits suffice) -> the frame's accumulators
  unsigned v[6] = {q.r, q.g, q.b, q.counted, q.dark, q.clipped};
#pragma unroll
  for (int c = 0; c < 6; ++c)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[c] += __shfl_xor_sync(0xffffffffu, v[c], o);
  if (lane == 0)
#pragma unroll
    for (int c = 0; c < 6; ++c) red[warp][c] = v[c];
  __syncthreads();
  AwbAcc &acc = p.acc[f];
  if (tid < 6) {
    unsigned long long s = 0;
    for (int w = 0; w < kAwbThreads / 32; ++w) s += red[w][tid];
    if (tid < 3) atomicAdd(&acc.sum[tid], s);
    else atomicAdd(tid == 3 ? &acc.counted : tid == 4 ? &acc.dark : &acc.clipped, (unsigned)s);
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) last = atomicAdd(&acc.ctas_done, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!last) return;

  // last CTA of the frame: every other CTA's sums are in (their fence precedes their ctas_done increment)
  __threadfence();
  uint8_t *out = p.ccm + (size_t)f * kCcmBytes;
  if (tid == 0) {
    volatile AwbAcc &va = acc;
    const unsigned long long S[3] = {va.sum[0], va.sum[1], va.sum[2]};
    const unsigned counted = va.counted, dark = va.dark, clipped = va.clipped;
    va.sum[0] = va.sum[1] = va.sum[2] = 0;          // ready for the next launch
    va.counted = va.dark = va.clipped = 0;
    va.ctas_done = 0;
    const unsigned long long A[3] = {2 * S[0], S[1], 2 * S[2]};
    const bool valid = counted >= (unsigned)p.cfg[2] && A[0] && A[1] && A[2];
    const unsigned long long amax = max(A[0], max(A[1], A[2]));
    int g[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const unsigned long long gc = valid ? (1024ull * amax + A[c] / 2) / A[c] : 1024ull;
      g[c] = (int)min(gc, (unsigned long long)p.cfg[3]);
    }
    const int *m = reinterpret_cast<const int *>(p.base);
#pragma unroll
    for (int k = 0; k < 9; ++k) mf[k] = min(max((m[k] * g[k % 3] + 512) >> 10, -32768), 32767);
    AwbRecord &r = p.rec[f];
    r.sum[0] = S[0]; r.sum[1] = S[1]; r.sum[2] = S[2];
    r.counted = counted; r.dark = dark; r.clipped = clipped;
    r.valid = valid ? 1 : 0;
    r.gain_q10[0] = g[0]; r.gain_q10[1] = g[1]; r.gain_q10[2] = g[2];
    r.reserved = 0;
  }
  __syncthreads();
  if (tid < 9) reinterpret_cast<int *>(out)[tid] = mf[tid];
  else if (tid < 12) reinterpret_cast<int *>(out)[tid] = 0;                                  // pad to kCcmTone
  if (tid < 3 * 256 / 4)
    reinterpret_cast<uint32_t *>(out + kCcmTone)[tid] = reinterpret_cast<const uint32_t *>(p.base + kCcmTone)[tid];
}

}  // namespace

cudaError_t launch_awb(const AwbParams &p, cudaStream_t s) {
  if (p.n <= 0) return cudaSuccess;
  if (p.chan_order < 2 || p.chan_order > 5 || p.src_w < 2 || p.src_h < 2 || p.n > 65535 || !p.cfg || !p.base ||
      !p.acc || !p.ccm || !p.rec || (!p.src && !p.src_indirect))
    return cudaErrorInvalidValue;
  const bool wide = (p.src_w & 15) == 0;
  const long long items = (long long)(p.src_h >> 1) * (wide ? (p.src_w >> 4) : (p.src_w >> 1));
  const long long per_cta = (long long)kAwbThreads * (wide ? kWideItems : kByteItems);
  const long long ctas = (items + per_cta - 1) / per_cta;
  if (ctas < 1 || ctas > 0x7fffffffLL) return cudaErrorInvalidValue;
  const dim3 grid((unsigned)ctas, (unsigned)p.n);
  if (wide) {
    if (p.raw_lut) awb_kernel<true, true><<<grid, kAwbThreads, 0, s>>>(p);
    else awb_kernel<true, false><<<grid, kAwbThreads, 0, s>>>(p);
  } else {
    if (p.raw_lut) awb_kernel<false, true><<<grid, kAwbThreads, 0, s>>>(p);
    else awb_kernel<false, false><<<grid, kAwbThreads, 0, s>>>(p);
  }
  return cudaGetLastError();
}

}  // namespace irmv
