// 10- / 12-bit and 12-bit packed Bayer frames -> the 8-bit mosaic the stems, the rotate kernel and the armor stage
// read (RawDecodeParams, common.cuh).  Every sample is masked to `bits` bits and mapped through the [2][2][1 << bits]
// table of its sensor site parity, staged in shared memory (16 KB at 12 bits).  This is the only kernel that knows
// the raw format; it streams the whole batch as one flat run of n * W * H samples, so a frame that does not start on
// a 16-byte boundary costs nothing extra.
#include "common.cuh"

namespace irmv {
namespace {

constexpr int kDecodeThreads = 256;
constexpr int kGroup = 16;          // samples per thread and step: one 16-byte store of the 8-bit mosaic

// Sample i of the batch, read byte by byte (any alignment).
template <bool PACKED>
__device__ __forceinline__ unsigned sample_at(const uint8_t *__restrict__ base, unsigned long long i) {
  if (PACKED) {
    const uint8_t *q = base + (i >> 1) * 3;
    return (i & 1) ? ((unsigned)q[2] << 4 | (unsigned)q[1] >> 4) : ((unsigned)q[0] << 4 | ((unsigned)q[1] & 15u));
  }
  return (unsigned)base[2 * i] | (unsigned)base[2 * i + 1] << 8;
}

// mw = ceil(2^64 / W): the batch row of sample i is umulhi(i, mw), exact while i * W < 2^64 (launch_raw_decode)
template <bool PACKED>
__global__ void __launch_bounds__(kDecodeThreads) raw_decode_kernel(RawDecodeParams p, unsigned long long mw) {
  extern __shared__ uint4 tab_vec[];
  const uint8_t *tab = reinterpret_cast<const uint8_t *>(tab_vec);
  const int bits = p.bits;
  const unsigned T = 1u << bits, mask = T - 1;
  for (unsigned k = threadIdx.x; k < T / 4; k += blockDim.x) tab_vec[k] = __ldg(reinterpret_cast<const uint4 *>(p.lut) + k);
  __syncthreads();

  const uint8_t *__restrict__ base = p.src_indirect ? *p.src_indirect : p.src;
  uint8_t *__restrict__ dst = p.dst;
  const unsigned W = p.src_w, H = p.src_h;
  const unsigned long long total = (unsigned long long)p.n * W * H, groups = total / kGroup;
  auto one = [&](unsigned long long i) {
    const unsigned long long row = __umul64hi(i, mw);
    const unsigned x = (unsigned)(i - row * W), y = (unsigned)row % H;
    dst[i] = tab[(((y & 1) * 2 + (x & 1)) << bits) + (sample_at<PACKED>(base, i) & mask)];
  };
  // Wide path: 32 (u16) or 24 (packed) input bytes per group in vector loads.  An even W puts every row start at an
  // even sample, so sample j of a group is on an x-parity j & 1 site, and W >= kGroup lets a group cross at most one
  // row end.
  const bool wide = W >= (unsigned)kGroup && !(W & 1) && ((uintptr_t)base & (PACKED ? 7 : 15)) == 0;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (unsigned long long g = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += stride) {
    const unsigned long long i0 = g * kGroup;
    if (!wide) {
      for (int j = 0; j < kGroup; ++j) one(i0 + j);
      continue;
    }
    unsigned s[kGroup];
    if (PACKED) {
      const uint2 *q = reinterpret_cast<const uint2 *>(base + (i0 >> 1) * 3);
      const uint2 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
      const uint32_t w[6] = {a.x, a.y, b.x, b.y, c.x, c.y};
#pragma unroll
      for (int m = 0; m < kGroup / 2; ++m) {
        const unsigned b0 = (w[(3 * m) >> 2] >> (((3 * m) & 3) * 8)) & 255u;
        const unsigned b1 = (w[(3 * m + 1) >> 2] >> (((3 * m + 1) & 3) * 8)) & 255u;
        const unsigned b2 = (w[(3 * m + 2) >> 2] >> (((3 * m + 2) & 3) * 8)) & 255u;
        s[2 * m] = b0 << 4 | (b1 & 15u);
        s[2 * m + 1] = b2 << 4 | b1 >> 4;
      }
    } else {
      const uint4 *q = reinterpret_cast<const uint4 *>(base + i0 * 2);
      const uint4 a = __ldg(q), b = __ldg(q + 1);
      const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
      for (int m = 0; m < kGroup / 2; ++m) {
        s[2 * m] = w[m] & mask;
        s[2 * m + 1] = (w[m] >> 16) & mask;
      }
    }
    // samples j < jb are on row y0, the others on the next row (row 0 of the next frame after a frame's last row)
    const unsigned long long row = __umul64hi(i0, mw);
    const unsigned x0 = (unsigned)(i0 - row * W), y0 = (unsigned)row % H;
    const unsigned y1 = y0 + 1 == H ? 0 : y0 + 1, jb = W - x0;
    const unsigned off0 = (y0 & 1) << (bits + 1), off1 = (y1 & 1) << (bits + 1);
    uint32_t o[kGroup / 4] = {0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < kGroup; ++j) {
      const unsigned v = tab[((unsigned)j < jb ? off0 : off1) + ((j & 1) ? T : 0u) + s[j]];
      o[j >> 2] |= v << ((j & 3) * 8);
    }
    *reinterpret_cast<uint4 *>(dst + i0) = make_uint4(o[0], o[1], o[2], o[3]);
  }
  // the last total % kGroup samples
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x < total - groups * kGroup) one(groups * kGroup + threadIdx.x);
}

}  // namespace

cudaError_t launch_raw_decode(const RawDecodeParams &p, int num_sms, cudaStream_t s) {
  if (p.n <= 0) return cudaSuccess;
  if ((p.bits != 10 && p.bits != 12) || (p.packed && (p.bits != 12 || (p.src_w & 1))) || p.src_w < 2 || p.src_h < 1 ||
      !p.lut || !p.dst || ((uintptr_t)p.dst & 15) || ((uintptr_t)p.lut & 15) || (!p.src && !p.src_indirect))
    return cudaErrorInvalidValue;
  const unsigned long long W = (unsigned)p.src_w, total = (unsigned long long)p.n * W * (unsigned)p.src_h;
  // exactness of the row division (i * W < 2^64) and 32-bit batch rows
  if (total > ~0ULL / W || (unsigned long long)p.n * (unsigned)p.src_h > 0xffffffffULL) return cudaErrorInvalidValue;
  const unsigned long long mw = ~0ULL / W + 1;
  const unsigned long long groups = total / kGroup;
  unsigned long long blocks = (groups + kDecodeThreads - 1) / kDecodeThreads;
  const size_t smem = (size_t)4 << p.bits;
  auto kernel = p.packed ? raw_decode_kernel<true> : raw_decode_kernel<false>;
  // one wave of resident CTAs walking the batch (the table is staged once per CTA)
  int per_sm = 0;
  cudaError_t err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kDecodeThreads, smem);
  if (err != cudaSuccess) return err;
  const unsigned long long cap = (unsigned long long)(num_sms > 0 ? num_sms : 1) * (per_sm > 0 ? per_sm : 1);
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  kernel<<<(unsigned)blocks, kDecodeThreads, smem, s>>>(p, mw);
  return cudaGetLastError();
}

}  // namespace irmv
