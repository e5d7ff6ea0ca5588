// Implicit-GEMM convolution on the 5th-gen tensor cores (tcgen05 + TMEM), sm_100a only.
// Replaces the TensorRT FP16 engine body of the reference (reference src/yolo_engine.cpp:100-105).
//
//   D[M = B*OH*OW pixels][N = cout] = im2col(A)[M][K = k*k*cin] * W[N][K]^T   (FP16 in, FP32 accum)
//
// Persistent, warp-specialised CTA (one per SM), 128-row tiles:
//   warps 0-7   A producers: gather im2col rows straight from the NHWC activation(s) with 16-byte
//               cp.async into a 128B-swizzled K-major smem ring.  The gather does the padding
//               (zero fill), the stride, concat-on-read (two segments) and nearest-2x
//               upsample-on-read, so no im2col / concat / upsample tensor ever touches HBM.
//   warp  13    weight loader: the host pre-swizzles W into the exact smem image, so whole
//               k-blocks arrive with TMA bulk copies (cp.async.bulk + mbarrier complete_tx);
//               resident for the CTA's lifetime when they fit, streamed per stage otherwise.
//   warp  12    MMA issuer: one lane issues tcgen05.mma (M=128, N=npad, K=16) from smem
//               descriptors; tcgen05.commit releases ring slots and publishes accumulators.
//   warps 8-11  epilogue: tcgen05.ld accumulator rows out of TMEM (double-buffered, 2*N columns),
//               + bias, SiLU, residual, FP16 pack, channel-slice store.
#include <cstdlib>

#include "common.cuh"

namespace irmv {
namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int A_STAGE = BM * BK * 2;          // 16 KB
constexpr int NPROD = 256;                    // warps 0-7
constexpr int EPI_WARP0 = 8;
constexpr int MMA_WARP = 12;
constexpr int BLD_WARP = 13;
constexpr int NTHREADS = 14 * 32;
constexpr int MAX_STAGES = 12;
constexpr int SMEM_BUDGET = 220 * 1024;       // the ring depth hides HBM latency; L1 is not relied on

struct Bars {
  uint64_t full[MAX_STAGES];
  uint64_t empty[MAX_STAGES];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint64_t bfull;
  uint32_t tmem_base;
  uint32_t pad;
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// try_wait with a suspend-time hint: the polling lane sleeps in hardware until the phase
// completes (or the hint expires) instead of re-issuing try_wait every few cycles -- measured:
// un-hinted spinning by the epilogue lanes was 35% of all executed instructions and slowed every
// other mbarrier operation on the SM.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)), "r"(parity), "r"(0x989680u) : "memory");
}
// One lane polls, the warp is released by __syncwarp: 32 lanes spinning on try_wait saturate the
// shared-memory sync unit (measured: ~600 cycles to return from an already-completed barrier).
__device__ __forceinline__ void mbar_wait_warp(uint64_t *bar, uint32_t parity, int lane) {
  if (lane == 0) mbar_wait(bar, parity);
  __syncwarp();
}
// elect.sync: ptxas knows exactly one lane runs the guarded region, so tcgen05 operands can live in
// uniform registers without the per-lane "waterfall" loop that `if (lane == 0)` produces.
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .b32 %%rx;\n"
      ".reg .pred %%px;\n"
      "elect.sync %%rx|%%px, %1;\n"
      "@%%px mov.s32 %0, 1;\n"
      "}" : "+r"(pred) : "r"(0xffffffffu));
  return pred;
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes)
               : "memory");
}
__device__ __forceinline__ void cp_async_mbar_arrive(uint64_t *bar) {
  asm volatile("cp.async.mbarrier.arrive.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// wait until at most n of this thread's cp.async groups are still in flight (n is an immediate)
__device__ __forceinline__ void cp_async_wait_lag(int n) {
  switch (n) {
    case 0: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
    case 1: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
    case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
    case 3: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
    case 4: asm volatile("cp.async.wait_group 4;" ::: "memory"); break;
    case 5: asm volatile("cp.async.wait_group 5;" ::: "memory"); break;
    case 6: asm volatile("cp.async.wait_group 6;" ::: "memory"); break;
    default: asm volatile("cp.async.wait_group 7;" ::: "memory"); break;
  }
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
               ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                           uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128B-swizzled operand: rows are 128 B apart, 8-row groups 1024 B apart.
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);        // start address
  d |= (uint64_t)1 << 16;                          // LBO (ignored for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                // SBO
  d |= (uint64_t)1 << 46;                          // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                          // SWIZZLE_128B
  return d;
}

// SiLU with one MUFU op per element: x*sigmoid(x) = h + h*tanh(h), h = x/2 (tanh.approx.f32,
// relative error ~2^-11, the size of the FP16 rounding that follows).
__device__ __forceinline__ float silu(float x) {
  const float h = 0.5f * x;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

struct TcArgs {
  ConvParams p;
  int M, num_tiles, KB, ksteps_last, stages, b_resident, tmem_cols, rev;
  int nsplit, npad_full;        // nsplit > 1: CTA b computes output channels [slice * p.npad, +p.npad) of tile b / nsplit, slice = b % nsplit
                                // (p.npad / p.cout are the slice's; npad_full is the row count of a k-block of w_tiled)
  uint32_t idesc;
  uint32_t mul_ow, mul_oh;      // ceil(2^34 / OW), ceil(2^34 / OH): q = (n * mul) >> 34, exact for n < 2^25
  uint32_t off_b, off_ktab, off_bias, off_bars;
};

__global__ void __launch_bounds__(NTHREADS, 1) conv_tc_kernel(const __grid_constant__ TcArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const ConvParams &p = a.p;
  uint8_t *sA = smem;
  uint8_t *sB = smem + a.off_b;
  int32_t *s_ktab = reinterpret_cast<int32_t *>(smem + a.off_ktab);
  float *s_bias = reinterpret_cast<float *>(smem + a.off_bias);
  Bars *bars = reinterpret_cast<Bars *>(smem + a.off_bars);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int npad = p.npad;
  const uint32_t b_block_bytes = (uint32_t)npad * 128u;
  // output-channel split for small replays (same idea as the raster kernel's, conv_raster.cu): a k-block of the
  // pre-swizzled weights is [npad_full rows][128 B], so a slice of rows (a multiple of 8) is a contiguous range
  // with the same swizzle phase
  const int nsplit = a.nsplit;
  const int bid = nsplit > 1 ? (int)(blockIdx.x / (unsigned)nsplit) : (int)blockIdx.x;
  const int gsz = nsplit > 1 ? (int)(gridDim.x / (unsigned)nsplit) : (int)gridDim.x;
  const int split = nsplit > 1 ? (int)(blockIdx.x % (unsigned)nsplit) : 0;
  const __half *const w_g = p.w_tiled + (size_t)split * npad * BK;
  const size_t w_kb_stride = (size_t)a.npad_full * BK;

  // Programmatic dependent launch: the next kernel may start its prologue now; this kernel's own prologue (tables,
  // barriers, TMEM, resident weights) runs under the previous kernel's tail and only the warps that touch
  // activations wait for it (griddepcontrol.wait below).
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  for (int i = tid; i < a.KB * 16; i += NTHREADS) s_ktab[i] = p.ktab[i];
  for (int i = tid; i < npad; i += NTHREADS) s_bias[i] = p.bias[split * npad + i];
  if (tid == 0) {
    for (int s = 0; s < a.stages; ++s) {
      mbar_init(&bars->full[s], 128 + (a.b_resident ? 0 : 1));   // the 128 threads of the owning producer group
      mbar_init(&bars->empty[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars->tmem_full[i], 1);
      mbar_init(&bars->tmem_empty[i], 4);                                // one arrive per epilogue warp
    }
    mbar_init(&bars->bfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == MMA_WARP) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(&bars->tmem_base)), "r"((uint32_t)a.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;
  if (warp != BLD_WARP) asm volatile("griddepcontrol.wait;" ::: "memory");   // weights are constants: their loader runs ahead

  if (warp < EPI_WARP0) {
    // ===================================================================== A producers
    // Two groups of 4 warps alternate k-blocks (group = k-block parity), so the serial latency of
    // one warp's loop body (barrier wait, table lookup, issue) is paid once per TWO k-blocks.
    // Per tile a thread decodes its 8 rows once (magic-number division) into a 32-bit element
    // offset per (segment, row) and a bitmask of the taps that fall inside the image; per
    // k-block one table lookup gives the tap's element offset, so a row costs a bit test, an
    // add and the cp.async.  Hand-off: each thread tracks its copies with cp.async groups and ONE
    // lane per warp arrives on the stage's mbarrier, `lag` of the group's k-blocks behind the
    // issue front (256 per-thread arrives per stage serialise on one smem word).
    const int grp = warp >> 2;
    const int ptid = tid & 127;
    const int chunk = ptid & 7;
    const int rbase = ptid >> 3;                      // 0..15, rows rbase + 16*i
    const uint32_t dst_off = (uint32_t)rbase * 128u + (uint32_t)((chunk ^ (rbase & 7)) << 4);
    const int H = p.H, W = p.W, OW = p.OW, OH = p.OH, cstr = p.stride, M = a.M;
    const bool k3 = p.k == 3;
    const uint32_t mul_ow = a.mul_ow, mul_oh = a.mul_oh;
    const __half *sp0 = p.seg[0].ptr, *sp1 = p.seg[1].ptr;
    const long long ps0 = p.seg[0].pstride, ps1 = p.seg[1].pstride;
    const int up0 = p.seg[0].up, up1 = p.seg[1].up;
    const int two = p.nseg > 1;
    const int Hh = H >> 1, Wh = W >> 1;
    const int stages = a.stages, KB = a.KB;
    const int lag = (stages - 1) / 2 < 7 ? (stages - 1) / 2 : 7;   // own k-blocks in flight = lag + 1
    int s = 0;                 // ring slot of the current k-block
    uint32_t ph = 0;           // its phase
    int par = 0;               // its parity (which group owns it)
    int own = 0;               // k-blocks this group has issued
    int s_pub = grp % stages;  // ring slot of the next k-block this group publishes
    int itp = 0;
    for (int tseq = bid; tseq < a.num_tiles; tseq += gsz, ++itp) {
      const int tile = a.rev ? a.num_tiles - 1 - tseq : tseq; (void)tile;
      const bool tr = p.trace && blockIdx.x == 0 && tid == 0 && itp < p.trace_cap;
      if (tr) p.trace[itp * 8 + 0] = clock64();
      int off0[8], off1[8];
      uint32_t mask[8];
      {
        // The eight lanes that share rbase (chunk = lane & 7) need the same eight rows rbase + 16*i: lane
        // `chunk` decodes row i = chunk only and the octet exchanges the results by shuffle (the decode was
        // 29 % of the kernel's instructions when every thread decoded all eight rows itself).
        const int m = tile * BM + rbase + 16 * chunk;
        const uint32_t t = (uint32_t)(((uint64_t)(uint32_t)m * mul_ow) >> 34);      // m / OW
        const int ox = m - (int)t * OW;
        const uint32_t bimg = (uint32_t)(((uint64_t)t * mul_oh) >> 34);             // t / OH
        const int oy = (int)t - (int)bimg * OH;
        const int iy0 = oy * cstr, ix0 = ox * cstr;
        const int full = ((int)bimg * (H + 1) + 1 + iy0) * (W + 1) + ix0;                       // PR layout
        const int half = ((int)bimg * (Hh + 1) + 1 + (iy0 >> 1)) * (Wh + 1) + (ix0 >> 1);
        const int my0 = (up0 ? half : full) * 8;           // halfs inside a plane
        const int my1 = two ? (up1 ? half : full) * 8 : 0;
        // the PR layout's zero row/column make every tap of a real output pixel readable
        const uint32_t vb = __ballot_sync(0xffffffffu, m < M) >> (lane & 24);
        const uint32_t mfull = k3 ? 0x1FFu : 1u;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          off0[i] = __shfl_sync(0xffffffffu, my0, (lane & 24) | i);
          off1[i] = two ? __shfl_sync(0xffffffffu, my1, (lane & 24) | i) : 0;
          mask[i] = ((vb >> i) & 1u) ? mfull : 0u;
        }
      }
      if (tr) p.trace[itp * 8 + 1] = clock64();
      for (int kb = 0; kb < KB; ++kb) {
        if (par == grp) {
          const int2 e = *reinterpret_cast<const int2 *>(&s_ktab[(kb * 8 + chunk) * 2]);
          const int tapbit = e.y & 15, sg = (e.y >> 4) & 1;
          const uint32_t kvalid = (uint32_t)(e.y >> 5) & 1u;
          const __half *sbase = (sg ? sp1 : sp0) + (long long)(e.y >> 8) * (sg ? ps1 : ps0) + (long long)e.x * 8;
          const uint32_t dst0 = smem_u32(sA + (size_t)s * A_STAGE) + dst_off;
          const bool tk = p.trace && blockIdx.x == 0 && ptid == 0 && itp == 3 && kb < 16;
          if (tk) p.trace[p.trace_cap * 8 + kb * 8 + 0] = clock64();
          mbar_wait_warp(&bars->empty[s], ph ^ 1u, lane);
          if (tk) p.trace[p.trace_cap * 8 + kb * 8 + 1] = clock64();
          if (tr && kb == 0) p.trace[itp * 8 + 2] = clock64();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const uint32_t ok = kvalid & (mask[i] >> tapbit);
            const __half *src = ok ? sbase + (sg ? off1[i] : off0[i]) : sp0;
            cp_async16(dst0 + (uint32_t)i * (16u * 128u), src, ok ? 16u : 0u);
          }
          // each thread's copies arrive on the stage barrier when they land (no thread blocks on
          // memory latency); .noinc: the arrival is one of the 128 the barrier was initialised with
          asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(&bars->full[s])) : "memory");
          if (tk) p.trace[p.trace_cap * 8 + kb * 8 + 2] = clock64();
          ++own;
          if (tr && kb >= KB - 2) p.trace[itp * 8 + 3] = clock64();
        }
        par ^= 1;
        if (++s == stages) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp < MMA_WARP) {
    // ===================================================================== epilogue
    const int ew = warp - EPI_WARP0;
    const int row = ew * 32 + lane;
    int it = 0;
    for (int tseq = bid; tseq < a.num_tiles; tseq += gsz, ++it) {
      const int tile = a.rev ? a.num_tiles - 1 - tseq : tseq; (void)tile;
      const int acc = it & 1;
      const uint32_t aph = (uint32_t)(it >> 1) & 1u;
      const bool tr = p.trace && blockIdx.x == 0 && tid == EPI_WARP0 * 32 && it < p.trace_cap;
      mbar_wait_warp(&bars->tmem_full[acc], aph, lane);
      tc_fence_after();
      if (tr) p.trace[it * 8 + 6] = clock64();
      const int m = tile * BM + row;
      const bool mok = m < a.M;
      size_t opix = 0;
      if (mok) {
        const uint32_t t = (uint32_t)(((uint64_t)(uint32_t)m * a.mul_ow) >> 34);
        const uint32_t bimg = (uint32_t)(((uint64_t)t * a.mul_oh) >> 34);
        opix = (size_t)pr_index((int)bimg, (int)t - (int)bimg * p.OH, m - (int)t * p.OW, p.OH, p.OW);
      }
      __half *orow = p.out + (size_t)(split * (npad >> 3)) * p.out_pstride + opix * 8;                      // + plane * out_pstride
      const __half *rrow = p.res ? p.res + (size_t)(split * (npad >> 3)) * p.res_pstride + opix * 8 : nullptr;
      const uint32_t tbase = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * npad);
      for (int c0 = 0; c0 < npad; c0 += 16) {
        uint32_t r[16];
        tc_ld16(tbase + (uint32_t)c0, r);
        tc_ld_wait();
        if (c0 + 16 >= npad) {           // accumulator fully read: hand it back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&bars->tmem_empty[acc]);
        }
        if (!mok || c0 >= p.cout) continue;
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          float x = __uint_as_float(r[j]) + s_bias[c0 + j];
          v[j] = p.act ? silu(x) : x;
        }
        const int pl = c0 >> 3;                              // first of the two 8-channel planes
        if (rrow) {
          uint4 q0 = *reinterpret_cast<const uint4 *>(rrow + (size_t)pl * p.res_pstride);
          uint4 q1 = *reinterpret_cast<const uint4 *>(rrow + (size_t)(pl + 1) * p.res_pstride);
          const __half2 *h0 = reinterpret_cast<const __half2 *>(&q0);
          const __half2 *h1 = reinterpret_cast<const __half2 *>(&q1);
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            float2 f0 = __half22float2(h0[t]), f1 = __half22float2(h1[t]);
            v[2 * t] += f0.x; v[2 * t + 1] += f0.y;
            v[8 + 2 * t] += f1.x; v[8 + 2 * t + 1] += f1.y;
          }
        }
        __half2 hv[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) hv[t] = __floats2half2_rn(v[2 * t], v[2 * t + 1]);
        *reinterpret_cast<uint4 *>(orow + (size_t)pl * p.out_pstride) = *reinterpret_cast<uint4 *>(&hv[0]);
        if (c0 + 8 < p.cout)
          *reinterpret_cast<uint4 *>(orow + (size_t)(pl + 1) * p.out_pstride) = *reinterpret_cast<uint4 *>(&hv[4]);
      }
      if (tr) p.trace[it * 8 + 7] = clock64();
    }
  } else if (warp == MMA_WARP) {
    // ===================================================================== MMA issuer
    if (a.b_resident) mbar_wait_warp(&bars->bfull, 0, lane);
    int it = 0, s = 0;
    uint32_t ph = 0;
    const int stages = a.stages, KB = a.KB;
    for (int tseq = bid; tseq < a.num_tiles; tseq += gsz, ++it) {
      const int tile = a.rev ? a.num_tiles - 1 - tseq : tseq; (void)tile;
      const int acc = it & 1;
      const uint32_t aph = (uint32_t)(it >> 1) & 1u;
      mbar_wait_warp(&bars->tmem_empty[acc], aph ^ 1u, lane);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + (uint32_t)(acc * npad);
      for (int kb = 0; kb < KB; ++kb) {
        const bool tk = p.trace && blockIdx.x == 0 && lane == 0 && it == 3 && kb < 16;
        if (tk) p.trace[p.trace_cap * 8 + kb * 8 + 5] = clock64();
        mbar_wait_warp(&bars->full[s], ph, lane);
        tc_fence_after();
        if (tk) p.trace[p.trace_cap * 8 + kb * 8 + 6] = clock64();
        if (p.trace && blockIdx.x == 0 && lane == 0 && it < p.trace_cap) {
          if (kb == 0) p.trace[it * 8 + 4] = clock64();
          if (kb == KB - 1) p.trace[it * 8 + 5] = clock64();
        }
        if (elect_one()) {
          const uint64_t adesc = make_desc(smem_u32(sA + (size_t)s * A_STAGE));
          const uint64_t bdesc = make_desc(smem_u32(sB + (size_t)(a.b_resident ? kb : s) * b_block_bytes));
          const int nks = (kb == KB - 1) ? a.ksteps_last : 4;
          for (int ks = 0; ks < nks; ++ks)
            tc_mma_f16(tmem_d, adesc + (uint64_t)(ks * 2), bdesc + (uint64_t)(ks * 2), a.idesc,
                       (uint32_t)((kb | ks) != 0));
          tc_commit(&bars->empty[s]);
          if (kb == KB - 1) tc_commit(&bars->tmem_full[acc]);
          if (tk) p.trace[p.trace_cap * 8 + kb * 8 + 7] = clock64();
        }
        __syncwarp();
        if (++s == stages) { s = 0; ph ^= 1u; }
      }
    }
  } else {
    // ===================================================================== weight loader
    if (elect_one()) {
      if (a.b_resident) {
        mbar_expect_tx(&bars->bfull, (uint32_t)a.KB * b_block_bytes);
        for (int kb = 0; kb < a.KB; ++kb)
          bulk_g2s(sB + (size_t)kb * b_block_bytes, w_g + (size_t)kb * w_kb_stride,
                   b_block_bytes, &bars->bfull);
      } else {
        int s = 0;
        uint32_t ph = 0;
        for (int tseq = bid; tseq < a.num_tiles; tseq += gsz) {
      const int tile = a.rev ? a.num_tiles - 1 - tseq : tseq; (void)tile;
          for (int kb = 0; kb < a.KB; ++kb) {
            mbar_wait(&bars->empty[s], ph ^ 1u);
            mbar_expect_tx(&bars->full[s], b_block_bytes);
            bulk_g2s(sB + (size_t)s * b_block_bytes, w_g + (size_t)kb * w_kb_stride,
                     b_block_bytes, &bars->full[s]);
            if (++s == a.stages) { s = 0; ph ^= 1u; }
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;"
                 ::"r"(tmem_base), "r"((uint32_t)a.tmem_cols) : "memory");
  }
}

}  // namespace

size_t conv_tc_smem_bytes(const ConvParams &p, int *stages_out, int *b_resident_out) {
  const int KB = p.kpad / BK;
  const size_t b_block = (size_t)p.npad * 128;
  const size_t misc = (size_t)KB * 16 * 4 + (size_t)p.npad * 4 + sizeof(Bars) + 256;
  int resident = 0, stages = 0;
  if ((size_t)KB * b_block + 4 * (size_t)A_STAGE + misc + 1024 <= (size_t)SMEM_BUDGET) {
    resident = 1;
    stages = (int)(((size_t)SMEM_BUDGET - (size_t)KB * b_block - misc - 1024) / A_STAGE);
  } else {
    stages = (int)(((size_t)SMEM_BUDGET - misc - 1024) / (A_STAGE + b_block));
  }
  if (stages > MAX_STAGES) stages = MAX_STAGES;
  if (stages < 2) stages = 2;
  if (stages_out) *stages_out = stages;
  if (b_resident_out) *b_resident_out = resident;
  size_t b_bytes = resident ? (size_t)KB * b_block : (size_t)stages * b_block;
  return (size_t)stages * A_STAGE + b_bytes + misc + 1024;
}

cudaError_t launch_conv_tc(const ConvParams &p_in, int num_sms, cudaStream_t s) {
  TcArgs a;
  ConvParams p = p_in;
  a.M = p.B * p.OH * p.OW;
  a.num_tiles = (a.M + BM - 1) / BM;
  a.nsplit = 1;
  a.npad_full = p.npad;
  if (p.npad >= 128 && p.npad % 64 == 0 && p.cout == p.npad && a.num_tiles * 4 <= num_sms) {
    a.nsplit = 4;
    p.npad /= 4;
    p.cout /= 4;
  }
  a.p = p;
  a.rev = p.rev_tiles;
  a.KB = p.kpad / BK;
  const int ksteps_total = (p.K + 15) / 16;
  a.ksteps_last = ksteps_total - (a.KB - 1) * 4;
  size_t smem = conv_tc_smem_bytes(p, &a.stages, &a.b_resident);
  int cols = 2 * p.npad;
  int alloc = 32;
  while (alloc < cols) alloc <<= 1;
  a.tmem_cols = alloc;
  // instruction descriptor: D=F32, A=B=F16, both K-major, N = npad, M = 128
  a.idesc = (1u << 4) | ((uint32_t)(p.npad >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
  const size_t b_block = (size_t)p.npad * 128;
  a.off_b = (uint32_t)((size_t)a.stages * A_STAGE);
  size_t b_bytes = a.b_resident ? (size_t)a.KB * b_block : (size_t)a.stages * b_block;
  a.off_ktab = (uint32_t)(a.off_b + b_bytes);
  a.off_bias = a.off_ktab + (uint32_t)a.KB * 16 * 4;
  a.mul_ow = (uint32_t)(((1ull << 34) + (uint64_t)p.OW - 1) / (uint64_t)p.OW);
  a.mul_oh = (uint32_t)(((1ull << 34) + (uint64_t)p.OH - 1) / (uint64_t)p.OH);
  a.off_bars = (a.off_bias + (uint32_t)p.npad * 4 + 15u) & ~15u;
  {   // per device, cheap: no process-wide flag
    cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)(227 * 1024));
    if (e != cudaSuccess) return e;
  }
  const int slots = num_sms / a.nsplit;
  const int grid = (a.num_tiles < slots ? a.num_tiles : slots) * a.nsplit;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(NTHREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, conv_tc_kernel, a);
}

}  // namespace irmv
