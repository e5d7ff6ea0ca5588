// Raster (halo-tile) implicit-GEMM convolution on tcgen05 + TMEM, sm_100a only.
// Covers the 3x3 / stride-1 / pad-1 and the 1x1 convolutions of YOLOv8n (about 85 % of its FLOPs),
// i.e. the bulk of what the reference runs inside its TensorRT engine
// (reference src/yolo_engine.cpp:100-105).
//
// Activations live in the zero-padded raster layout (common.cuh): pixel q of the flat raster has
// its 3x3 neighbours at q + (ky-1)*Wp + (kx-1), with the padding pixels really being zero.  A tile
// of TM = 128*R consecutive raster pixels therefore needs ONE contiguous range of input pixels
// (TM + 2*Wp + 2 of them), and all nine taps are the same shared-memory tile read at nine
// different row offsets:
//
//   warp 8 (one lane)  TMA producer: the activation planes are [pixel][8 channels] arrays, so the
//                      halo range of one plane is ONE contiguous byte range and one
//                      cp.async.bulk per plane fills the tile  [cin/8][PP pixels][8 halfs]  -- the
//                      K-major, unswizzled UMMA operand layout, in which a tap shift is just
//                      +16 bytes per pixel on the descriptor's start address.  One mbarrier
//                      (expect_tx) hand-off per TILE.  Weights: resident (one load per CTA) when
//                      they fit next to two activation stages, otherwise streamed tap by tap
//                      through a small ring (layers with cin*cout >= 128*128).
//   warp 9 (one lane)  issues R * taps * cin/16 tcgen05.mma per tile back to back.  The loop is
//                      written so that every operand is a warp-uniform add on the previous one
//                      (descriptor low words, TMEM column): measured with scripts/mma_probe.cu the
//                      tensor pipe sustains max(N/2, 32 + N/4) cycles per M128 x N x K16 MMA for
//                      ANY operand layout, but a single thread that rebuilds 64-bit descriptors
//                      per MMA only issues one every 90-200 cycles.
//   warps 0-7          epilogue out of double-buffered TMEM: bias, SiLU, residual, FP16; a warp
//                      stores 32 consecutive pixels of one plane = 512 contiguous bytes; padding
//                      pixels are skipped so the zero border is preserved.  tcgen05.ld of the
//                      next 16-column chunk is in flight while the current one is processed.
#include <cstdlib>

#include "common.cuh"

namespace irmv {
namespace {

// warps 0..NEPI-1: epilogue (TMEM lane quarter = warp % 4); warp NEPI: TMA producer; warp NEPI+1: MMA issuer.
// NEPI = 8 when two CTAs share an SM (16 epilogue warps per SM either way), 16 otherwise.
constexpr int MAX_STAGES = 4;
constexpr int MAX_BSTAGES = 4;
constexpr int SMEM_BUDGET = 226 * 1024;     // 232448 B is the opt-in maximum per CTA

struct Bars {
  uint64_t full[MAX_STAGES];
  uint64_t empty[MAX_STAGES];
  uint64_t bw_full[MAX_BSTAGES];
  uint64_t bw_empty[MAX_BSTAGES];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint64_t mid_full, mid_empty;           // fused tail: intermediate tile written / consumed
  uint64_t ext_full[2], ext_empty[2];     // fused tail: the tail's other input planes loaded / consumed (1 or 2 buffers)
  uint64_t tail_full[2], tail_empty[2];   // fused tail: second accumulator set
  uint64_t bfull;
  uint32_t tmem_base;
  uint32_t pad;
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
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
// non-blocking probe: has the phase with this parity completed?
__device__ __forceinline__ bool mbar_test(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "mbarrier.test_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
      "selp.u32 %0, 1, 0, P1;\n"
      "}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_warp(uint64_t *bar, uint32_t parity, int lane) {
  if (lane == 0) mbar_wait(bar, parity);
  __syncwarp();
}
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
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// descriptors as (lo, hi) words: only the low word (start address, LBO) ever changes
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi,
                                           uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b64 da, db;\n"
      "setp.ne.b32 p, %6, 0;\n"
      "mov.b64 da, {%1, %2};\n"
      "mov.b64 db, {%3, %4};\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n"
      "}" ::"r"(tmem_d), "r"(alo), "r"(ahi), "r"(blo), "r"(bhi), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major operand without swizzle: 8x(16 B) core matrices; SBO = bytes between 8-row groups
// (128, rows are 16 B apart), LBO = bytes between the two 16-byte K halves of one MMA.
// Low word: start address >> 4 | (LBO >> 4) << 16; high word: SBO >> 4, descriptor version 1
// (bit 46), layout type 0 = no swizzle.
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) {
  return ((saddr & 0x3FFFFu) >> 4) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}
constexpr uint32_t kDescHi = (128u >> 4) | (1u << 14);

struct RArgs {
  ConvParams p;
  int R, TM, PP, halo_front, npix_need;   // rows = 128*R; PP = plane pitch (pixels); halo before q0
  int NCH, NP, taps, Wp, Hp1;             // cin/8, planes per stage, 1 or 9, OW+1, OH+1
  int q_begin, q_end, num_tiles, stages, tmem_cols, ctas_per_sm;
  int b_stream, b_stages;                 // weights streamed chunk by chunk through b_stages ring slots
  int nchunks, chunk_pairs;               // K chunks (a tap, or 64 channels of a wide 1x1) and K16 steps per chunk
  long long npix;                         // raster pixels of the tensors for this batch
  uint32_t idesc, mul_wp, mul_hp1;        // magic dividers (q / Wp, row / (H+1)), >> 34
  uint32_t a_stage_bytes, b_bytes, b_tap_bytes, off_b, off_bias, off_bars;
  uint32_t tap_a[9];                      // per chunk: A start offset inside a stage, 16-byte units
  // fused 1x1 tail (ConvParams::tail_w): intermediate tile [cout/8][TM][8], tail weights, tail bias
  uint32_t off_mid, off_ext, off_bt, off_tbias, bt_bytes, tail_idesc;
  int ext_planes;                         // tail input planes that come from global memory (ConvParams::tail_ext)
  int ext_stages;                         // buffers for them (2 when shared memory allows: the load of tile j+1 runs under tail(j))
  int rev;                                // walk the tiles from the last to the first (ConvParams::rev_tiles)
  int tmem_tail0;                         // first TMEM column of the tail accumulators
  int nsplit;                             // > 1: CTA b computes output-channel slice b % nsplit of tile b / nsplit (ConvParams::w_raster_split);
                                          // p.cout / p.npad are then the slice's, b_bytes the slice's weight bytes
};

// One 16-column chunk of one accumulator: bias, SiLU, residual, FP16, two 16-byte plane stores.
// hb: bias / 2 (ACT: folded into the SiLU argument) or the bias itself.
__device__ __forceinline__ void st_shared_v4(uint32_t addr, const uint4 &v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// padding pixels of the intermediate tile of a fused tail: finite values (their output rows are never stored)
__device__ __forceinline__ void st_shared_zero2(uint32_t addr, uint32_t plane_bytes) {
  const uint4 z = make_uint4(0, 0, 0, 0);
  st_shared_v4(addr, z);
  st_shared_v4(addr + plane_bytes, z);
}

// RES: 0 = none; 1 = residual of the same pixel added after the activation (C2f bottleneck shortcut); 2 = partial
// sum of the same channels added BEFORE the activation (r0 / r1 come from a half-resolution tensor: the
// upsampled half of a 1x1 conv over concat(upsample(a), b), computed at a's resolution -- ConvParams::res_up)
template <bool ACT, int RES, bool MID = false>
__device__ __forceinline__ void epi_chunk(const uint32_t (&v32)[16], const float *hb, __half *o, long long out_ps,
                                          __half *o2, long long out2_ps, const uint4 &r0, const uint4 &r1,
                                          uint32_t mid = 0, uint32_t mid_plane_bytes = 0) {
  float b[16];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 t = *reinterpret_cast<const float4 *>(hb + 4 * j);   // same address in every lane: broadcast
    b[4 * j] = t.x; b[4 * j + 1] = t.y; b[4 * j + 2] = t.z; b[4 * j + 3] = t.w;
  }
  if (RES == 2) {
    const float sc = ACT ? 0.5f : 1.0f;                    // ACT: b is bias / 2 and the accumulator is halved below
    const __half2 *h0 = reinterpret_cast<const __half2 *>(&r0);
    const __half2 *h1 = reinterpret_cast<const __half2 *>(&r1);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const float2 f0 = __half22float2(h0[t]), f1 = __half22float2(h1[t]);
      b[2 * t] = fmaf(f0.x, sc, b[2 * t]); b[2 * t + 1] = fmaf(f0.y, sc, b[2 * t + 1]);
      b[8 + 2 * t] = fmaf(f1.x, sc, b[8 + 2 * t]); b[8 + 2 * t + 1] = fmaf(f1.y, sc, b[8 + 2 * t + 1]);
    }
  }
  float v[16];
  if (ACT) {
    // SiLU(x) = x * sigmoid(x) = h + h * tanh(h), h = x / 2: one MUFU per element
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float h = fmaf(__uint_as_float(v32[j]), 0.5f, b[j]);
      float t;
      asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
      v[j] = fmaf(h, t, h);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(v32[j]) + b[j];
  }
  if (RES == 1) {
    const __half2 *h0 = reinterpret_cast<const __half2 *>(&r0);
    const __half2 *h1 = reinterpret_cast<const __half2 *>(&r1);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const float2 f0 = __half22float2(h0[t]), f1 = __half22float2(h1[t]);
      v[2 * t] += f0.x; v[2 * t + 1] += f0.y;
      v[8 + 2 * t] += f1.x; v[8 + 2 * t + 1] += f1.y;
    }
  }
  __half2 hv[8];
#pragma unroll
  for (int t = 0; t < 8; ++t) hv[t] = __floats2half2_rn(v[2 * t], v[2 * t + 1]);
  if (o) {
    *reinterpret_cast<uint4 *>(o) = *reinterpret_cast<uint4 *>(&hv[0]);
    *reinterpret_cast<uint4 *>(o + out_ps) = *reinterpret_cast<uint4 *>(&hv[4]);
  }
  if (o2) {                                                 // parity-split twin (stride-2 consumer)
    *reinterpret_cast<uint4 *>(o2) = *reinterpret_cast<uint4 *>(&hv[0]);
    *reinterpret_cast<uint4 *>(o2 + out2_ps) = *reinterpret_cast<uint4 *>(&hv[4]);
  }
  if (MID) {                                                // A operand of the fused 1x1 tail: [plane][pixel][8 channels]
    st_shared_v4(mid, *reinterpret_cast<uint4 *>(&hv[0]));
    st_shared_v4(mid + mid_plane_bytes, *reinterpret_cast<uint4 *>(&hv[4]));
  }
}

// TAIL: 0 = none, 1 = fused 1x1 consumer without activation, 2 = with SiLU
template <int R, int NEPI, bool ACT, int RES, int TAIL>
__global__ void __launch_bounds__((NEPI + 2) * 32, NEPI == 8 ? 2 : 1) conv_raster_kernel(const __grid_constant__ RArgs a) {
  constexpr int NTHREADS = (NEPI + 2) * 32;
  constexpr int TMA_WARP = NEPI, MMA_WARP = NEPI + 1;
  extern __shared__ __align__(1024) uint8_t smem[];
  const ConvParams &p = a.p;
  uint8_t *sA = smem;
  uint8_t *sB = smem + a.off_b;
  float *s_hb = reinterpret_cast<float *>(smem + a.off_bias);
  uint8_t *sMid = smem + a.off_mid;
  uint8_t *sExt = smem + a.off_ext;
  uint8_t *sBt = smem + a.off_bt;
  float *s_tb = reinterpret_cast<float *>(smem + a.off_tbias);
  Bars *bars = reinterpret_cast<Bars *>(smem + a.off_bars);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int npad = p.npad;
  // output-channel split (small replays): CTA -> (tile stream bid of gsz, slice)
  const int nsplit = a.nsplit;
  const int bid = nsplit > 1 ? (int)(blockIdx.x / (unsigned)nsplit) : (int)blockIdx.x;
  const int gsz = nsplit > 1 ? (int)(gridDim.x / (unsigned)nsplit) : (int)gridDim.x;
  const int split = nsplit > 1 ? (int)(blockIdx.x % (unsigned)nsplit) : 0;
  const float *const bias_g = p.bias + split * npad;
  const uint8_t *const w_g = reinterpret_cast<const uint8_t *>(p.w_raster) + (size_t)split * a.b_bytes;
  // debug trace rows cap+15 (CTA 0) / cap+14 (last CTA): {entry, setup done, exit} clocks + globaltimer ns
  long long *trow = (p.trace && tid == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1))
                        ? p.trace + (size_t)(p.trace_cap + (blockIdx.x == 0 ? 15 : 14)) * 8 : nullptr;
  if (trow) {
    trow[0] = clock64();
    unsigned long long g;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
    trow[3] = (long long)g;
  }

  // Programmatic dependent launch: let the next kernel of the stream start its prologue now; its
  // own griddepcontrol.wait still blocks until this grid has completed and flushed.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  // act: bias / 2 (folded into the SiLU argument), otherwise the bias itself
  for (int i = tid; i < npad; i += NTHREADS) s_hb[i] = ACT ? 0.5f * bias_g[i] : bias_g[i];
  if (TAIL)
    for (int i = tid; i < p.tail_npad; i += NTHREADS) s_tb[i] = TAIL == 2 ? 0.5f * p.tail_bias[i] : p.tail_bias[i];
  if (tid == 0) {
    for (int s = 0; s < a.stages; ++s) {
      mbar_init(&bars->full[s], 1);
      mbar_init(&bars->empty[s], 1);
    }
    for (int s = 0; s < MAX_BSTAGES; ++s) {
      mbar_init(&bars->bw_full[s], 1);
      mbar_init(&bars->bw_empty[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars->tmem_full[i], 1);
      mbar_init(&bars->tmem_empty[i], NEPI);
    }
    mbar_init(&bars->bfull, 1);
    mbar_init(&bars->mid_full, NEPI);
    mbar_init(&bars->mid_empty, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars->ext_full[i], 1);
      mbar_init(&bars->ext_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars->tail_full[i], 1);
      mbar_init(&bars->tail_empty[i], NEPI);
    }
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
  if (trow) trow[1] = clock64();
  // Resident weights are constants: start loading them before waiting for the producer kernel.
  if (warp == TMA_WARP && !a.b_stream && elect_one()) {
    const uint32_t bar = smem_u32(&bars->bfull), sB_u = smem_u32(sB);
    mbar_expect_tx(bar, a.b_bytes + (TAIL ? a.bt_bytes : 0u));
    for (uint32_t off = 0; off < a.b_bytes; off += 65536u) {
      const uint32_t n = a.b_bytes - off < 65536u ? a.b_bytes - off : 65536u;
      bulk_g2s(sB_u + off, w_g + off, n, bar);
    }
    if (TAIL) bulk_g2s(smem_u32(sBt), p.tail_w, a.bt_bytes, bar);
  }
  // Everything above overlapped the tail of the previous kernel (PDL); activations, residuals
  // and output buffers may only be touched once it has completed.
  asm volatile("griddepcontrol.wait;" ::: "memory");

  if (warp < NEPI) {
    // ===================================================================== epilogue
    // warp w reads TMEM lanes 32*(w%4)..+31 (hardware rule); the two warps of a lane quarter split
    // the (accumulator, 16-column chunk) work items between them.  Software pipeline: the
    // tcgen05.ld of item i+1 is issued before item i is processed (tcgen05.wait::ld waits for
    // every outstanding load, so exactly one load is in flight while the other chunk is computed).
    // warp w reads TMEM lanes 32*(w%4)..+31 (hardware rule); the NEPI/4 warps of a lane quarter split
    // the (accumulator, 16-column chunk) work items between them.  Software pipeline: the
    // tcgen05.ld of the warp's next item is issued before the current one is processed
    // (tcgen05.wait::ld waits for every outstanding load, so exactly one load is in flight while
    // the other chunk is computed).
    constexpr int NSUB = NEPI / 4;
    const int ew = warp & 3, sub = warp >> 2;
    const int chunk_shift = 31 - __clz(npad >> 4);          // npad / 16 is a power of two
    const int chunk_mask = (npad >> 4) - 1;
    const int items = R << chunk_shift;
    const uint32_t lane_base = tmem_base + ((uint32_t)(ew * 32) << 16);
    __half *const out = p.out ? p.out + (long long)(split * (npad >> 3)) * p.out_pstride : nullptr;
    const __half *const res = p.res ? p.res + (long long)(split * (npad >> 3)) * p.res_pstride : nullptr;
    const long long out_ps = p.out_pstride, res_ps = p.res_pstride;
    const int orl = p.out_runs;
    const long long out_ps_pair = orl == 1 ? 2 * out_ps : out_ps;   // distance between the two planes of a 16-channel chunk
    const int cout = p.cout;
    const int Wp = a.Wp, Hp1 = a.Hp1, W = p.OW, q_end = a.q_end, TM = a.TM;
    __half *const out2 = p.out2;
    const long long out2_ps = p.out2_pstride;
    const int Wp2 = (p.OW >> 1) + 1, Hp2 = (p.OH >> 1) + 1, cpl = cout >> 3;
    const uint32_t mul_wp = a.mul_wp, mul_hp1 = a.mul_hp1;
    const int q_lane = a.q_begin + ew * 32 + lane;
    const int num_tiles = a.num_tiles;
    long long *const trace = p.trace;
    const int trace_cap = p.trace_cap;
    // real pixel? (not the zero column x == W, not a zero row, inside the batch) -- per accumulator
    auto valid_mask = [&](int q_tile) -> uint32_t {
      uint32_t m = 0;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const int qi = q_tile + r * 128;
        const uint32_t row = (uint32_t)(((uint64_t)(uint32_t)qi * mul_wp) >> 34);
        const int x = qi - (int)row * Wp;
        const uint32_t img = (uint32_t)(((uint64_t)row * mul_hp1) >> 34);
        const int yrow = (int)row - (int)img * Hp1;
        if (qi < q_end && x < W && yrow != 0) m |= 1u << r;
      }
      return m;
    };
    // Fused tail, second epilogue: accumulators of tile number `jt` (TMEM set jt & 1) -> bias,
    // activation, FP16 -> the tail's output planes.
    const int tnp = TAIL ? p.tail_npad : 16;
    const int tshift = 31 - __clz(tnp >> 4), tmask = (tnp >> 4) - 1;
    __half *const tout = p.tail_out;
    const long long tout_ps = p.tail_out_pstride;
    __half *const tout2 = p.tail_out2;
    const long long tout2_ps = p.tail_out2_pstride;
    const int tcout = p.tail_cout;
    auto tail_epilogue = [&](int jt, int tile_j) {
      const int tb = jt & 1;
      const int q_tile = q_lane + tile_j * TM;
      const uint32_t okm = valid_mask(q_tile);
      mbar_wait_warp(&bars->tail_full[tb], (uint32_t)(jt >> 1) & 1u, lane);
      tc_fence_after();
      const uint32_t tcol = lane_base + (uint32_t)(a.tmem_tail0 + tb * R * tnp);
      const int items2 = R << tshift;
      const uint4 z = make_uint4(0, 0, 0, 0);
      for (int w = sub; w < items2; w += NSUB) {
        const int r = w >> tshift, c0 = (w & tmask) << 4;
        uint32_t v[16];
        tc_ld16(tcol + (uint32_t)(r * tnp + c0), v);
        tc_ld_wait();
        if (((okm >> r) & 1u) && c0 < tcout) {
          __half *o = tout ? tout + (long long)(c0 >> 3) * tout_ps + (long long)(q_tile + r * 128) * 8 : nullptr;
          __half *o2 = nullptr;
          if (tout2) {                                      // parity twin of the tail's output
            const int qi = q_tile + r * 128;
            const uint32_t row = (uint32_t)(((uint64_t)(uint32_t)qi * mul_wp) >> 34);
            const int x = qi - (int)row * Wp;
            const uint32_t img = (uint32_t)(((uint64_t)row * mul_hp1) >> 34);
            const int y = (int)row - (int)img * Hp1 - 1;
            const int px2 = ((int)img * Hp2 + 1 + (y >> 1)) * Wp2 + (x >> 1);
            o2 = tout2 + (long long)(((y & 1) * 2 + (x & 1)) * (tcout >> 3) + (c0 >> 3)) * tout2_ps + (long long)px2 * 8;
          }
          epi_chunk<TAIL == 2, false>(v, s_tb + c0, o, tout_ps, o2, tout2_ps, z, z);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->tail_empty[tb]);
    };
    int it = 0, prev_tile = -1;
    for (int tseq = bid; tseq < num_tiles; tseq += gsz, ++it) {
      const int tile = a.rev ? num_tiles - 1 - tseq : tseq;
      const int buf = it & 1;
      const uint32_t aph = (uint32_t)(it >> 1) & 1u;
      const bool tr = trace && blockIdx.x == 0 && tid == 0 && it < trace_cap;
      const int q_tile = q_lane + tile * TM;
      const uint32_t okmask = valid_mask(q_tile);
      __half *const out_q = out + (long long)q_tile * 8;
      const __half *const res_q = RES == 1 ? res + (long long)q_tile * 8 : nullptr;
      mbar_wait_warp(&bars->tmem_full[buf], aph, lane);
      // fused tail: the intermediate tile is free once the tail MMAs of the previous tile have read it
      if (TAIL) mbar_wait_warp(&bars->mid_empty, (uint32_t)(it & 1) ^ 1u, lane);
      tc_fence_after();
      if (tr) trace[it * 8 + 6] = clock64();
      const uint32_t tcol0 = lane_base + (uint32_t)(buf * R * npad);
      const uint32_t mid_lane = smem_u32(sMid) + (uint32_t)(ew * 32 + lane) * 16u;   // + (plane * TM + r * 128) * 16
      // item w -> accumulator r = w / chunks, chunk c = w % chunks; this warp takes w = sub, sub+NSUB, ...
      struct Item { int c0; bool ok; __half *o, *o2; uint32_t mid; uint4 r0, r1; };
      auto setup = [&](int w, Item &t) -> uint32_t {
        const int r = w >> chunk_shift;
        t.c0 = (w & chunk_mask) << 4;
        t.ok = ((okmask >> r) & 1u) && t.c0 < cout;
        const long long off = (long long)run_plane(t.c0 >> 3, orl) * out_ps + r * 1024;
        t.o = out ? out_q + off : nullptr;
        t.o2 = nullptr;
        t.mid = TAIL ? mid_lane + (uint32_t)((t.c0 >> 3) * TM + r * 128) * 16u : 0u;
        if (out2) {                                         // parity twin: plane group and half-resolution pixel of this lane
          const int qi = q_tile + r * 128;
          const uint32_t row = (uint32_t)(((uint64_t)(uint32_t)qi * mul_wp) >> 34);
          const int x = qi - (int)row * Wp;
          const uint32_t img = (uint32_t)(((uint64_t)row * mul_hp1) >> 34);
          const int y = (int)row - (int)img * Hp1 - 1;
          const int px2 = ((int)img * Hp2 + 1 + (y >> 1)) * Wp2 + (x >> 1);
          t.o2 = out2 + (long long)(((y & 1) * 2 + (x & 1)) * cpl + (t.c0 >> 3)) * out2_ps + (long long)px2 * 8;
        }
        if (RES == 1 && t.ok) {                             // residual: issue the loads early
          const __half *rp = res_q + (long long)(t.c0 >> 3) * res_ps + r * 1024;
          t.r0 = *reinterpret_cast<const uint4 *>(rp);
          t.r1 = *reinterpret_cast<const uint4 *>(rp + res_ps);
        }
        if (RES == 2 && t.ok) {                             // half-resolution partial sum: pixel (y / 2, x / 2) of its raster
          const int qi = q_tile + r * 128;
          const uint32_t row = (uint32_t)(((uint64_t)(uint32_t)qi * mul_wp) >> 34);
          const int x = qi - (int)row * Wp;
          const uint32_t img = (uint32_t)(((uint64_t)row * mul_hp1) >> 34);
          const int y = (int)row - (int)img * Hp1 - 1;
          const int px2 = ((int)img * Hp2 + 1 + (y >> 1)) * Wp2 + (x >> 1);
          const __half *rp = res + (long long)(t.c0 >> 3) * res_ps + (long long)px2 * 8;
          t.r0 = __ldg(reinterpret_cast<const uint4 *>(rp));
          t.r1 = __ldg(reinterpret_cast<const uint4 *>(rp + res_ps));
        }
        return tcol0 + (uint32_t)(r * npad + t.c0);
      };
      uint32_t va[16], vb[16];
      Item ia, ib;
      ia.r0 = ia.r1 = ib.r0 = ib.r1 = make_uint4(0, 0, 0, 0);
      int w = sub;
      if (w < items) tc_ld16(setup(w, ia), va);
      while (w < items) {
        tc_ld_wait();                                       // va ready
        const bool more_b = w + NSUB < items;
        if (more_b) tc_ld16(setup(w + NSUB, ib), vb);
        if (ia.ok) epi_chunk<ACT, RES, TAIL != 0>(va, s_hb + ia.c0, ia.o, out_ps_pair, ia.o2, out2_ps, ia.r0, ia.r1, ia.mid, (uint32_t)TM * 16u);
        else if (TAIL) st_shared_zero2(ia.mid, (uint32_t)TM * 16u);
        if (!more_b) break;
        tc_ld_wait();                                       // vb ready
        const bool more_a = w + 2 * NSUB < items;
        if (more_a) tc_ld16(setup(w + 2 * NSUB, ia), va);
        if (ib.ok) epi_chunk<ACT, RES, TAIL != 0>(vb, s_hb + ib.c0, ib.o, out_ps_pair, ib.o2, out2_ps, ib.r0, ib.r1, ib.mid, (uint32_t)TM * 16u);
        else if (TAIL) st_shared_zero2(ib.mid, (uint32_t)TM * 16u);
        if (!more_a) break;
        w += 2 * NSUB;
      }
      // all of this warp's TMEM reads of the buffer are done: hand it back to the MMA warp
      if (TAIL) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // st.shared -> tcgen05.mma operand reads
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&bars->tmem_empty[buf]);
        if (TAIL) mbar_arrive(&bars->mid_full);
      }
      if (tr) trace[it * 8 + 7] = clock64();
      if (TAIL && it > 0) tail_epilogue(it - 1, prev_tile);
      prev_tile = tile;
    }
    if (TAIL && it > 0) tail_epilogue(it - 1, prev_tile);
  } else if (warp == TMA_WARP) {
    // ===================================================================== TMA producer
    if (elect_one()) {
      const uint32_t sA_u = smem_u32(sA), sB_u = smem_u32(sB);
      int s = 0, itl = 0, bs = 0;
      uint32_t ph = 0, bph = 0;
      const uint32_t plane_bytes = (uint32_t)a.npix_need * 16u;
      const uint32_t pitch_bytes = (uint32_t)a.PP * 16u;
      const uint32_t tile_tx = plane_bytes * (uint32_t)a.NP;
      const int n0 = p.in_parity ? a.NP : p.seg[0].c >> 3, n1 = p.nseg > 1 ? p.seg[1].c >> 3 : 0;
      const size_t ps0 = (size_t)p.seg[0].pstride * 2, ps1 = (size_t)p.seg[1].pstride * 2;
      const int rl0 = p.in_parity ? 0 : p.seg[0].runs;
      // fused tail over a concat: the tail's other input planes for tile number j (no halo).  They do not
      // depend on this kernel's own progress, so they are loaded as early as their buffer is free.
      const uint32_t ext_bytes = (uint32_t)a.TM * 16u;
      const uint32_t ext_buf_bytes = ext_bytes * (uint32_t)a.ext_planes;
      auto issue_ext = [&](int j, int tile_j) {
        const int eb = a.ext_stages == 2 ? (j & 1) : 0;
        const uint32_t bar = smem_u32(&bars->ext_full[eb]);
        mbar_expect_tx(bar, ext_buf_bytes);
        uint32_t dst = smem_u32(sExt) + (uint32_t)eb * ext_buf_bytes;
        const uint8_t *src = reinterpret_cast<const uint8_t *>(p.tail_ext.ptr) + ((long long)a.q_begin + (long long)tile_j * a.TM) * 16;
        const size_t pse = (size_t)p.tail_ext.pstride * 2;
        for (int c = 0; c < a.ext_planes; ++c, dst += ext_bytes, src += pse) bulk_g2s(dst, src, ext_bytes, bar);
      };
      auto issue_main = [&](int tile, int itl) {
        const bool tr = p.trace && blockIdx.x == 0 && itl < p.trace_cap;
        const long long qlo = (long long)a.q_begin + (long long)tile * a.TM - a.halo_front;
        if (tr) p.trace[itl * 8 + 1] = clock64();
        const uint32_t bar = smem_u32(&bars->full[s]);
        mbar_expect_tx(bar, tile_tx);
        uint32_t dst = sA_u + (uint32_t)s * a.a_stage_bytes;
        const uint8_t *src = reinterpret_cast<const uint8_t *>(p.seg[0].ptr) + qlo * 16;
        if (rl0 == 0) {
          for (int c = 0; c < n0; ++c, dst += pitch_bytes, src += ps0) bulk_g2s(dst, src, plane_bytes, bar);
        } else {                                            // planes in runs (ConvSeg::runs)
          for (int c = 0; c < n0; ++c, dst += pitch_bytes) bulk_g2s(dst, src + (size_t)run_plane(c, rl0) * ps0, plane_bytes, bar);
        }
        src = reinterpret_cast<const uint8_t *>(p.seg[1].ptr) + qlo * 16;
        for (int c = 0; c < n1; ++c, dst += pitch_bytes, src += ps1) bulk_g2s(dst, src, plane_bytes, bar);
        if (tr) p.trace[itl * 8 + 2] = clock64();
        if (++s == a.stages) { s = 0; ph ^= 1u; }
      };
      auto tile_of = [&](int seq) { return a.rev ? a.num_tiles - 1 - seq : seq; };
      if (TAIL && a.ext_planes) {
        // Two independent streams of loads (main tiles, ext tiles) issued by one thread: poll both
        // barriers without blocking, so a full ext buffer never holds back the next main tile (the
        // blocking order main(j+1) -> ext(j) serialised the loads: one main tile in flight at a time,
        // its DRAM latency exposed on every tile -- scripts/trace_conv.py, profiles/r2_summary.md).
        const int mine = a.num_tiles > bid ? (a.num_tiles - 1 - bid) / gsz + 1 : 0;
        int mi = 0, ei = 0;
        while (mi < mine || ei < mine) {
          bool progressed = false;
          if (mi < mine && mbar_test(&bars->empty[s], ph ^ 1u)) {
            if (p.trace && blockIdx.x == 0 && mi < p.trace_cap) p.trace[mi * 8 + 0] = clock64();
            issue_main(tile_of(bid + mi * gsz), mi);
            ++mi;
            progressed = true;
          }
          if (ei < mine) {
            const int eb = a.ext_stages == 2 ? (ei & 1) : 0;
            const uint32_t eph = a.ext_stages == 2 ? ((uint32_t)(ei >> 1) & 1u) : ((uint32_t)ei & 1u);
            if (mbar_test(&bars->ext_empty[eb], eph ^ 1u)) {
              issue_ext(ei, tile_of(bid + ei * gsz));
              ++ei;
              progressed = true;
            }
          }
          if (!progressed) __nanosleep(64);
        }
      } else {
        for (int tseq = bid; tseq < a.num_tiles; tseq += gsz, ++itl) {
          const int tile = tile_of(tseq);
          if (p.trace && blockIdx.x == 0 && itl < p.trace_cap) p.trace[itl * 8 + 0] = clock64();
          mbar_wait(&bars->empty[s], ph ^ 1u);
          issue_main(tile, itl);
          if (a.b_stream) {
            const uint8_t *wsrc = w_g;
            for (int t = 0; t < a.nchunks; ++t, wsrc += a.b_tap_bytes) {
              mbar_wait(&bars->bw_empty[bs], bph ^ 1u);
              const uint32_t bbar = smem_u32(&bars->bw_full[bs]);
              mbar_expect_tx(bbar, a.b_tap_bytes);
              bulk_g2s(sB_u + (uint32_t)bs * a.b_tap_bytes, wsrc, a.b_tap_bytes, bbar);
              if (++bs == a.b_stages) { bs = 0; bph ^= 1u; }
            }
          }
        }
      }
    }
  } else {
    // ===================================================================== MMA issuer
    if (!a.b_stream) mbar_wait_warp(&bars->bfull, 0, lane);
    int it = 0, s = 0, bs = 0;
    uint32_t ph = 0, bph = 0;
    const uint32_t a_lo0 = desc_lo(smem_u32(sA), (uint32_t)a.PP * 16u);
    const uint32_t b_lo0 = desc_lo(smem_u32(sB), (uint32_t)npad * 16u);
    const uint32_t a_stage_u = a.a_stage_bytes >> 4;       // descriptor address units are 16 bytes
    const uint32_t a_pair_u = 2u * (uint32_t)a.PP;         // two 8-channel planes per K16 step
    const uint32_t b_pair_u = 2u * (uint32_t)npad;
    const uint32_t b_tap_u = a.b_tap_bytes >> 4;
    const int pairs = a.chunk_pairs, nchunks = a.nchunks;
    // Fused tail: MMAs of the pointwise consumer for tile number j, issued one tile behind the main
    // MMAs (tile j+1's main MMAs keep the pipe busy while the epilogue produces tile j's operand).
    const int tnp = TAIL ? p.tail_npad : 16;
    const uint32_t mid_lo0 = desc_lo(smem_u32(sMid), (uint32_t)a.TM * 16u);
    const uint32_t ext_lo0 = desc_lo(smem_u32(sExt), (uint32_t)a.TM * 16u);
    const uint32_t bt_lo0 = desc_lo(smem_u32(sBt), (uint32_t)tnp * 16u);
    auto issue_tail = [&](int j) {
      const int tb = j & 1;
      const int eb = a.ext_stages == 2 ? (j & 1) : 0;
      const uint32_t eph = a.ext_stages == 2 ? ((uint32_t)(j >> 1) & 1u) : ((uint32_t)j & 1u);
      mbar_wait_warp(&bars->mid_full, (uint32_t)j & 1u, lane);
      if (a.ext_planes) mbar_wait_warp(&bars->ext_full[eb], eph, lane);
      mbar_wait_warp(&bars->tail_empty[tb], ((uint32_t)(j >> 1) & 1u) ^ 1u, lane);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t td0 = tmem_base + (uint32_t)(a.tmem_tail0 + tb * R * tnp);
        // K of the tail = [planes loaded from global (older concat chunks) | the intermediate tile]
        uint32_t bl = bt_lo0, acc = 0;
        uint32_t al = ext_lo0 + (uint32_t)eb * (uint32_t)(a.ext_planes * a.TM);     // 16-byte units: planes x TM pixels per buffer
        for (int kk = 0; kk < (a.ext_planes >> 1); ++kk, al += 2u * (uint32_t)a.TM, bl += 2u * (uint32_t)tnp) {
#pragma unroll
          for (int r = 0; r < R; ++r)
            tc_mma_f16(td0 + (uint32_t)(r * tnp), al + (uint32_t)(r * 128), kDescHi, bl, kDescHi, a.tail_idesc, acc);
          acc = 1;
        }
        al = mid_lo0;
        for (int kk = 0; kk < (npad >> 4); ++kk, al += 2u * (uint32_t)a.TM, bl += 2u * (uint32_t)tnp) {
#pragma unroll
          for (int r = 0; r < R; ++r)
            tc_mma_f16(td0 + (uint32_t)(r * tnp), al + (uint32_t)(r * 128), kDescHi, bl, kDescHi, a.tail_idesc, acc);
          acc = 1;
        }
        tc_commit(&bars->tail_full[tb]);
        tc_commit(&bars->mid_empty);
        if (a.ext_planes) tc_commit(&bars->ext_empty[eb]);
      }
      __syncwarp();
    };
    for (int tile = bid; tile < a.num_tiles; tile += gsz, ++it) {
      const int buf = it & 1;
      const uint32_t aph = (uint32_t)(it >> 1) & 1u;
      const bool tr = p.trace && blockIdx.x == 0 && lane == 0 && it < p.trace_cap;
      if (tr) p.trace[it * 8 + 3] = clock64();
      mbar_wait_warp(&bars->tmem_empty[buf], aph ^ 1u, lane);
      mbar_wait_warp(&bars->full[s], ph, lane);
      tc_fence_after();
      if (tr) p.trace[it * 8 + 4] = clock64();
      const uint32_t tmem_d0 = tmem_base + (uint32_t)(buf * R * npad);
      const uint32_t a_stage_lo = a_lo0 + (uint32_t)s * a_stage_u;
      if (!a.b_stream) {
        if (elect_one()) {
          // MMAs into the R accumulators of the tile are interleaved (r innermost); every operand
          // below is a uniform add.
          uint32_t acc = 0;
          uint32_t bl_t = b_lo0;
          for (int t = 0; t < nchunks; ++t, bl_t += b_tap_u) {
            uint32_t al = a_stage_lo + a.tap_a[t], bl = bl_t;
            for (int j = 0; j < pairs; ++j, al += a_pair_u, bl += b_pair_u) {
#pragma unroll
              for (int r = 0; r < R; ++r)
                tc_mma_f16(tmem_d0 + (uint32_t)(r * npad), al + (uint32_t)(r * 128), kDescHi, bl, kDescHi, a.idesc, acc);
              acc = 1;
            }
          }
          tc_commit(&bars->empty[s]);
          tc_commit(&bars->tmem_full[buf]);
        }
        __syncwarp();
      } else {
        for (int t = 0; t < nchunks; ++t) {
          mbar_wait_warp(&bars->bw_full[bs], bph, lane);
          tc_fence_after();
          if (elect_one()) {
            uint32_t al = a_stage_lo + a.tap_a[t], bl = b_lo0 + (uint32_t)bs * b_tap_u;
            for (int j = 0; j < pairs; ++j, al += a_pair_u, bl += b_pair_u) {
#pragma unroll
              for (int r = 0; r < R; ++r)
                tc_mma_f16(tmem_d0 + (uint32_t)(r * npad), al + (uint32_t)(r * 128), kDescHi, bl, kDescHi, a.idesc,
                           (t | j) != 0 ? 1u : 0u);
            }
            tc_commit(&bars->bw_empty[bs]);
            if (t == nchunks - 1) {
              tc_commit(&bars->empty[s]);
              tc_commit(&bars->tmem_full[buf]);
            }
          }
          __syncwarp();
          if (++bs == a.b_stages) { bs = 0; bph ^= 1u; }
        }
      }
      if (tr) p.trace[it * 8 + 5] = clock64();
      if (++s == a.stages) { s = 0; ph ^= 1u; }
      if (TAIL && it > 0) issue_tail(it - 1);
    }
    if (TAIL && it > 0) issue_tail(it - 1);
  }

  tc_fence_before();
  __syncthreads();
  if (trow) {
    trow[2] = clock64();
    unsigned long long g;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
    trow[4] = (long long)g;
  }
  if (warp == MMA_WARP) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)a.tmem_cols) : "memory");
  }
}

bool plan(const ConvParams &p_in, int num_sms, RArgs &a) {
  ConvParams p = p_in;
  // Small replays: a launch with fewer 128-pixel tiles than a quarter of the SMs gives every tile to `split_ways`
  // CTAs, one per slice of output channels (ConvParams::w_raster_split).
  a.nsplit = 1;
  if (p.w_raster_split && p.split_ways > 1 && p.stride == 1 && !p.in_parity && !p.tail_w && !p.out2 && !p.out_runs &&
      !p.seg[0].runs && !p.res_up && p.out && p.cout == p.npad && p.npad % (16 * p.split_ways) == 0) {
    const long long m = (long long)p.B * (p.OH + 1) * (p.OW + 1) - (p.OW + 1);
    if ((m + 127) / 128 * p.split_ways <= num_sms) {
      a.nsplit = p.split_ways;
      p.w_raster = p.w_raster_split;
      p.cout /= a.nsplit;
      p.npad /= a.nsplit;
    }
  }
  const bool s2 = p.stride == 2;
  if (s2) {
    // stride 2: 3x3 / pad 1 over the parity-split twin of the input (common.cuh)
    if (!p.in_parity || p.k != 3 || p.pad != 1 || p.nseg != 1 || (p.H & 1) || (p.W & 1)) return false;
  } else {
    if (p.in_parity || p.stride != 1 || !(p.k == 1 || p.k == 3) || (p.k == 3 && p.pad != 1) || (p.k == 1 && p.pad != 0)) return false;
  }
  if (p.cin % 16 != 0 || p.npad % 16 != 0 || p.npad > 256) return false;
  for (int i = 0; i < p.nseg; ++i) if (p.seg[i].up || p.seg[i].c % 8) return false;
  if (p.OW + 2 + 8 > kGuardFront || p.cout % 16 != 0) return false;
  if (p.out2 && ((p.OH & 1) || (p.OW & 1))) return false;
  if (p.res_up && (!p.res || !p.act || p.tail_w || s2 || (p.OH & 1) || (p.OW & 1))) return false;
  // planes in runs: plain 1x1 / 3x3 convs only (no twin, residual, tail or second segment)
  if ((p.out_runs || p.seg[0].runs) && (p.out2 || p.res || p.tail_w || p.in_parity || p.nseg != 1)) return false;
  a.p = p;
  a.rev = p.rev_tiles;
  a.NCH = p.cin / 8;
  a.NP = s2 ? 4 * a.NCH : a.NCH;                     // planes per activation stage
  a.taps = p.k * p.k;
  // raster geometry of the OUTPUT grid (identical to the input grid for stride 1, and to each
  // parity sub-raster of the input for stride 2)
  a.Wp = p.OW + 1;
  a.Hp1 = p.OH + 1;
  a.npix = pr_pixels(p.B, p.OH, p.OW);
  a.q_begin = a.Wp;                                  // first pixel of raster row 1
  a.q_end = (p.B * (p.OH + 1)) * a.Wp;              // end of the last image row
  const long long Mr = (long long)a.q_end - a.q_begin;
  a.b_bytes = (uint32_t)((size_t)a.taps * p.cin * p.npad * 2);
  // K chunks: a tap of a 3x3, or (streamed wide 1x1) 64 input channels
  a.nchunks = a.taps;
  a.chunk_pairs = a.NCH >> 1;
  a.b_tap_bytes = (uint32_t)((size_t)p.cin * p.npad * 2);
  const bool tail = p.tail_w != nullptr;
  if (tail && (p.tail_npad % 16 || p.tail_npad > 256 || p.tail_cout % 16 || p.cout != p.npad || (!p.tail_out && !p.tail_out2))) return false;
  if (tail && p.res && !(p.act && p.tail_act)) return false;
  const int tnp = tail ? p.tail_npad : 0;
  const int ext_c = tail ? p.tail_ext.c : 0;         // tail input channels that come from global memory
  if (ext_c % 16 || (tail && p.tail_ext.up) || (tail && p.tail_out2 && ((p.OH & 1) || (p.OW & 1)))) return false;
  a.ext_planes = ext_c / 8;
  a.bt_bytes = tail ? (uint32_t)((size_t)(p.npad + ext_c) * tnp * 2) : 0u;
  // fused tail: the FP16 intermediate tile [cout/8][TM][8] (and the tail's other input planes) stay in shared memory
  // (two buffers for the tail's other input planes when they fit: their load then runs a tile ahead)
  int ext_stages = 1;
  auto tail_bytes = [&](int R) { return tail ? (size_t)a.bt_bytes + (size_t)(p.npad + ext_c * ext_stages) * 128 * R * 2 + 256 : (size_t)0; };
  const size_t misc = (size_t)p.npad * 4 + (size_t)tnp * 4 + sizeof(Bars) + 1024 + 256;
  const int halo = p.k == 3 ? (s2 ? a.Wp + 1 : 2 * a.Wp + 2) : 0;
  // Bulk copies run fastest when source, destination and size are multiples of 128 bytes (8
  // pixels): the copied range starts `delta` pixels early so that it begins on an 8-pixel boundary
  // of the plane (delta is the same for every tile because TM is a multiple of 128), and the tap
  // offsets absorb the shift.
  const int halo_front = p.k == 3 ? a.Wp + 1 : 0;
  const int delta = (((a.q_begin - halo_front) % 8) + 8) % 8;
  auto plane_pixels = [&](int R) { return (128 * R + halo + delta + 7) & ~7; };
  auto stage_bytes = [&](int R) { return (size_t)a.NP * plane_pixels(R) * 16; };
  int best_R = 0;
  a.b_stream = 0;
  for (int R = 4; R >= 1 && !best_R; R >>= 1) {
    if (2 * R * (p.npad + tnp) > 512) continue;
    long long tiles = (Mr + 128 * R - 1) / (128 * R);
    if (R > 1 && tiles < 2LL * num_sms) continue;    // keep every SM busy at small batch
    for (ext_stages = ext_c ? 2 : 1; ext_stages >= 1; --ext_stages) {
      if (a.b_bytes + tail_bytes(R) + 2 * stage_bytes(R) + misc > (size_t)SMEM_BUDGET) continue;
      best_R = R;
      break;
    }
  }
  if (ext_stages < 1) ext_stages = 1;
  a.ext_stages = ext_stages;
  if (!best_R && tail) return false;                 // a fused tail needs resident weights
  if (!best_R) {
    // weights do not fit next to two activation stages: stream them chunk by chunk.  Larger tiles
    // amortise the weight traffic (all of the weights once per tile), so prefer the largest R that
    // still leaves one tile per SM.
    if (p.k == 1) {
      if (a.NCH % 8 != 0 || a.NCH / 8 > 9) return false;
      a.nchunks = a.NCH / 8;
      a.chunk_pairs = 4;
      a.b_tap_bytes = (uint32_t)((size_t)64 * p.npad * 2);
    }
    for (int R = 4; R >= 1; R >>= 1) {
      if (2 * R * p.npad > 512) continue;
      if (2 * (size_t)a.b_tap_bytes + stage_bytes(R) + misc > (size_t)SMEM_BUDGET) continue;
      long long tiles = (Mr + 128 * R - 1) / (128 * R);
      if (R > 1 && tiles < (long long)num_sms) continue;
      best_R = R;
      a.b_stream = 1;
      break;
    }
  }
  if (!best_R) return false;
  a.R = best_R;
  a.TM = 128 * a.R;
  a.halo_front = halo_front + delta;
  a.npix_need = plane_pixels(a.R);
  a.PP = a.npix_need;
  a.a_stage_bytes = (uint32_t)stage_bytes(a.R);
  int cols = 2 * a.R * (p.npad + tnp), alloc = 32;
  while (alloc < cols) alloc <<= 1;
  a.tmem_cols = alloc;
  a.tmem_tail0 = 2 * a.R * p.npad;
  a.num_tiles = (int)((Mr + a.TM - 1) / a.TM);
  size_t b_smem = a.b_bytes;
  if (a.b_stream) {
    // split what is left between activation stages (at most 2) and weight ring slots (at most 4)
    a.ctas_per_sm = 1;
    size_t left = (size_t)SMEM_BUDGET - misc;
    a.stages = (left >= 2 * (size_t)a.a_stage_bytes + 2 * (size_t)a.b_tap_bytes) ? 2 : 1;
    left -= (size_t)a.stages * a.a_stage_bytes;
    a.b_stages = (int)(left / a.b_tap_bytes);
    if (a.b_stages > MAX_BSTAGES) a.b_stages = MAX_BSTAGES;
    b_smem = (size_t)a.b_stages * a.b_tap_bytes;
  } else {
    // The per-tile chain load -> MMA -> epilogue has latency bubbles, so when two CTAs fit on an SM
    // (shared memory and TMEM halves) run two: their phases interleave.
    const size_t half_budget = 112 * 1024;
    const size_t fixed = a.b_bytes + tail_bytes(a.R) + misc;
    const bool two = alloc <= 256 && fixed + 2 * (size_t)a.a_stage_bytes <= half_budget;
    a.ctas_per_sm = two ? 2 : 1;
    const size_t budget = two ? half_budget : (size_t)SMEM_BUDGET;
    a.stages = (int)((budget - fixed) / a.a_stage_bytes);
    if (a.stages > MAX_STAGES) a.stages = MAX_STAGES;
    a.b_stages = 0;
  }
  a.idesc = (1u << 4) | ((uint32_t)(p.npad >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  a.mul_wp = (uint32_t)(((1ull << 34) + (uint64_t)a.Wp - 1) / (uint64_t)a.Wp);
  a.mul_hp1 = (uint32_t)(((1ull << 34) + (uint64_t)a.Hp1 - 1) / (uint64_t)a.Hp1);
  a.off_b = (uint32_t)((size_t)a.stages * a.a_stage_bytes);
  a.off_mid = (uint32_t)((a.off_b + b_smem + 127u) & ~(size_t)127u);
  a.off_ext = a.off_mid + (tail ? (uint32_t)((size_t)p.npad * a.TM * 2) : 0u);
  a.off_bt = a.off_ext + (uint32_t)((size_t)ext_c * a.ext_stages * a.TM * 2);
  a.off_bias = (uint32_t)((a.off_bt + a.bt_bytes + 127u) & ~(size_t)127u);
  a.off_tbias = a.off_bias + (uint32_t)p.npad * 4;
  a.off_bars = (a.off_tbias + (uint32_t)tnp * 4 + 15u) & ~15u;
  a.tail_idesc = (1u << 4) | ((uint32_t)((tail ? tnp : 16) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  for (int t = 0; t < 9; ++t) {
    const int ky = t / 3, kx = t % 3;
    if (s2) {
      // tap (ky, kx) reads parity group g at offset (ky == 0 ? -Wp : 0) + (kx == 0 ? -1 : 0)
      const int g = (ky != 1) * 2 + (kx != 1);
      a.tap_a[t] = (uint32_t)(g * a.NCH * a.PP + delta + (ky == 0 ? 0 : a.Wp) + (kx == 0 ? 0 : 1));
    } else if (a.taps == 9) {
      a.tap_a[t] = (uint32_t)(delta + ky * a.Wp + kx);                    // tap shift in pixels
    } else {
      a.tap_a[t] = (uint32_t)(delta + t * 8 * a.PP);                      // 64-channel chunk = 8 planes
    }
  }
  return true;
}

template <int R, int NEPI, bool ACT, int RES, int TAIL>
cudaError_t launch_k(const RArgs &a, int grid, size_t smem, cudaStream_t s) {
  {   // the attribute is per device: no process-wide flag (several engines / devices per process); the call is cheap
    cudaError_t e = cudaFuncSetAttribute(conv_raster_kernel<R, NEPI, ACT, RES, TAIL>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((NEPI + 2) * 32);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, conv_raster_kernel<R, NEPI, ACT, RES, TAIL>, a);
}

template <int R, int NEPI>
cudaError_t launch_r(const RArgs &a, int grid, size_t smem, cudaStream_t s) {
  const bool act = a.p.act != 0, res = a.p.res != nullptr;
  if (res && a.p.res_up) {                           // 1x1 over concat(upsample(a), b), the a half precomputed at a's resolution
    if (!act || a.p.tail_w) return cudaErrorInvalidValue;
    return launch_k<R, NEPI, true, 2, 0>(a, grid, smem, s);
  }
  if (a.p.tail_w) {                                  // fused 1x1 consumer
    if (res) {                                       // bottleneck with shortcut + C2f.cv2: SiLU on both
      if (!act || !a.p.tail_act) return cudaErrorInvalidValue;
      return launch_k<R, NEPI, true, 1, 2>(a, grid, smem, s);
    }
    if (a.p.tail_act) return act ? launch_k<R, NEPI, true, 0, 2>(a, grid, smem, s) : launch_k<R, NEPI, false, 0, 2>(a, grid, smem, s);
    return act ? launch_k<R, NEPI, true, 0, 1>(a, grid, smem, s) : launch_k<R, NEPI, false, 0, 1>(a, grid, smem, s);
  }
  if (act) return res ? launch_k<R, NEPI, true, 1, 0>(a, grid, smem, s) : launch_k<R, NEPI, true, 0, 0>(a, grid, smem, s);
  return res ? launch_k<R, NEPI, false, 1, 0>(a, grid, smem, s) : launch_k<R, NEPI, false, 0, 0>(a, grid, smem, s);
}

}  // namespace

// Debug: the kernel instantiation and tiling plan() picks for this layer instance:
// {R, NEPI, b_stream, ctas_per_sm, stages, b_stages, tail (0/1/2), tiles}.
bool conv_raster_plan_info(const ConvParams &p, int num_sms, int out[8]) {
  RArgs a;
  if (!p.w_raster || !plan(p, num_sms, a)) return false;
  out[0] = a.R; out[1] = a.ctas_per_sm == 2 ? 8 : 16; out[2] = a.b_stream; out[3] = a.ctas_per_sm; out[4] = a.stages;
  out[5] = a.b_stages; out[6] = p.tail_w ? (p.tail_act ? 2 : 1) : 0; out[7] = a.num_tiles;
  return true;
}

bool conv_raster_fits(const ConvParams &p) {
  RArgs a;
  return p.w_raster != nullptr && plan(p, 148, a);
}

cudaError_t launch_conv_raster(const ConvParams &p, int num_sms, cudaStream_t s) {
  RArgs a;
  if (!plan(p, num_sms, a)) return cudaErrorInvalidValue;
  const size_t smem = (size_t)a.off_bars + sizeof(Bars) + 64;
  const int slots = num_sms * a.ctas_per_sm / a.nsplit;
  const int grid = (a.num_tiles < slots ? a.num_tiles : slots) * a.nsplit;
  if (a.ctas_per_sm == 2) {
    switch (a.R) {
      case 4: return launch_r<4, 8>(a, grid, smem, s);
      case 2: return launch_r<2, 8>(a, grid, smem, s);
      default: return launch_r<1, 8>(a, grid, smem, s);
    }
  }
  switch (a.R) {
    case 4: return launch_r<4, 16>(a, grid, smem, s);
    case 2: return launch_r<2, 16>(a, grid, smem, s);
    default: return launch_r<1, 16>(a, grid, smem, s);
  }
}

}  // namespace irmv
