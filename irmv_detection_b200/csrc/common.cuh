// Shared declarations for the sm_100a kernels and the host engine.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

namespace irmv {

constexpr int kNet = 640;           // network input side (reference: src/yolo_engine.cpp:98-99)
constexpr int kInC = 8;             // conv0 input is NHWC8: RGB + 5 zero channels (16-byte pixels)
constexpr int kRegMax = 16;
constexpr int kNumAnchors = 8400;   // 80*80 + 40*40 + 20*20
constexpr int kClsPad = 16;         // class-logit channels padded 14 -> 16
constexpr int kMaxCand = 4096;      // pre-NMS top-k (oracle/nms_ref.py MAX_CAND)

// ---------------------------------------------------------------- activation layout
// Activations are channel-blocked: a tensor of C channels is C/8 PLANES, each plane holding 8
// channels (16 bytes) per pixel: plane[q][8].  A channel slice or a concatenation is a list of
// planes, a tile of one plane is a contiguous byte range (one TMA bulk copy), and 32 lanes storing
// 32 consecutive pixels of a plane write 512 contiguous bytes.
// Inside a plane the pixels form a zero-padded raster ("PR" layout): row pitch Wp = W + 1
// (one zero pixel after each row -- it is the right neighbour of x = W-1 and the left neighbour of
// x = 0 of the next row), H + 1 rows per image (one zero row before each image -- it is the bottom
// neighbour of the previous image and the top neighbour of this one) and one trailing zero row.
// A 3x3 / pad-1 tap is then a constant raster offset (ky-1)*Wp + (kx-1) with no bounds test, which
// is what lets the raster convolution kernel feed all 9 taps from one shared-memory halo tile.
// Planes carry kGuardFront / kGuardBack zero pixels so halo tiles never leave the allocation.
__host__ __device__ inline int pr_wp(int W) { return W + 1; }
__host__ __device__ inline long long pr_pixels(int B, int H, int W) { return ((long long)B * (H + 1) + 1) * (W + 1); }
__host__ __device__ inline long long pr_index(int b, int y, int x, int H, int W) {
  return ((long long)b * (H + 1) + 1 + y) * (W + 1) + x;
}
constexpr int kGuardFront = 384;    // >= Wp + 1 of the widest raster-kernel layer (320 + 2)
constexpr int kGuardBack = 1024;    // >= 512-row tile overhang + Wp + 1

void set_error(const std::string &msg);
bool cuda_ok(cudaError_t e, const char *what, const char *file, int line);

#define IRMV_CUDA(call)                                              \
  do {                                                               \
    if (!::irmv::cuda_ok((call), #call, __FILE__, __LINE__)) return 1; \
  } while (0)

// ---------------------------------------------------------------- preprocess
struct PreprocessParams {
  const uint8_t *src;          // [n][H][W][3] or [n][H][W] (Bayer); used when src_indirect == null
  const uint8_t *const *src_indirect;  // device word holding the frame base pointer (batch path)
  __half *dst;                 // PR layout of [n][640][640][8]
  uint8_t *rotated;            // optional [n][H][W][3] rotated RGB image, may be null
  int n, src_w, src_h;
  int frame0;                  // index of the first source frame of this launch (chunked replays)
  int rev_order;               // 1: CTAs walk frames and strips from the last to the first (see ConvParams::rev_tiles)
  int chan_order, rotate180, resize_mode, quantize_u8;
  // filled by letterbox_geometry(): the resized image is new_w x new_h at (pad_x, pad_y) of the
  // 640 x 640 network input (stretch modes: 640 x 640 at (0, 0))
  int pad_x, pad_y, new_w, new_h;
  // Raw-domain colour stage of a Bayer source (irmv_engine_set_raw_lut): [2][2][256] bytes, sample s at sensor
  // position (y, x) reads as raw_lut[y & 1][x & 1][s] before anything else uses it; null = off
  const uint8_t *raw_lut;
  // Colour-correction stage of a Bayer source (irmv_engine_set_color_matrix): a kCcmBytes device block (layout
  // below) applied to every demosaiced pixel, after the raw table and before rot180 / resize; null = off
  const uint8_t *ccm;
  // Bytes between the colour-correction blocks of consecutive frames: 0 = one block for every frame (the user's
  // matrix), kCcmBytes = one block per source frame (auto white balance, awb.cu); frame f reads ccm + f * ccm_stride
  int ccm_stride;
};
// Device block of the colour-correction stage: int32 m[3][3] (row-major, units of 1/1024) at byte 0, u8 tone[3][256]
// at byte kCcmTone.  A demosaiced pixel (R, G, B) becomes, per output channel c,
//   tone[c][clamp((m[c][0] R + m[c][1] G + m[c][2] B + 512) >> 10, 0, 255)]
// (raw_lut.apply_color_matrix is the definition).  Staged in shared memory by the kernels that read it per pixel.
constexpr int kCcmTone = 48, kCcmBytes = kCcmTone + 3 * 256;
__device__ __forceinline__ int ccm_channel(const int *m, const uint8_t *tone, int R, int G, int B) {
  return tone[min(max((m[0] * R + m[1] * G + m[2] * B + 512) >> 10, 0), 255)];
}
__device__ __forceinline__ void apply_ccm(const uint8_t *ccm, int &R, int &G, int &B) {
  const int *m = reinterpret_cast<const int *>(ccm);
  const uint8_t *tone = ccm + kCcmTone;
  const int r = R, g = G, b = B;
  R = ccm_channel(m, tone, r, g, b);
  G = ccm_channel(m + 3, tone + 256, r, g, b);
  B = ccm_channel(m + 6, tone + 512, r, g, b);
}
// Copies the block to shared memory (dst 16-byte aligned, nthreads >= kCcmBytes / 4); visible after the next barrier.
__device__ __forceinline__ void stage_ccm(uint8_t *dst, const uint8_t *ccm, int tid) {
  if (tid < kCcmBytes / 4) reinterpret_cast<uint32_t *>(dst)[tid] = reinterpret_cast<const uint32_t *>(ccm)[tid];
}
// Resize geometry of a src_w x src_h frame.  LETTERBOX (resize_mode 1) follows ultralytics'
// LetterBox: r = min(640/w, 640/h), new = round(size * r), centred, pad value 114, pixel-centre
// bilinear resize.  (The reference itself stretches, src/yolo_engine.cpp:186-190; north_star and
// BASELINE configs[0] name the letterboxed form.)
inline void letterbox_geometry(int src_w, int src_h, int resize_mode, int *pad_x, int *pad_y, int *new_w, int *new_h) {
  *pad_x = *pad_y = 0; *new_w = *new_h = kNet;
  if (resize_mode != 1) return;
  const double rw = (double)kNet / src_w, rh = (double)kNet / src_h, r = rw < rh ? rw : rh;
  *new_w = (int)(src_w * r + 0.5); *new_h = (int)(src_h * r + 0.5);
  if (*new_w > kNet) *new_w = kNet;
  if (*new_h > kNet) *new_h = kNet;
  const double dw = (kNet - *new_w) / 2.0, dh = (kNet - *new_h) / 2.0;
  *pad_x = (int)(dw - 0.1 + 0.5); *pad_y = (int)(dh - 0.1 + 0.5);
  if (*pad_x < 0) *pad_x = 0;
  if (*pad_y < 0) *pad_y = 0;
}
cudaError_t launch_preprocess(const PreprocessParams &p, cudaStream_t s);
// rotated packed-RGB frame only (what get_rotated_image() exposes, reference include/irmv_detection/yolo_engine.hpp:34)
cudaError_t launch_rotate(const PreprocessParams &p, cudaStream_t s);
// Fused preprocess + conv0 (3x3 s2, 3->16, SiLU): w = [16][9 taps][3] FP32, writes two planes.
// out2 (optional): parity-split twin of the output (see ConvParams); the camera-case kernel writes one of the two.
// fast_tab: device table block of stem_bayer2x_tables() (null: always the generic kernel).
cudaError_t launch_stem(const PreprocessParams &p, const float *w, const float *bias, const uint32_t *fast_tab, __half *out,
                        long long out_pstride, __half *out2, long long out2_pstride, cudaStream_t s);
// Camera-case stem (stem_bayer.cu): Bayer or packed source of width 1280, reference resize, 8-bit intermediate,
// shared memory within a block's limit; with p.raw_lut, only where the table keeps the CTAs per SM.
bool stem_bayer2x_applies(const PreprocessParams &p);
// CTAs per SM of the camera-case kernel for p (with its raw table if p.raw_lut), 0 where it does not apply
int stem_bayer2x_ctas(const PreprocessParams &p);
// w [16][9 taps][3], bias [16]; the tables depend on the source height, the Bayer pattern and the rotation
std::vector<uint32_t> stem_bayer2x_tables(const float *w, const float *bias, int src_h, int chan_order, int rotate180);
cudaError_t launch_stem_bayer2x(const PreprocessParams &p, int frame0, const uint32_t *tab, __half *out,
                                long long out_ps, __half *out2, long long out2_ps, cudaStream_t s);

// ---------------------------------------------------------------- raw decode (raw_decode.cu)
// 10- / 12-bit and 12-bit packed Bayer frames -> the 8-bit mosaic every other kernel reads.  Frames are row-major
// without line padding: one little-endian u16 per sample (value in the low `bits` bits, the bits above are ignored),
// or two samples in three bytes (packed: B0 = p0[11:4], B1 = p1[3:0] << 4 | p0[3:0], B2 = p1[11:4]).
struct RawDecodeParams {
  const uint8_t *src;                  // [n] frames; used when src_indirect == null; any alignment
  const uint8_t *const *src_indirect;  // device word holding the frame base pointer (batch path)
  uint8_t *dst;                        // [n][H][W] 8-bit mosaic, 16-byte aligned
  const uint8_t *lut;                  // [2][2][1 << bits]: sample s at sensor position (y, x) -> lut[y & 1][x & 1][s]
  int n, src_w, src_h;
  int bits;                            // 10 or 12
  int packed;                          // 1: 12-bit packed (src_w even)
};
cudaError_t launch_raw_decode(const RawDecodeParams &p, int num_sms, cudaStream_t s);

// ---------------------------------------------------------------- auto white balance (awb.cu)
// Per frame: statistics over the 2x2 quads of the 8-bit mosaic, grey-world gains, and the frame's colour-correction
// block = the base block's matrix times diag(gains) plus its tone table (raw_lut.awb_statistics / awb_gains /
// awb_matrix are the definition).
struct AwbAcc {                        // per-frame accumulators; zero before a launch, left zero after it
  unsigned long long sum[3];           // SR, SG (both green sites), SB over the counted quads
  unsigned int counted, dark, clipped;
  unsigned int ctas_done;              // CTAs of the frame that have added their sums
};
struct AwbRecord {                     // == irmv_awb (include/irmv_cabi.h, static_assert in engine.cu)
  unsigned long long sum[3];
  unsigned int counted, dark, clipped;
  int valid;
  int gain_q10[3];
  int reserved;
};
struct AwbParams {
  const uint8_t *src;                  // [n][H][W] 8-bit mosaics; used when src_indirect == null
  const uint8_t *const *src_indirect;  // device word holding the frame base pointer (batch path)
  int n, src_w, src_h, chan_order;
  const uint8_t *raw_lut;              // [2][2][256] raw-domain colour table (PreprocessParams::raw_lut), or null
  const int *cfg;                      // device {dark_level, clip_level, min_quads, gain_max_q10} (irmv_awb_params)
  const uint8_t *base;                 // kCcmBytes block: the user's matrix and tone table, or the identity
  AwbAcc *acc;                         // [n]
  uint8_t *ccm;                        // [n][kCcmBytes] out: the block frame f is demosaiced with
  AwbRecord *rec;                      // [n] out
};
cudaError_t launch_awb(const AwbParams &p, cudaStream_t s);

// ---------------------------------------------------------------- convolution
struct ConvSeg {
  const __half *ptr;    // pixel 0 of the first plane of the slice read
  long long pstride;    // halfs between consecutive planes
  int c;                // channels read (multiple of 8)
  int up;               // 1: tensor is half resolution, read with nearest 2x upsampling
  int runs;             // raster kernel: 0 = the planes are contiguous; k > 0 = they form runs of r = 1 << (k-1)
                        // planes, one run every 2r planes (plane i of the slice = plane (i / r) * 2r + i % r
                        // counted from ptr).  The ShuffleNetV2 units process every second run of a stage
                        // buffer in place (channel split + shuffle cost zero bytes).
};
__host__ __device__ inline int run_plane(int i, int runs) {
  return runs == 0 ? i : (((i >> (runs - 1)) << runs) + (i & ((1 << (runs - 1)) - 1)));
}

struct ConvParams {
  ConvSeg seg[2];
  int nseg;
  int B, H, W;        // input grid (after upsampling)
  int OH, OW;
  int k, stride, pad;
  int cin;            // seg[0].c + seg[1].c
  int cout;           // stored output channels (multiple of 8)
  int npad;           // GEMM N (multiple of 16)
  int K;              // k*k*cin
  int kpad;           // K rounded up to 64
  int act;            // 1 = SiLU
  const __half *w_plain;   // [npad][kpad], k = (ky*k+kx)*cin + c          (direct kernel)
  const __half *w_tiled;   // [kpad/64][npad][64] with the 128B swizzle     (tcgen05 gather kernel)
  const __half *w_raster;  // [k*k][cin/8][npad][8]                          (tcgen05 raster kernel)
  const int32_t *ktab;     // [kpad/8][2] {pixel offset of the tap, meta} (tcgen05 gather kernel)
  const float *bias;       // [npad]
  __half *out;             // pixel 0 of the first output plane (raster kernel: null = only the parity twin is written)
  long long out_pstride;
  int out_runs;            // output planes in runs like ConvSeg::runs (raster kernel, no tail / twin / residual)
  const __half *res;       // residual added after the activation (same grid as out); may be null
  long long res_pstride;
  int res_up;              // raster kernel: 1 = `res` is a HALF-resolution tensor (OH/2 x OW/2) whose pixel (y/2, x/2) is
                           // added BEFORE the activation: the a-half of a 1x1 conv over concat(upsample(a), b), computed at
                           // a's resolution (a 1x1 conv commutes with nearest upsampling)
  // Parity-split twin tensors (raster kernel only).  A tensor of C channels on an H x W grid is
  // stored a second time as 4 * C/8 planes ordered [parity g = (y&1)*2 + (x&1)][C/8], each a padded
  // raster of the (H/2) x (W/2) pixels of that parity.  A 3x3 / stride-2 / pad-1 tap (ky, kx) then
  // reads parity ((ky != 1), (kx != 1)) at the constant raster offset (ky == 0 ? -Wp : 0) +
  // (kx == 0 ? -1 : 0) of the OUTPUT raster, so stride-2 layers run on the halo-tile kernel too.
  // Fused 1x1 consumer ("tail", raster kernel only): the epilogue's FP16 output tile stays in
  // shared memory as the A operand of a second, pointwise GEMM (K = cout of this conv), so the
  // intermediate tensor never goes to HBM when nobody else reads it (out == null).
  const __half *tail_w;    // [cout/8][tail_npad][8] = the 1x1 conv's w_raster image; null = no tail
  const float *tail_bias;  // [tail_npad]
  int tail_npad, tail_cout, tail_act;
  __half *tail_out;        // pixel 0 of the first output plane of the tail (null: only the parity twin)
  long long tail_out_pstride;
  __half *tail_out2;       // parity twin of the tail's output, or null
  long long tail_out2_pstride;
  ConvSeg tail_ext;        // channels that precede the intermediate in the tail's input concat (C2f.cv2 over
                           // [older chunks | the bottleneck output just computed]); c == 0: none
  int in_parity;           // 1: seg[0].ptr / pstride describe the parity twin of the input
  __half *out2;            // parity twin of the output (written in addition to `out` unless that is null); may be null
  long long out2_pstride;
  int rev_tiles;           // 1: process the tiles from the last to the first.  Consecutive layers alternate the
                           // direction, so a layer starts with the part of its input the producer wrote last --
                           // the part that is still in the 126 MB L2 (tensors of a 128-frame replay are 100-400 MB)
  long long *trace;        // debug: CTA 0 writes per-tile clock64 stamps [tile][8]; null in production
  int trace_cap;
  // Raster kernel, small replays: the same weights as `split_ways` slices of npad / split_ways output channels,
  // [slice][k*k][cin/8][npad / split_ways][8].  When a launch has fewer tiles than SMs / split_ways (the 20x20 layers
  // of a batch-1 replay are 4 tiles), each tile is computed by split_ways CTAs, one per slice: a CTA then pulls a
  // quarter of the weights through its SM and issues N/4-wide MMAs.  Null = never split.
  const __half *w_raster_split;
  int split_ways;
};
cudaError_t launch_conv_direct(const ConvParams &p, cudaStream_t s);
cudaError_t launch_conv_tc(const ConvParams &p, int num_sms, cudaStream_t s);
size_t conv_tc_smem_bytes(const ConvParams &p, int *stages, int *b_resident);
// Raster (halo-tile) kernel: 3x3/stride-1/pad-1 and 1x1 convolutions whose weights fit in shared
// memory.  w_raster: [tap][cin/8][npad][8] (no swizzle).  Returns false from the fit test when the
// layer has to take the gather kernel instead.
bool conv_raster_fits(const ConvParams &p);
bool conv_raster_plan_info(const ConvParams &p, int num_sms, int out[8]);
cudaError_t launch_conv_raster(const ConvParams &p, int num_sms, cudaStream_t s);

// ktab meta: bits 0-3 tap index (ky*k+kx), 4 segment, 5 valid, 8.. plane index inside the segment.
// The pixel offset is (ky-pad)*Wp + (kx-pad) relative to pixel (oy*stride, ox*stride); 0 for an
// upsample-on-read segment (1x1 convs only).
__host__ __device__ inline int32_t ktab_meta(int tap, int seg, int valid, int plane) {
  return tap | (seg << 4) | (valid << 5) | (plane << 8);
}

// ---------------------------------------------------------------- depthwise 3x3 (ShuffleNetV2 units)
struct DwParams {
  const __half *in;        // pixel 0 of the first input plane (padded raster layout)
  long long in_ps;         // halfs between planes
  __half *out;             // pixel 0 of the first output plane
  long long out_ps;
  const __half *w;         // [planes][9 taps][8 channels]
  const float *bias;       // [planes][8]
  int planes, B, H, W;     // input grid
  int stride;              // 1 or 2 (pad 1)
  int rev;                 // walk blocks from the last to the first (see ConvParams::rev_tiles)
};
cudaError_t launch_dwconv3x3(const DwParams &p, cudaStream_t s);

// ---------------------------------------------------------------- fused ShuffleNetV2 units (shuffle_unit.cu)
// The unit's constants as ONE blob the kernel fetches with a single bulk copy (byte offsets, all 16-byte
// aligned): 1x1 weights as [h][K + 8] halves (pw1: cin -> h, pw2: h -> h, down only: branch-1 1x1 cin -> h);
// depthwise weights as the B-operand table of the block-diagonal GEMM the kernel runs them as,
// [planes][10 taps (9 + a zero tap)][8 channels] 32-bit words = the FP16 weight in the half its channel parity
// selects (dw on the 1x1 -> dw -> 1x1 path, down only: dwa on the input); FP32 biases b1[h] b2[h] ba[h] dwb[h] dwab[cin].
struct ShuffleBlobLayout { int w1, w2, wa, dw, dwa, bias, bytes; };
__host__ __device__ inline ShuffleBlobLayout shuffle_blob_layout(int down, int cin, int h) {
  ShuffleBlobLayout L;
  L.w1 = 0;
  L.w2 = L.w1 + h * (cin + 8) * 2;
  L.wa = L.w2 + h * (h + 8) * 2;
  L.dw = L.wa + (down ? h * (cin + 8) * 2 : 0);
  L.dwa = L.dw + (h / 8) * 80 * 4;
  L.bias = L.dwa + (down ? (cin / 8) * 80 * 4 : 0);
  L.bytes = L.bias + (4 * h + cin) * 4;
  return L;
}
struct ShuffleUnitParams {
  int down;                      // 1: down unit (input grid 2H x 2W), 0: basic unit
  const __half *in;              // plane 0 of the input (down: the previous stage / stem output; basic: the stage buffer read)
  long long in_ps;
  __half *out;                   // plane 0 of the stage buffer written
  long long out_ps;
  int B, H, W;                   // output grid
  int cin, h;                    // input channels of the 1x1 convs on the input (basic: = h), half of the stage's channels
  int first_plane, runs;         // basic: the planes of the right half (ConvSeg::runs); the left half lies one run before
  const uint8_t *blob;           // shuffle_blob_layout(down, cin, h)
  int TH;                        // output rows per tile (divides H)
  int rev;
  int num_sms;
};
size_t shuffle_unit_smem(const ShuffleUnitParams &p);
int shuffle_unit_ctas_per_sm(const ShuffleUnitParams &p);
cudaError_t launch_shuffle_unit(const ShuffleUnitParams &p, cudaStream_t s);

// ---------------------------------------------------------------- SPPF pooling
// in: planes [0, c/8) of `buf`; writes maxpool5, maxpool5^2, maxpool5^3 to the three following
// groups of c/8 planes of the same tensor (ultralytics SPPF).
cudaError_t launch_sppf_pool(__half *buf, int B, int H, int W, long long pstride, int c, cudaStream_t s);

// ---------------------------------------------------------------- decode + NMS
struct HeadPtrs {
  const __half *box[3];   // 8 planes of [B][hw][hw] (PR layout)
  const __half *cls[3];   // 2 planes
  long long box_ps[3], cls_ps[3];   // plane strides (halfs)
  int padded;             // 1: planar PR layout (engine); 0: dense [B][hw*hw][C] (irmv_decode stage entry)
};
struct DetOut {            // per frame, device
  int32_t *num_dets;      // [B]
  float *boxes;           // [B][max_det][4]  network pixels
  float *scores;          // [B][max_det]
  int32_t *classes;       // [B][max_det]
  int32_t *index;         // [B][max_det]  flat anchor*nc+class
};
struct NmsScratch {
  float *boxes;                    // [B][A][4]
  unsigned long long *keys;        // [B][A*nc]
  int32_t *counts;                 // [B]
};
cudaError_t launch_decode(const HeadPtrs &h, int B, int nc, float score_thr, NmsScratch sc,
                          float *scores_or_null, cudaStream_t s);
cudaError_t launch_score_filter(const float *scores, int B, int A, int nc, float score_thr,
                                NmsScratch sc, cudaStream_t s);
cudaError_t launch_nms(NmsScratch sc, int B, int A, int nc, float iou_thr, int max_det, DetOut out,
                       cudaStream_t s);

// ---------------------------------------------------------------- light bars -> armors
// GPU form of IrmDetector::extract_armors (reference src/irm_detector.cpp:292-355): per detection,
// ROI of the rotated frame -> gray -> threshold -> top-level outer contours -> minimum-area
// rectangle -> light filter -> first two lights -> armor.  One CTA per detection.
struct ArmorOut {            // == irmv_armor (include/irmv_cabi.h)
  float pts[8];              // left.bottom, left.top, right.top, right.bottom (pixels of the rotated frame)
  float center[2];
  float score;
  int32_t class_id;
  int32_t size;              // 0 small, 1 large
  int32_t valid;
};
struct ArmorParams {
  const uint8_t *src;                   // [n] frames as the camera wrote them; used when src_indirect == null
  const uint8_t *const *src_indirect;   // device word holding the frame base pointer (batch path)
  int n, src_w, src_h, chan_order, rotate180;
  const int32_t *num;                   // [n] detections per frame
  const float *boxes;                   // [n][max_det][4] xyxy
  const float *scores;                  // [n][max_det]
  const int32_t *classes;               // [n][max_det]
  int max_det;
  float box_sx, box_sy, box_px, box_py; // box -> source pixels: (b - p) * s (engine: network pixels; 1/0 otherwise)
  int binary_threshold;
  float min_ratio, max_ratio, max_angle;
  double min_small, max_small, min_large, max_large;
  ArmorOut *out;                        // [n][max_det]
  int *slot_locks;                      // head of the scratch allocation (64 words, unused since every CTA owns a slot)
  uint32_t *scratch;                    // slots for ROIs that do not fit in shared memory (scratch allocation + 64 words)
  size_t scratch_words_per_cta;         // words per slot
  int grid;
  unsigned long long *prof;             // debug: cycles summed over ROIs {bitmap, flood, walks, armor, rois, flood rounds}; null in production
  const uint8_t *raw_lut;               // [2][2][256] raw-domain colour stage of a Bayer source (PreprocessParams::raw_lut), or null
  const uint8_t *ccm;                   // colour-correction block of a Bayer source (PreprocessParams::ccm), or null
  int ccm_stride;                       // PreprocessParams::ccm_stride
};
int armors_grid(int num_sms);
// null when the stage takes src_w x src_h frames, else why not (checked where the stage is set up, not per launch)
const char *armors_geometry_error(int src_w, int src_h);
size_t armors_scratch_words_per_cta(int src_w, int src_h);
size_t armors_scratch_total_words(int src_w, int src_h, int grid);   // allocate this many words (one slot per CTA of the grid)
cudaError_t launch_extract_armors(const ArmorParams &p, cudaStream_t s);
// armor corners -> PnP quads in the calibration frame; slots without an armor get a fixed valid quad
cudaError_t launch_quads_from_armors(const ArmorOut *armors, int total, float sx, float sy, float *pts, float *centers, cudaStream_t s);
cudaError_t launch_mask_pose_ok(const ArmorOut *armors, int total, uint8_t *ok, cudaStream_t s);

// ---------------------------------------------------------------- PnP
struct PnpConsts {
  double fx, fy, cx, cy;
  double k1, k2, p1, p2, k3;
  double half_w[2], half_h[2];   // small, large armor half extents (m)
};
struct PnpOut {
  double *rvec, *tvec;           // [n][3]
  uint8_t *ok;                   // [n]
  double *quat;                  // [n][4] or null
  double *rvec2, *tvec2, *rmse;  // second solution / [n][2] rmse, or null
  // distance_to_image_center (reference src/irm_detector.cpp:229, src/pnp_solver.cpp:54-59, the intended
  // computation): |centre - (cx, cy)| in FP32; centre = centers[i] when given (Armor::center in the
  // calibration frame), else the mean of the four image points.  dist may be null.
  float *dist;                   // [n] or null
  const float *centers;          // [n][2] or null
};
cudaError_t launch_pnp(const PnpConsts &c, const float *pts, int n, int large, PnpOut out,
                       cudaStream_t s);
// Optional Levenberg-Marquardt refinement of (rvec, tvec) in place on the pixel reprojection error
// (not in the reference's call; oracle cv2.solvePnPRefineLM).  quat may be null.
cudaError_t launch_pnp_refine_lm(const PnpConsts &c, const float *pts, int n, int large, int max_iters, double *rvec,
                                 double *tvec, double *quat, cudaStream_t s);

}  // namespace irmv
