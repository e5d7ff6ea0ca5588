// Host side of libirmv_b200.so: weight loading and re-layout, the YOLOv8n layer program, CUDA
// graphs on per-lane streams, pinned source slots, and the C ABI of include/irmv_cabi.h.
//
// Reference behaviour mirrored here (reference src/yolo_engine.cpp):
//   :24-117  constructor: allocate buffers, bind, capture {preprocess, network} into a graph
//   :153-177 detect(): graph launch, stream sync, parse_output
//   :202-220 parse_output(): scale boxes by (W/640, H/640), class id -> ArmorClass/UNKNOWN
// What changed: unified memory -> pinned host slots + device buffers; TensorRT/NPP -> the kernels
// in this directory; batch-1 -> sub-batches replayed on several lanes (streams).
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <exception>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/irmv_cabi.h"
#include "common.cuh"
#include "result_layout.h"

namespace irmv {

static thread_local std::string g_err;
void set_error(const std::string &msg) { g_err = msg; }
bool cuda_ok(cudaError_t e, const char *what, const char *file, int line) {
  if (e == cudaSuccess) return true;
  char buf[512];
  snprintf(buf, sizeof buf, "%s:%d: %s -> %s", file, line, what, cudaGetErrorString(e));
  set_error(buf);
  return false;
}

// Every device / pinned allocation of this file goes through these two, so that a test can assert
// that the per-frame calls allocate nothing (irmv_debug_alloc_count, include/irmv_cabi.h).
static std::atomic<long long> g_allocs{0};
cudaError_t dev_malloc(void **p, size_t bytes) { g_allocs.fetch_add(1); return cudaMalloc(p, bytes); }
cudaError_t host_malloc(void **p, size_t bytes) { g_allocs.fetch_add(1); return cudaHostAlloc(p, bytes, cudaHostAllocDefault); }

// Nothing may throw across the C ABI: entry points that build std containers from caller data run
// their body under this guard.
#define IRMV_ABI_TRY try {
#define IRMV_ABI_CATCH                                                                   \
  } catch (const std::exception &ex) {                                                   \
    ::irmv::set_error(std::string("internal error: ") + ex.what());                      \
    return 90;                                                                           \
  } catch (...) {                                                                        \
    ::irmv::set_error("internal error");                                                 \
    return 90;                                                                           \
  }

namespace {

struct HostConv {   // one GEMM as the kernels see it (possibly several reference convs merged)
  int cin_eff = 0, cout = 0, k = 1, stride = 1, act = 1;
  int npad = 0, K = 0, kpad = 0;
  std::vector<int> seg_c;            // channels per input segment (sum = cin_eff)
  std::vector<__half> w_plain;       // [npad][kpad]
  std::vector<__half> w_tiled;       // [kpad/64][npad][64] swizzled
  std::vector<__half> w_raster;      // [k*k][cin/8][npad][8] unswizzled (raster kernel)
  std::vector<float> bias;           // [npad]
  std::vector<int32_t> ktab;         // [kpad/8]
  __half *d_plain = nullptr, *d_tiled = nullptr, *d_raster = nullptr;
  __half *d_raster_split = nullptr;  // [split_ways][k*k][cin/8][npad / split_ways][8] (ConvParams::w_raster_split)
  int split_ways = 0;
  float *d_bias = nullptr;
  int32_t *d_ktab = nullptr;
  // a 1x1 conv over concat(upsample(a), b) split into W_a (at a's resolution, no bias / activation) and W_b (at
  // full resolution, + bias, + upsampled partial sum before the activation: ConvParams::res_up); null = not split
  std::shared_ptr<HostConv> up_a, up_b;
};

struct FileConv {
  int cin, cout, k, stride, act, groups = 1;
  std::vector<float> w, b;   // w [cout][cin / groups][k][k]
};

constexpr int kArchYolov8n = 0, kArchShuffleKpt = 1;   // irmv_detection_b200/weights.py ARCH_*

bool read_weights(const char *path, int &nc, int &arch, std::vector<FileConv> &out) {
  FILE *f = fopen(path, "rb");
  if (!f) { set_error(std::string("cannot open weight file ") + path); return false; }
  auto fail = [&](const std::string &why) { fclose(f); set_error(std::string(path) + ": " + why); return false; };
  if (fseek(f, 0, SEEK_END) != 0) return fail("cannot seek");
  const long long file_bytes = ftell(f);
  rewind(f);
  char magic[4];
  uint32_t hdr[3];
  if (fread(magic, 1, 4, f) != 4 || memcmp(magic, "IRMW", 4) != 0 || fread(hdr, 4, 3, f) != 3 || (hdr[0] != 1 && hdr[0] != 2))
    return fail("not an IRMW v1/v2 weight file");
  const bool v2 = hdr[0] == 2;          // v2: + architecture id in the header, + groups per convolution
  arch = kArchYolov8n;
  if (v2) {
    uint32_t a = 0;
    if (fread(&a, 4, 1, f) != 1 || a > 1) return fail("unknown architecture id");
    arch = (int)a;
  }
  // nothing in the header is trusted: counts and shapes are bounded before anything is allocated
  if (hdr[2] < 1 || hdr[2] > 512) return fail("implausible convolution count");
  nc = (int)hdr[1];
  out.resize(hdr[2]);
  long long left = file_bytes - (v2 ? 20 : 16);
  for (auto &c : out) {
    uint32_t h[6] = {0, 0, 0, 0, 0, 1};
    const size_t nh = v2 ? 6 : 5;
    if (left < (long long)nh * 4 || fread(h, 4, nh, f) != nh) return fail("truncated weight file");
    left -= (long long)nh * 4;
    if (h[0] < 1 || h[0] > 4096 || h[1] < 1 || h[1] > 4096 || !(h[2] == 1 || h[2] == 3) || !(h[3] == 1 || h[3] == 2) || h[4] > 1 ||
        !(h[5] == 1 || (h[5] == h[0] && h[0] == h[1])))
      return fail("bad convolution header (cin/cout in 1..4096, k in {1,3}, stride in {1,2}, act in {0,1}, groups 1 or depthwise)");
    c.cin = (int)h[0]; c.cout = (int)h[1]; c.k = (int)h[2]; c.stride = (int)h[3]; c.act = (int)h[4]; c.groups = (int)h[5];
    const long long nw = (long long)c.cout * (c.cin / c.groups) * c.k * c.k, need = (nw + c.cout) * 4;
    if (need > left) return fail("truncated weight file");
    c.w.resize((size_t)nw);
    c.b.resize((size_t)c.cout);
    if (fread(c.w.data(), 4, c.w.size(), f) != c.w.size() || fread(c.b.data(), 4, c.b.size(), f) != c.b.size())
      return fail("truncated weight file");
    left -= need;
  }
  fclose(f);
  return true;
}

// The convolutions the engine's layer program expects, in file order (irmv_detection_b200/weights.py
// conv_specs; ultralytics yolov8.yaml scale n, nc = 14, optional Pose branch kpt_shape [4, 2]).
struct Spec { int cin, cout, k, stride, act, groups = 1; };
struct ShuffleStage { int cin, cout, units; };
// the four stride-2 stages of the ShuffleNetV2-style backbone (irmv_detection_b200/weights.py shuffle_stage_plan)
const ShuffleStage kShuffleStages[4] = {{16, 32, 0}, {32, 64, 1}, {64, 128, 3}, {128, 256, 1}};
// stages with half-width <= this run as one fused kernel per unit (shuffle_unit.cu); the last stage (h = 128 on
// 20 x 20 maps) is weight-heavy and keeps one tcgen05 launch per convolution
constexpr int kShuffleFuseMaxH = 64;

std::vector<Spec> expected_specs(bool pose, int arch = kArchYolov8n) {
  std::vector<Spec> s;
  if (arch == kArchShuffleKpt) {
    // weights.py shuffle_conv_specs: stem, per stage a down unit {b1.dw, b1.pw, b2.pw1, b2.dw, b2.pw2} and
    // basic units {pw1, dw, pw2}, then everything of YOLOv8n-pose from m9.cv1 on
    s.push_back({3, 16, 3, 2, 1});
    for (const ShuffleStage &st : kShuffleStages) {
      const int h = st.cout / 2;
      s.push_back({st.cin, st.cin, 3, 2, 0, st.cin});
      s.push_back({st.cin, h, 1, 1, 1});
      s.push_back({st.cin, h, 1, 1, 1});
      s.push_back({h, h, 3, 2, 0, h});
      s.push_back({h, h, 1, 1, 1});
      for (int u = 0; u < st.units; ++u) {
        s.push_back({h, h, 1, 1, 1});
        s.push_back({h, h, 3, 1, 0, h});
        s.push_back({h, h, 1, 1, 1});
      }
    }
    const std::vector<Spec> y = expected_specs(true, kArchYolov8n);
    s.insert(s.end(), y.begin() + 25, y.end());
    return s;
  }
  auto c2f = [&](int c1, int c2, int n) {
    const int c = c2 / 2;
    s.push_back({c1, 2 * c, 1, 1, 1});
    for (int i = 0; i < n; ++i) { s.push_back({c, c, 3, 1, 1}); s.push_back({c, c, 3, 1, 1}); }
    s.push_back({(2 + n) * c, c2, 1, 1, 1});
  };
  s.push_back({3, 16, 3, 2, 1});
  s.push_back({16, 32, 3, 2, 1});
  c2f(32, 32, 1);
  s.push_back({32, 64, 3, 2, 1});
  c2f(64, 64, 2);
  s.push_back({64, 128, 3, 2, 1});
  c2f(128, 128, 2);
  s.push_back({128, 256, 3, 2, 1});
  c2f(256, 256, 1);
  s.push_back({256, 128, 1, 1, 1});
  s.push_back({512, 256, 1, 1, 1});
  c2f(384, 128, 1);
  c2f(192, 64, 1);
  s.push_back({64, 64, 3, 2, 1});
  c2f(192, 128, 1);
  s.push_back({128, 128, 3, 2, 1});
  c2f(384, 256, 1);
  const int chs[3] = {64, 128, 256};
  for (int i = 0; i < 3; ++i) {
    s.push_back({chs[i], 64, 3, 1, 1}); s.push_back({64, 64, 3, 1, 1}); s.push_back({64, 64, 1, 1, 0});
    s.push_back({chs[i], 64, 3, 1, 1}); s.push_back({64, 64, 3, 1, 1}); s.push_back({64, IRMV_NUM_CLASSES, 1, 1, 0});
  }
  if (pose)
    for (int i = 0; i < 3; ++i) { s.push_back({chs[i], 16, 3, 1, 1}); s.push_back({16, 16, 3, 1, 1}); s.push_back({16, 8, 1, 1, 0}); }
  return s;
}

bool check_specs(const std::vector<FileConv> &fc, bool pose, int arch) {
  const std::vector<Spec> want = expected_specs(pose, arch);
  if (fc.size() != want.size()) { set_error("weight file does not hold the convolutions of its architecture"); return false; }
  for (size_t i = 0; i < fc.size(); ++i) {
    const FileConv &c = fc[i];
    const Spec &w = want[i];
    if (c.cin != w.cin || c.cout != w.cout || c.k != w.k || c.stride != w.stride || c.act != w.act || c.groups != w.groups) {
      char buf[200];
      snprintf(buf, sizeof buf, "weight file: convolution %zu is %d->%d k%d s%d act%d, the layer program needs %d->%d k%d s%d act%d",
               i, c.cin, c.cout, c.k, c.stride, c.act, w.cin, w.cout, w.k, w.stride, w.act);
      set_error(buf);
      return false;
    }
  }
  return true;
}

// Build the GEMM operand images.  `parts` are reference convs sharing input/k/stride whose
// outputs are concatenated along N (the Detect head's box.0 | cls.0 pair); cin_pad >= cin.
HostConv make_conv(const std::vector<const FileConv *> &parts, int cin_pad,
                   const std::vector<int> &seg_c) {
  HostConv h;
  const FileConv &f0 = *parts[0];
  h.cin_eff = cin_pad; h.k = f0.k; h.stride = f0.stride; h.act = f0.act;
  int cout_real = 0;
  for (auto *p : parts) cout_real += p->cout;
  h.cout = (cout_real + 7) / 8 * 8;
  h.npad = (cout_real + 15) / 16 * 16;
  if (h.cout < h.npad) h.cout = h.npad;   // stored channels == GEMM N (cls head: 14 -> 16)
  h.K = h.k * h.k * cin_pad;
  h.kpad = (h.K + 63) / 64 * 64;
  h.seg_c = seg_c;
  h.w_plain.assign((size_t)h.npad * h.kpad, __float2half(0.f));
  h.bias.assign(h.npad, 0.f);
  int n0 = 0;
  for (auto *p : parts) {
    for (int n = 0; n < p->cout; ++n) {
      h.bias[n0 + n] = p->b[n];
      for (int c = 0; c < p->cin; ++c)
        for (int ky = 0; ky < p->k; ++ky)
          for (int kx = 0; kx < p->k; ++kx) {
            float v = p->w[(((size_t)n * p->cin + c) * p->k + ky) * p->k + kx];
            size_t kk = (size_t)(ky * p->k + kx) * cin_pad + c;
            h.w_plain[(size_t)(n0 + n) * h.kpad + kk] = __float2half(v);
          }
    }
    n0 += p->cout;
  }
  // tensor-core image: [kb][n][64] with the 16-byte chunk index XORed by (n & 7)
  const int KB = h.kpad / 64;
  h.w_tiled.assign((size_t)KB * h.npad * 64, __float2half(0.f));
  for (int kb = 0; kb < KB; ++kb)
    for (int n = 0; n < h.npad; ++n)
      for (int kk = 0; kk < 64; ++kk) {
        int chunk = (kk >> 3) ^ (n & 7);
        h.w_tiled[((size_t)kb * h.npad + n) * 64 + chunk * 8 + (kk & 7)] =
            h.w_plain[(size_t)n * h.kpad + kb * 64 + kk];
      }
  // raster-kernel image: [tap][cin/8][npad][8]
  {
    const int taps = h.k * h.k, nch = cin_pad / 8;
    h.w_raster.assign((size_t)taps * nch * h.npad * 8, __float2half(0.f));
    for (int t = 0; t < taps; ++t)
      for (int c = 0; c < nch; ++c)
        for (int n = 0; n < h.npad; ++n)
          for (int e = 0; e < 8; ++e)
            h.w_raster[(((size_t)t * nch + c) * h.npad + n) * 8 + e] =
                h.w_plain[(size_t)n * h.kpad + (size_t)t * cin_pad + c * 8 + e];
  }
  // chunk table (one entry per 8-channel chunk of K): {tap, segment, channel offset}; the
  // device tap table is derived per layer instance in add_conv (it needs W and the pixel strides)
  h.ktab.assign((size_t)(h.kpad / 8) * 3, -1);
  for (int q = 0; q < h.K / 8; ++q) {
    int kk = q * 8, tap = kk / cin_pad, c = kk % cin_pad;
    int sg = 0, off = c;
    if (seg_c.size() > 1 && c >= seg_c[0]) { sg = 1; off = c - seg_c[0]; }
    h.ktab[q * 3 + 0] = tap; h.ktab[q * 3 + 1] = sg; h.ktab[q * 3 + 2] = off;
  }
  return h;
}

// Input channels [c0, c1) of a convolution as a convolution of its own (bias / activation kept or dropped).
FileConv slice_cin(const FileConv &f, int c0, int c1, bool keep_bias_act) {
  FileConv r = f;
  const int kk = f.k * f.k;
  r.cin = c1 - c0;
  r.w.assign((size_t)f.cout * r.cin * kk, 0.f);
  for (int n = 0; n < f.cout; ++n)
    for (int c = c0; c < c1; ++c)
      for (int t = 0; t < kk; ++t) r.w[((size_t)n * r.cin + (c - c0)) * kk + t] = f.w[((size_t)n * f.cin + c) * kk + t];
  if (!keep_bias_act) { r.act = 0; std::fill(r.b.begin(), r.b.end(), 0.f); }
  return r;
}

// The ShuffleNetV2 units never move channels: a stage lives in one buffer, a unit rewrites every second
// run of its planes in place, and channel split / concat / shuffle become a logical -> physical channel
// map that is folded into the weights of whoever reads or writes the buffer.
// in_map[k] = logical input channel held by physical input channel k; out_map[n] likewise for outputs.
FileConv permuted(const FileConv &f, const std::vector<int> &in_map, const std::vector<int> &out_map) {
  FileConv r = f;
  const int kk = f.k * f.k;
  for (int n = 0; n < f.cout; ++n) {
    const int ln = out_map.empty() ? n : out_map[n];
    r.b[n] = f.b[ln];
    for (int c = 0; c < f.cin; ++c) {
      const int lc = in_map.empty() ? c : in_map[c];
      for (int t = 0; t < kk; ++t) r.w[((size_t)n * f.cin + c) * kk + t] = f.w[((size_t)ln * f.cin + lc) * kk + t];
    }
  }
  return r;
}

struct HostDw {              // depthwise 3x3: [planes][9 taps][8] FP16 + [planes][8] FP32 bias, physical channel order
  int c = 0, stride = 1;
  std::vector<__half> w;
  std::vector<float> b;
  __half *d_w = nullptr;
  float *d_b = nullptr;
};

HostDw make_dw(const FileConv &f, const std::vector<int> &map) {   // map[physical channel] = logical channel
  HostDw h;
  h.c = f.cout; h.stride = f.stride;
  h.w.assign((size_t)f.cout * 9, __float2half(0.f));
  h.b.assign(f.cout, 0.f);
  for (int pc = 0; pc < f.cout; ++pc) {
    const int lc = map.empty() ? pc : map[pc];
    h.b[pc] = f.b[lc];
    for (int t = 0; t < 9; ++t) h.w[((size_t)(pc / 8) * 9 + t) * 8 + pc % 8] = __float2half(f.w[(size_t)lc * 9 + t]);
  }
  return h;
}

bool upload(HostConv &h) {
  auto up = [](void **d, const void *src, size_t bytes) {
    if (!cuda_ok(dev_malloc(d, bytes), "dev_malloc(weights)", __FILE__, __LINE__)) return false;
    return cuda_ok(cudaMemcpy(*d, src, bytes, cudaMemcpyHostToDevice), "cudaMemcpy(weights)",
                   __FILE__, __LINE__);
  };
  // output-channel slices for the small-replay split (layers with at least 128 output channels)
  if (h.npad >= 128 && h.npad % 64 == 0 && !h.w_raster.empty() && h.w_raster.size() % ((size_t)h.npad * 8) == 0) {
    const int ways = 4, ns = h.npad / ways;
    const size_t rows = h.w_raster.size() / ((size_t)h.npad * 8);          // k*k * cin/8
    std::vector<__half> sp(h.w_raster.size());
    for (int sl = 0; sl < ways; ++sl)
      for (size_t r = 0; r < rows; ++r)
        for (int n = 0; n < ns; ++n)
          for (int j = 0; j < 8; ++j)
            sp[(((size_t)sl * rows + r) * ns + n) * 8 + j] = h.w_raster[(r * h.npad + (size_t)sl * ns + n) * 8 + j];
    if (!up((void **)&h.d_raster_split, sp.data(), sp.size() * 2)) return false;
    h.split_ways = ways;
  }
  return up((void **)&h.d_plain, h.w_plain.data(), h.w_plain.size() * 2) &&
         up((void **)&h.d_tiled, h.w_tiled.data(), h.w_tiled.size() * 2) &&
         up((void **)&h.d_raster, h.w_raster.data(), h.w_raster.size() * 2) &&
         up((void **)&h.d_bias, h.bias.data(), h.bias.size() * 4);
}

struct Tensor {            // channel-blocked planar PR layout (common.cuh)
  __half *p = nullptr;     // pixel 0 of plane 0
  long long pstride = 0;   // halfs between planes
  int H = 0, W = 0, C = 0;
  __half *pp = nullptr;    // parity-split twin (4 * C/8 planes of (H/2) x (W/2) rasters), or null
  long long pp_stride = 0;
  bool parity_only = false;  // the producer writes only the twin (every consumer reads the twin)
  std::vector<int> cmap;     // logical -> physical channel (ShuffleNetV2 stage buffers); empty = identity
};

struct Op {
  enum Kind { CONV, POOL, DW, SHUF } kind = CONV;
  DwParams dw{};
  ShuffleUnitParams su{};
  ConvParams cp{};
  bool raster = false;       // raster (halo-tile) kernel, else the per-tap gather kernel
  // Small replays (issue_replay): independent sub-graphs run on side streams.  `stream` 0 is the lane's own
  // stream; before the op its stream waits for event `wait`, after it the stream records event `signal`.
  int stream = 0, wait = -1, signal = -1;
  __half *pool_buf = nullptr;
  int pH = 0, pW = 0, pC = 0;
  long long pStride = 0;
};

DetOut det_out(uint8_t *blk, const ResultLayout &L) {
  return {L.at<int32_t>(blk, kNum), L.at<float>(blk, kBoxes), L.at<float>(blk, kScores), L.at<int32_t>(blk, kClasses),
          L.at<int32_t>(blk, kIndex)};
}

struct Lane {
  cudaStream_t stream = nullptr;
  cudaEvent_t done = nullptr;
  std::vector<void *> allocs;
  struct Raster { const __half *p; long long pstride; int planes, H, W; };   // every padded raster of the lane (normal layouts and parity twins)
  std::vector<Raster> rasters;
  std::map<std::string, Tensor> taps;
  std::vector<Op> ops;
  Tensor in8, stem_out;
  HeadPtrs heads{};
  NmsScratch nms{};
  uint8_t *results = nullptr;              // everything a replay hands back: irmv_engine::lane_res
  DetOut det{};                            // the detection fields of `results`
  const uint8_t **src_word = nullptr;      // device word: base pointer of the frames of this replay
  uint8_t *rotated = nullptr;
  std::map<int, cudaGraphExec_t> graphs;   // keyed by frames in the replay
  static constexpr int kSide = 9, kSig = 6;
  cudaStream_t side[kSide] = {};           // side streams of the branched schedule (index 0 unused)
  cudaEvent_t side_done[kSide] = {}, sig[kSig] = {};
  int launches_per_replay = 0;
  float *pnp_pts = nullptr;                // [S*max_det][8]
  double *pnp_rvec = nullptr, *pnp_tvec = nullptr;
  uint8_t *pnp_ok = nullptr;
  double *pnp_quat = nullptr;              // [S*max_det][4] tf2 quaternion (x, y, z, w) of the pose
  float *pnp_dist = nullptr;               // [S*max_det] distance_to_image_center
  float *pnp_centers = nullptr;            // [S*max_det][2] Armor::center in the calibration frame (armor stage only)
  const __half *kpt[3] = {nullptr, nullptr, nullptr};   // keypoint-branch outputs per scale (plane 0 = the 8 raw values)
  float *kpts = nullptr;                   // [S*max_det][8] decoded keypoints of the kept detections, network pixels
  ArmorOut *armors = nullptr;              // [S*max_det], allocated by irmv_engine_enable_armors
  uint32_t *armor_scratch = nullptr;       // per-CTA bitmaps of ROIs that do not fit in shared memory
  cudaEvent_t stage_ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

__global__ void set_src_kernel(const uint8_t **word, const uint8_t *ptr) { *word = ptr; }

// Debug (irmv_debug_check_padding): counts the pixels of one padded raster plane set that must be zero -- guard
// pixels, the zero row before every image and after the last, the zero column -- and are not.  Every kernel that
// writes activations relies on that padding being intact, so a stray store shows up here.
__global__ void __launch_bounds__(256) check_padding_kernel(const __half *p, long long pstride, int planes, int S, int H, int W,
                                                            unsigned long long *bad) {
  const long long real = pr_pixels(S, H, W), total = (long long)kGuardFront + real + kGuardBack;
  const int plane = blockIdx.y;
  const uint4 *base = reinterpret_cast<const uint4 *>(p + (long long)plane * pstride) - kGuardFront;
  unsigned long long n = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long q = i - kGuardFront;
    bool must_be_zero = q < 0 || q >= real;
    if (!must_be_zero) {
      const long long row = q / (W + 1);
      const int x = (int)(q - row * (W + 1));
      must_be_zero = x == W || row % (H + 1) == 0;
    }
    if (must_be_zero) {
      const uint4 v = base[i];
      n += (v.x | v.y | v.z | v.w) != 0u;
    }
  }
  if (n) atomicAdd(bad, n);
  (void)planes;
}

// Detections -> PnP corner quads {LB, LT, RT, RB} (reference order, src/pnp_solver.cpp:41-44).
// Until the light-bar extractor (reference src/irm_detector.cpp:292-355) is on the GPU the four
// corners are the box corners, scaled from network pixels to the calibration frame.
__global__ void quads_from_dets_kernel(const int32_t *num, const float *boxes, int n, int max_det,
                                       float sx, float sy, float px, float py, float *pts) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * max_det) return;
  int f = i / max_det, k = i - f * max_det;
  float4 b = make_float4(150.f + px, 140.f + py, 200.f + px, 160.f + py);     // inactive slots: a fixed valid quad
  if (k < num[f]) b = reinterpret_cast<const float4 *>(boxes)[i];
  float x1 = (b.x - px) * sx, y1 = (b.y - py) * sy, x2 = (b.z - px) * sx, y2 = (b.w - py) * sy;
  float4 *o = reinterpret_cast<float4 *>(pts + (size_t)i * 8);
  o[0] = make_float4(x1, y2, x1, y1);
  o[1] = make_float4(x2, y1, x2, y2);
}

// Keypoint branch (ultralytics Pose, kpt_shape [4, 2]): for every kept detection, the 8 raw values at
// its anchor -> (raw * 2 + grid) * stride, network pixels (oracle/yolov8n_ref.decode_keypoints).
// index = flat anchor * nc + class, anchors scale-major 80x80 | 40x40 | 20x20.
__global__ void kpts_from_dets_kernel(const int32_t *num, const int32_t *index, int n, int max_det, int nc,
                                      const __half *k0, const __half *k1, const __half *k2, float *kpts) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * max_det) return;
  const int f = i / max_det, k = i - f * max_det;
  float4 lo = make_float4(0.f, 0.f, 0.f, 0.f), hi = lo;
  if (k < num[f]) {
    int a = index[i] / nc;
    const __half *base = k0;
    int hw = 80;
    float stride = 8.f;
    if (a >= 8000) { a -= 8000; base = k2; hw = 20; stride = 32.f; }
    else if (a >= 6400) { a -= 6400; base = k1; hw = 40; stride = 16.f; }
    const int gy = a / hw, gx = a - gy * hw;
    const uint4 raw = *reinterpret_cast<const uint4 *>(base + pr_index(f, gy, gx, hw, hw) * 8);
    const __half2 *h = reinterpret_cast<const __half2 *>(&raw);
    float v[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 p = __half22float2(h[j]);
      v[2 * j] = __fmul_rn(__fadd_rn(__fmul_rn(p.x, 2.f), (float)gx), stride);
      v[2 * j + 1] = __fmul_rn(__fadd_rn(__fmul_rn(p.y, 2.f), (float)gy), stride);
    }
    lo = make_float4(v[0], v[1], v[2], v[3]);
    hi = make_float4(v[4], v[5], v[6], v[7]);
  }
  float4 *o = reinterpret_cast<float4 *>(kpts + (size_t)i * 8);
  o[0] = lo; o[1] = hi;
}

// Keypoints -> PnP quads (the four keypoints are the armor corners in PnPSolver's order LB, LT, RT, RB,
// reference src/pnp_solver.cpp:41-44), scaled from network pixels to the calibration frame.
__global__ void quads_from_kpts_kernel(const int32_t *num, const float *kpts, int n, int max_det, float sx, float sy,
                                       float px, float py, float *pts) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * max_det) return;
  const int f = i / max_det, k = i - f * max_det;
  float q[8] = {150.f, 160.f, 150.f, 140.f, 200.f, 140.f, 200.f, 160.f};    // inactive slots: a fixed valid quad
  if (k < num[f]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      q[2 * j] = (kpts[(size_t)i * 8 + 2 * j] - px) * sx;
      q[2 * j + 1] = (kpts[(size_t)i * 8 + 2 * j + 1] - py) * sy;
    }
  }
  float4 *o = reinterpret_cast<float4 *>(pts + (size_t)i * 8);
  o[0] = make_float4(q[0], q[1], q[2], q[3]);
  o[1] = make_float4(q[4], q[5], q[6], q[7]);
}

}  // namespace
}  // namespace irmv

using namespace irmv;

constexpr int kSets = 3;    // batches in flight in the pipelined hand-off

struct irmv_engine {
  irmv_engine_config cfg{};
  int nc = IRMV_NUM_CLASSES;
  int num_sms = 148;
  int S = 1, L = 1;
  size_t frame_bytes = 0;
  std::vector<std::unique_ptr<HostConv>> convs;
  int arch = kArchYolov8n;
  std::vector<std::unique_ptr<HostDw>> dws;       // depthwise convs of the ShuffleNetV2 backbone, execution order
  struct ShuffleUnit { int first_plane, runs; };  // planes a basic unit rewrites in place (ConvSeg::runs)
  std::vector<std::vector<ShuffleUnit>> sh_units; // per stage
  std::vector<std::vector<int>> sh_map;           // per stage: logical -> physical channel of the stage output
  // fused units (shuffle_unit.cu): one constant blob (shuffle_blob_layout) per unit of the stages it serves, in execution order
  std::vector<uint8_t *> sh_blobs;
  bool up_split = true;                           // 1x1 over concat(upsample(a), b) as two raster launches (HostConv::up_a / up_b)
  bool sh_fused = true;                           // cfg.reserved[2] != 0: one launch per conv instead (unfused reference path)
  std::vector<Lane> lanes;
  cudaStream_t main_stream = nullptr;
  cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
  std::vector<uint8_t *> slots_host;      // pinned
  uint8_t *slot_dev = nullptr;            // device copy of the frame being detected
  uint8_t *batch_dev = nullptr;           // staging for host-resident batches
  ResultLayout lane_res, res;             // result block of a lane (S frames) and of a pinned set (max_batch frames)
  // Pipelined hand-off (irmv_engine_submit_batch / _collect): three result sets so that the H2D copy
  // of batch k+1 (copy stream) runs under the kernels of batch k while the host still parses batch k-1 -- the B200 form of the
  // reference's camera/detector overlap through its TripleBuffer (reference README.md:60-63).
  struct Set {
    uint8_t *res_host = nullptr;          // pinned results of this set
    uint8_t *batch_dev = nullptr;         // device staging of this set's frames
    cudaEvent_t done = nullptr;           // all lanes finished (results in res_host)
    std::vector<cudaEvent_t> h2d;         // per chunk: frames arrived on the device
    int n = 0;
    long long ticket = -1;                // ticket whose results the set holds (-1: a synchronous call / nothing)
    bool in_flight = false;               // submitted and not yet collected
  } sets[kSets];
  cudaStream_t copy_stream = nullptr;
  long long next_ticket = 0;
  double profile_ms = 0.0, device_ms = 0.0;
  bool pnp_on = false;
  bool fused_stem = true;               // preprocess + conv0 in one kernel (input never materialised)
  float *d_stem_w = nullptr, *d_stem_b = nullptr;
  uint32_t *d_stem_tab = nullptr;        // table block of the camera-case stem (stem_bayer.cu), or null
  PnpConsts pnp_c{};
  float net_sx = 1.f, net_sy = 1.f, net_px = 0.f, net_py = 0.f;   // network -> source pixels: (v - p) * s (parse_output)
  float pnp_sx = 1.f, pnp_sy = 1.f, pnp_px = 0.f, pnp_py = 0.f;
  float corner_sx = 1.f, corner_sy = 1.f;   // source pixels -> calibration frame (irmv_engine_enable_pnp)
  bool pose = false;                        // the weight file holds the keypoint branch (72 convs)
  bool armors_on = false;                   // light-bar extraction between NMS and PnP
  irmv_armor_params armor_prm{};
  int last_slot = -1;
  int last_n = 0;
  // get_rotated_image(): address-stable pinned buffers (one per source slot) refreshed by every
  // detect() once enabled -- the reference's cv::Mat is a view of the buffer its graph rotates in
  // place (include/irmv_detection/yolo_engine.hpp:34, src/yolo_engine.cpp:182-184)
  bool rotated_on = false;
  uint8_t *rot_dev = nullptr;
  std::vector<uint8_t *> rot_host;
  std::vector<char> rot_valid;
  std::vector<irmv_bbox> parse_tmp;        // detect(): max_det boxes, sized once
  unsigned long long h2d_bytes = 0, d2h_bytes = 0;   // bytes of every host<->device copy queued so far
};

namespace {

bool lane_alloc(Lane &ln, void **p, size_t bytes) {
  if (!cuda_ok(dev_malloc(p, bytes), "dev_malloc(activation)", __FILE__, __LINE__)) return false;
  ln.allocs.push_back(*p);
  return cuda_ok(cudaMemset(*p, 0, bytes), "cudaMemset", __FILE__, __LINE__);
}

bool new_tensor(Lane &ln, int S, int H, int W, int C, Tensor &t, const char *tap = nullptr) {
  t.H = H; t.W = W; t.C = C;
  // C/8 zeroed planes of [guard | PR raster | guard] pixels x 8 channels
  // planes start on 128-byte boundaries (8 pixels): the raster kernel's bulk copies rely on it
  const size_t plane_px = ((size_t)kGuardFront + (size_t)pr_pixels(S, H, W) + kGuardBack + 7) & ~(size_t)7;
  t.pstride = (long long)plane_px * 8;
  __half *base = nullptr;
  if (!lane_alloc(ln, (void **)&base, (size_t)(C / 8) * plane_px * 16)) return false;
  t.p = base + (size_t)kGuardFront * 8;
  ln.rasters.push_back({t.p, t.pstride, C / 8, H, W});
  if (tap) ln.taps[tap] = t;
  return true;
}

// Parity-split twin of `t` (written by t's producer next to the normal layout, read by a
// stride-2 consumer running on the raster kernel; ConvParams in common.cuh).
bool add_parity_twin(Lane &ln, int S, Tensor &t, bool only) {
  t.parity_only = only;
  const size_t plane_px = ((size_t)kGuardFront + (size_t)pr_pixels(S, t.H / 2, t.W / 2) + kGuardBack + 7) & ~(size_t)7;
  t.pp_stride = (long long)plane_px * 8;
  __half *base = nullptr;
  if (!lane_alloc(ln, (void **)&base, (size_t)(4 * (t.C / 8)) * plane_px * 16)) return false;
  t.pp = base + (size_t)kGuardFront * 8;
  ln.rasters.push_back({t.pp, t.pp_stride, 4 * (t.C / 8), t.H / 2, t.W / 2});
  return true;
}

struct SegRef { const Tensor *t; int coff; int c; int up; };

void add_conv(irmv_engine *e, Lane &ln, HostConv &hc, std::vector<SegRef> in, int H, int W,
              const Tensor &out, int out_coff, const Tensor *res = nullptr, int res_coff = 0, int res_up = 0) {
  Op op;
  op.kind = Op::CONV;
  ConvParams &p = op.cp;
  p.nseg = (int)in.size();
  int cin = 0;
  for (int i = 0; i < p.nseg; ++i) {
    p.seg[i].ptr = in[i].t->p + (long long)(in[i].coff / 8) * in[i].t->pstride;
    p.seg[i].pstride = in[i].t->pstride;
    p.seg[i].c = in[i].c; p.seg[i].up = in[i].up;
    cin += in[i].c;
  }
  if (p.nseg == 1) p.seg[1] = p.seg[0];
  p.B = e->S; p.H = H; p.W = W;
  p.k = hc.k; p.stride = hc.stride; p.pad = hc.k / 2;
  p.OH = (H + 2 * p.pad - hc.k) / hc.stride + 1;
  p.OW = (W + 2 * p.pad - hc.k) / hc.stride + 1;
  p.cin = cin; p.cout = hc.cout; p.npad = hc.npad; p.K = hc.K; p.kpad = hc.kpad; p.act = hc.act;
  p.w_plain = hc.d_plain; p.w_tiled = hc.d_tiled; p.w_raster = hc.d_raster; p.bias = hc.d_bias;
  p.w_raster_split = hc.d_raster_split; p.split_ways = hc.split_ways;
  {
    // device tap table for this layer instance
    const int nq = hc.kpad / 8;
    std::vector<int32_t> tab((size_t)nq * 2, 0);
    for (int q = 0; q < nq; ++q) {
      int tap = hc.ktab[q * 3 + 0], sg = hc.ktab[q * 3 + 1], off = hc.ktab[q * 3 + 2];
      if (tap < 0) { tab[q * 2 + 0] = 0; tab[q * 2 + 1] = ktab_meta(0, 0, 0, 0); continue; }
      const ConvSeg &g = p.seg[sg];
      int ky = tap / hc.k, kx = tap % hc.k;
      tab[q * 2 + 0] = g.up ? 0 : (ky - p.pad) * (W + 1) + (kx - p.pad);   // pixel offset, PR pitch
      tab[q * 2 + 1] = ktab_meta(tap, sg, 1, off / 8);
    }
    int32_t *d = nullptr;
    dev_malloc((void **)&d, tab.size() * 4);
    cudaMemcpy(d, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice);
    ln.allocs.push_back(d);
    p.ktab = d;
  }
  p.out = out.p + (long long)(out_coff / 8) * out.pstride; p.out_pstride = out.pstride;
  p.res = res ? res->p + (long long)(res_coff / 8) * res->pstride : nullptr;
  p.res_pstride = res ? res->pstride : 0;
  p.res_up = res ? res_up : 0;
  p.sync_mode = 0;
  p.trace = nullptr; p.trace_cap = 0;
  p.in_parity = 0;
  p.out2 = nullptr; p.out2_pstride = 0;
  if (out.pp && out_coff == 0 && hc.cout == out.C) {
    p.out2 = out.pp; p.out2_pstride = out.pp_stride;
    if (out.parity_only) p.out = nullptr;
  }
  if (hc.stride == 2 && p.nseg == 1 && in[0].t->pp && in[0].coff == 0 && in[0].c == in[0].t->C &&
      !getenv("IRMV_NO_RASTER") && !getenv("IRMV_NO_S2_RASTER")) {
    ConvParams q = p;                       // try the raster kernel on the parity twin of the input
    q.in_parity = 1;
    q.seg[0].ptr = in[0].t->pp; q.seg[0].pstride = in[0].t->pp_stride;
    q.seg[1] = q.seg[0];
    if (conv_raster_fits(q)) p = q;
    else if (in[0].t->parity_only) fprintf(stderr, "irmv: internal: stride-2 consumer of a parity-only tensor does not fit the raster kernel\n");
  }
  op.raster = conv_raster_fits(p) && !getenv("IRMV_NO_RASTER");
  if (p.out2 && !op.raster) { p.out2 = nullptr; p.out = out.p; }   // conv0 as a stand-alone op: the stem kernel writes the twin
  ln.ops.push_back(op);
}

// C2f (ultralytics): cv1 -> split -> n bottlenecks chained on the last chunk -> cv2 over all chunks.
// All chunks live in one buffer so split and concat are channel offsets.
bool add_c2f(irmv_engine *e, Lane &ln, size_t &ci, std::vector<SegRef> in, int H, int W, int c2,
             int n, bool shortcut, Tensor &out, const char *tap, int parity_out = 0) {   // 1: twin only, 2: both layouts
  const int c = c2 / 2;
  Tensor buf, tmp;
  if (!new_tensor(ln, e->S, H, W, (2 + n) * c, buf) || !new_tensor(ln, e->S, H, W, c, tmp) ||
      !new_tensor(ln, e->S, H, W, c2, out, tap))
    return false;
  if (parity_out) {
    if (!add_parity_twin(ln, e->S, out, parity_out == 1)) return false;
    if (tap) ln.taps[tap] = out;
  }
  // cv1 of the neck C2f blocks reads concat(upsample(a), b).  A 1x1 conv commutes with nearest upsampling:
  // conv1x1(upsample(a)) == upsample(conv1x1(a)), so W_a runs at half resolution and its partial sum joins the
  // full-resolution accumulator in the epilogue, before the activation.  (Round 1 built this with the extra epilogue
  // state in EVERY instantiation: residual layers spilled and the replay got slower.  As its own template value --
  // conv_raster_kernel<.., RES = 2, ..> -- it takes m15.cv1 + m12.cv1 from 198 us on the gather kernel to about
  // 130 us on four raster launches per 128 frames.)
  HostConv &cv1 = *e->convs[ci++];
  bool split = false;
  if (cv1.up_a && in.size() == 2 && in[0].up && !in[1].up) {
    // cv1 over concat(upsample(a), b): W_a . a at a's resolution (no bias, no activation), then W_b . b at full
    // resolution with the upsampled partial sum added before the activation -- both on the raster kernel
    Tensor ya;
    if (!new_tensor(ln, e->S, H / 2, W / 2, cv1.cout, ya)) return false;
    add_conv(e, ln, *cv1.up_a, {{in[0].t, in[0].coff, in[0].c, 0}}, H / 2, W / 2, ya, 0);
    const bool ok_a = ln.ops.back().raster;
    add_conv(e, ln, *cv1.up_b, {in[1]}, H, W, buf, 0, &ya, 0, 1);
    if (ok_a && ln.ops.back().raster) split = true;
    else { ln.ops.pop_back(); ln.ops.pop_back(); }          // does not fit the raster kernel: the gather kernel does the concat
  }
  if (!split) add_conv(e, ln, cv1, in, H, W, buf, 0);
  for (int i = 0; i < n; ++i) {
    add_conv(e, ln, *e->convs[ci++], {{&buf, (1 + i) * c, c, 0}}, H, W, tmp, 0);
    add_conv(e, ln, *e->convs[ci++], {{&tmp, 0, c, 0}}, H, W, buf, (2 + i) * c,
             shortcut ? &buf : nullptr, (1 + i) * c);
  }
  add_conv(e, ln, *e->convs[ci++], {{&buf, 0, (2 + n) * c, 0}}, H, W, out, 0);
  return true;
}

// Fuse a pointwise (1x1, stride 1) conv into the raster conv that produces its only input: the
// producer keeps its FP16 output tile in shared memory as the A operand of a second GEMM
// (ConvParams::tail_*), so the intermediate tensor is neither written nor re-read and one launch
// disappears (m1 -> m2.cv1 and the Detect towers' 3x3 -> 1x1 pairs).  Only when nobody else reads
// the intermediate and the fused operands fit (conv_raster_fits decides).
void fuse_tails(irmv_engine *e, Lane &ln) {
  if (e->cfg.conv_impl == IRMV_CONV_DIRECT || e->cfg.reserved[1] || getenv("IRMV_NO_TAIL")) return;
  auto overlaps = [](const __half *a0, const __half *a1, const __half *b0, const __half *b1) { return a0 < b1 && b0 < a1; };
  for (size_t i = 0; i + 1 < ln.ops.size(); ++i) {
    Op &m = ln.ops[i];
    const Op &t = ln.ops[i + 1];
    if (m.kind != Op::CONV || t.kind != Op::CONV || !m.raster || !t.raster) continue;
    const ConvParams &tp = t.cp;
    ConvParams mp = m.cp;
    if (tp.k != 1 || tp.stride != 1 || tp.nseg != 1 || tp.res || tp.in_parity || tp.seg[0].up || tp.tail_w) continue;
    if (mp.out2 || mp.tail_w || !mp.out) continue;
    if (tp.seg[0].runs || tp.out_runs || mp.seg[0].runs || mp.out_runs) continue;   // ShuffleNetV2 in-place units
    // the tail reads [ext channels | this conv's output]: either exactly the output (ext = 0) or a
    // concat whose LAST chunk it is (C2f.cv2 right after the last bottleneck conv)
    const int ext = tp.seg[0].c - mp.cout;
    if (ext < 0 || tp.seg[0].pstride != mp.out_pstride) continue;
    if (tp.seg[0].ptr + (long long)(ext / 8) * tp.seg[0].pstride != mp.out) continue;
    if (tp.H != mp.OH || tp.W != mp.OW) continue;
    const __half *o0 = mp.out, *o1 = mp.out + (long long)(mp.cout / 8) * mp.out_pstride;
    bool other = false;
    for (size_t j = 0; j < ln.ops.size() && !other; ++j) {
      if (j == i || j == i + 1) continue;
      const Op &q = ln.ops[j];
      if (q.kind == Op::POOL) { other = overlaps(o0, o1, q.pool_buf, q.pool_buf + 4LL * (q.pC / 8) * q.pStride); continue; }
      if (q.kind == Op::DW) { other = overlaps(o0, o1, q.dw.in, q.dw.in + (long long)q.dw.planes * q.dw.in_ps); continue; }
      if (q.kind == Op::SHUF) { other = overlaps(o0, o1, q.su.in, q.su.in + (long long)(q.su.down ? q.su.cin / 8 : q.su.h / 4) * q.su.in_ps); continue; }
      for (int sgi = 0; sgi < q.cp.nseg; ++sgi) {
        const ConvSeg &g = q.cp.seg[sgi];
        if (!q.cp.in_parity && overlaps(o0, o1, g.ptr, g.ptr + (long long)(g.c / 8) * g.pstride)) other = true;
      }
      if (q.cp.res && overlaps(o0, o1, q.cp.res, q.cp.res + (long long)(q.cp.cout / 8) * q.cp.res_pstride)) other = true;
    }
    for (int h = 0; h < 3 && !other; ++h)
      if (ln.heads.box[h] == mp.out || ln.heads.cls[h] == mp.out) other = true;
    if (other) continue;
    mp.tail_w = tp.w_raster; mp.tail_bias = tp.bias; mp.tail_npad = tp.npad; mp.tail_cout = tp.cout; mp.tail_act = tp.act;
    mp.tail_out = tp.out; mp.tail_out_pstride = tp.out_pstride;
    mp.tail_out2 = tp.out2; mp.tail_out2_pstride = tp.out2_pstride;
    mp.tail_ext = tp.seg[0]; mp.tail_ext.c = ext;
    mp.out = nullptr;
    if (!conv_raster_fits(mp)) continue;
    m.cp = mp;
    if (t.signal >= 0) m.signal = t.signal;                   // the fused launch now produces what the tail produced
    for (auto it = ln.taps.begin(); it != ln.taps.end();)     // the intermediate is no longer materialised
      it = (it->second.p == o0) ? ln.taps.erase(it) : std::next(it);
    ln.ops.erase(ln.ops.begin() + (long)i + 1);
  }
}

bool build_lane(irmv_engine *e, Lane &ln) {
  const int S = e->S;
  if (!cuda_ok(cudaStreamCreateWithFlags(&ln.stream, cudaStreamNonBlocking), "cudaStreamCreate",
               __FILE__, __LINE__) ||
      !cuda_ok(cudaEventCreateWithFlags(&ln.done, cudaEventDisableTiming), "cudaEventCreate",
               __FILE__, __LINE__))
    return false;
  for (int i = 1; i < Lane::kSide; ++i)
    if (!cuda_ok(cudaStreamCreateWithFlags(&ln.side[i], cudaStreamNonBlocking), "cudaStreamCreate", __FILE__, __LINE__) ||
        !cuda_ok(cudaEventCreateWithFlags(&ln.side_done[i], cudaEventDisableTiming), "cudaEventCreate", __FILE__, __LINE__))
      return false;
  for (auto &ev : ln.sig)
    if (!cuda_ok(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming), "cudaEventCreate", __FILE__, __LINE__)) return false;
  if (!new_tensor(ln, S, kNet, kNet, kInC, ln.in8, "input")) return false;
  size_t ci = 0;
  Tensor t0, t1, x2, t3, x4, t5, x6, t7, x8, sp, x9, x12, x15, t16, x18, t19, x21;
  // stride-2 3x3 layers whose operands fit run on the raster kernel from parity-split twins of
  // their inputs (m1, m3, m5, m16); the producers write the twin next to the normal layout
  const bool par = e->cfg.conv_impl != IRMV_CONV_DIRECT && !getenv("IRMV_NO_RASTER") && !getenv("IRMV_NO_S2_RASTER");
  const bool fused = e->fused_stem && e->cfg.conv_impl != IRMV_CONV_DIRECT;
  // x4 / x15 also feed stride-1 consumers, so their producers would write both layouts (m5, m16)
  const bool par2 = par && getenv("IRMV_S2_DUAL");
  const bool shuffle = e->arch == kArchShuffleKpt;
  if (!new_tensor(ln, S, 320, 320, 16, t0, "m0")) return false;
  if (!shuffle && par && fused && !add_parity_twin(ln, S, t0, true)) return false;
  ln.taps["m0"] = t0;
  add_conv(e, ln, *e->convs[ci++], {{&ln.in8, 0, kInC, 0}}, 640, 640, t0, 0);
  ln.ops.back().cp.out2 = nullptr;                 // conv0 as a stand-alone op never writes the twin
  ln.stem_out = t0;
  if (shuffle) {
    // ShuffleNetV2-style backbone (weights.py shuffle_conv_specs).  A stage is ONE buffer X of cout channels:
    // the down unit writes its two branches into the two halves, every basic unit rewrites the planes of
    // its "right half" in place (engine->sh_units: runs of planes), and split / concat / shuffle are the
    // channel map folded into the weights at load time (irmv_engine_create).
    size_t di = 0, bi = 0;
    const Tensor *prev = &ln.stem_out;
    Tensor stage_out[4];
    int hw = 320;
    auto add_dw = [&](const HostDw &d, const Tensor &in, int in_plane0, int H, const Tensor &out) {
      Op op;
      op.kind = Op::DW;
      op.dw.in = in.p + (long long)in_plane0 * in.pstride; op.dw.in_ps = in.pstride;
      op.dw.out = out.p; op.dw.out_ps = out.pstride;
      op.dw.w = d.d_w; op.dw.bias = d.d_b;
      op.dw.planes = d.c / 8; op.dw.B = e->S; op.dw.H = H; op.dw.W = H; op.dw.stride = d.stride; op.dw.rev = 0;
      ln.ops.push_back(op);
    };
    for (int sgi = 0; sgi < 4; ++sgi) {
      const ShuffleStage &st = kShuffleStages[sgi];
      const int h = st.cout / 2, oh = hw / 2;
      Tensor X, Ta, Tb, Tc, T1, T2;
      char nm[8];
      snprintf(nm, sizeof nm, "d%d", sgi + 1);
      if (e->sh_fused && h <= kShuffleFuseMaxH) {
        // one kernel per unit (shuffle_unit.cu); basic units ping-pong between two stage buffers (their
        // depthwise conv reads a halo other CTAs may already have rewritten, so not in place)
        Tensor XB;
        if (!new_tensor(ln, S, oh, oh, st.cout, X) || (st.units && !new_tensor(ln, S, oh, oh, st.cout, XB))) return false;
        static const int th_force = getenv("IRMV_UNIT_TH") ? atoi(getenv("IRMV_UNIT_TH")) : 0;
        auto pick_th = [&](ShuffleUnitParams q) {                          // most rows per tile that still leave two CTAs per SM
          for (int th : {8, 4, 2}) {
            if (oh % th) continue;
            q.TH = th;
            if (th == th_force || (!th_force && shuffle_unit_ctas_per_sm(q) >= 2)) return th;
          }
          return 1;
        };
        Op op;
        op.kind = Op::SHUF;
        ShuffleUnitParams &q = op.su;
        q.down = 1; q.in = prev->p; q.in_ps = prev->pstride; q.out = X.p; q.out_ps = X.pstride;
        q.B = S; q.H = oh; q.W = oh; q.cin = st.cin; q.h = h; q.first_plane = 0; q.runs = 0;
        q.blob = e->sh_blobs[bi++];
        q.rev = 0; q.num_sms = e->num_sms;
        q.TH = pick_th(q);
        ln.ops.push_back(op);
        ci += 3; di += 2;
        Tensor *cur = &X, *oth = &XB;
        for (int u = 0; u < st.units; ++u) {
          const irmv_engine::ShuffleUnit &su = e->sh_units[sgi][u];
          const int run_planes = su.runs ? (1 << (su.runs - 1)) : h / 8;
          if (su.first_plane != run_planes) { set_error("internal: shuffle unit planes do not start one run in"); return false; }
          Op ob;
          ob.kind = Op::SHUF;
          ShuffleUnitParams &r = ob.su;
          r.down = 0; r.in = cur->p; r.in_ps = cur->pstride; r.out = oth->p; r.out_ps = oth->pstride;
          r.B = S; r.H = oh; r.W = oh; r.cin = h; r.h = h; r.first_plane = su.first_plane; r.runs = su.runs;
          r.blob = e->sh_blobs[bi++];
          r.rev = 0; r.num_sms = e->num_sms;
          r.TH = pick_th(r);
          ln.ops.push_back(ob);
          ci += 2; di += 1;
          std::swap(cur, oth);
        }
        X = *cur;                                                          // the buffer that holds the stage output
        X.cmap = e->sh_map[sgi];
        ln.taps[nm] = X;
      } else {
      if (!new_tensor(ln, S, oh, oh, st.cout, X) || !new_tensor(ln, S, oh, oh, st.cin, Ta) ||
          !new_tensor(ln, S, hw, hw, h, Tb) || !new_tensor(ln, S, oh, oh, h, Tc))
        return false;
      X.cmap = e->sh_map[sgi];
      ln.taps[nm] = X;
      add_dw(*e->dws[di++], *prev, 0, hw, Ta);                                              // b1.dw  (stride 2)
      add_conv(e, ln, *e->convs[ci++], {{&Ta, 0, st.cin, 0}}, oh, oh, X, 0);                // b1.pw  -> X[0, h)
      add_conv(e, ln, *e->convs[ci++], {{prev, 0, st.cin, 0}}, hw, hw, Tb, 0);              // b2.pw1
      add_dw(*e->dws[di++], Tb, 0, hw, Tc);                                                 // b2.dw  (stride 2)
      add_conv(e, ln, *e->convs[ci++], {{&Tc, 0, h, 0}}, oh, oh, X, h);                     // b2.pw2 -> X[h, 2h)
      if (st.units && (!new_tensor(ln, S, oh, oh, h, T1) || !new_tensor(ln, S, oh, oh, h, T2))) return false;
      for (int u = 0; u < st.units; ++u) {
        const irmv_engine::ShuffleUnit &su = e->sh_units[sgi][u];
        add_conv(e, ln, *e->convs[ci++], {{&X, su.first_plane * 8, h, 0}}, oh, oh, T1, 0);  // pw1: the unit's planes -> T1
        ln.ops.back().cp.seg[0].runs = su.runs; ln.ops.back().cp.seg[1].runs = su.runs;
        add_dw(*e->dws[di++], T1, 0, oh, T2);                                               // dw
        add_conv(e, ln, *e->convs[ci++], {{&T2, 0, h, 0}}, oh, oh, X, su.first_plane * 8);  // pw2: T2 -> the same planes
        ln.ops.back().cp.out_runs = su.runs;
      }
      }
      stage_out[sgi] = X;
      ln.taps[nm] = X;
      prev = &stage_out[sgi];
      hw = oh;
    }
    for (size_t k = 1; k < ln.ops.size(); ++k)
      if (ln.ops[k].kind == Op::CONV && !ln.ops[k].raster) { set_error("internal: a ShuffleNetV2 1x1 conv does not fit the raster kernel"); return false; }
    if (di != e->dws.size() || ci != 23) { set_error("internal: backbone conv count mismatch"); return false; }
    x4 = stage_out[1]; x6 = stage_out[2]; x8 = stage_out[3];
  } else {
  if (!new_tensor(ln, S, 160, 160, 32, t1, "m1")) return false;
  add_conv(e, ln, *e->convs[ci++], {{&t0, 0, 16, 0}}, 320, 320, t1, 0);
  if (!add_c2f(e, ln, ci, {{&t1, 0, 32, 0}}, 160, 160, 32, 1, true, x2, "m2", par ? 1 : 0)) return false;
  if (!new_tensor(ln, S, 80, 80, 64, t3, "m3")) return false;
  add_conv(e, ln, *e->convs[ci++], {{&x2, 0, 32, 0}}, 160, 160, t3, 0);
  if (!add_c2f(e, ln, ci, {{&t3, 0, 64, 0}}, 80, 80, 64, 2, true, x4, "m4", par2 ? 2 : 0)) return false;
  if (!new_tensor(ln, S, 40, 40, 128, t5, "m5")) return false;
  add_conv(e, ln, *e->convs[ci++], {{&x4, 0, 64, 0}}, 80, 80, t5, 0);
  if (!add_c2f(e, ln, ci, {{&t5, 0, 128, 0}}, 40, 40, 128, 2, true, x6, "m6")) return false;
  if (!new_tensor(ln, S, 20, 20, 256, t7, "m7")) return false;
  add_conv(e, ln, *e->convs[ci++], {{&x6, 0, 128, 0}}, 40, 40, t7, 0);
  if (!add_c2f(e, ln, ci, {{&t7, 0, 256, 0}}, 20, 20, 256, 1, true, x8, "m8")) return false;
  }
  // SPPF: cv1 -> [pool x3 into the next slices] -> cv2
  if (!new_tensor(ln, S, 20, 20, 512, sp) || !new_tensor(ln, S, 20, 20, 256, x9, "m9")) return false;
  add_conv(e, ln, *e->convs[ci++], {{&x8, 0, 256, 0}}, 20, 20, sp, 0);
  {
    Op op; op.kind = Op::POOL; op.pool_buf = sp.p; op.pH = 20; op.pW = 20; op.pC = 128; op.pStride = sp.pstride;
    ln.ops.push_back(op);
  }
  add_conv(e, ln, *e->convs[ci++], {{&sp, 0, 512, 0}}, 20, 20, x9, 0);
  // neck: upsample and concat happen in the consumers' gathers
  if (!add_c2f(e, ln, ci, {{&x9, 0, 256, 1}, {&x6, 0, 128, 0}}, 40, 40, 128, 1, false, x12, "m12")) return false;
  if (!add_c2f(e, ln, ci, {{&x12, 0, 128, 1}, {&x4, 0, 64, 0}}, 80, 80, 64, 1, false, x15, "m15", par2 ? 2 : 0)) return false;
  ln.ops.back().signal = 0;                        // P3 feature ready: its Detect / keypoint towers may start
  if (!new_tensor(ln, S, 40, 40, 64, t16, "m16")) return false;
  add_conv(e, ln, *e->convs[ci++], {{&x15, 0, 64, 0}}, 80, 80, t16, 0);
  if (!add_c2f(e, ln, ci, {{&t16, 0, 64, 0}, {&x12, 0, 128, 0}}, 40, 40, 128, 1, false, x18, "m18")) return false;
  ln.ops.back().signal = 1;                        // P4
  if (!new_tensor(ln, S, 20, 20, 128, t19, "m19")) return false;
  add_conv(e, ln, *e->convs[ci++], {{&x18, 0, 128, 0}}, 40, 40, t19, 0);
  if (!add_c2f(e, ln, ci, {{&t19, 0, 128, 0}, {&x9, 0, 256, 0}}, 20, 20, 256, 1, false, x21, "m21")) return false;
  ln.ops.back().signal = 2;                        // P5
  // Detect head: box.0|cls.0 merged (N=128), then the two towers
  const Tensor *feat[3] = {&x15, &x18, &x21};
  const int hw[3] = {80, 40, 20};
  for (int i = 0; i < 3; ++i) {
    Tensor h0, hb, hc, bo, co;
    char nb[8], ncn[8];
    snprintf(nb, sizeof nb, "box%d", i);
    snprintf(ncn, sizeof ncn, "cls%d", i);
    if (!new_tensor(ln, S, hw[i], hw[i], 128, h0) || !new_tensor(ln, S, hw[i], hw[i], 64, hb) ||
        !new_tensor(ln, S, hw[i], hw[i], 64, hc) || !new_tensor(ln, S, hw[i], hw[i], 64, bo, nb) ||
        !new_tensor(ln, S, hw[i], hw[i], kClsPad, co, ncn))
      return false;
    // branched schedule: scale i's towers start as soon as its feature exists (the P3 towers run beside the
    // rest of the neck); box and cls towers of a scale run side by side; P5's first conv stays on the trunk
    const int s_box = i < 2 ? 1 + 2 * i : 0, s_cls = i < 2 ? 2 + 2 * i : 5;
    add_conv(e, ln, *e->convs[ci++], {{feat[i], 0, feat[i]->C, 0}}, hw[i], hw[i], h0, 0);
    ln.ops.back().stream = s_box; ln.ops.back().wait = i; ln.ops.back().signal = 3 + i;
    add_conv(e, ln, *e->convs[ci++], {{&h0, 0, 64, 0}}, hw[i], hw[i], hb, 0);
    ln.ops.back().stream = s_box;
    add_conv(e, ln, *e->convs[ci++], {{&hb, 0, 64, 0}}, hw[i], hw[i], bo, 0);
    ln.ops.back().stream = s_box;
    add_conv(e, ln, *e->convs[ci++], {{&h0, 64, 64, 0}}, hw[i], hw[i], hc, 0);
    ln.ops.back().stream = s_cls; ln.ops.back().wait = 3 + i;
    add_conv(e, ln, *e->convs[ci++], {{&hc, 0, 64, 0}}, hw[i], hw[i], co, 0);
    ln.ops.back().stream = s_cls;
    ln.heads.box[i] = bo.p; ln.heads.box_ps[i] = bo.pstride;
    ln.heads.cls[i] = co.p; ln.heads.cls_ps[i] = co.pstride;
    ln.heads.padded = 1;
  }
  if (e->pose)
    for (int i = 0; i < 3; ++i) {          // keypoint branch: 3x3 ch->16, 3x3 16->16, 1x1 16->8 (padded to 16 planes-wise)
      Tensor k0, k1, ko;
      char nk[8];
      snprintf(nk, sizeof nk, "kpt%d", i);
      if (!new_tensor(ln, S, hw[i], hw[i], 16, k0) || !new_tensor(ln, S, hw[i], hw[i], 16, k1) ||
          !new_tensor(ln, S, hw[i], hw[i], 16, ko, nk))
        return false;
      add_conv(e, ln, *e->convs[ci++], {{feat[i], 0, feat[i]->C, 0}}, hw[i], hw[i], k0, 0);
      ln.ops.back().stream = 6 + i; ln.ops.back().wait = i;
      add_conv(e, ln, *e->convs[ci++], {{&k0, 0, 16, 0}}, hw[i], hw[i], k1, 0);
      ln.ops.back().stream = 6 + i;
      add_conv(e, ln, *e->convs[ci++], {{&k1, 0, 16, 0}}, hw[i], hw[i], ko, 0);
      ln.ops.back().stream = 6 + i;
      ln.kpt[i] = ko.p;
    }
  if (ci != e->convs.size()) { set_error("internal: conv count mismatch"); return false; }
  fuse_tails(e, ln);
  // decode / NMS scratch and outputs
  if (!lane_alloc(ln, (void **)&ln.nms.boxes, (size_t)S * kNumAnchors * 16) ||
      !lane_alloc(ln, (void **)&ln.nms.keys, (size_t)S * kNumAnchors * e->nc * 8) ||
      !lane_alloc(ln, (void **)&ln.nms.counts, (size_t)S * 4))
    return false;
  if (!lane_alloc(ln, (void **)&ln.src_word, sizeof(void *))) return false;
  const size_t slots = (size_t)S * e->cfg.max_det;
  // Everything a replay hands back lives in ONE device block per lane, laid out like the pinned result set.
  // When a replay covers the whole batch the copies back then merge into two or three cudaMemcpyAsync calls
  // instead of ten (each costs 5-10 us of stream time: 0.1 ms of a 4.6 ms step, and a tenth of the batch-1
  // detect() latency).
  const ResultLayout &R = e->lane_res;
  if (!lane_alloc(ln, (void **)&ln.results, R.bytes)) return false;
  ln.det = det_out(ln.results, R);
  ln.pnp_rvec = R.at<double>(ln.results, kRvec);
  ln.pnp_tvec = R.at<double>(ln.results, kTvec);
  ln.pnp_ok = R.at<uint8_t>(ln.results, kOk);
  ln.armors = R.at<ArmorOut>(ln.results, kArmors);
  ln.kpts = R.at<float>(ln.results, kKpts);
  ln.pnp_quat = R.at<double>(ln.results, kQuat);
  ln.pnp_dist = R.at<float>(ln.results, kDist);
  if (!lane_alloc(ln, (void **)&ln.pnp_pts, slots * 32) || !lane_alloc(ln, (void **)&ln.pnp_centers, slots * 8)) return false;
  for (auto &ev : ln.stage_ev)
    if (!cuda_ok(cudaEventCreate(&ev), "cudaEventCreate", __FILE__, __LINE__)) return false;
  Tensor bt; bt.p = reinterpret_cast<__half *>(ln.nms.boxes); bt.H = 1; bt.W = kNumAnchors; bt.C = 4; bt.pstride = 0;
  ln.taps["boxes"] = bt;
  return true;
}

// Enqueue one replay (n frames) of the whole pipeline on the lane stream.  With `stage_events`
// the lane's events are recorded between stages (profiling pass, never inside a graph).
int issue_replay(irmv_engine *e, Lane &ln, int n, cudaStream_t st, int *launches,
                 bool stage_events = false, std::vector<cudaEvent_t> *op_events = nullptr) {
  int cnt = 0;
  auto op_mark = [&]() {
    if (!op_events) return;
    cudaEvent_t ev = nullptr;
    cudaEventCreate(&ev);
    cudaEventRecord(ev, st);
    op_events->push_back(ev);
  };
  auto mark = [&](int i) -> int {
    if (stage_events) IRMV_CUDA(cudaEventRecord(ln.stage_ev[i], st));
    return 0;
  };
  if (mark(0)) return 1;
  PreprocessParams pp{};
  pp.src = nullptr; pp.src_indirect = ln.src_word; pp.dst = ln.in8.p; pp.rotated = ln.rotated;
  pp.n = n; pp.src_w = e->cfg.src_width; pp.src_h = e->cfg.src_height; pp.frame0 = 0;
  pp.chan_order = e->cfg.chan_order; pp.rotate180 = e->cfg.rotate180;
  pp.resize_mode = e->cfg.resize_mode; pp.quantize_u8 = e->cfg.quantize_u8;
  const bool fused = e->fused_stem && e->cfg.conv_impl != IRMV_CONV_DIRECT;
  if (fused) IRMV_CUDA(launch_stem(pp, e->d_stem_w, e->d_stem_b, e->d_stem_tab, ln.stem_out.parity_only ? nullptr : ln.stem_out.p, ln.stem_out.pstride, ln.stem_out.pp, ln.stem_out.pp_stride, st));
  else IRMV_CUDA(launch_preprocess(pp, st));
  cnt += 1 + (ln.rotated ? 1 : 0);
  if (mark(1)) return 1;
  op_mark();
  // Consecutive kernels walk their tiles in opposite directions (ConvParams::rev_tiles): a layer then
  // starts with the end of the tensor its producer has just finished writing, which is what the L2 still holds.
  static const bool pingpong = !getenv("IRMV_NO_PINGPONG");
  // Branched schedule for small replays: at batch 1 a Detect tower launch occupies 4-52 of the 148 SMs and the
  // replay is a chain of ~57 launch latencies, so the towers of a scale run on side streams next to the rest of the
  // neck and next to each other (fork / join by events; inside a CUDA graph these become parallel branches).  Measured
  // (scripts/ab_small.py, device time of a replay, one stream -> branched): 1 frame 392 -> 346 us, 8 frames 548 -> 525,
  // 64 frames 1438 -> 1411 (the towers fill the other launches' partial last waves); at 128 / 256 frames every launch
  // fills the machine and the two schedules time the same, so those stay on one stream.
  static const int branch_max = getenv("IRMV_BRANCH_MAX") ? atoi(getenv("IRMV_BRANCH_MAX")) : 64;
  const bool branched = n <= branch_max && !stage_events && !op_events && e->cfg.conv_impl != IRMV_CONV_DIRECT;
  unsigned side_used = 0;
  const cudaStream_t trunk = st;
  int seq = 0;
  bool first = true;
  for (auto &op : ln.ops) {
    if (first && fused) { first = false; continue; }        // conv0 ran inside the stem kernel
    first = false;
    ++seq;
    st = trunk;
    if (branched) {
      if (op.stream > 0) { st = ln.side[op.stream]; side_used |= 1u << op.stream; }
      if (op.wait >= 0) IRMV_CUDA(cudaStreamWaitEvent(st, ln.sig[op.wait], 0));
    }
    if (op.kind == Op::CONV) {
      ConvParams p = op.cp;
      p.B = n;
      p.rev_tiles = pingpong ? (seq & 1) : 0;
      if (e->cfg.conv_impl == IRMV_CONV_DIRECT) IRMV_CUDA(launch_conv_direct(p, st));
      else if (op.raster) IRMV_CUDA(launch_conv_raster(p, e->num_sms, st));
      else IRMV_CUDA(launch_conv_tc(p, e->num_sms, st));
    } else if (op.kind == Op::SHUF) {
      ShuffleUnitParams q = op.su;
      q.B = n;
      q.rev = pingpong ? (seq & 1) : 0;
      IRMV_CUDA(launch_shuffle_unit(q, st));
    } else if (op.kind == Op::DW) {
      DwParams d = op.dw;
      d.B = n;
      d.rev = pingpong ? (seq & 1) : 0;
      IRMV_CUDA(launch_dwconv3x3(d, st));
    } else {
      IRMV_CUDA(launch_sppf_pool(op.pool_buf, n, op.pH, op.pW, op.pStride, op.pC, st));
    }
    ++cnt;
    if (branched && op.signal >= 0) IRMV_CUDA(cudaEventRecord(ln.sig[op.signal], st));
    op_mark();
    if (getenv("IRMV_SYNC_EACH")) {
      cudaError_t ce = cudaStreamSynchronize(st);
      if (ce != cudaSuccess) {
        char buf[256];
        snprintf(buf, sizeof buf, "op %d (%s k=%d s=%d cin=%d cout=%d H=%d) failed: %s", cnt - 2,
                 op.kind == Op::POOL ? "pool" : (op.kind == Op::DW ? "dw" : (op.kind == Op::SHUF ? "shuffle-unit" : (op.raster ? "raster" : "gather"))), op.cp.k, op.cp.stride, op.cp.cin,
                 op.cp.cout, op.cp.H, cudaGetErrorString(ce));
        set_error(buf);
        return 1;
      }
    }
  }
  st = trunk;
  for (int i = 1; i < Lane::kSide; ++i)                      // join the side streams
    if (side_used & (1u << i)) {
      IRMV_CUDA(cudaEventRecord(ln.side_done[i], ln.side[i]));
      IRMV_CUDA(cudaStreamWaitEvent(st, ln.side_done[i], 0));
    }
  if (mark(2)) return 1;
  IRMV_CUDA(launch_decode(ln.heads, n, e->nc, e->cfg.score_thr, ln.nms, nullptr, st)); ++cnt;
  IRMV_CUDA(launch_nms(ln.nms, n, kNumAnchors, e->nc, e->cfg.iou_thr, e->cfg.max_det, ln.det, st)); ++cnt;
  if (e->pose) {
    const int total = n * e->cfg.max_det;
    kpts_from_dets_kernel<<<(total + 127) / 128, 128, 0, st>>>(ln.det.num_dets, ln.det.index, n, e->cfg.max_det, e->nc,
                                                              ln.kpt[0], ln.kpt[1], ln.kpt[2], ln.kpts);
    IRMV_CUDA(cudaGetLastError());
    ++cnt;
  }
  if (mark(3)) return 1;
  if (e->armors_on) {
    // reference message_callback: extract_armors(get_rotated_image(), bboxes), then solvePnP per armor
    // (src/irm_detector.cpp:183,204-208)
    ArmorParams ap{};
    ap.src = nullptr; ap.src_indirect = ln.src_word;
    ap.n = n; ap.src_w = e->cfg.src_width; ap.src_h = e->cfg.src_height;
    ap.chan_order = e->cfg.chan_order; ap.rotate180 = e->cfg.rotate180;
    ap.num = ln.det.num_dets; ap.boxes = ln.det.boxes; ap.scores = ln.det.scores; ap.classes = ln.det.classes;
    ap.max_det = e->cfg.max_det;
    ap.box_sx = e->net_sx; ap.box_sy = e->net_sy; ap.box_px = e->net_px; ap.box_py = e->net_py;   // parse()'s transform
    const irmv_armor_params &q = e->armor_prm;
    ap.binary_threshold = q.binary_threshold;
    ap.min_ratio = q.light_min_ratio; ap.max_ratio = q.light_max_ratio; ap.max_angle = q.light_max_angle;
    ap.min_small = q.min_small_center_distance; ap.max_small = q.max_small_center_distance;
    ap.min_large = q.min_large_center_distance; ap.max_large = q.max_large_center_distance;
    ap.out = ln.armors; ap.slot_locks = reinterpret_cast<int *>(ln.armor_scratch); ap.scratch = ln.armor_scratch + 64;
    ap.scratch_words_per_cta = armors_scratch_words_per_cta(e->cfg.src_width, e->cfg.src_height);
    ap.grid = armors_grid(e->num_sms);
    IRMV_CUDA(launch_extract_armors(ap, st)); ++cnt;
    if (e->pnp_on) {
      const int total = n * e->cfg.max_det;
      IRMV_CUDA(launch_quads_from_armors(ln.armors, total, e->corner_sx, e->corner_sy, ln.pnp_pts, ln.pnp_centers, st));
      PnpOut po{ln.pnp_rvec, ln.pnp_tvec, ln.pnp_ok, ln.pnp_quat, nullptr, nullptr, nullptr, ln.pnp_dist, ln.pnp_centers};
      IRMV_CUDA(launch_pnp(e->pnp_c, ln.pnp_pts, total, 0, po, st));
      IRMV_CUDA(launch_mask_pose_ok(ln.armors, total, ln.pnp_ok, st));
      cnt += 3;
    }
  } else if (e->pnp_on) {
    const int total = n * e->cfg.max_det;
    if (e->pose)    // the keypoints are the armor corners
      quads_from_kpts_kernel<<<(total + 127) / 128, 128, 0, st>>>(ln.det.num_dets, ln.kpts, n, e->cfg.max_det, e->pnp_sx,
                                                                 e->pnp_sy, e->pnp_px, e->pnp_py, ln.pnp_pts);
    else
      quads_from_dets_kernel<<<(total + 127) / 128, 128, 0, st>>>(ln.det.num_dets, ln.det.boxes, n, e->cfg.max_det,
                                                                 e->pnp_sx, e->pnp_sy, e->pnp_px, e->pnp_py, ln.pnp_pts);
    IRMV_CUDA(cudaGetLastError());
    PnpOut po{ln.pnp_rvec, ln.pnp_tvec, ln.pnp_ok, ln.pnp_quat, nullptr, nullptr, nullptr, ln.pnp_dist, nullptr};
    IRMV_CUDA(launch_pnp(e->pnp_c, ln.pnp_pts, total, 0, po, st));
    cnt += 2;
  }
  if (mark(4)) return 1;
  if (launches) *launches = cnt;
  return 0;
}

static_assert(sizeof(ArmorOut) == sizeof(irmv_armor) && sizeof(irmv_armor) == 56, "ArmorOut mirrors irmv_armor");

int run_replay(irmv_engine *e, Lane &ln, int n) {
  if (!e->cfg.use_graph) return issue_replay(e, ln, n, ln.stream, &ln.launches_per_replay);
  auto it = ln.graphs.find(n);
  if (it == ln.graphs.end()) {
    cudaGraph_t g = nullptr;
    cudaGraphExec_t ge = nullptr;
    // one eager pass first (function attributes, module load), like the reference's
    // enqueueV3 before capture (src/yolo_engine.cpp:100-101)
    if (int rc0 = issue_replay(e, ln, n, ln.stream, &ln.launches_per_replay)) return rc0;
    IRMV_CUDA(cudaStreamBeginCapture(ln.stream, cudaStreamCaptureModeThreadLocal));
    int rc = issue_replay(e, ln, n, ln.stream, &ln.launches_per_replay);
    cudaError_t ce = cudaStreamEndCapture(ln.stream, &g);
    if (rc) return rc;
    IRMV_CUDA(ce);
    IRMV_CUDA(cudaGraphInstantiate(&ge, g, 0));
    cudaGraphDestroy(g);
    it = ln.graphs.emplace(n, ge).first;
  }
  IRMV_CUDA(cudaGraphLaunch(it->second, ln.stream));
  return 0;
}

// frames_dev: device pointer to n contiguous frames.  Results land in sets[set].res_host (pinned).
// frames_host != null: the frames are still on the host; each chunk is copied on its lane's stream
// right before its replay, so the H2D of one lane overlaps the compute of the others.
int enqueue(irmv_engine *e, const uint8_t *frames_dev, int n, const uint8_t *frames_host = nullptr, int set = 0,
            bool copy_stream = false) {
  irmv_engine::Set &rs = e->sets[set];
  IRMV_CUDA(cudaEventRecord(e->ev_start, e->main_stream));
  // Pipelined host batches (submit_batch) are replayed in chunks of at most 128 frames: a chunk starts as soon as its
  // own frames have landed, under the copy of the next one.  Measured on 256-frame batches (end to end, frames/s):
  // one 256-frame replay 40.7-40.8 k, two chunks of 128 41.3-41.4 k (0.977 of the H2D ceiling), four of 64 37.6 k.
  static const int host_chunk = getenv("IRMV_HOST_CHUNK") ? atoi(getenv("IRMV_HOST_CHUNK")) : 128;
  const int S = (frames_host && copy_stream && host_chunk > 0 && host_chunk < e->S) ? host_chunk : e->S;
  const int chunks = (n + S - 1) / S;
  const int used = chunks < e->L ? chunks : e->L;
  unsigned fields = 1u << kNum | 1u << kBoxes | 1u << kScores | 1u << kClasses | 1u << kIndex;
  if (e->pnp_on) fields |= 1u << kRvec | 1u << kTvec | 1u << kOk | 1u << kQuat | 1u << kDist;
  if (e->armors_on) fields |= 1u << kArmors;
  if (e->pose) fields |= 1u << kKpts;
  // (pipelined submissions keep the lanes free-running: stream order already serialises a lane)
  if (!copy_stream)
    for (int l = 0; l < used; ++l) IRMV_CUDA(cudaStreamWaitEvent(e->lanes[l].stream, e->ev_start, 0));
  for (int c = 0; c < chunks; ++c) {
    Lane &ln = e->lanes[c % e->L];
    const int f0 = c * S, nf = (n - f0) < S ? (n - f0) : S;
    if (frames_host && copy_stream) {
      // all H2D copies go back to back on the copy stream; the lane only waits for its own chunk
      while ((int)rs.h2d.size() <= c) {
        cudaEvent_t ev = nullptr;
        IRMV_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        rs.h2d.push_back(ev);
      }
      // (alternating the chunks between two copy streams was measured on the 8-GPU box: no faster, the
      // link is saturated by one stream)
      cudaStream_t cs = e->copy_stream;
      IRMV_CUDA(cudaMemcpyAsync(const_cast<uint8_t *>(frames_dev) + (size_t)f0 * e->frame_bytes,
                                frames_host + (size_t)f0 * e->frame_bytes, (size_t)nf * e->frame_bytes,
                                cudaMemcpyHostToDevice, cs));
      e->h2d_bytes += (size_t)nf * e->frame_bytes;
      IRMV_CUDA(cudaEventRecord(rs.h2d[c], cs));
      IRMV_CUDA(cudaStreamWaitEvent(ln.stream, rs.h2d[c], 0));
    } else if (frames_host) {
      IRMV_CUDA(cudaMemcpyAsync(const_cast<uint8_t *>(frames_dev) + (size_t)f0 * e->frame_bytes,
                                frames_host + (size_t)f0 * e->frame_bytes, (size_t)nf * e->frame_bytes,
                                cudaMemcpyHostToDevice, ln.stream));
      e->h2d_bytes += (size_t)nf * e->frame_bytes;
    }
    set_src_kernel<<<1, 1, 0, ln.stream>>>(ln.src_word, frames_dev + (size_t)f0 * e->frame_bytes);
    IRMV_CUDA(cudaGetLastError());
    if (int rc = run_replay(e, ln, nf)) return rc;
    // results: the lane's block -> the slots of its frames in the pinned set
    static const bool merge = !getenv("IRMV_NO_D2H_MERGE");   // A/B knob
    const CopyPlan plan = plan_copies(e->lane_res, e->res, fields, (size_t)f0, (size_t)nf, merge);
    for (int i = 0; i < plan.n; ++i) {
      const CopyRange &r = plan.r[i];
      e->d2h_bytes += r.bytes;
      IRMV_CUDA(cudaMemcpyAsync(rs.res_host + r.host_off, ln.results + r.dev_off, r.bytes, cudaMemcpyDeviceToHost, ln.stream));
    }
  }
  for (int l = 0; l < used; ++l) {
    IRMV_CUDA(cudaEventRecord(e->lanes[l].done, e->lanes[l].stream));
    IRMV_CUDA(cudaStreamWaitEvent(e->main_stream, e->lanes[l].done, 0));
  }
  IRMV_CUDA(cudaEventRecord(e->ev_stop, e->main_stream));
  IRMV_CUDA(cudaEventRecord(rs.done, e->main_stream));
  rs.n = n;
  e->last_n = n;
  return 0;
}

// reference parse_output (src/yolo_engine.cpp:202-220)
void parse(irmv_engine *e, int n, irmv_bbox *out, int *counts, int set = 0) {
  const int md = e->cfg.max_det;
  const ResultLayout &R = e->res;
  const uint8_t *h = e->sets[set].res_host;
  const int32_t *num = R.at<const int32_t>(h, kNum), *cls = R.at<const int32_t>(h, kClasses);
  const float *boxes = R.at<const float>(h, kBoxes), *scores = R.at<const float>(h, kScores);
  const float sx = e->net_sx, sy = e->net_sy, px = e->net_px, py = e->net_py;
  for (int f = 0; f < n; ++f) {
    int k = num[f];
    if (counts) counts[f] = k;
    for (int i = 0; i < k; ++i) {
      const float *b = boxes + ((size_t)f * md + i) * 4;
      irmv_bbox &o = out[(size_t)f * md + i];
      o.xyxy[0] = (b[0] - px) * sx; o.xyxy[1] = (b[1] - py) * sy; o.xyxy[2] = (b[2] - px) * sx; o.xyxy[3] = (b[3] - py) * sy;
      o.score = scores[(size_t)f * md + i];
      int c = cls[(size_t)f * md + i];
      o.class_id = (c >= 0 && c < IRMV_NUM_CLASSES) ? c : IRMV_CLASS_UNKNOWN;
    }
  }
}

// rvec / tvec / ok of the first n frames of result set h
void copy_poses(const irmv_engine *e, const uint8_t *h, int n, double *rvecs, double *tvecs, uint8_t *ok) {
  const ResultLayout &R = e->res;
  memcpy(rvecs, h + R.offset[kRvec], (size_t)n * R.frame_bytes[kRvec]);
  memcpy(tvecs, h + R.offset[kTvec], (size_t)n * R.frame_bytes[kTvec]);
  if (ok) memcpy(ok, h + R.offset[kOk], (size_t)n * R.frame_bytes[kOk]);
}

// The synchronous entry points share set 0, lane 0's buffers and the main stream with the pipelined
// hand-off: they are refused while a submitted batch has not been collected.
bool pipeline_busy(irmv_engine *e) {
  for (auto &st : e->sets)
    if (st.in_flight) { set_error("pipelined batches are in flight: collect them before a synchronous call"); return true; }
  return false;
}

// Refresh the rotated frame of `slot` from the device copy of the frame (slot_dev) on the main stream.
int refresh_rotated(irmv_engine *e, int slot) {
  PreprocessParams pp{};
  pp.src = e->slot_dev; pp.rotated = e->rot_dev; pp.n = 1;
  pp.src_w = e->cfg.src_width; pp.src_h = e->cfg.src_height; pp.chan_order = e->cfg.chan_order;
  pp.rotate180 = e->cfg.rotate180;
  IRMV_CUDA(launch_rotate(pp, e->main_stream));
  IRMV_CUDA(cudaMemcpyAsync(e->rot_host[slot], e->rot_dev, (size_t)e->cfg.src_width * e->cfg.src_height * 3,
                            cudaMemcpyDeviceToHost, e->main_stream));
  e->d2h_bytes += (size_t)e->cfg.src_width * e->cfg.src_height * 3;
  e->rot_valid[slot] = 1;
  return 0;
}

}  // namespace

// =============================================================================== C ABI
extern "C" {

const char *irmv_last_error(void) { return g_err.c_str(); }

int irmv_chan_order_from_media_type(uint32_t t) {
  switch (t) {
    case IRMV_MV_MEDIA_TYPE_BAYRG8: return IRMV_CH_BAYER_RGGB;
    case IRMV_MV_MEDIA_TYPE_BAYGR8: return IRMV_CH_BAYER_GRBG;
    case IRMV_MV_MEDIA_TYPE_BAYGB8: return IRMV_CH_BAYER_GBRG;
    case IRMV_MV_MEDIA_TYPE_BAYBG8: return IRMV_CH_BAYER_BGGR;
    case IRMV_MV_MEDIA_TYPE_RGB8: return IRMV_CH_PASSTHROUGH;     // the reference feeds the ISP's RGB8 as is
    case IRMV_MV_MEDIA_TYPE_BGR8: return IRMV_CH_SWAP_RB;
    default: return -1;
  }
}
int irmv_version(void) { return 100; }

int irmv_engine_config_default(irmv_engine_config *c) {
  if (!c) return 1;
  memset(c, 0, sizeof *c);
  c->src_width = 1280; c->src_height = 1024;
  c->chan_order = IRMV_CH_PASSTHROUGH; c->rotate180 = 1; c->resize_mode = IRMV_RESIZE_STRETCH;
  c->quantize_u8 = 1; c->max_batch = 1; c->sub_batch = 0; c->num_lanes = 0; c->num_slots = 3;
  c->device = 0; c->conv_impl = IRMV_CONV_TCGEN05; c->max_det = 100;
  c->score_thr = 0.25f; c->iou_thr = 0.45f; c->use_graph = 1;
  return 0;
}

int irmv_engine_create(const char *weights_path, const irmv_engine_config *cfg, irmv_engine **out) {
  if (!weights_path || !cfg || !out) { set_error("null argument"); return 1; }
  IRMV_ABI_TRY
  if (cfg->max_batch < 1 || cfg->src_width < 2 || cfg->src_height < 2 || cfg->max_det < 1 || cfg->max_det > 1024) {
    set_error("bad engine config"); return 2;
  }
  int ndev = 0;
  IRMV_CUDA(cudaGetDeviceCount(&ndev));
  if (cfg->device < 0 || cfg->device >= ndev) { set_error("no such CUDA device"); return 3; }
  IRMV_CUDA(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  IRMV_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) { set_error("libirmv_b200 needs an sm_100 (Blackwell) GPU"); return 3; }
  std::unique_ptr<irmv_engine> e(new irmv_engine);
  e->cfg = *cfg;
  e->num_sms = prop.multiProcessorCount;
  std::vector<FileConv> fc;
  if (!read_weights(weights_path, e->nc, e->arch, fc)) return 4;
  if (e->nc != IRMV_NUM_CLASSES) { set_error("weight file is not an nc=14 detector"); return 4; }
  if (e->arch == kArchYolov8n && fc.size() != 63 && fc.size() != 72) { set_error("weight file is not YOLOv8n nc=14"); return 4; }
  e->pose = e->arch == kArchShuffleKpt || fc.size() == 72;    // + keypoint branch (kpt_shape [4, 2])
  if (!check_specs(fc, e->pose, e->arch)) return 4;            // make_conv / build_lane index by the expected shapes
  if (e->arch == kArchShuffleKpt && (cfg->conv_impl == IRMV_CONV_DIRECT || getenv("IRMV_NO_RASTER"))) {
    set_error("the ShuffleNetV2 variant runs on the tcgen05 raster kernel only"); return 2;
  }
  e->up_split = cfg->conv_impl != IRMV_CONV_DIRECT && cfg->reserved[3] == 0 && !getenv("IRMV_NO_RASTER") && !getenv("IRMV_NO_UP_SPLIT");
  // 63 reference convs -> 60 GEMMs (Detect box.0|cls.0 merged per scale)
  auto single = [&](size_t i, int cin_pad, std::vector<int> seg) {
    e->convs.emplace_back(new HostConv(make_conv({&fc[i]}, cin_pad, seg)));
  };
  auto single_p = [&](const FileConv &f, int cin_pad, std::vector<int> seg) {
    e->convs.emplace_back(new HostConv(make_conv({&f}, cin_pad, seg)));
  };
  size_t i = 0;
  single(i++, kInC, {kInC});                                   // m0: 3 -> 8 input channels
  size_t neck0 = 27;                                           // first neck conv (m12.cv1) in file order
  std::vector<int> inv4, inv6, inv8;                           // physical -> logical channel of x4 / x6 / x8 (empty: identity)
  if (e->arch == kArchYolov8n) {
    for (; i < 25; ++i) single(i, fc[i].cin, {fc[i].cin});     // m1 .. m8.cv2
  } else {
    // ShuffleNetV2 backbone: build every conv with the channel maps folded in (see permuted())
    neck0 = 38;
    std::vector<int> Lp;                                       // logical -> physical of the stage input (stem: identity)
    for (int c = 0; c < 16; ++c) Lp.push_back(c);
    auto inverse = [](const std::vector<int> &L) { std::vector<int> r(L.size()); for (size_t j = 0; j < L.size(); ++j) r[L[j]] = (int)j; return r; };
    for (const ShuffleStage &st : kShuffleStages) {
      const int h = st.cout / 2;
      const std::vector<int> pinv = inverse(Lp);               // physical -> logical of the stage input
      e->dws.emplace_back(new HostDw(make_dw(fc[i++], pinv)));                              // b1.dw on the input
      single_p(permuted(fc[i], pinv, {}), st.cin, {st.cin}); ++i;                           // b1.pw  -> X[0, h)
      single_p(permuted(fc[i], pinv, {}), st.cin, {st.cin}); ++i;                           // b2.pw1 -> Tb
      e->dws.emplace_back(new HostDw(make_dw(fc[i++], {})));                                // b2.dw
      single(i, h, {h}); ++i;                                                               // b2.pw2 -> X[h, 2h)
      std::vector<int> L(2 * h);                               // shuffle of concat(b1, b2)
      for (int j = 0; j < h; ++j) { L[2 * j] = j; L[2 * j + 1] = h + j; }
      std::vector<irmv_engine::ShuffleUnit> units;
      for (int u = 0; u < st.units; ++u) {
        // x2 = logical [h, 2h): the physical planes it occupies, ascending
        std::vector<int> phys(L.begin() + h, L.end());
        std::sort(phys.begin(), phys.end());
        std::vector<int> planes;
        for (int j = 0; j < h; j += 8) {
          for (int q = 1; q < 8; ++q)
            if (phys[j + q] != phys[j] + q || phys[j] % 8) { set_error("internal: shuffle unit is not plane aligned"); return 6; }
          planes.push_back(phys[j] / 8);
        }
        int run = 1;
        while (run < (int)planes.size() && planes[run] == planes[0] + run) ++run;
        int runs = 0;
        if (run < (int)planes.size()) { runs = 1; while ((1 << (runs - 1)) < run) ++runs; }
        for (size_t q = 0; q < planes.size(); ++q)
          if (planes[q] != planes[0] + run_plane((int)q, runs)) { set_error("internal: shuffle unit planes are not regular runs"); return 6; }
        units.push_back({planes[0], runs});
        const std::vector<int> Linv = inverse(L);
        std::vector<int> m(h);                                 // physical position in the slice -> logical index inside x2 / b
        for (int j = 0; j < h; ++j) m[j] = Linv[planes[j / 8] * 8 + j % 8] - h;
        single_p(permuted(fc[i], m, {}), h, {h}); ++i;                                      // pw1: x2 -> T1
        e->dws.emplace_back(new HostDw(make_dw(fc[i++], {})));                              // dw:  T1 -> T2
        single_p(permuted(fc[i], {}, m), h, {h}); ++i;                                      // pw2: T2 -> x2's planes
        std::vector<int> Ln(2 * h);                            // b[j] sits where x2[j] was; shuffle(concat(x1, b))
        for (int j = 0; j < h; ++j) { Ln[2 * j] = L[j]; Ln[2 * j + 1] = L[h + j]; }
        L = Ln;
      }
      e->sh_units.push_back(units);
      e->sh_map.push_back(L);
      Lp = L;
    }
    inv4 = inverse(e->sh_map[1]); inv6 = inverse(e->sh_map[2]); inv8 = inverse(e->sh_map[3]);
  }
  if (i != neck0 - 2) { set_error("internal: backbone conv count mismatch"); return 6; }
  // SPPF + neck (file order from m9.cv1 on is the same for both architectures)
  {
    const size_t b9 = neck0 - 2;
    if (inv8.empty()) single(b9, fc[b9].cin, {fc[b9].cin}); else single_p(permuted(fc[b9], inv8, {}), fc[b9].cin, {fc[b9].cin});
    single(b9 + 1, fc[b9 + 1].cin, {fc[b9 + 1].cin});
    for (size_t k = 0; k < 18; ++k) {
      const size_t fi = neck0 + k;
      int cin = fc[fi].cin;
      std::vector<int> seg{cin};
      std::vector<int> in_map;
      // concat-on-read layers: first conv of m12, m15, m18, m21 (cv1 over two sources)
      if (k == 0) { seg = {256, 128}; if (!inv6.empty()) { for (int c = 0; c < 256; ++c) in_map.push_back(c); for (int c : inv6) in_map.push_back(256 + c); } }
      if (k == 4) { seg = {128, 64}; if (!inv4.empty()) { for (int c = 0; c < 128; ++c) in_map.push_back(c); for (int c : inv4) in_map.push_back(128 + c); } }
      if (k == 9) seg = {64, 128};
      if (k == 14) seg = {128, 256};
      const FileConv f = in_map.empty() ? fc[fi] : permuted(fc[fi], in_map, {});
      single_p(f, cin, seg);
      if ((k == 0 || k == 4) && e->up_split) {               // m12.cv1 / m15.cv1: split over the upsampled half (add_c2f)
        HostConv &hc = *e->convs.back();
        const FileConv fa = slice_cin(f, 0, seg[0], false), fb = slice_cin(f, seg[0], cin, true);
        hc.up_a.reset(new HostConv(make_conv({&fa}, seg[0], {seg[0]})));
        hc.up_b.reset(new HostConv(make_conv({&fb}, seg[1], {seg[1]})));
      }
    }
  }
  const size_t head0 = neck0 + 18;
  for (int sc = 0; sc < 3; ++sc) {
    size_t b = head0 + (size_t)sc * 6;
    e->convs.emplace_back(new HostConv(make_conv({&fc[b + 0], &fc[b + 3]}, fc[b].cin, {fc[b].cin})));
    single(b + 1, 64, {64});
    single(b + 2, 64, {64});
    single(b + 4, 64, {64});
    single(b + 5, 64, {64});
  }
  if (e->pose)
    for (int sc = 0; sc < 3; ++sc) {
      size_t b = head0 + 18 + (size_t)sc * 3;
      single(b + 0, fc[b].cin, {fc[b].cin});
      single(b + 1, 16, {16});
      single(b + 2, 16, {16});
    }
  e->sh_fused = e->arch == kArchShuffleKpt && cfg->reserved[2] == 0 && !getenv("IRMV_NO_SHUFFLE_FUSE");
  if (e->sh_fused) {
    // convs[1 .. 22] are the backbone's 1x1 convs (3 per down unit: b1.pw, b2.pw1, b2.pw2; 2 per basic unit),
    // dws[] its depthwise convs (2 per down unit: b1.dw, b2.dw; 1 per basic unit), both in execution order
    size_t ci = 1, di = 0;
    auto put_pw = [&](std::vector<uint8_t> &blob, int off, const HostConv &hc, int boff, int h) {
      const int K = hc.cin_eff;
      __half *w = reinterpret_cast<__half *>(blob.data() + off);
      // every 1x1 of a unit ends in SiLU(x) = x/2 + x/2 * tanh(x/2): the 1/2 is folded into weights and bias (exact in FP16
      // short of subnormals), so the kernel's accumulator is x/2 already
      for (int n = 0; n < h; ++n)
        for (int c = 0; c < K; ++c) w[(size_t)n * (K + 8) + c] = __float2half(0.5f * __half2float(hc.w_plain[(size_t)n * hc.kpad + c]));
      float *bb = reinterpret_cast<float *>(blob.data() + boff);
      for (int n = 0; n < h; ++n) bb[n] = 0.5f * hc.bias[n];
    };
    auto put_dw = [&](std::vector<uint8_t> &blob, int off, const HostDw &d, int boff) {
      // d.w is [planes][9 taps][8 channels] FP16 -> [planes][10][8] words, the weight in the half of its channel parity
      uint32_t *w = reinterpret_cast<uint32_t *>(blob.data() + off);
      const int planes = d.c / 8;
      for (int p = 0; p < planes; ++p)
        for (int t = 0; t < 9; ++t)
          for (int c = 0; c < 8; ++c) {
            uint16_t bits;
            const __half hv = d.w[((size_t)p * 9 + t) * 8 + c];
            memcpy(&bits, &hv, 2);
            w[(p * 10 + t) * 8 + c] = (c & 1) ? ((uint32_t)bits << 16) : (uint32_t)bits;
          }
      memcpy(blob.data() + boff, d.b.data(), d.b.size() * 4);
    };
    for (int sgi = 0; sgi < 4; ++sgi) {
      const ShuffleStage &st = kShuffleStages[sgi];
      const int h = st.cout / 2;
      const bool fuse = h <= kShuffleFuseMaxH;
      for (int u = -1; u < st.units; ++u) {
        const bool down = u < 0;
        if (fuse) {
          const int cin = down ? st.cin : h;
          const ShuffleBlobLayout L = shuffle_blob_layout(down, cin, h);
          std::vector<uint8_t> blob(L.bytes, 0);
          if (down) {
            put_pw(blob, L.wa, *e->convs[ci], L.bias + 2 * h * 4, h);
            put_pw(blob, L.w1, *e->convs[ci + 1], L.bias, h);
            put_pw(blob, L.w2, *e->convs[ci + 2], L.bias + h * 4, h);
            put_dw(blob, L.dwa, *e->dws[di], L.bias + 4 * h * 4);
            put_dw(blob, L.dw, *e->dws[di + 1], L.bias + 3 * h * 4);
          } else {
            put_pw(blob, L.w1, *e->convs[ci], L.bias, h);
            put_pw(blob, L.w2, *e->convs[ci + 1], L.bias + h * 4, h);
            put_dw(blob, L.dw, *e->dws[di], L.bias + 3 * h * 4);
          }
          uint8_t *d = nullptr;
          IRMV_CUDA(dev_malloc((void **)&d, blob.size()));
          IRMV_CUDA(cudaMemcpy(d, blob.data(), blob.size(), cudaMemcpyHostToDevice));
          e->sh_blobs.push_back(d);
        }
        ci += down ? 3 : 2;
        di += down ? 2 : 1;
      }
    }
  }
  for (auto &d : e->dws) {
    IRMV_CUDA(dev_malloc((void **)&d->d_w, d->w.size() * 2));
    IRMV_CUDA(dev_malloc((void **)&d->d_b, d->b.size() * 4));
    IRMV_CUDA(cudaMemcpy(d->d_w, d->w.data(), d->w.size() * 2, cudaMemcpyHostToDevice));
    IRMV_CUDA(cudaMemcpy(d->d_b, d->b.data(), d->b.size() * 4, cudaMemcpyHostToDevice));
  }
  for (auto &c : e->convs) {
    if (!upload(*c)) return 5;
    if (c->up_a && (!upload(*c->up_a) || !upload(*c->up_b))) return 5;
  }
  {
    // stem weights: conv0 as FP32 [16][9 taps][3] + bias
    const HostConv &c0 = *e->convs[0];
    std::vector<float> w(16 * 27), b(16);
    for (int n = 0; n < 16; ++n) {
      b[n] = c0.bias[n];
      for (int t = 0; t < 9; ++t)
        for (int c = 0; c < 3; ++c) w[n * 27 + t * 3 + c] = __half2float(c0.w_plain[(size_t)n * c0.kpad + t * kInC + c]);
    }
    IRMV_CUDA(dev_malloc((void **)&e->d_stem_w, w.size() * 4));
    IRMV_CUDA(dev_malloc((void **)&e->d_stem_b, b.size() * 4));
    IRMV_CUDA(cudaMemcpy(e->d_stem_w, w.data(), w.size() * 4, cudaMemcpyHostToDevice));
    IRMV_CUDA(cudaMemcpy(e->d_stem_b, b.data(), b.size() * 4, cudaMemcpyHostToDevice));
    e->fused_stem = cfg->reserved[0] == 0;
    PreprocessParams probe{};
    probe.src_w = cfg->src_width; probe.src_h = cfg->src_height; probe.chan_order = cfg->chan_order;
    probe.resize_mode = cfg->resize_mode; probe.quantize_u8 = cfg->quantize_u8;
    if (stem_bayer2x_applies(probe)) {
      const std::vector<uint32_t> tab = stem_bayer2x_tables(w.data(), b.data(), cfg->src_height, cfg->chan_order, cfg->rotate180);
      IRMV_CUDA(dev_malloc((void **)&e->d_stem_tab, tab.size() * 4));
      IRMV_CUDA(cudaMemcpy(e->d_stem_tab, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice));
    }
  }

  const bool bayer = cfg->chan_order >= 2;
  e->frame_bytes = (size_t)cfg->src_width * cfg->src_height * (bayer ? 1 : 3);
  // defaults from the bench sweeps: replays of up to 256 frames (a launch carries ~7 us of fixed cost whatever
  // its size, so one 256-frame replay beats two of 128 by 3 %); two lanes when the batch needs several replays
  e->S = cfg->sub_batch > 0 ? cfg->sub_batch : (cfg->max_batch < 256 ? cfg->max_batch : 256);
  if (e->S > cfg->max_batch) e->S = cfg->max_batch;
  int chunks = (cfg->max_batch + e->S - 1) / e->S;
  e->L = cfg->num_lanes > 0 ? cfg->num_lanes : (chunks < 2 ? chunks : 2);
  if (e->L > chunks) e->L = chunks;
  e->lane_res = ResultLayout(e->S, cfg->max_det);
  e->res = ResultLayout(cfg->max_batch, cfg->max_det);
  {
    // reference parse_output scales by (W/640, H/640) (src/yolo_engine.cpp:211-214); with LETTERBOX the
    // resized image sits at (pad_x, pad_y) and is new_w x new_h, so boxes are shifted back first
    int pad_x, pad_y, new_w, new_h;
    letterbox_geometry(cfg->src_width, cfg->src_height, cfg->resize_mode, &pad_x, &pad_y, &new_w, &new_h);
    e->net_sx = (float)cfg->src_width / new_w; e->net_sy = (float)cfg->src_height / new_h;
    e->net_px = (float)pad_x; e->net_py = (float)pad_y;
  }
  e->lanes.resize(e->L);
  IRMV_CUDA(cudaStreamCreateWithFlags(&e->main_stream, cudaStreamNonBlocking));
  IRMV_CUDA(cudaEventCreate(&e->ev_start));
  IRMV_CUDA(cudaEventCreate(&e->ev_stop));
  for (auto &ln : e->lanes) if (!build_lane(e.get(), ln)) return 6;
  int nslots = cfg->num_slots > 0 ? cfg->num_slots : 1;
  e->slots_host.resize(nslots, nullptr);
  for (auto &s : e->slots_host) {
    IRMV_CUDA(host_malloc((void **)&s, e->frame_bytes));
    memset(s, 0, e->frame_bytes);
  }
  IRMV_CUDA(dev_malloc((void **)&e->slot_dev, e->frame_bytes));
  IRMV_CUDA(host_malloc((void **)&e->sets[0].res_host, e->res.bytes));
  memset(e->sets[0].res_host, 0, e->res.bytes);
  IRMV_CUDA(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
  for (auto &st : e->sets) IRMV_CUDA(cudaEventCreateWithFlags(&st.done, cudaEventDisableTiming));
  e->rot_host.assign(nslots, nullptr);
  e->rot_valid.assign(nslots, 0);
  IRMV_CUDA(cudaDeviceSynchronize());
  *out = e.release();
  return 0;
  IRMV_ABI_CATCH
}

void irmv_engine_destroy(irmv_engine *e) {
  if (!e) return;
  cudaSetDevice(e->cfg.device);
  cudaDeviceSynchronize();
  for (auto &ln : e->lanes) {
    for (auto &g : ln.graphs) cudaGraphExecDestroy(g.second);
    for (void *p : ln.allocs) cudaFree(p);
    if (ln.rotated) cudaFree(ln.rotated);
    if (ln.stream) cudaStreamDestroy(ln.stream);
    if (ln.done) cudaEventDestroy(ln.done);
    for (auto ev : ln.stage_ev) if (ev) cudaEventDestroy(ev);
    for (auto st : ln.side) if (st) cudaStreamDestroy(st);
    for (auto ev : ln.side_done) if (ev) cudaEventDestroy(ev);
    for (auto ev : ln.sig) if (ev) cudaEventDestroy(ev);
  }
  for (auto &c : e->convs) {
    cudaFree(c->d_plain); cudaFree(c->d_tiled); cudaFree(c->d_raster); cudaFree(c->d_bias); cudaFree(c->d_raster_split);
    for (HostConv *u : {c->up_a.get(), c->up_b.get()})
      if (u) { cudaFree(u->d_plain); cudaFree(u->d_tiled); cudaFree(u->d_raster); cudaFree(u->d_bias); cudaFree(u->d_raster_split); }
  }
  for (auto &d : e->dws) { cudaFree(d->d_w); cudaFree(d->d_b); }
  for (uint8_t *b : e->sh_blobs) cudaFree(b);

  for (auto s : e->slots_host) cudaFreeHost(s);
  for (auto s : e->rot_host) if (s) cudaFreeHost(s);
  if (e->rot_dev) cudaFree(e->rot_dev);
  cudaFree(e->slot_dev);
  cudaFree(e->d_stem_w); cudaFree(e->d_stem_b); cudaFree(e->d_stem_tab);
  if (e->batch_dev) cudaFree(e->batch_dev);
  for (int i = 1; i < kSets; ++i)
    if (e->sets[i].batch_dev) cudaFree(e->sets[i].batch_dev);
  for (auto &st : e->sets) {
    if (st.res_host) cudaFreeHost(st.res_host);
    if (st.done) cudaEventDestroy(st.done);
    for (auto ev : st.h2d) cudaEventDestroy(ev);
  }
  if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
  cudaEventDestroy(e->ev_start); cudaEventDestroy(e->ev_stop);
  cudaStreamDestroy(e->main_stream);
  delete e;
}

uint8_t *irmv_engine_src_buffer(irmv_engine *e, int slot) {
  if (!e || slot < 0 || slot >= (int)e->slots_host.size()) { set_error("bad slot"); return nullptr; }
  return e->slots_host[slot];
}

int irmv_engine_detect(irmv_engine *e, int slot, irmv_bbox *out, int cap, int *n) {
  if (!e || !n || slot < 0 || slot >= (int)e->slots_host.size()) { set_error("bad argument"); return 1; }
  if (pipeline_busy(e)) return 5;
  auto t0 = std::chrono::high_resolution_clock::now();
  IRMV_CUDA(cudaSetDevice(e->cfg.device));
  IRMV_CUDA(cudaMemcpyAsync(e->slot_dev, e->slots_host[slot], e->frame_bytes, cudaMemcpyHostToDevice, e->main_stream));
  e->h2d_bytes += e->frame_bytes;
  if (int rc = enqueue(e, e->slot_dev, 1)) return rc;
  if (e->rotated_on) { if (int rc = refresh_rotated(e, slot)) return rc; }
  else if (!e->rot_valid.empty()) e->rot_valid[slot] = 0;
  IRMV_CUDA(cudaStreamSynchronize(e->main_stream));
  e->sets[0].ticket = -1;
  if ((int)e->parse_tmp.size() < e->cfg.max_det) e->parse_tmp.resize(e->cfg.max_det);   // once
  int k = 0;
  parse(e, 1, e->parse_tmp.data(), &k);
  *n = k < cap ? k : cap;
  if (out) memcpy(out, e->parse_tmp.data(), sizeof(irmv_bbox) * (size_t)*n);
  e->last_slot = slot;
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e->ev_start, e->ev_stop);
  e->device_ms = ms;
  auto t1 = std::chrono::high_resolution_clock::now();
  e->profile_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
  return 0;
}

int irmv_engine_enqueue_batch(irmv_engine *e, const uint8_t *frames_dev, int nframes) {
  if (!e || !frames_dev || nframes < 1 || nframes > e->cfg.max_batch) { set_error("bad argument"); return 1; }
  if (pipeline_busy(e)) return 5;
  IRMV_CUDA(cudaSetDevice(e->cfg.device));
  e->sets[0].ticket = -1;
  return enqueue(e, frames_dev, nframes);
}

int irmv_engine_sync(irmv_engine *e) {
  if (!e) return 1;
  IRMV_CUDA(cudaStreamSynchronize(e->main_stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e->ev_start, e->ev_stop);
  e->device_ms = ms;
  return 0;
}

int irmv_engine_fetch(irmv_engine *e, int nframes, irmv_bbox *out, int *counts) {
  if (!e || !out || nframes < 1 || nframes > e->cfg.max_batch) { set_error("bad argument"); return 1; }
  parse(e, nframes, out, counts);
  return 0;
}

int irmv_engine_detect_batch(irmv_engine *e, const uint8_t *frames, int on_device, int nframes,
                             irmv_bbox *out, int *counts) {
  if (!e || !frames || !out || nframes < 1 || nframes > e->cfg.max_batch) { set_error("bad argument"); return 1; }
  if (pipeline_busy(e)) return 5;
  auto t0 = std::chrono::high_resolution_clock::now();
  IRMV_CUDA(cudaSetDevice(e->cfg.device));
  e->sets[0].ticket = -1;
  const uint8_t *dev = frames;
  if (!on_device) {
    if (!e->batch_dev) IRMV_CUDA(dev_malloc((void **)&e->batch_dev, e->frame_bytes * (size_t)e->cfg.max_batch));
    e->sets[0].batch_dev = e->batch_dev;
    dev = e->batch_dev;
  }
  // host frames of a large batch take the pipelined route (copy stream, 128-frame chunks): the second chunk's copy
  // runs under the first chunk's kernels (256 Bayer frames: 10.7 -> 8.6 ms per call)
  const bool chunked = !on_device && nframes > 128 && e->S > 128;
  if (int rc = enqueue(e, dev, nframes, on_device ? nullptr : frames, 0, chunked)) return rc;
  if (int rc = irmv_engine_sync(e)) return rc;
  parse(e, nframes, out, counts);
  auto t1 = std::chrono::high_resolution_clock::now();
  e->profile_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
  return 0;
}

// Pipelined form of detect_batch for host-resident frames: submit returns as soon as the work is
// queued (H2D on the copy stream, kernels on the lanes, D2H of the results); collect waits for
// that batch and parses it.  Up to three batches may be in flight: submit(k+1) before collect(k) puts
// the copy of batch k+1 under the kernels of batch k, submit(k+2) keeps the copy engine busy while the
// host parses.  Tickets must be collected in order.
int irmv_engine_submit_batch(irmv_engine *e, const uint8_t *frames_host, int nframes, int *ticket) {
  if (!e || !frames_host || !ticket || nframes < 1 || nframes > e->cfg.max_batch) { set_error("bad argument"); return 1; }
  IRMV_CUDA(cudaSetDevice(e->cfg.device));
  const int set = (int)(e->next_ticket % kSets);
  irmv_engine::Set &rs = e->sets[set];
  if (rs.in_flight) {
    char buf[128];
    snprintf(buf, sizeof buf, "three batches are in flight: collect ticket %lld before submitting another", rs.ticket);
    set_error(buf);
    return 6;
  }
  if (!rs.res_host) {
    IRMV_CUDA(host_malloc((void **)&rs.res_host, e->res.bytes));
    memset(rs.res_host, 0, e->res.bytes);
  }
  if (!rs.batch_dev) {
    if (set == 0 && e->batch_dev) rs.batch_dev = e->batch_dev;
    else IRMV_CUDA(dev_malloc((void **)&rs.batch_dev, e->frame_bytes * (size_t)e->cfg.max_batch));
    if (set == 0) e->batch_dev = rs.batch_dev;
  }
  // the set's staging buffer and result block are free once its previous batch has finished
  IRMV_CUDA(cudaStreamWaitEvent(e->copy_stream, rs.done, 0));
  if (int rc = enqueue(e, rs.batch_dev, nframes, frames_host, set, true)) return rc;
  rs.ticket = e->next_ticket & 0x7fffffff;
  rs.in_flight = true;
  *ticket = (int)(e->next_ticket++ & 0x7fffffff);
  return 0;
}

int irmv_engine_collect(irmv_engine *e, int ticket, irmv_bbox *out, int *counts, double *rvecs, double *tvecs,
                        uint8_t *ok) {
  if (!e || !out) { set_error("bad argument"); return 1; }
  IRMV_CUDA(cudaSetDevice(e->cfg.device));
  if (ticket < 0) { set_error("bad ticket"); return 2; }
  const int set = ticket % kSets;
  irmv_engine::Set &rs = e->sets[set];
  if (rs.n < 1 || rs.ticket != ticket || !rs.in_flight) {
    set_error("this ticket is not in flight (never submitted, already collected, or its result set was reused)");
    return 2;
  }
  // tickets complete in submission order; an older uncollected ticket would be overtaken silently
  for (auto &o : e->sets)
    if (o.in_flight && o.ticket < rs.ticket) { set_error("collect tickets in submission order"); return 2; }
  IRMV_CUDA(cudaEventSynchronize(rs.done));
  rs.in_flight = false;
  parse(e, rs.n, out, counts, set);
  if (rvecs && tvecs && e->pnp_on) copy_poses(e, rs.res_host, rs.n, rvecs, tvecs, ok);
  return 0;
}

// Bytes of every host->device / device->host copy the engine has queued since it was created (bench.py
// reports the per-step difference as e2e.h2d_bytes_per_step / d2h_bytes_per_step).
int irmv_engine_copy_bytes(irmv_engine *e, unsigned long long *h2d, unsigned long long *d2h) {
  if (!e) return 1;
  if (h2d) *h2d = e->h2d_bytes;
  if (d2h) *d2h = e->d2h_bytes;
  return 0;
}

double irmv_engine_profile_ms(irmv_engine *e) { return e ? e->profile_ms : 0.0; }
double irmv_engine_last_device_ms(irmv_engine *e) { return e ? e->device_ms : 0.0; }
void *irmv_engine_stream(irmv_engine *e) { return e ? (void *)e->main_stream : nullptr; }

int irmv_engine_kernel_launches(irmv_engine *e, int nframes) {
  if (!e) return 0;
  int chunks = (nframes + e->S - 1) / e->S;
  return chunks * (e->lanes[0].launches_per_replay + 1);
}

// get_rotated_image() (reference include/irmv_detection/yolo_engine.hpp:34): the first call switches the
// engine to "rotated frames on": from then on every detect() also writes the rotated packed-RGB
// frame of its slot into an address-stable pinned buffer (one rotate kernel + one D2H on the main
// stream, no allocation, no re-upload), and this call is a pointer return.  The first call itself
// rotates the frame of the last detect() from the device copy that is still there.
int irmv_engine_rotated_view(irmv_engine *e, int slot, const uint8_t **view) {
  if (!e || !view || slot < 0 || slot >= (int)e->slots_host.size()) { set_error("bad argument"); return 1; }
  const size_t bytes = (size_t)e->cfg.src_width * e->cfg.src_height * 3;
  if (!e->rotated_on || !e->rot_host[slot] || !e->rot_valid[slot]) {
    if (pipeline_busy(e)) return 5;
    IRMV_CUDA(cudaSetDevice(e->cfg.device));
    if (!e->rot_dev) IRMV_CUDA(dev_malloc((void **)&e->rot_dev, bytes));
    for (auto &h : e->rot_host)
      if (!h) { IRMV_CUDA(host_malloc((void **)&h, bytes)); memset(h, 0, bytes); }
    e->rotated_on = true;
    if (e->last_slot != slot)      // the device copy holds another slot's frame: bring this one over
      IRMV_CUDA(cudaMemcpyAsync(e->slot_dev, e->slots_host[slot], e->frame_bytes, cudaMemcpyHostToDevice, e->main_stream));
    if (int rc = refresh_rotated(e, slot)) return rc;
    IRMV_CUDA(cudaStreamSynchronize(e->main_stream));
    e->last_slot = slot;
  }
  *view = e->rot_host[slot];
  return 0;
}

int irmv_engine_rotated_image(irmv_engine *e, int slot, uint8_t *dst) {
  if (!dst) { set_error("bad argument"); return 1; }
  const uint8_t *v = nullptr;
  if (int rc = irmv_engine_rotated_view(e, slot, &v)) return rc;
  memcpy(dst, v, (size_t)e->cfg.src_width * e->cfg.src_height * 3);
  return 0;
}

long long irmv_debug_alloc_count(void) { return g_allocs.load(); }

int irmv_debug_check_padding(irmv_engine *e, long long *bad_pixels) {
  IRMV_ABI_TRY
  if (!e || !bad_pixels) { set_error("null argument"); return 1; }
  IRMV_CUDA(cudaSetDevice(e->cfg.device));
  IRMV_CUDA(cudaDeviceSynchronize());
  unsigned long long *d = nullptr;
  IRMV_CUDA(cudaMalloc((void **)&d, 8));
  IRMV_CUDA(cudaMemset(d, 0, 8));
  for (const Lane &ln : e->lanes)
    for (const Lane::Raster &r : ln.rasters)
      check_padding_kernel<<<dim3(64, (unsigned)r.planes), 256>>>(r.p, r.pstride, r.planes, e->S, r.H, r.W, d);
  unsigned long long h = 0;
  const cudaError_t err = cudaMemcpy(&h, d, 8, cudaMemcpyDeviceToHost);
  cudaFree(d);
  IRMV_CUDA(err);
  *bad_pixels = (long long)h;
  return 0;
  IRMV_ABI_CATCH
}

int irmv_engine_read_tensor(irmv_engine *e, const char *name, void *dst, int64_t cap, int32_t dims[5]) {
  if (!e || !name || !dims) { set_error("bad argument"); return 1; }
  IRMV_CUDA(cudaSetDevice(e->cfg.device));
  Lane &ln = e->lanes[0];
  auto it = ln.taps.find(name);
  if (it == ln.taps.end()) { set_error(std::string("no tensor named ") + name); return 2; }
  const Tensor &t = it->second;
  const bool is_boxes = strcmp(name, "boxes") == 0;
  int es = is_boxes ? 4 : 2;
  int nb = e->last_n < e->S ? (e->last_n > 0 ? e->last_n : 1) : e->S;
  dims[0] = nb; dims[1] = t.H; dims[2] = t.W; dims[3] = t.C; dims[4] = es;
  int64_t bytes = (int64_t)nb * t.H * t.W * t.C * es;
  if (dst) {
    if (bytes > cap) { set_error("destination too small"); return 3; }
    IRMV_CUDA(cudaDeviceSynchronize());
    if (is_boxes) {
      IRMV_CUDA(cudaMemcpy(dst, t.p, (size_t)bytes, cudaMemcpyDeviceToHost));
    } else {
      // device tensors are channel-blocked planes in the padded raster layout: gather to dense NHWC
      const size_t px = (size_t)pr_pixels(nb, t.H, t.W);
      const int planes = t.C / 8;
      std::vector<uint16_t> tmp(px * 8);
      uint16_t *o = static_cast<uint16_t *>(dst);
      for (int pl = 0; pl < planes && !t.parity_only; ++pl) {
        IRMV_CUDA(cudaMemcpy(tmp.data(), t.p + (long long)pl * t.pstride, tmp.size() * 2, cudaMemcpyDeviceToHost));
        for (int b = 0; b < nb; ++b)
          for (int y = 0; y < t.H; ++y)
            for (int x = 0; x < t.W; ++x)
              memcpy(o + ((((size_t)b * t.H + y) * t.W + x) * t.C + pl * 8),
                     tmp.data() + (size_t)pr_index(b, y, x, t.H, t.W) * 8, 16);
      }
      if (!t.cmap.empty()) {             // ShuffleNetV2 stage buffer: physical channel order -> logical
        std::vector<uint16_t> px(t.C);
        for (size_t q = 0; q < (size_t)nb * t.H * t.W; ++q) {
          memcpy(px.data(), o + q * t.C, (size_t)t.C * 2);
          for (int c = 0; c < t.C; ++c) o[q * t.C + c] = px[t.cmap[c]];
        }
      }
      if (t.parity_only) {               // only the parity-split twin exists: planes [g][C/8] of (H/2) x (W/2)
        const size_t px2 = (size_t)pr_pixels(nb, t.H / 2, t.W / 2);
        tmp.resize(px2 * 8);
        for (int g = 0; g < 4; ++g)
          for (int pl = 0; pl < planes; ++pl) {
            IRMV_CUDA(cudaMemcpy(tmp.data(), t.pp + (long long)(g * planes + pl) * t.pp_stride, tmp.size() * 2, cudaMemcpyDeviceToHost));
            for (int b = 0; b < nb; ++b)
              for (int y = g >> 1; y < t.H; y += 2)
                for (int x = g & 1; x < t.W; x += 2)
                  memcpy(o + ((((size_t)b * t.H + y) * t.W + x) * t.C + pl * 8),
                         tmp.data() + (size_t)pr_index(b, y >> 1, x >> 1, t.H / 2, t.W / 2) * 8, 16);
          }
      }
    }
  }
  return 0;
}

int irmv_engine_read_kept_indices(irmv_engine *e, int frame, int32_t *idx, int cap, int *n) {
  if (!e || !idx || !n || frame < 0 || frame >= e->cfg.max_batch) { set_error("bad argument"); return 1; }
  const uint8_t *h = e->sets[0].res_host;
  const int k = e->res.at<const int32_t>(h, kNum)[frame];
  *n = k < cap ? k : cap;
  memcpy(idx, e->res.at<const int32_t>(h, kIndex) + (size_t)frame * e->cfg.max_det, (size_t)*n * 4);
  return 0;
}

int irmv_engine_enable_pnp(irmv_engine *e, const double K[9], const double D[5], float corner_sx, float corner_sy) {
  if (!e || !K || !D) { set_error("bad argument"); return 1; }
  e->pnp_c.fx = K[0]; e->pnp_c.cx = K[2]; e->pnp_c.fy = K[4]; e->pnp_c.cy = K[5];
  e->pnp_c.k1 = D[0]; e->pnp_c.k2 = D[1]; e->pnp_c.p1 = D[2]; e->pnp_c.p2 = D[3]; e->pnp_c.k3 = D[4];
  e->pnp_c.half_w[0] = 135.0 / 2.0 / 1000.0; e->pnp_c.half_h[0] = 55.0 / 2.0 / 1000.0;
  e->pnp_c.half_w[1] = 225.0 / 2.0 / 1000.0; e->pnp_c.half_h[1] = 55.0 / 2.0 / 1000.0;
  // boxes are in network pixels: first to the source frame (parse_output's scale), then to the calibration frame
  {
    int pad_x, pad_y, new_w, new_h;
    letterbox_geometry(e->cfg.src_width, e->cfg.src_height, e->cfg.resize_mode, &pad_x, &pad_y, &new_w, &new_h);
    e->pnp_sx = corner_sx * (float)e->cfg.src_width / (float)new_w;
    e->pnp_sy = corner_sy * (float)e->cfg.src_height / (float)new_h;
    e->pnp_px = (float)pad_x; e->pnp_py = (float)pad_y;
  }
  e->corner_sx = corner_sx; e->corner_sy = corner_sy;
  e->pnp_on = true;
  IRMV_CUDA(cudaSetDevice(e->cfg.device));
  IRMV_CUDA(cudaDeviceSynchronize());
  for (auto &ln : e->lanes) {             // the pipeline changed: drop captured graphs
    for (auto &g : ln.graphs) cudaGraphExecDestroy(g.second);
    ln.graphs.clear();
  }
  return 0;
}

int irmv_engine_fetch_poses(irmv_engine *e, int nframes, double *rvecs, double *tvecs, uint8_t *ok) {
  if (!e || !rvecs || !tvecs || nframes < 1 || nframes > e->cfg.max_batch) { set_error("bad argument"); return 1; }
  if (!e->pnp_on) { set_error("PnP stage not enabled"); return 2; }
  copy_poses(e, e->sets[0].res_host, nframes, rvecs, tvecs, ok);
  return 0;
}

// Result block of a finished call: ticket < 0 = the last synchronous call (set 0), else a collected
// pipelined batch whose set has not been reused yet.
static const uint8_t *result_block(irmv_engine *e, int ticket) {
  if (ticket < 0) {
    if (e->sets[0].ticket != -1) { set_error("set 0 holds a pipelined batch: pass its ticket"); return nullptr; }
    return e->sets[0].res_host;
  }
  const irmv_engine::Set &rs = e->sets[ticket % kSets];
  if (!rs.res_host || rs.ticket != ticket) { set_error("this ticket's results are gone (never submitted, or its result set was reused)"); return nullptr; }
  if (rs.in_flight) { set_error("collect the ticket first"); return nullptr; }
  return rs.res_host;
}

static_assert(sizeof(irmv_pose) == 88, "irmv_pose layout");
// The fields IrmDetector::message_callback fills per armor (reference src/irm_detector.cpp:213-230),
// straight from the fused replay: position = tvec, orientation = tf2 quaternion of Rodrigues(rvec),
// distance_to_image_center.  out: nframes*max_det entries, slot-aligned with the detections.
int irmv_engine_fetch_armor_poses(irmv_engine *e, int ticket, int nframes, irmv_pose *out) {
  if (!e || !out || nframes < 1 || nframes > e->cfg.max_batch) { set_error("bad argument"); return 1; }
  if (!e->pnp_on) { set_error("PnP stage not enabled"); return 2; }
  const uint8_t *h = result_block(e, ticket);
  if (!h) return 2;
  const size_t md = e->cfg.max_det;
  const ResultLayout &R = e->res;
  const double *rv = R.at<const double>(h, kRvec), *tv = R.at<const double>(h, kTvec), *q = R.at<const double>(h, kQuat);
  const uint8_t *ok = R.at<const uint8_t>(h, kOk);
  const float *d = R.at<const float>(h, kDist);
  const int32_t *num = R.at<const int32_t>(h, kNum);
  for (size_t f = 0; f < (size_t)nframes; ++f)
    for (size_t i = 0; i < md; ++i) {
      const size_t k = f * md + i;
      irmv_pose &o = out[k];
      for (int c = 0; c < 3; ++c) { o.position[c] = tv[k * 3 + c]; o.rvec[c] = rv[k * 3 + c]; }
      for (int c = 0; c < 4; ++c) o.orientation[c] = q[k * 4 + c];
      o.distance_to_image_center = d[k];
      o.ok = ((int)i < num[f] && ok[k]) ? 1 : 0;
    }
  return 0;
}

int irmv_armor_params_default(irmv_armor_params *p) {
  if (!p) return 1;
  // node parameter defaults, reference src/irm_detector.cpp:152,162-173
  p->binary_threshold = 150;
  p->light_min_ratio = 0.1f; p->light_max_ratio = 0.4f; p->light_max_angle = 40.0f;
  p->min_small_center_distance = 0.8; p->max_small_center_distance = 3.2;
  p->min_large_center_distance = 3.2; p->max_large_center_distance = 5.5;
  return 0;
}

int irmv_engine_enable_armors(irmv_engine *e, const irmv_armor_params *prm) {
  if (!e) { set_error("bad argument"); return 1; }
  if (prm) e->armor_prm = *prm; else irmv_armor_params_default(&e->armor_prm);
  IRMV_CUDA(cudaSetDevice(e->cfg.device));
  IRMV_CUDA(cudaDeviceSynchronize());
  const size_t slots = (size_t)e->S * e->cfg.max_det;
  const size_t words = armors_scratch_total_words(e->cfg.src_width, e->cfg.src_height, armors_grid(e->num_sms));
  for (auto &ln : e->lanes) {
    if (!ln.armor_scratch) {                                    // (the armor slots are part of the lane's result block)
      if (!lane_alloc(ln, (void **)&ln.armor_scratch, words * 4)) return 3;
      IRMV_CUDA(cudaMemset(ln.armors, 0, slots * sizeof(ArmorOut)));
      IRMV_CUDA(cudaMemset(ln.armor_scratch, 0, 256));         // slot locks
    }
    for (auto &g : ln.graphs) cudaGraphExecDestroy(g.second);   // the pipeline changed: drop captured graphs
    ln.graphs.clear();
  }
  e->armors_on = true;
  return 0;
}

int irmv_engine_fetch_armors(irmv_engine *e, int ticket, int nframes, irmv_armor *out) {
  if (!e || !out || nframes < 1 || nframes > e->cfg.max_batch) { set_error("bad argument"); return 1; }
  if (!e->armors_on) { set_error("armor stage not enabled"); return 2; }
  const uint8_t *h = result_block(e, ticket);
  if (!h) return 2;
  memcpy(out, h + e->res.offset[kArmors], (size_t)nframes * e->res.frame_bytes[kArmors]);
  return 0;
}

static thread_local double g_armors_ms = 0.0;
static thread_local unsigned long long g_armors_prof[8] = {0, 0, 0, 0, 0, 0, 0, 0};
double irmv_extract_armors_last_device_ms(void) { return g_armors_ms; }
// Debug: per-phase SM cycles of the last stand-alone call, summed over ROIs:
// {bitmap, flood, walks + lights, armor, ROIs processed, flood rounds, recording walks (warp cycles),
// hull + rectangle + light (warp cycles)}.  Collected only when the
// environment variable IRMV_ARMOR_PROF is set.
int irmv_extract_armors_last_profile(unsigned long long out[8]) {
  if (!out) return 1;
  for (int i = 0; i < 8; ++i) out[i] = g_armors_prof[i];
  return 0;
}

int irmv_engine_has_keypoints(irmv_engine *e) { return e && e->pose ? 1 : 0; }

// Keypoints of the kept detections in source pixels (the same shift and scale parse() applies to the
// boxes, reference src/yolo_engine.cpp:211-214): kpts[nframes][max_det][4][2].
int irmv_engine_fetch_keypoints(irmv_engine *e, int ticket, int nframes, float *kpts) {
  if (!e || !kpts || nframes < 1 || nframes > e->cfg.max_batch) { set_error("bad argument"); return 1; }
  if (!e->pose) { set_error("the weight file has no keypoint branch"); return 2; }
  const uint8_t *h = result_block(e, ticket);
  if (!h) return 2;
  const float *src = e->res.at<const float>(h, kKpts);
  const float sx = e->net_sx, sy = e->net_sy, px = e->net_px, py = e->net_py;
  for (size_t i = 0; i < (size_t)nframes * e->cfg.max_det * 4; ++i) {
    kpts[2 * i] = (src[2 * i] - px) * sx;
    kpts[2 * i + 1] = (src[2 * i + 1] - py) * sy;
  }
  return 0;
}

// Stand-alone stage entry: extract_armors over n frames and their detections (boxes in source pixels).
int irmv_extract_armors(const uint8_t *frames, int frames_on_device, int nframes, int src_w, int src_h, int chan_order,
                        int rotate180, const irmv_bbox *boxes, const int *counts, int max_det,
                        const irmv_armor_params *prm, int device, irmv_armor *out) {
  if (!frames || !boxes || !counts || !out || nframes < 1 || max_det < 1 || src_w < 2 || src_h < 2) { set_error("bad argument"); return 1; }
  irmv_armor_params q;
  if (prm) q = *prm; else irmv_armor_params_default(&q);
  IRMV_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  IRMV_CUDA(cudaGetDeviceProperties(&prop, device));
  const size_t fb = (size_t)src_w * src_h * (chan_order >= 2 ? 1 : 3), slots = (size_t)nframes * max_det;
  uint8_t *d_frames = nullptr;
  int32_t *d_num = nullptr, *d_cls = nullptr;
  float *d_boxes = nullptr, *d_scores = nullptr;
  ArmorOut *d_out = nullptr;
  uint32_t *d_scratch = nullptr;
  std::vector<float> hb(slots * 4, 0.f), hs(slots, 0.f);
  std::vector<int32_t> hc(slots, 0);
  for (size_t i = 0; i < slots; ++i) {
    for (int k = 0; k < 4; ++k) hb[i * 4 + k] = boxes[i].xyxy[k];
    hs[i] = boxes[i].score; hc[i] = boxes[i].class_id;
  }
  const int grid = armors_grid(prop.multiProcessorCount);
  const size_t wpc = armors_scratch_words_per_cta(src_w, src_h), wtotal = armors_scratch_total_words(src_w, src_h, grid);
  int rc = 0;
  auto body = [&]() -> int {
    if (!frames_on_device) {
      IRMV_CUDA(dev_malloc((void **)&d_frames, fb * nframes));
      IRMV_CUDA(cudaMemcpy(d_frames, frames, fb * nframes, cudaMemcpyHostToDevice));
    }
    IRMV_CUDA(dev_malloc((void **)&d_num, (size_t)nframes * 4));
    IRMV_CUDA(dev_malloc((void **)&d_cls, slots * 4));
    IRMV_CUDA(dev_malloc((void **)&d_boxes, slots * 16));
    IRMV_CUDA(dev_malloc((void **)&d_scores, slots * 4));
    IRMV_CUDA(dev_malloc((void **)&d_out, slots * sizeof(ArmorOut)));
    IRMV_CUDA(dev_malloc((void **)&d_scratch, wtotal * 4));
    IRMV_CUDA(cudaMemset(d_scratch, 0, 256));                  // slot locks
    IRMV_CUDA(cudaMemcpy(d_num, counts, (size_t)nframes * 4, cudaMemcpyHostToDevice));
    IRMV_CUDA(cudaMemcpy(d_cls, hc.data(), slots * 4, cudaMemcpyHostToDevice));
    IRMV_CUDA(cudaMemcpy(d_boxes, hb.data(), slots * 16, cudaMemcpyHostToDevice));
    IRMV_CUDA(cudaMemcpy(d_scores, hs.data(), slots * 4, cudaMemcpyHostToDevice));
    IRMV_CUDA(cudaMemset(d_out, 0, slots * sizeof(ArmorOut)));
    ArmorParams ap{};
    ap.src = frames_on_device ? frames : d_frames; ap.src_indirect = nullptr;
    ap.n = nframes; ap.src_w = src_w; ap.src_h = src_h; ap.chan_order = chan_order; ap.rotate180 = rotate180;
    ap.num = d_num; ap.boxes = d_boxes; ap.scores = d_scores; ap.classes = d_cls; ap.max_det = max_det;
    ap.box_sx = 1.f; ap.box_sy = 1.f; ap.box_px = 0.f; ap.box_py = 0.f;
    ap.binary_threshold = q.binary_threshold;
    ap.min_ratio = q.light_min_ratio; ap.max_ratio = q.light_max_ratio; ap.max_angle = q.light_max_angle;
    ap.min_small = q.min_small_center_distance; ap.max_small = q.max_small_center_distance;
    ap.min_large = q.min_large_center_distance; ap.max_large = q.max_large_center_distance;
    ap.out = d_out; ap.slot_locks = reinterpret_cast<int *>(d_scratch); ap.scratch = d_scratch + 64;
    ap.scratch_words_per_cta = wpc; ap.grid = grid;
    unsigned long long *d_prof = nullptr;
    if (getenv("IRMV_ARMOR_PROF")) {
      IRMV_CUDA(dev_malloc((void **)&d_prof, 64));
      IRMV_CUDA(cudaMemset(d_prof, 0, 64));
    }
    ap.prof = d_prof;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    IRMV_CUDA(cudaEventCreate(&e0));
    IRMV_CUDA(cudaEventCreate(&e1));
    IRMV_CUDA(cudaEventRecord(e0, nullptr));
    IRMV_CUDA(launch_extract_armors(ap, nullptr));
    IRMV_CUDA(cudaEventRecord(e1, nullptr));
    IRMV_CUDA(cudaDeviceSynchronize());
    float ms = 0.f;
    IRMV_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    g_armors_ms = ms;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (d_prof) {
      IRMV_CUDA(cudaMemcpy(g_armors_prof, d_prof, 64, cudaMemcpyDeviceToHost));
      cudaFree(d_prof);
    }
    IRMV_CUDA(cudaMemcpy(out, d_out, slots * sizeof(ArmorOut), cudaMemcpyDeviceToHost));
    return 0;
  };
  rc = body();
  cudaFree(d_frames); cudaFree(d_num); cudaFree(d_cls); cudaFree(d_boxes); cudaFree(d_scores); cudaFree(d_out); cudaFree(d_scratch);
  return rc;
}

// One eager (non-graph) replay of up to sub_batch frames on lane 0 with CUDA events between the
// stages: ms[0] preprocess, ms[1] convolutions (+SPPF pool), ms[2] decode+NMS, ms[3] PnP, ms[4] total.
int irmv_engine_profile_stages(irmv_engine *e, const uint8_t *frames_dev, int nframes, float ms[5]) {
  if (!e || !frames_dev || !ms || nframes < 1) { set_error("bad argument"); return 1; }
  IRMV_CUDA(cudaSetDevice(e->cfg.device));
  Lane &ln = e->lanes[0];
  const int n = nframes < e->S ? nframes : e->S;
  IRMV_CUDA(cudaDeviceSynchronize());
  set_src_kernel<<<1, 1, 0, ln.stream>>>(ln.src_word, frames_dev);
  IRMV_CUDA(cudaGetLastError());
  int launches = 0;
  if (int rc = issue_replay(e, ln, n, ln.stream, &launches, true)) return rc;
  IRMV_CUDA(cudaStreamSynchronize(ln.stream));
  for (int i = 0; i < 4; ++i) IRMV_CUDA(cudaEventElapsedTime(&ms[i], ln.stage_ev[i], ln.stage_ev[i + 1]));
  IRMV_CUDA(cudaEventElapsedTime(&ms[4], ln.stage_ev[0], ln.stage_ev[4]));
  return n;
}

// One eager replay with a CUDA event after every kernel of the network stage: ms[i] = duration of
// op i (op 0 = conv0 is inside the stem kernel and reported as 0 when fused).  Returns ops timed.
int irmv_engine_profile_ops(irmv_engine *e, const uint8_t *frames_dev, int nframes, float *ms, int cap) {
  if (!e || !frames_dev || !ms || nframes < 1) { set_error("bad argument"); return -1; }
  cudaSetDevice(e->cfg.device);
  Lane &ln = e->lanes[0];
  const int n = nframes < e->S ? nframes : e->S;
  cudaDeviceSynchronize();
  set_src_kernel<<<1, 1, 0, ln.stream>>>(ln.src_word, frames_dev);
  std::vector<cudaEvent_t> evs;
  int launches = 0;
  if (issue_replay(e, ln, n, ln.stream, &launches, false, &evs)) return -1;
  if (cudaStreamSynchronize(ln.stream) != cudaSuccess) { set_error("profile_ops: replay failed"); return -1; }
  int k = 0;
  for (size_t i = 1; i < evs.size() && k < cap; ++i, ++k) cudaEventElapsedTime(&ms[k], evs[i - 1], evs[i]);
  for (auto ev : evs) cudaEventDestroy(ev);
  return k;
}

// Debug: one line per kernel of the network stage of a replay, in issue order:
// "conv k s cin cout hw raster tail_cout" or "pool".  Returns the number of bytes written.
int irmv_engine_describe_ops(irmv_engine *e, char *buf, int cap) {
  if (!e || !buf || cap < 1) return -1;
  std::string out;
  bool first = true;
  const bool fused = e->fused_stem && e->cfg.conv_impl != IRMV_CONV_DIRECT;
  for (auto &o : e->lanes[0].ops) {
    if (first && fused) { first = false; continue; }       // conv0 runs inside the stem kernel
    first = false;
    char line[160];
    if (o.kind == Op::POOL) snprintf(line, sizeof line, "pool\n");
    else if (o.kind == Op::DW) snprintf(line, sizeof line, "dw %d %d %d\n", o.dw.stride, o.dw.planes * 8, o.dw.H / o.dw.stride);
    else if (o.kind == Op::SHUF) snprintf(line, sizeof line, "unit %d %d %d %d %d\n", o.su.down, o.su.cin, o.su.h, o.su.H, o.su.TH);
    else snprintf(line, sizeof line, "conv %d %d %d %d %d %d %d\n", o.cp.k, o.cp.stride, o.cp.cin, o.cp.cout, o.cp.OH,
                  o.raster ? 1 : 0, o.cp.tail_w ? o.cp.tail_cout : 0);
    out += line;
  }
  if ((int)out.size() + 1 > cap) { set_error("buffer too small"); return -1; }
  memcpy(buf, out.c_str(), out.size() + 1);
  return (int)out.size();
}

// Debug: the tiling plan of every network-stage kernel for a replay of `nframes` frames, one line per
// launch in issue order: "raster k s cin cout hw R nepi b_stream ctas_per_sm stages b_stages tail act res tiles",
// "gather k s cin cout hw" or "pool".  plan() depends on the tile count, so the kernel instantiations
// differ between replay sizes; tests use this to show which ones an oracle-compared run covers.
int irmv_engine_describe_plans(irmv_engine *e, int nframes, char *buf, int cap) {
  if (!e || !buf || cap < 1 || nframes < 1) return -1;
  std::string out;
  bool first = true;
  const bool fused = e->fused_stem && e->cfg.conv_impl != IRMV_CONV_DIRECT;
  const int n = nframes < e->S ? nframes : e->S;
  for (auto &o : e->lanes[0].ops) {
    if (first && fused) { first = false; continue; }
    first = false;
    char line[200];
    if (o.kind == Op::POOL) { out += "pool\n"; continue; }
    if (o.kind == Op::DW) { snprintf(line, sizeof line, "dw %d %d %d\n", o.dw.stride, o.dw.planes * 8, o.dw.H / o.dw.stride); out += line; continue; }
    if (o.kind == Op::SHUF) { snprintf(line, sizeof line, "unit %d %d %d %d %d\n", o.su.down, o.su.cin, o.su.h, o.su.H, o.su.TH); out += line; continue; }
    ConvParams p = o.cp;
    p.B = n;
    int info[8];
    if (o.raster && conv_raster_plan_info(p, e->num_sms, info))
      snprintf(line, sizeof line, "raster %d %d %d %d %d %d %d %d %d %d %d %d %d %d %d\n", p.k, p.stride, p.cin, p.cout, p.OH,
               info[0], info[1], info[2], info[3], info[4], info[5], info[6], p.act, p.res ? 1 : 0, info[7]);
    else
      snprintf(line, sizeof line, "gather %d %d %d %d %d\n", p.k, p.stride, p.cin, p.cout, p.OH);
    out += line;
  }
  if ((int)out.size() + 1 > cap) { set_error("buffer too small"); return -1; }
  memcpy(buf, out.c_str(), out.size() + 1);
  return (int)out.size();
}

// Debug: re-run GEMM number `op_index` of lane 0 on whatever its input buffers hold, with CTA 0
// writing clock64 stamps per tile: {tile start, before empty wait, after, last k-block issued,
// MMA first full, MMA last full, epilogue start, epilogue end}.  Returns tiles traced.
int irmv_engine_trace_conv(irmv_engine *e, int op_index, int nframes, long long *out, int cap_tiles, float *kernel_ms) {
  if (!e || !out || cap_tiles < 1) { set_error("bad argument"); return -1; }
  cudaSetDevice(e->cfg.device);
  Lane &ln = e->lanes[0];
  int ci = -1;
  Op *op = nullptr;
  for (auto &o : ln.ops) if (o.kind == Op::CONV && ++ci == op_index) { op = &o; break; }
  if (!op) { set_error("no such conv"); return -1; }
  long long *d = nullptr;
  dev_malloc((void **)&d, (size_t)(cap_tiles + 16) * 64);
  cudaMemset(d, 0, (size_t)(cap_tiles + 16) * 64);
  ConvParams p = op->cp;
  p.B = nframes < e->S ? nframes : e->S;
  p.trace = d; p.trace_cap = cap_tiles;
  if (const char *dbg = getenv("IRMV_TC_DEBUG")) p.sync_mode = atoi(dbg);
  cudaDeviceSynchronize();
  cudaEventRecord(ln.stage_ev[0], ln.stream);
  if (op->raster) launch_conv_raster(p, e->num_sms, ln.stream); else launch_conv_tc(p, e->num_sms, ln.stream);
  cudaEventRecord(ln.stage_ev[1], ln.stream);
  cudaError_t ce = cudaStreamSynchronize(ln.stream);
  if (kernel_ms) cudaEventElapsedTime(kernel_ms, ln.stage_ev[0], ln.stage_ev[1]);
  cudaMemcpy(out, d, (size_t)(cap_tiles + 16) * 64, cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (ce != cudaSuccess) { set_error(cudaGetErrorString(ce)); return -1; }
  int M = p.B * p.OH * p.OW, tiles = (M + 127) / 128;
  if (op->raster) return cap_tiles;   // rows past the CTA's last tile stay zero
  int per_cta = (tiles + (tiles < e->num_sms ? tiles : e->num_sms) - 1) / (tiles < e->num_sms ? tiles : e->num_sms);
  return per_cta < cap_tiles ? per_cta : cap_tiles;
}

// ------------------------------------------------------------------ stage entry points
int irmv_preprocess(const uint8_t *src, int n, int src_w, int src_h, int chan_order, int rotate180,
                    int resize_mode, int quantize_u8, uint16_t *dst, uint8_t *rotated, int device) {
  if (!src || !dst || n < 1) { set_error("bad argument"); return 1; }
  IRMV_CUDA(cudaSetDevice(device));
  const size_t fb = (size_t)src_w * src_h * (chan_order >= 2 ? 1 : 3);
  const size_t ob = (size_t)pr_pixels(n, kNet, kNet) * kInC * 2;     // kernel writes the PR layout
  uint8_t *ds = nullptr, *dr = nullptr;
  __half *dd = nullptr;
  IRMV_CUDA(dev_malloc((void **)&ds, fb * n));
  IRMV_CUDA(dev_malloc((void **)&dd, ob));
  IRMV_CUDA(cudaMemset(dd, 0, ob));
  if (rotated) IRMV_CUDA(dev_malloc((void **)&dr, (size_t)src_w * src_h * 3 * n));
  IRMV_CUDA(cudaMemcpy(ds, src, fb * n, cudaMemcpyHostToDevice));
  PreprocessParams pp{};
  pp.src = ds; pp.dst = dd; pp.rotated = dr; pp.n = n; pp.src_w = src_w; pp.src_h = src_h;
  pp.chan_order = chan_order; pp.rotate180 = rotate180; pp.resize_mode = resize_mode; pp.quantize_u8 = quantize_u8;
  cudaError_t ce = launch_preprocess(pp, 0);
  if (ce == cudaSuccess) ce = cudaDeviceSynchronize();
  std::vector<uint16_t> tmp(ob / 2);
  if (ce == cudaSuccess) ce = cudaMemcpy(tmp.data(), dd, ob, cudaMemcpyDeviceToHost);
  if (ce == cudaSuccess && rotated) ce = cudaMemcpy(rotated, dr, (size_t)src_w * src_h * 3 * n, cudaMemcpyDeviceToHost);
  cudaFree(ds); cudaFree(dd); if (dr) cudaFree(dr);
  IRMV_CUDA(ce);
  for (int b = 0; b < n; ++b)
    for (int y = 0; y < kNet; ++y)
      memcpy(dst + (((size_t)b * kNet + y) * kNet) * kInC, tmp.data() + (size_t)pr_index(b, y, 0, kNet, kNet) * kInC,
             (size_t)kNet * kInC * 2);
  return 0;
}

// NMS scratch and a result block (its detection fields) for n frames
static int alloc_nms(int n, int A, int nc, const ResultLayout &L, NmsScratch &sc, uint8_t *&det) {
  IRMV_CUDA(dev_malloc((void **)&sc.boxes, (size_t)n * A * 16));
  IRMV_CUDA(dev_malloc((void **)&sc.keys, (size_t)n * A * nc * 8));
  IRMV_CUDA(dev_malloc((void **)&sc.counts, (size_t)n * 4));
  IRMV_CUDA(cudaMemset(sc.counts, 0, (size_t)n * 4));
  IRMV_CUDA(dev_malloc((void **)&det, L.end(kIndex)));
  IRMV_CUDA(cudaMemset(det, 0, L.end(kIndex)));
  return 0;
}

int irmv_nms(const float *boxes, const float *scores, int n, int A, int nc, float score_thr,
             float iou_thr, int max_det, int32_t *num_dets, float *det_boxes, float *det_scores,
             int32_t *det_classes, int32_t *det_index, int device) {
  if (!boxes || !scores || !num_dets || n < 1 || A < 1 || nc < 1 || max_det < 1) { set_error("bad argument"); return 1; }
  IRMV_CUDA(cudaSetDevice(device));
  NmsScratch sc{};
  const ResultLayout L(n, max_det);
  uint8_t *det = nullptr;
  if (int rc = alloc_nms(n, A, nc, L, sc, det)) return rc;
  float *ds = nullptr;
  IRMV_CUDA(dev_malloc((void **)&ds, (size_t)n * A * nc * 4));
  IRMV_CUDA(cudaMemcpy(sc.boxes, boxes, (size_t)n * A * 16, cudaMemcpyHostToDevice));
  IRMV_CUDA(cudaMemcpy(ds, scores, (size_t)n * A * nc * 4, cudaMemcpyHostToDevice));
  cudaError_t ce = launch_score_filter(ds, n, A, nc, score_thr, sc, 0);
  if (ce == cudaSuccess) ce = launch_nms(sc, n, A, nc, iou_thr, max_det, det_out(det, L), 0);
  if (ce == cudaSuccess) ce = cudaDeviceSynchronize();
  std::vector<uint8_t> host(L.end(kIndex));
  if (ce == cudaSuccess) ce = cudaMemcpy(host.data(), det, host.size(), cudaMemcpyDeviceToHost);
  cudaFree(sc.boxes); cudaFree(sc.keys); cudaFree(sc.counts); cudaFree(det); cudaFree(ds);
  IRMV_CUDA(ce);
  auto out = [&](void *dst, ResultField f) { if (dst) memcpy(dst, host.data() + L.offset[f], (size_t)n * L.frame_bytes[f]); };
  out(num_dets, kNum); out(det_boxes, kBoxes); out(det_scores, kScores); out(det_classes, kClasses); out(det_index, kIndex);
  return 0;
}

int irmv_decode(const uint16_t *box, const uint16_t *cls, int n, float *boxes, float *scores, int device) {
  if (!box || !cls || !boxes || !scores || n < 1) { set_error("bad argument"); return 1; }
  IRMV_CUDA(cudaSetDevice(device));
  const int nc = IRMV_NUM_CLASSES;
  NmsScratch sc{};
  uint8_t *det = nullptr;
  if (int rc = alloc_nms(n, kNumAnchors, nc, ResultLayout(n, 1), sc, det)) return rc;
  // inputs arrive in anchor order [n][A][C]; the kernel wants one tensor per scale [n][hw*hw][C]
  const int cnt[3] = {6400, 1600, 400}, off[3] = {0, 6400, 8000};
  HeadPtrs h{};
  __half *db[3], *dc[3];
  float *dscores = nullptr;
  IRMV_CUDA(dev_malloc((void **)&dscores, (size_t)n * kNumAnchors * nc * 4));
  for (int s = 0; s < 3; ++s) {
    IRMV_CUDA(dev_malloc((void **)&db[s], (size_t)n * cnt[s] * 64 * 2));
    IRMV_CUDA(dev_malloc((void **)&dc[s], (size_t)n * cnt[s] * kClsPad * 2));
    for (int f = 0; f < n; ++f) {
      IRMV_CUDA(cudaMemcpy(db[s] + (size_t)f * cnt[s] * 64, box + ((size_t)f * kNumAnchors + off[s]) * 64,
                           (size_t)cnt[s] * 64 * 2, cudaMemcpyHostToDevice));
      IRMV_CUDA(cudaMemcpy(dc[s] + (size_t)f * cnt[s] * kClsPad, cls + ((size_t)f * kNumAnchors + off[s]) * kClsPad,
                           (size_t)cnt[s] * kClsPad * 2, cudaMemcpyHostToDevice));
    }
    h.box[s] = db[s]; h.cls[s] = dc[s];
  }
  h.padded = 0;
  cudaError_t ce = launch_decode(h, n, nc, 2.0f /* no candidates */, sc, dscores, 0);
  if (ce == cudaSuccess) ce = cudaDeviceSynchronize();
  if (ce == cudaSuccess) ce = cudaMemcpy(boxes, sc.boxes, (size_t)n * kNumAnchors * 16, cudaMemcpyDeviceToHost);
  if (ce == cudaSuccess) ce = cudaMemcpy(scores, dscores, (size_t)n * kNumAnchors * nc * 4, cudaMemcpyDeviceToHost);
  for (int s = 0; s < 3; ++s) { cudaFree(db[s]); cudaFree(dc[s]); }
  cudaFree(sc.boxes); cudaFree(sc.keys); cudaFree(sc.counts); cudaFree(det); cudaFree(dscores);
  IRMV_CUDA(ce);
  return 0;
}

}  // extern "C"

// =============================================================================== PnP
struct irmv_pnp {
  PnpConsts c{};
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  double last_ms = 0.0;
  int lm_iters = 0;             // > 0: Levenberg-Marquardt refinement after IPPE (not in the reference's call)
  // small persistent buffers for the single-armor call
  float *d_pts1 = nullptr;
  double *d_out1 = nullptr;   // rvec[3] tvec[3]
  uint8_t *d_ok1 = nullptr;
  float *h_pts1 = nullptr;    // pinned
  double *h_out1 = nullptr;
  uint8_t *h_ok1 = nullptr;
  // grow-only device buffers of the batch call: no allocation per call once they are large enough
  size_t cap = 0;             // armors the buffers below hold
  float *d_pts = nullptr;
  double *d_rv = nullptr, *d_tv = nullptr, *d_q = nullptr, *d_rv2 = nullptr, *d_tv2 = nullptr, *d_e = nullptr;
  uint8_t *d_ok = nullptr;
};

static void pnp_free_batch(irmv_pnp *p) {
  cudaFree(p->d_pts); cudaFree(p->d_rv); cudaFree(p->d_tv); cudaFree(p->d_q); cudaFree(p->d_rv2); cudaFree(p->d_tv2);
  cudaFree(p->d_e); cudaFree(p->d_ok);
  p->d_pts = nullptr; p->d_rv = p->d_tv = p->d_q = p->d_rv2 = p->d_tv2 = p->d_e = nullptr; p->d_ok = nullptr;
  p->cap = 0;
}

static int pnp_reserve(irmv_pnp *p, size_t n) {
  if (n <= p->cap) return 0;
  size_t cap = p->cap ? p->cap : 1024;
  while (cap < n) cap *= 2;
  IRMV_CUDA(cudaStreamSynchronize(p->stream));
  pnp_free_batch(p);
  IRMV_CUDA(irmv::dev_malloc((void **)&p->d_pts, cap * 32));
  IRMV_CUDA(irmv::dev_malloc((void **)&p->d_rv, cap * 24));
  IRMV_CUDA(irmv::dev_malloc((void **)&p->d_tv, cap * 24));
  IRMV_CUDA(irmv::dev_malloc((void **)&p->d_q, cap * 32));
  IRMV_CUDA(irmv::dev_malloc((void **)&p->d_rv2, cap * 24));
  IRMV_CUDA(irmv::dev_malloc((void **)&p->d_tv2, cap * 24));
  IRMV_CUDA(irmv::dev_malloc((void **)&p->d_e, cap * 16));
  IRMV_CUDA(irmv::dev_malloc((void **)&p->d_ok, cap));
  p->cap = cap;
  return 0;
}

extern "C" {

int irmv_pnp_create(const double K[9], const double D[5], int device, irmv_pnp **out) {
  if (!K || !D || !out) { set_error("null argument"); return 1; }
  int ndev = 0;
  IRMV_CUDA(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) { set_error("no such CUDA device"); return 3; }
  IRMV_CUDA(cudaSetDevice(device));
  std::unique_ptr<irmv_pnp> p(new irmv_pnp);
  p->device = device;
  // reference src/pnp_solver.cpp:10-15: K row-major 3x3, D first five coefficients
  p->c.fx = K[0]; p->c.cx = K[2]; p->c.fy = K[4]; p->c.cy = K[5];
  p->c.k1 = D[0]; p->c.k2 = D[1]; p->c.p1 = D[2]; p->c.p2 = D[3]; p->c.k3 = D[4];
  // reference include/irmv_detection/pnp_solver.hpp:30-33 (mm) and src/pnp_solver.cpp:18-21
  p->c.half_w[0] = 135.0 / 2.0 / 1000.0; p->c.half_h[0] = 55.0 / 2.0 / 1000.0;
  p->c.half_w[1] = 225.0 / 2.0 / 1000.0; p->c.half_h[1] = 55.0 / 2.0 / 1000.0;
  IRMV_CUDA(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
  IRMV_CUDA(cudaEventCreate(&p->ev0));
  IRMV_CUDA(cudaEventCreate(&p->ev1));
  IRMV_CUDA(dev_malloc((void **)&p->d_pts1, 32));
  IRMV_CUDA(dev_malloc((void **)&p->d_out1, 48));
  IRMV_CUDA(dev_malloc((void **)&p->d_ok1, 4));
  IRMV_CUDA(host_malloc((void **)&p->h_pts1, 32));
  IRMV_CUDA(host_malloc((void **)&p->h_out1, 48));
  IRMV_CUDA(host_malloc((void **)&p->h_ok1, 4));
  *out = p.release();
  return 0;
}

void irmv_pnp_destroy(irmv_pnp *p) {
  if (!p) return;
  cudaSetDevice(p->device);
  cudaStreamSynchronize(p->stream);
  pnp_free_batch(p);
  cudaFree(p->d_pts1); cudaFree(p->d_out1); cudaFree(p->d_ok1);
  cudaFreeHost(p->h_pts1); cudaFreeHost(p->h_out1); cudaFreeHost(p->h_ok1);
  cudaEventDestroy(p->ev0); cudaEventDestroy(p->ev1);
  cudaStreamDestroy(p->stream);
  delete p;
}

int irmv_pnp_solve(irmv_pnp *p, const float img_pts[8], double rvec[3], double tvec[3], int *ok) {
  if (!p || !img_pts || !rvec || !tvec) { set_error("null argument"); return 1; }
  IRMV_CUDA(cudaSetDevice(p->device));
  memcpy(p->h_pts1, img_pts, 32);
  IRMV_CUDA(cudaMemcpyAsync(p->d_pts1, p->h_pts1, 32, cudaMemcpyHostToDevice, p->stream));
  PnpOut o{p->d_out1, p->d_out1 + 3, p->d_ok1, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  IRMV_CUDA(launch_pnp(p->c, p->d_pts1, 1, 0 /* reference: small_armor = true, src/pnp_solver.cpp:47 */, o, p->stream));
  if (p->lm_iters > 0)
    IRMV_CUDA(launch_pnp_refine_lm(p->c, p->d_pts1, 1, 0, p->lm_iters, p->d_out1, p->d_out1 + 3, nullptr, p->stream));
  IRMV_CUDA(cudaMemcpyAsync(p->h_out1, p->d_out1, 48, cudaMemcpyDeviceToHost, p->stream));
  IRMV_CUDA(cudaMemcpyAsync(p->h_ok1, p->d_ok1, 1, cudaMemcpyDeviceToHost, p->stream));
  IRMV_CUDA(cudaStreamSynchronize(p->stream));
  memcpy(rvec, p->h_out1, 24);
  memcpy(tvec, p->h_out1 + 3, 24);
  if (ok) *ok = p->h_ok1[0];
  return 0;
}

int irmv_pnp_solve_batch_ex(irmv_pnp *p, const float *img_pts, int n, int on_device, int large,
                            double *rvecs, double *tvecs, uint8_t *ok, double *quats,
                            double *rvecs2, double *tvecs2, double *rmse2) {
  if (!p || !img_pts || !rvecs || !tvecs || n < 1) { set_error("bad argument"); return 1; }
  IRMV_CUDA(cudaSetDevice(p->device));
  const bool want2 = rvecs2 && tvecs2 && rmse2;
  if (int rc = pnp_reserve(p, (size_t)n)) return rc;
  const float *dp = img_pts;
  if (!on_device) {
    IRMV_CUDA(cudaMemcpyAsync(p->d_pts, img_pts, (size_t)n * 32, cudaMemcpyHostToDevice, p->stream));
    dp = p->d_pts;
  }
  double *dq = quats ? p->d_q : nullptr;
  PnpOut o{p->d_rv, p->d_tv, p->d_ok, dq, want2 ? p->d_rv2 : nullptr, want2 ? p->d_tv2 : nullptr, want2 ? p->d_e : nullptr,
           nullptr, nullptr};
  IRMV_CUDA(cudaEventRecord(p->ev0, p->stream));
  IRMV_CUDA(launch_pnp(p->c, dp, n, large, o, p->stream));
  if (p->lm_iters > 0) IRMV_CUDA(launch_pnp_refine_lm(p->c, dp, n, large, p->lm_iters, p->d_rv, p->d_tv, dq, p->stream));
  IRMV_CUDA(cudaEventRecord(p->ev1, p->stream));
  IRMV_CUDA(cudaMemcpyAsync(rvecs, p->d_rv, (size_t)n * 24, cudaMemcpyDeviceToHost, p->stream));
  IRMV_CUDA(cudaMemcpyAsync(tvecs, p->d_tv, (size_t)n * 24, cudaMemcpyDeviceToHost, p->stream));
  if (ok) IRMV_CUDA(cudaMemcpyAsync(ok, p->d_ok, (size_t)n, cudaMemcpyDeviceToHost, p->stream));
  if (quats) IRMV_CUDA(cudaMemcpyAsync(quats, p->d_q, (size_t)n * 32, cudaMemcpyDeviceToHost, p->stream));
  if (want2) {
    IRMV_CUDA(cudaMemcpyAsync(rvecs2, p->d_rv2, (size_t)n * 24, cudaMemcpyDeviceToHost, p->stream));
    IRMV_CUDA(cudaMemcpyAsync(tvecs2, p->d_tv2, (size_t)n * 24, cudaMemcpyDeviceToHost, p->stream));
    IRMV_CUDA(cudaMemcpyAsync(rmse2, p->d_e, (size_t)n * 16, cudaMemcpyDeviceToHost, p->stream));
  }
  IRMV_CUDA(cudaStreamSynchronize(p->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, p->ev0, p->ev1);
  p->last_ms = ms;
  return 0;
}

int irmv_pnp_solve_batch(irmv_pnp *p, const float *img_pts, int n, int on_device, int large,
                         double *rvecs, double *tvecs, uint8_t *ok) {
  return irmv_pnp_solve_batch_ex(p, img_pts, n, on_device, large, rvecs, tvecs, ok, nullptr, nullptr,
                                 nullptr, nullptr);
}

int irmv_pnp_set_refine_lm(irmv_pnp *p, int max_iters) {
  if (!p || max_iters < 0 || max_iters > 1000) { set_error("bad argument"); return 1; }
  p->lm_iters = max_iters;
  return 0;
}

double irmv_pnp_last_device_ms(irmv_pnp *p) { return p ? p->last_ms : 0.0; }

// The reference reads its CV_64F camera matrix with .at<float> (src/pnp_solver.cpp:56-57), which
// yields garbage principal-point values (SURVEY.md section 0.8).  This implements the intended
// computation: distance from the image point to (cx, cy).
float irmv_pnp_distance_to_center(irmv_pnp *p, float x, float y) {
  if (!p) return 0.f;
  float dx = x - (float)p->c.cx, dy = y - (float)p->c.cy;
  return sqrtf(dx * dx + dy * dy);
}

}  // extern "C"
