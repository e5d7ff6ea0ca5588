// Byte layout of the per-frame results of a replay.  A lane's device block and a pinned result set are
// the same layout, for the lane's S frames and for max_batch frames, so that the copies between them
// merge wherever both sides are contiguous.  Plain C++ (no CUDA) so that the CPU tests compile it.
#pragma once
#include <cstddef>

namespace irmv {

// In memory order.  Each field is `frames` consecutive per-frame arrays.
enum ResultField { kNum, kBoxes, kScores, kClasses, kIndex, kRvec, kTvec, kOk, kArmors, kKpts, kQuat, kDist, kNumResultFields };

struct ResultFieldSpec { size_t frame_fixed, per_det, align; };   // bytes per frame = frame_fixed + per_det * max_det
constexpr ResultFieldSpec kResultFields[kNumResultFields] = {
    {4, 0, 4},     // num: i32 kept detections
    {0, 16, 16},   // boxes: xyxy f32, network pixels (float4 stores)
    {0, 4, 4},     // scores: f32
    {0, 4, 4},     // classes: i32
    {0, 4, 4},     // index: i32 flat anchor * nc + class
    {0, 24, 16},   // rvec: f64[3]
    {0, 24, 16},   // tvec: f64[3]
    {0, 1, 1},     // ok: u8
    {0, 56, 16},   // armors: ArmorOut == irmv_armor (static_assert in engine.cu)
    {0, 32, 16},   // kpts: f32[4][2], network pixels (float4 stores)
    {0, 32, 16},   // quat: f64[4] tf2 quaternion (x, y, z, w)
    {0, 4, 4},     // dist: f32 distance_to_image_center
};

struct ResultLayout {
  size_t frames = 0;
  size_t offset[kNumResultFields] = {}, frame_bytes[kNumResultFields] = {};
  size_t bytes = 0;   // the whole block

  explicit ResultLayout(size_t frames_ = 0, size_t max_det = 0) : frames(frames_) {
    for (int f = 0; f < kNumResultFields; ++f) {
      const ResultFieldSpec &s = kResultFields[f];
      frame_bytes[f] = s.frame_fixed + s.per_det * max_det;
      offset[f] = (bytes + s.align - 1) / s.align * s.align;
      bytes = end(ResultField(f));
    }
  }
  size_t end(ResultField f) const { return offset[f] + frames * frame_bytes[f]; }
  template <class T, class Byte> T *at(Byte *base, ResultField f) const { return reinterpret_cast<T *>(base + offset[f]); }
};

struct CopyRange { size_t host_off, dev_off, bytes; };
struct CopyPlan { CopyRange r[kNumResultFields]; int n = 0; };

// Copies of frames [f0, f0 + n) from a device block (frames 0 .. n-1 of `dev`) to their slots in a host
// set: one range per field of `fields` (bit i = field i), in table order.  With `merge`, a range that
// continues the previous one on both sides extends it.
inline CopyPlan plan_copies(const ResultLayout &dev, const ResultLayout &host, unsigned fields, size_t f0, size_t n,
                            bool merge = true) {
  CopyPlan p;
  for (int f = 0; f < kNumResultFields; ++f) {
    if (!(fields >> f & 1u)) continue;
    const CopyRange c{host.offset[f] + f0 * host.frame_bytes[f], dev.offset[f], n * dev.frame_bytes[f]};
    CopyRange *last = p.n ? &p.r[p.n - 1] : nullptr;
    if (merge && last && last->host_off + last->bytes == c.host_off && last->dev_off + last->bytes == c.dev_off) last->bytes += c.bytes;
    else p.r[p.n++] = c;
  }
  return p;
}

}  // namespace irmv
