// irmv_detection_b200/csrc/result_layout.h: field placement for every batch size the engine builds, and the
// device -> host copy plan of the engine's configurations (copies and bytes per call).  CPU-only.
#include <cstdio>
#include <initializer_list>
#include "result_layout.h"
using namespace irmv;

static int failures = 0;
#define CHECK(c, ...) do { if (!(c)) { ++failures; printf("FAIL %s:%d: ", __FILE__, __LINE__); printf(__VA_ARGS__); printf("\n"); } } while (0)

// One engine call: n frames replayed in chunks of `chunk` frames on lane blocks laid out for `lane_frames`,
// landing in a result set laid out for `max_batch` frames.
static void check_plan(const char *name, size_t max_batch, size_t lane_frames, size_t chunk, size_t n, unsigned fields,
                       int want_copies, size_t want_bytes) {
  const ResultLayout dev(lane_frames, 100), host(max_batch, 100);
  int copies = 0;
  size_t bytes = 0;
  for (size_t f0 = 0; f0 < n; f0 += chunk) {
    const size_t nf = n - f0 < chunk ? n - f0 : chunk;
    const CopyPlan p = plan_copies(dev, host, fields, f0, nf);
    copies += p.n;
    for (int i = 0; i < p.n; ++i) {
      bytes += p.r[i].bytes;
      CHECK(p.r[i].dev_off + p.r[i].bytes <= dev.bytes && p.r[i].host_off + p.r[i].bytes <= host.bytes, "%s: range %d out of bounds", name, i);
    }
    CHECK(plan_copies(dev, host, fields, f0, nf, false).n == __builtin_popcount(fields), "%s: unmerged plan", name);
  }
  CHECK(copies == want_copies && bytes == want_bytes, "%s: %d copies / %zu bytes, want %d / %zu", name, copies, bytes,
        want_copies, want_bytes);
}

int main() {
  for (size_t md : {1, 7, 100, 1024})
    for (size_t frames : {1, 2, 3, 5, 64, 128, 256}) {
      const ResultLayout L(frames, md);
      for (int f = 0; f < kNumResultFields; ++f) {
        CHECK(L.offset[f] % kResultFields[f].align == 0, "md %zu frames %zu: field %d at %zu", md, frames, f, L.offset[f]);
        CHECK(L.frame_bytes[f] == (f == kNum ? 4 : kResultFields[f].per_det * md), "md %zu: field %d size", md, f);
        if (f) CHECK(L.offset[f] >= L.end(ResultField(f - 1)), "md %zu frames %zu: field %d overlaps field %d", md, frames, f, f - 1);
      }
      CHECK(L.bytes >= L.end(kDist), "md %zu frames %zu: bytes %zu", md, frames, L.bytes);
    }

  const unsigned det = 1u << kNum | 1u << kBoxes | 1u << kScores | 1u << kClasses | 1u << kIndex;
  const unsigned pnp = det | 1u << kRvec | 1u << kTvec | 1u << kOk | 1u << kQuat | 1u << kDist;
  // max_det 100; copies and bytes of the engine before the layout had one description
  check_plan("bench main", 256, 256, 256, 256, pnp, 2, 2893824);
  check_plan("bench end to end", 256, 256, 128, 256, pnp, 20, 2893824);
  check_plan("batch-1 detect", 1, 1, 1, 1, pnp, 3, 11304);
  check_plan("armor bench", 128, 64, 64, 128, pnp | 1u << kArmors, 22, 2163712);
  check_plan("keypoint variant", 64, 64, 64, 64, pnp | 1u << kKpts, 2, 928256);
  check_plan("B3 S3 armors", 3, 3, 3, 3, pnp | 1u << kArmors, 4, 50712);
  check_plan("B7 S3 detections", 7, 3, 3, 7, det, 15, 19628);
  check_plan("B5 S2 all", 5, 2, 2, 5, pnp | 1u << kArmors | 1u << kKpts, 36, 100520);

  if (failures) return 1;
  printf("RESULT_LAYOUT_OK\n");
  return 0;
}
