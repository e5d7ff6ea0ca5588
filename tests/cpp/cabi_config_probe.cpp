// Prints sizeof(irmv_engine_config) and the offsets of reserved[] and raw_format as the C compiler lays them out,
// for tests/test_raw_bits.py to compare with the ctypes mirror (irmv_detection_b200/_lib.py EngineConfig).
#include <cstddef>
#include <cstdio>

#include "irmv_cabi.h"

int main() {
  std::printf("%zu %zu %zu\n", sizeof(irmv_engine_config), offsetof(irmv_engine_config, reserved),
              offsetof(irmv_engine_config, raw_format));
  return 0;
}
