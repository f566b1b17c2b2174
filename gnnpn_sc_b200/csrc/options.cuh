// Library-wide run-time options (gnnpn_set_option / gnnpn_get_option, include/gnnpn_b200.h).  The matching
// environment variables are read ONCE, when the library is loaded, to set the initial values; kernels and dispatchers
// read the atomics -- nothing on a call path reads the environment.
#pragma once
#include <atomic>

namespace gnnpn {

struct Options {
  std::atomic<int> scan{-1};         // "scan": -1 auto (by batch size), 0 CTA-pair scan, 1 column-split cluster scan   [GNNPN_COLSPLIT]
  std::atomic<int> scan_groups{0};   // "scan_groups": 0 auto, 1 / 2 / 3 instance groups per column-split encoder cluster  [GNNPN_COLSPLIT_G]
  std::atomic<int> persistent{3};    // "persistent": bit 0 encoder, bit 1 decoder run as ONE persistent launch           [GNNPN_SEQ]
  std::atomic<int> bptt{1};          // "bptt": 1 = REINFORCE backward as two persistent cluster scans, 0 = two launches per step   [GNNPN_BPTT]
  std::atomic<int> prof{0};          // "prof": in-kernel wait-cycle counters, printed to stderr (debug, synchronous)     [GNNPN_SEQ_PROF]
};
Options& options();

}  // namespace gnnpn
