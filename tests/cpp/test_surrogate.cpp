// The near-miss measures through the C++ façade (include/pp.hpp): a small IDM job, its record and
// totals read back with Rollouts::surrogate() / surrogate_totals() and written as raw arrays, in
// the order of pp_rollout_surrogate then the totals, for tests/test_surrogate.py to compare with
// the Python binding.
//   test_surrogate <highway_map.csv> <out.bin>
#include <cstdio>
#include <vector>

#include "pp.hpp"

template <class T>
static void put(std::FILE *f, const std::vector<T> &v) {
  if (!v.empty()) std::fwrite(v.data(), sizeof(T), v.size(), f);
}

int main(int argc, char **argv) {
  if (argc < 3) return 1;
  try {
    pp::Map map;
    map.InitFromCsv(argv[1]);
    pp::Rollouts ro(map, 300, 12, 11, 5);
    ro.set_traffic(PP_TRAFFIC_IDM);
    ro.set_surrogate();
    ro.run(40, 1);
    ro.run(20, 3);
    const pp::Rollouts::Surrogate s = ro.surrogate();
    const std::vector<int64_t> tot = ro.surrogate_totals();
    std::FILE *f = std::fopen(argv[2], "wb");
    if (!f) return 1;
    put(f, s.min_ttc_front);
    put(f, s.min_ttc_rear);
    put(f, s.min_thw);
    put(f, s.min_ttc_front_tick);
    put(f, s.time_hist);
    put(f, tot);
    std::fclose(f);
    std::printf("surrogate facade ok\n");
  } catch (const pp::Error &e) {
    std::printf("pp::Error: %s\n", e.what());
    return 2;
  }
  return 0;
}
