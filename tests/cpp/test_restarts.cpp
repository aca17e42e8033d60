// Episode restarts through the C++ façade (include/pp.hpp): a small IDM job that restarts on every
// kind but collision_rear and on a non-finite distance, its record and totals read back with
// Rollouts::restarts() / restart_totals() and written as raw arrays, in the order of
// pp_rollout_restarts then the totals, for tests/test_restarts.py to compare with the Python
// binding.
//   test_restarts <highway_map.csv> <out.bin>
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
    ro.set_restart(((1u << (PP_REC_NONFINITE + 1)) - 1) & ~(1u << PP_INC_COLLISION_REAR));
    ro.set_traffic(PP_TRAFFIC_IDM);
    ro.run(40, 1);
    ro.run(20, 3);
    const pp::Rollouts::Restarts s = ro.restarts();
    const std::vector<int64_t> tot = ro.restart_totals();
    std::FILE *f = std::fopen(argv[2], "wb");
    if (!f) return 1;
    put(f, s.episodes);
    put(f, s.by_bit);
    put(f, s.episode_tick);
    put(f, s.episode_m);
    put(f, s.ended_m);
    put(f, s.ended_lap);
    put(f, tot);
    std::fclose(f);
    std::printf("restarts facade ok\n");
  } catch (const pp::Error &e) {
    std::printf("pp::Error: %s\n", e.what());
    return 2;
  }
  return 0;
}
