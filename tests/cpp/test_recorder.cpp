// The flight recorder through the C++ façade (include/pp.hpp): a small IDM job with a wrapping
// window, read back with Rollouts::recording() and written as raw arrays, in the order of
// pp_rollout_recording, for tests/test_recorder.py to compare with the Python binding.
//   test_recorder <highway_map.csv> <out.bin>
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
    ro.set_recorder(7, 0xFDu);  // every kind but collision_rear, and a non-finite distance
    ro.run(5, 1);
    ro.run(9, 3);
    const pp::Rollouts::Recording r = ro.recording({0, 17, 299, 17});
    std::FILE *f = std::fopen(argv[2], "wb");
    if (!f) return 1;
    put(f, r.trigger_tick);
    put(f, r.trigger_bits);
    put(f, r.tick);
    put(f, r.consume_k);
    for (const auto *v : {&r.ego_x, &r.ego_y, &r.ego_yaw_deg, &r.ego_speed_mph, &r.prev_x, &r.prev_y,
                          &r.car_x, &r.car_y, &r.car_vx, &r.car_vy})
      put(f, *v);
    for (const auto *v : {&r.prev_n, &r.target_lane_in, &r.n_cars, &r.car_id}) put(f, *v);
    std::fclose(f);
    std::printf("recorder facade ok\n");
  } catch (const pp::Error &e) {
    std::printf("pp::Error: %s\n", e.what());
    return 2;
  }
  return 0;
}
