// C++ host driving libmrsb through the façade the way a multi-UAV node does every tick, without stalling the GPU: the commands
// that arrived since the last tick go up as mixed-mode rows (Swarm::setInputRowsAsync, a UAV may appear twice: the later row wins),
// one tick of makeStep + handleCollisions (Swarm::run), then positions and odometry | IMU | range rows of a followed subset come
// down (Swarm::getPositionsAsync / getObservationsAsync).  Host buffers are two deep: the rows of tick t are written while tick
// t - 1 may still compute, and the downloads of tick t - 1 are read while tick t computes.  256 x500 on a 2 m grid, 40 ticks.
// Prints a few facts as JSON; tests/test_node_io_gpu.py compares them with the same flight driven through the blocking Python calls.
#include <cstdio>
#include <vector>

#include "mrsb/uav_system.hpp"

static const int kN = 256, kTicks = 40, kSub = 96, kStride = 4;

// The commands of tick t: UAV i gets one when (7 i + 3 t) % 8 == 0, in the mode (i / 8 + t) % 4 picks; the first of them also gets a
// second row in the next mode (the later one wins).  Rows of 4 doubles.
static void commands(int t, std::vector<int32_t>& idx, std::vector<int32_t>& modes, std::vector<double>& rows) {
  static const int32_t kModes[4] = {MRSB_VELOCITY_HDG_RATE_CMD, MRSB_VELOCITY_HDG_CMD, MRSB_POSITION_CMD, MRSB_ACCELERATION_HDG_RATE_CMD};
  idx.clear(), modes.clear(), rows.clear();
  auto add = [&](int i, int m) {
    idx.push_back(i);
    modes.push_back(kModes[m]);
    if (kModes[m] == MRSB_POSITION_CMD) {
      rows.insert(rows.end(), {2.0 * (i % 16) + 0.5, 2.0 * (i / 16) - 0.5, 3.0 + 0.25 * (t % 4), 0.3});
    } else if (kModes[m] == MRSB_ACCELERATION_HDG_RATE_CMD) {
      rows.insert(rows.end(), {0.2 * ((i + t) % 3 - 1), 0.1, 0.0, 0.05});
    } else {
      rows.insert(rows.end(), {0.1 * ((i + t) % 7 - 3), 0.1 * ((3 * i + t) % 5 - 2), 0.05 * ((i + 2 * t) % 3), 0.01 * (i % 100)});
    }
  };
  for (int i = 0; i < kN; i++)
    if ((7 * i + 3 * t) % 8 == 0) add(i, (i / 8 + t) % 4);
  if (!idx.empty()) add(idx[0], (idx[0] + t + 1) % 4);
}

int main() {
  try {
    mrsb_model_params x500     = mrsb::defaultModelParams();
    x500.takeoff_patch_enabled = 0;
    x500.ground_enabled        = 1;
    x500.ground_z              = 0.0;
    std::vector<std::array<double, 3>> spawn;
    std::vector<double>                heading(kN, 0.0);
    for (int i = 0; i < kN; i++) spawn.push_back({2.0 * (i % 16), 2.0 * (i / 16), 3.0});
    mrsb::Swarm swarm({x500}, {}, spawn, heading);
    swarm.setCollisions(true, false, 100.0);
    std::vector<int32_t> sub(kSub);
    for (int j = 0; j < kSub; j++) sub[size_t(j)] = int32_t((37 * j + 11) % kN);  // a followed subset in scrambled order
    swarm.setPositionSubset(kSub, sub.data());
    std::vector<double> hover(size_t(kN) * kStride, 0.0);
    swarm.setInputAsync(MRSB_VELOCITY_HDG_RATE_CMD, hover.data(), kStride);

    std::vector<int32_t> idx[2], modes[2];
    std::vector<double>  rows[2], pos[2], obs[2];
    for (int k = 0; k < 2; k++) pos[k].resize(size_t(kSub) * 3), obs[k].resize(size_t(kSub) * 17);
    double pos_sum = 0.0, obs_sum = 0.0;
    int    n_rows  = 0;
    auto   publish = [&](int k) {  // what the node publishes from the downloads of one tick
      for (int j = 0; j < kSub; j++) {
        const double* p = &pos[k][size_t(j) * 3];
        const double* o = &obs[k][size_t(j) * 17];
        pos_sum += p[0] + 2.0 * p[1] + 3.0 * p[2];
        obs_sum += o[0] + o[3] + o[6] + o[7] + o[13] + o[16];
      }
    };
    for (int t = 0; t < kTicks; t++) {
      const int k = t & 1;
      swarm.waitUploads();  // the rows of tick t - 2 (and t - 1) are on the device: buffer k may be refilled
      commands(t, idx[k], modes[k], rows[k]);
      n_rows += int(idx[k].size());
      swarm.setInputRowsAsync(int64_t(idx[k].size()), idx[k].data(), modes[k].data(), rows[k].data(), kStride);
      swarm.run(0.01, 1);
      if (t > 0) {
        swarm.waitDownloads();  // the downloads of tick t - 1, while tick t computes
        publish(k ^ 1);
      }
      swarm.getPositionsAsync(pos[k].data());
      swarm.getObservationsAsync(obs[k].data());
    }
    swarm.sync();
    publish((kTicks - 1) & 1);
    std::printf("{\"pos\": %.17g, \"obs\": %.17g, \"rows\": %d, \"pairs\": %zu}\n", pos_sum, obs_sum, n_rows, swarm.collisionPairs().size());
    return 0;
  } catch (const std::exception& e) {
    std::fprintf(stderr, "error: %s\n", e.what());
    return 3;
  }
}
