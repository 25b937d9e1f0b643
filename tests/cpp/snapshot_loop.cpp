// C++ host branching rollouts through the façade: 512 x500 fly position commands with collisions; a snapshot taken after 100
// ticks is the start of three branches of 50 ticks (the first continues, the second restores every UAV's own record, the third
// gives UAV i the record of UAV (i + 34) % 512), and its host image resumes on a second Swarm.  Prints a few facts as JSON;
// tests/test_snapshot_gpu.py compares them with the same branches driven through the Python mirror.
#include <cstdio>
#include <vector>

#include "mrsb/uav_system.hpp"

static double checksum(mrsb::Swarm& swarm) {
  double sum = 0.0;
  for (int i = 0; i < swarm.size(); i++) {
    const mrsb::State s = swarm[i].getState();
    sum += s.x[0] + 2.0 * s.x[1] + 3.0 * s.x[2] + s.v[2];
  }
  return sum;
}

int main() {
  try {
    const int         n    = 512;
    mrsb_model_params x500 = mrsb::defaultModelParams();
    x500.ground_enabled        = 1;
    x500.ground_z              = 0.0;
    x500.takeoff_patch_enabled = 1;
    std::vector<mrsb::Vec3> spawn;
    std::vector<double>     heading;
    for (int i = 0; i < n; i++) {
      spawn.push_back({1.5 * (i % 32), 1.5 * (i / 32), 0.0});
      heading.push_back(0.01 * i);
    }
    mrsb::Swarm swarm({x500}, {}, spawn, heading);
    swarm.setCollisions(true, false, 100.0);
    for (int i = 0; i < n; i++) {
      mrsb::reference::Position cmd;
      cmd.position = {spawn[i][0] + 0.5 * (i % 5), spawn[i][1] - 0.25 * (i % 3), 2.0 + 0.1 * (i % 7)};
      cmd.heading  = 0.3;
      swarm[i].setInput(cmd);
    }
    swarm.run(0.01, 100);
    const int32_t id = swarm.snapshotCreate();
    swarm.snapshotSave(id);
    std::vector<double> sums;
    for (int branch = 0; branch < 3; branch++) {
      if (branch == 1) swarm.snapshotRestore(id, n);
      if (branch == 2) {
        std::vector<int32_t> src(n);
        for (int i = 0; i < n; i++) src[size_t(i)] = (i + 34) % n;
        swarm.snapshotRestore(id, n, nullptr, src.data());
      }
      swarm.run(0.01, 50);
      sums.push_back(checksum(swarm));
    }
    const std::vector<unsigned char> image = swarm.snapshotImage(id);
    swarm.snapshotFree(id);

    mrsb::Swarm twin({x500}, {}, spawn, heading);
    twin.setCollisions(true, false, 100.0);
    const int32_t tid = twin.snapshotCreate();
    twin.snapshotLoad(tid, image);
    twin.snapshotRestore(tid, n);
    twin.run(0.01, 50);
    std::printf("{\"sums\": [%.17g, %.17g, %.17g], \"resumed\": %.17g, \"image_bytes\": %zu, \"pairs\": %zu}\n", sums[0], sums[1], sums[2],
                checksum(twin), image.size(), swarm.collisionPairs().size());
    return 0;
  } catch (const std::exception& e) {
    std::fprintf(stderr, "error: %s\n", e.what());
    return 3;
  }
}
