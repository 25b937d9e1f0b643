// C++ host running RL-style episodes through the façade: 512 x500 fly position commands; every 50 ticks the UAVs that are "done"
// (crashed, or past their target) start a new episode through Swarm::respawn, one more through UavSystem::respawn, and all of
// them get a new command.  Prints a few facts as JSON; tests/test_respawn_gpu.py compares them with the same episodes driven
// through the Python mirror.
#include <cstdio>
#include <vector>

#include "mrsb/uav_system.hpp"

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
      spawn.push_back({4.0 * (i % 32), 4.0 * (i / 32), 0.0});
      heading.push_back(0.01 * i);
    }
    mrsb::Swarm swarm({x500}, {}, spawn, heading);
    int respawned = 0;
    for (int episode = 0; episode < 4; episode++) {
      for (int i = 0; i < n; i++) {
        mrsb::reference::Position cmd;
        cmd.position = {spawn[i][0] + 0.5 * ((i + episode) % 5), spawn[i][1] - 0.25 * ((i + episode) % 3), 2.0 + 0.1 * (i % 7)};
        cmd.heading  = 0.1 * episode;
        swarm[i].setInput(cmd);
      }
      if (episode == 1)
        for (int i = 0; i < n; i += 9) swarm[i].crash();
      swarm.run(0.01, 50, 2, false);
      std::vector<int32_t> done;
      std::vector<double>  xyz, hdg;
      for (int i = 0; i < n; i++) {
        const mrsb::State s = swarm[i].getState();
        if (swarm[i].hasCrashed() || s.x[0] > spawn[i][0] + 1.0) {
          done.push_back(i);
          xyz.insert(xyz.end(), {spawn[i][0], spawn[i][1], 0.5 * episode});
          hdg.push_back(-0.02 * i);
        }
      }
      swarm.respawn(int64_t(done.size()), done.data(), xyz.data(), hdg.data());
      swarm[1].respawn({1.0, 2.0, 3.0}, 0.5);
      respawned += int(done.size()) + 1;
    }
    double sum = 0.0;
    int    crashed = 0;
    for (int i = 0; i < n; i++) {
      const mrsb::State s = swarm[i].getState();
      sum += s.x[0] + 2.0 * s.x[1] + 3.0 * s.x[2] + s.v[2] + s.motor_rpm[0];
      crashed += swarm[i].hasCrashed() ? 1 : 0;
    }
    const mrsb::State one = swarm[1].getState();
    std::printf("{\"sum\": %.17g, \"respawned\": %d, \"crashed\": %d, \"one_x\": [%.17g, %.17g, %.17g], \"one_rpm0\": %.17g, \"one_takeoff\": %d}\n", sum,
                respawned, crashed, one.x[0], one.x[1], one.x[2], one.motor_rpm[0], swarm[1].getParams().takeoff_patch_enabled);
    return 0;
  } catch (const std::exception& e) {
    std::fprintf(stderr, "error: %s\n", e.what());
    return 3;
  }
}
