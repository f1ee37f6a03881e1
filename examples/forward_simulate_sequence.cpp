// A plan executed as one call: 64 SE(2) particles are pushed into a wall, pulled back to where they started and driven to a
// third waypoint by fksgpu::GpuSimulator::ForwardSimulateRobotsSequence, and the same three legs are run again on a fresh
// simulator as three consecutive ForwardSimulateRobots calls, each starting from the previous call's end states.
//   g++ -std=c++11 -Iinclude examples/forward_simulate_sequence.cpp -Lfast_kinematic_simulator_b200 -lfksgpu -Wl,-rpath,... -o /tmp/seq
// Exit code 0 and "ok" when both give the same end states and counters for every leg and particle; 3 when no GPU is present
// (the library has no CPU fallback and says so).
#include <cstdio>
#include <cstring>

#include "fksgpu_simulator.hpp"

int main() {
    fks_obstacle wall;
    const double pose[12] = {1, 0, 0, 1.25, 0, 1, 0, 0.0, 0, 0, 1, 0.05};
    for (int i = 0; i < 12; i++) wall.pose[i] = pose[i];
    wall.extents[0] = 0.25; wall.extents[1] = 2.0; wall.extents[2] = 0.5;
    wall.object_id = 1; wall._pad = 0;
    fksgpu::Environment env(std::vector<fks_obstacle>(1, wall), 0.125);

    const double point[3] = {0.0, 0.0, 0.0};
    const int32_t link0 = 0;
    fks_axis_params axes[3];
    for (int i = 0; i < 3; i++) {
        axes[i].kp = 1.0; axes[i].ki = 0.0; axes[i].kd = 0.0; axes[i].integral_clamp = 0.0;
        axes[i].velocity_limit = (i < 2) ? 1.0 : 0.5;
        axes[i].proportional_noise = 0.1; axes[i].minimum_noise = 0.01; axes[i].noise_sigma = 0.5;
    }
    fks_robot_desc robot;
    std::memset(&robot, 0, sizeof(robot));
    robot.kind = FKS_ROBOT_SE2; robot.n_links = 1; robot.n_joints = 0; robot.n_dof = 3; robot.n_points = 1;
    robot.points_xyz = point; robot.point_link = &link0; robot.axes = axes;
    robot.position_distance_weight = 1.0; robot.rotation_distance_weight = 1.0;

    try {
        typedef std::vector<std::vector<double>> Configs;
        const Configs starts(64, std::vector<double>{0.6, 0.0, 0.0});
        std::vector<Configs> legs;
        legs.push_back(Configs(1, std::vector<double>{1.4, 0.0, 0.0}));   // into the wall
        legs.push_back(Configs(1, std::vector<double>{0.6, 0.0, 0.0}));   // back to the start
        legs.push_back(Configs(1, std::vector<double>{0.4, 0.5, 0.3}));   // a third waypoint
        fksgpu::GpuSimulatorPtr seq = fksgpu::MakeGpuSE2Simulator(env.Description(), robot, fksgpu::GetDefaultSolverParameters(), 25.0, 42, 0);
        const auto sequence = seq->ForwardSimulateRobotsSequence(starts, legs, true);

        fksgpu::GpuSimulatorPtr chain = fksgpu::MakeGpuSE2Simulator(env.Description(), robot, fksgpu::GetDefaultSolverParameters(), 25.0, 42, 0);
        Configs at = starts;
        int differ = 0, contacts = 0;
        for (size_t k = 0; k < legs.size(); k++) {
            const auto step = chain->ForwardSimulateRobots(at, legs[k], true);
            for (size_t i = 0; i < step.size(); i++) {
                const auto& a = sequence[k][i];
                const auto& b = step[i];
                if (a.result_config != b.result_config || a.flags != b.flags || a.n_microsteps != b.n_microsteps ||
                    a.n_resolver_iterations != b.n_resolver_iterations || a.n_steps != b.n_steps)
                    differ++;
                at[i] = b.result_config;
            }
        }
        for (const auto& r : sequence[0]) contacts += r.did_contact ? 1 : 0;
        const auto s1 = seq->GetStatistics(), s2 = chain->GetStatistics();
        if (s1 != s2) differ++;
        // legs with different target counts are an argument error
        bool rejected = false;
        std::vector<Configs> ragged = legs;
        ragged[1] = Configs(2, std::vector<double>{0.6, 0.0, 0.0});
        try {
            seq->ForwardSimulateRobotsSequence(starts, ragged, true);
        } catch (const std::invalid_argument&) {
            rejected = true;
        }
        const bool ok = differ == 0 && contacts == 64 && rejected;
        std::printf("%zu legs x %zu particles, %d in contact on leg 0, %d records / statistics differ from the chain of single calls, "
                    "ragged legs %s\n%s\n", sequence.size(), starts.size(), contacts, differ, rejected ? "rejected" : "ACCEPTED",
                    ok ? "ok" : "FAILED");
        return ok ? 0 : 1;
    } catch (const std::exception& e) {
        std::printf("no device path: %s\n", e.what());
        return 3;
    }
}
