// C++ host adapter above the C ABI (include/fksgpu.h): the GPU sibling of
// simple_particle_contact_simulator::SimpleParticleContactSimulator for the batch calls.
//
// It mirrors the reference's interface for this path -- same names, argument meaning and error behaviour:
//   ForwardSimulateRobots / ReverseSimulateRobots   simple_particle_contact_simulator.hpp:788-804 / :806-822
//   GetStatistics / ResetStatistics                 :488-512
//   MakeGpu{SE2,SE3,Linked}Simulator                fast_kinematic_simulator.hpp:18-22 (same argument order)
//   GetDefaultSolverParameters                      fast_kinematic_simulator.hpp:13-16
// but carries no Eigen / ROS / arc_utilities types: configurations are the flat layouts of the C ABI
// (SE2: x, y, theta; SE3: row-major 3x4 [R|t]; linked: one value per active joint).  include/fksgpu_glue.hpp holds the
// glue that converts the reference's own types (Eigen::Matrix<double,3,1>, Eigen::Isometry3d, sdf_tools grids) behind
// FKSGPU_WITH_EIGEN / FKSGPU_WITH_SDF_TOOLS; INTEGRATION.md shows how a maintainer wires it into the factories.
//
// Errors: the reference asserts (asserts are live in its build, CMakeLists.txt:66).  Here argument errors and
// device errors throw std::runtime_error with the library's message; conditions the reference would abort on
// inside the simulation are reported per particle in SimulationResult::flags (FKS_FLAG_WOULD_ASSERT_*).
#ifndef FKSGPU_SIMULATOR_HPP
#define FKSGPU_SIMULATOR_HPP

#include <cstdint>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "fksgpu.h"

namespace fksgpu {

inline void Check(int code) {
    if (code != FKS_OK) throw std::runtime_error(std::string("fksgpu: ") + fks_last_error_string());
}

inline fks_solver_params GetDefaultSolverParameters() {
    fks_solver_params p;
    fks_default_solver_params(&p);
    return p;
}

// simple_simulator_interface::SimulationResult<Configuration> (spcs.hpp:918) + the per-particle counters
template <typename Configuration>
struct SimulationResult {
    Configuration result_config;
    Configuration actual_target;
    bool did_contact;
    bool outcome_is_nominal;
    uint32_t flags, n_microsteps, n_resolver_iterations, n_steps;
};

// simple_simulator_interface::ForwardSimulationStepTrace (filled at spcs.hpp:1583-1617, :1703, :1714, :1778): one entry per
// controller step holding the control input, its per-microstep share, and per microstep the configurations the resolver
// went through (post-action configuration, every correction step, the returned previous configuration on a stop).
template <typename Configuration>
struct ForwardSimulationContactResolverStepTrace {
    std::vector<Configuration> contact_resolution_steps;
};
template <typename Configuration>
struct ForwardSimulationResolverTrace {
    std::vector<double> control_input;
    std::vector<double> control_input_step;
    std::vector<ForwardSimulationContactResolverStepTrace<Configuration>> contact_resolver_steps;
};
template <typename Configuration>
struct ForwardSimulationStepTrace {
    std::vector<ForwardSimulationResolverTrace<Configuration>> resolver_steps;
};

// Environment = what the reference simulator copies at construction (spcs.hpp:420)
class Environment {
public:
    // BuildCompleteEnvironment (simulator_environment_builder.cpp:470-476)
    Environment(const std::vector<fks_obstacle>& obstacles, double resolution) : built_(nullptr) {
        Check(fks_build_environment(obstacles.data(), obstacles.size(), resolution, &built_));
    }
    ~Environment() { fks_built_env_destroy(built_); }
    Environment(const Environment&) = delete;
    Environment& operator=(const Environment&) = delete;
    const fks_env_desc& Description() const { return *fks_built_env_desc(built_); }

private:
    fks_built_env* built_;
};

// The same environment built by CUDA kernels directly in device memory (fks_env_build_device): no host grids.
class DeviceEnvironment {
public:
    // BuildCompleteEnvironment (simulator_environment_builder.cpp:470-476) on `device`
    DeviceEnvironment(const std::vector<fks_obstacle>& obstacles, double resolution, int device = 0) : env_(nullptr) {
        Check(fks_env_build_device(device, obstacles.data(), obstacles.size(), resolution, &env_));
    }
    ~DeviceEnvironment() { fks_env_destroy(env_); }
    DeviceEnvironment(const DeviceEnvironment&) = delete;
    DeviceEnvironment& operator=(const DeviceEnvironment&) = delete;
    fks_env* Handle() const { return env_; }
    // milliseconds: total, rasterise, z / y / x passes, surface marking, normal emit, distance-field check, table allocation
    std::vector<double> BuildTimingsMs() const {
        std::vector<double> ms(9, 0.0);
        Check(fks_env_build_timings(env_, ms.data(), (int)ms.size()));
        return ms;
    }

private:
    fks_env* env_;
};

template <typename Configuration>
struct ConfigTraits;  // Flatten(config, double*) / Unflatten(const double*, stride) -> config

template <>
struct ConfigTraits<std::vector<double>> {
    static void Flatten(const std::vector<double>& c, double* out, int stride) {
        if ((int)c.size() != stride) throw std::invalid_argument("fksgpu: configuration has the wrong size");
        std::memcpy(out, c.data(), sizeof(double) * (size_t)stride);
    }
    static std::vector<double> Unflatten(const double* in, int stride) { return std::vector<double>(in, in + stride); }
};

// Clean-room shim of the part of simple_simulator_interface::SimulatorInterface<Configuration, RNG, ConfigAlloc> this
// path sits behind (upstream header, absent from the reference tree; the overrides at spcs.hpp:488-512, :788-843 and :1398
// give the signatures).  The robot argument of the reference calls (`const std::shared_ptr<BaseRobotType>& immutable_robot`)
// is the robot the simulator was created with here -- the reference clones it per particle and never mutates it (:826) --
// and the display callback takes an opaque pointer instead of visualization_msgs::MarkerArray.  include/fksgpu_glue.hpp
// adapts both to the reference's own types when they are available.
template <typename Configuration>
class SimulatorInterface {
public:
    typedef SimulationResult<Configuration> Result;
    typedef std::function<void(const void*)> DisplayFn;
    virtual ~SimulatorInterface() {}
    virtual std::vector<Result> ForwardSimulateRobots(const std::vector<Configuration>& start_positions,
                                                      const std::vector<Configuration>& target_positions, bool allow_contacts,
                                                      const DisplayFn& display_fn = nullptr) = 0;                      // :788
    virtual std::vector<Result> ReverseSimulateRobots(const std::vector<Configuration>& start_positions,
                                                      const std::vector<Configuration>& target_positions, bool allow_contacts,
                                                      const DisplayFn& display_fn = nullptr) = 0;                      // :806
    virtual Result ForwardSimulateRobot(const Configuration& start, const Configuration& target, bool allow_contacts) = 0;  // :824
    virtual Result ForwardSimulateRobot(const Configuration& start, const Configuration& target, bool allow_contacts,
                                        ForwardSimulationStepTrace<Configuration>& trace, bool enable_tracing) = 0;     // :824
    virtual bool CheckConfigCollision(const Configuration& config, double inflation_ratio) = 0;                         // :1398
    virtual std::map<std::string, double> GetStatistics() = 0;                                                          // :488
    virtual void ResetStatistics() = 0;                                                                                 // :502
    virtual int32_t GetDebugLevel() const = 0;                                                                          // :446
    virtual int32_t SetDebugLevel(int32_t debug_level) = 0;                                                             // :451
};

// A recorded run of the reference (or of the CPU oracle) for the parity mode: the truncated-normal draws each particle
// consumed and, optionally, the decisions of its contact solves (fks_noise_tape in fksgpu.h).
struct NoiseTape {
    std::vector<double> draws;
    std::vector<uint64_t> offsets;           // [n + 1]
    std::vector<uint64_t> decisions;         // records of 2 + n_dof words, may be empty
    std::vector<uint64_t> decision_offsets;  // [n + 1] when decisions are given
    fks_noise_tape View() const {
        fks_noise_tape t;
        t.draws = draws.data();
        t.offsets = offsets.data();
        t.decisions = decisions.empty() ? nullptr : decisions.data();
        t.decision_offsets = decision_offsets.empty() ? nullptr : decision_offsets.data();
        return t;
    }
};

// flattens the inputs of a sequence call (starts [n][stride], targets [leg][n_targets][stride]) and returns n_targets; throws
// std::invalid_argument when there is no leg or the legs' target counts differ or are not 1 / n
template <typename Configuration>
size_t FlattenSequence(const std::vector<Configuration>& starts, const std::vector<std::vector<Configuration>>& targets_per_leg, int stride,
                       std::vector<double>* hs, std::vector<double>* ht) {
    const size_t n = starts.size(), s = (size_t)stride;
    if (targets_per_leg.empty()) throw std::invalid_argument("fksgpu: a sequence needs at least one leg");
    const size_t n_targets = targets_per_leg[0].size();
    for (const auto& leg : targets_per_leg)
        if (leg.size() != n_targets || !(n_targets == 1 || n_targets == n))
            throw std::invalid_argument("fksgpu: every leg needs the same number of targets, 1 or one per start");
    hs->resize(n * s);
    ht->resize(targets_per_leg.size() * n_targets * s);
    for (size_t i = 0; i < n; i++) ConfigTraits<Configuration>::Flatten(starts[i], hs->data() + i * s, stride);
    for (size_t k = 0; k < targets_per_leg.size(); k++)
        for (size_t i = 0; i < n_targets; i++) ConfigTraits<Configuration>::Flatten(targets_per_leg[k][i], ht->data() + (k * n_targets + i) * s, stride);
    return n_targets;
}

template <typename Configuration>
class GpuParticleContactSimulator : public SimulatorInterface<Configuration> {
public:
    typedef SimulationResult<Configuration> Result;

    GpuParticleContactSimulator(const fks_env_desc& environment, const fks_robot_desc& robot, const fks_solver_params& solver_config,
                                double simulation_controller_frequency, uint64_t prng_seed, int32_t debug_level, int device = 0)
        : env_(nullptr), robot_(nullptr), sim_(nullptr) {
        try {
            Check(fks_env_create(device, &environment, &env_));
            Check(fks_robot_create(device, &robot, &robot_));
            Check(fks_sim_create(env_, robot_, &solver_config, simulation_controller_frequency, prng_seed, debug_level, &sim_));
        } catch (...) {
            Release();
            throw;
        }
        stride_ = fks_robot_config_stride(robot_);
        record_ = fks_sim_result_stride(sim_);
        dof_ = robot.n_dof;
        debug_level_ = debug_level;
    }
    // same, in an environment that already lives on the device (shared, must outlive the simulator)
    GpuParticleContactSimulator(const std::shared_ptr<DeviceEnvironment>& environment, const fks_robot_desc& robot,
                                const fks_solver_params& solver_config, double simulation_controller_frequency, uint64_t prng_seed,
                                int32_t debug_level, int device = 0)
        : shared_env_(environment), env_(nullptr), robot_(nullptr), sim_(nullptr) {
        if (!environment) throw std::invalid_argument("fksgpu: null device environment");
        try {
            Check(fks_robot_create(device, &robot, &robot_));
            Check(fks_sim_create(environment->Handle(), robot_, &solver_config, simulation_controller_frequency, prng_seed, debug_level, &sim_));
        } catch (...) {
            Release();
            throw;
        }
        stride_ = fks_robot_config_stride(robot_);
        record_ = fks_sim_result_stride(sim_);
        dof_ = robot.n_dof;
        debug_level_ = debug_level;
    }
    ~GpuParticleContactSimulator() { Release(); }
    GpuParticleContactSimulator(const GpuParticleContactSimulator&) = delete;
    GpuParticleContactSimulator& operator=(const GpuParticleContactSimulator&) = delete;

    // spcs.hpp:788: one result per start; target_positions.size() must be 1 or start_positions.size() (assert :790-793)
    std::vector<Result> ForwardSimulateRobots(const std::vector<Configuration>& start_positions,
                                              const std::vector<Configuration>& target_positions, bool allow_contacts,
                                              const std::function<void(const void*)>& display_fn = nullptr) override {
        (void)display_fn;  // RViz markers: not on the hot path (spcs.hpp:1725-1736 only fires at debug_level >= 2)
        return Simulate(start_positions, target_positions, allow_contacts, false);
    }
    // spcs.hpp:806 (ReverseSimulateMutableRobot forwards to the forward path, :838-841)
    std::vector<Result> ReverseSimulateRobots(const std::vector<Configuration>& start_positions,
                                              const std::vector<Configuration>& target_positions, bool allow_contacts,
                                              const std::function<void(const void*)>& display_fn = nullptr) override {
        (void)display_fn;
        return Simulate(start_positions, target_positions, allow_contacts, true);
    }
    // spcs.hpp:824: single particle
    Result ForwardSimulateRobot(const Configuration& start, const Configuration& target, bool allow_contacts) override {
        return ForwardSimulateRobots(std::vector<Configuration>(1, start), std::vector<Configuration>(1, target), allow_contacts)[0];
    }

    // spcs.hpp:824 with the trace arguments: single particle, trace filled when enable_tracing is set
    Result ForwardSimulateRobot(const Configuration& start, const Configuration& target, bool allow_contacts,
                                ForwardSimulationStepTrace<Configuration>& trace, bool enable_tracing) override {
        if (!enable_tracing) return ForwardSimulateRobot(start, target, allow_contacts);
        std::vector<double> s0((size_t)stride_), t0((size_t)stride_);
        ConfigTraits<Configuration>::Flatten(start, s0.data(), stride_);
        ConfigTraits<Configuration>::Flatten(target, t0.data(), stride_);
        const size_t rec = fks_sim_trace_stride(sim_);
        std::vector<unsigned char> result(record_), records;
        size_t capacity = 4096, n = 0;
        for (;;) {  // grow until the whole trace fits (the simulation is deterministic in the particle id)
            records.resize(capacity * rec);
            Check(fks_forward_simulate_traced(sim_, s0.data(), t0.data(), allow_contacts ? 1 : 0, FKS_NOISE_PHILOX, nullptr,
                                              next_particle_id_, result.data(), records.data(), capacity, &n));
            if (n <= capacity) break;
            capacity = n;
        }
        next_particle_id_ += 1;
        for (size_t i = 0; i < n; i++) {
            fks_trace_header h;
            std::memcpy(&h, records.data() + i * rec, sizeof(h));
            const double* v = reinterpret_cast<const double*>(records.data() + i * rec + sizeof(h));
            if (h.kind == FKS_TRACE_CONTROL_INPUT) {
                trace.resolver_steps.emplace_back();
                trace.resolver_steps.back().control_input.assign(v, v + dof_);
            } else if (h.kind == FKS_TRACE_CONTROL_INPUT_STEP) {
                trace.resolver_steps.back().control_input_step.assign(v, v + dof_);
            } else {
                auto& steps = trace.resolver_steps.back().contact_resolver_steps;
                if (h.kind == FKS_TRACE_POST_ACTION) steps.emplace_back();
                steps.back().contact_resolution_steps.push_back(ConfigTraits<Configuration>::Unflatten(v, stride_));
            }
        }
        return Unpack(result.data(), target);
    }

    // M consecutive ForwardSimulateRobot legs per particle in one call (fks_forward_simulate_sequence): leg k drives every
    // particle from where leg k-1 left it to targets_per_leg[k] (1 target or one per start, the same count for every leg).
    // Returns [leg][particle]; equal to M consecutive ForwardSimulateRobots calls (the particle id advances by n * M).
    std::vector<std::vector<Result>> ForwardSimulateRobotsSequence(const std::vector<Configuration>& start_positions,
                                                                   const std::vector<std::vector<Configuration>>& targets_per_leg,
                                                                   bool allow_contacts) {
        const size_t n = start_positions.size(), m = targets_per_leg.size();
        std::vector<double> hs, ht;
        const size_t n_targets = FlattenSequence(start_positions, targets_per_leg, stride_, &hs, &ht);
        std::vector<unsigned char> rec(m * n * record_);
        fks_noise_tape view;
        const fks_noise_tape* tape = nullptr;
        if (noise_mode_ == FKS_NOISE_INJECTED) {
            if (!tape_ || tape_->offsets.size() != n + 1) throw std::invalid_argument("fksgpu: the noise tape does not match the batch");
            view = tape_->View();
            tape = &view;
        }
        Check(fks_forward_simulate_sequence(sim_, hs.data(), ht.data(), n, n_targets, m, allow_contacts ? 1 : 0, noise_mode_, tape,
                                            next_particle_id_, rec.data()));
        next_particle_id_ += n * m;
        if (noise_mode_ == FKS_NOISE_INJECTED) SetNoiseMode(FKS_NOISE_PHILOX);  // a tape describes one call
        std::vector<std::vector<Result>> out(m, std::vector<Result>(n));
        for (size_t k = 0; k < m; k++)
            for (size_t i = 0; i < n; i++)
                out[k][i] = Unpack(rec.data() + (k * n + i) * record_, n_targets == 1 ? targets_per_leg[k][0] : targets_per_leg[k][i]);
        return out;
    }

    // spcs.hpp:1398: planner-side static query (environment inflated by inflation_ratio cells, self collisions)
    bool CheckConfigCollision(const Configuration& config, double inflation_ratio) override {
        std::vector<double> flat((size_t)stride_);
        ConfigTraits<Configuration>::Flatten(config, flat.data(), stride_);
        uint8_t out = 0;
        Check(fks_check_config_collision(sim_, flat.data(), 1, inflation_ratio, &out));
        return out != 0;
    }
    std::vector<uint8_t> CheckConfigCollisions(const std::vector<Configuration>& configs, double inflation_ratio) {
        std::vector<double> flat(configs.size() * (size_t)stride_);
        for (size_t i = 0; i < configs.size(); i++) ConfigTraits<Configuration>::Flatten(configs[i], flat.data() + i * (size_t)stride_, stride_);
        std::vector<uint8_t> out(configs.size(), 0);
        Check(fks_check_config_collision(sim_, flat.data(), configs.size(), inflation_ratio, out.data()));
        return out;
    }

    // spcs.hpp:488-500, same keys
    std::map<std::string, double> GetStatistics() override {
        uint64_t s[FKS_NUM_STATS];
        Check(fks_get_statistics(sim_, s));
        std::map<std::string, double> out;
        out["successful_resolves"] = (double)s[FKS_STAT_SUCCESSFUL_RESOLVES];
        out["unsuccessful_resolves"] = (double)s[FKS_STAT_UNSUCCESSFUL_RESOLVES];
        out["free_resolves"] = (double)s[FKS_STAT_FREE_RESOLVES];
        out["collision_resolves"] = (double)s[FKS_STAT_COLLISION_RESOLVES];
        out["fallback_resolves"] = (double)s[FKS_STAT_FALLBACK_RESOLVES];
        out["unsuccessful_self_collision_resolves"] = (double)s[FKS_STAT_UNSUCCESSFUL_SELF_COLLISION_RESOLVES];
        out["unsuccessful_env_collision_resolves"] = (double)s[FKS_STAT_UNSUCCESSFUL_ENV_COLLISION_RESOLVES];
        out["recovered_unsuccessful_resolves"] = (double)s[FKS_STAT_RECOVERED_UNSUCCESSFUL_RESOLVES];
        return out;
    }
    void ResetStatistics() override { Check(fks_reset_statistics(sim_)); }  // spcs.hpp:502-512
    int32_t GetDebugLevel() const override { return debug_level_; }               // spcs.hpp:446-449
    int32_t SetDebugLevel(int32_t debug_level) override {                         // spcs.hpp:451-455 (messages only; no device effect)
        debug_level_ = debug_level;
        return debug_level_;
    }

    // noise: Philox keyed by (prng_seed, first_particle_id + index); the id offset advances per call so that
    // successive calls draw fresh noise, as the reference's per-thread generators do
    void SetNextParticleId(uint64_t id) { next_particle_id_ = id; }
    // FKS_NOISE_PHILOX (default) or FKS_NOISE_NONE for the calls that follow
    void SetNoiseMode(int noise_mode) {
        if (noise_mode != FKS_NOISE_PHILOX && noise_mode != FKS_NOISE_NONE)
            throw std::invalid_argument("fksgpu: SetNoiseMode takes FKS_NOISE_PHILOX or FKS_NOISE_NONE; a tape goes through SetNoiseTape");
        noise_mode_ = noise_mode;
        tape_.reset();
    }
    // parity mode: the NEXT batch call consumes this recorded run (one entry per start position) instead of drawing noise
    void SetNoiseTape(const std::shared_ptr<const NoiseTape>& tape) {
        if (!tape || tape->offsets.size() < 2) throw std::invalid_argument("fksgpu: empty noise tape");
        tape_ = tape;
        noise_mode_ = FKS_NOISE_INJECTED;
    }
    int ConfigStride() const { return stride_; }
    const char* KernelInfo() { return fks_sim_kernel_info(sim_); }

private:
    std::vector<Result> Simulate(const std::vector<Configuration>& starts, const std::vector<Configuration>& targets,
                                 bool allow_contacts, bool reverse) {
        const size_t n = starts.size();
        if (!(targets.size() == 1 || targets.size() == n)) throw std::invalid_argument("fksgpu: need 1 target or one per start");
        std::vector<double> hs(n * (size_t)stride_), ht(targets.size() * (size_t)stride_);
        for (size_t i = 0; i < n; i++) ConfigTraits<Configuration>::Flatten(starts[i], hs.data() + i * (size_t)stride_, stride_);
        for (size_t i = 0; i < targets.size(); i++) ConfigTraits<Configuration>::Flatten(targets[i], ht.data() + i * (size_t)stride_, stride_);
        std::vector<unsigned char> rec(n * record_);
        fks_noise_tape view;
        const fks_noise_tape* tape = nullptr;
        if (noise_mode_ == FKS_NOISE_INJECTED) {
            if (!tape_ || tape_->offsets.size() != n + 1) throw std::invalid_argument("fksgpu: the noise tape does not match the batch");
            view = tape_->View();
            tape = &view;
        }
        Check((reverse ? fks_reverse_simulate : fks_forward_simulate)(sim_, hs.data(), ht.data(), n, targets.size(), allow_contacts ? 1 : 0,
                                                                     noise_mode_, tape, next_particle_id_, rec.data()));
        next_particle_id_ += n;
        if (noise_mode_ == FKS_NOISE_INJECTED) SetNoiseMode(FKS_NOISE_PHILOX);  // a tape describes one batch
        std::vector<Result> out(n);
        for (size_t i = 0; i < n; i++) out[i] = Unpack(rec.data() + i * record_, targets.size() == 1 ? targets[0] : targets[i]);
        return out;
    }
    Result Unpack(const unsigned char* r, const Configuration& target) const {
        Result out;
        fks_result_tail tail;
        std::memcpy(&tail, r + sizeof(double) * (size_t)stride_, sizeof(tail));
        out.result_config = ConfigTraits<Configuration>::Unflatten(reinterpret_cast<const double*>(r), stride_);
        out.actual_target = target;
        out.did_contact = (tail.flags & FKS_FLAG_DID_CONTACT) != 0;  // spcs.hpp:918
        out.outcome_is_nominal = true;                               // always true in the reference (:918)
        out.flags = tail.flags;
        out.n_microsteps = tail.n_microsteps;
        out.n_resolver_iterations = tail.n_resolver_iters;
        out.n_steps = tail.n_steps;
        return out;
    }
    void Release() {
        fks_sim_destroy(sim_);
        fks_robot_destroy(robot_);
        fks_env_destroy(env_);
        sim_ = nullptr;
        robot_ = nullptr;
        env_ = nullptr;
    }

    std::shared_ptr<DeviceEnvironment> shared_env_;  // set when the environment is not owned (env_ stays null)
    fks_env* env_;
    fks_robot* robot_;
    fks_sim* sim_;
    int stride_ = 0, dof_ = 0;
    size_t record_ = 0;
    uint64_t next_particle_id_ = 0;
    int noise_mode_ = FKS_NOISE_PHILOX;
    int32_t debug_level_ = 0;
    std::shared_ptr<const NoiseTape> tape_;
};

// The same batch calls over several GPUs of one box (fks_multi_* in fksgpu.h): contiguous particle shards, environment and
// robot replicated per device, records independent of the device count (Philox noise is keyed by the global particle id).
template <typename Configuration>
class MultiGpuParticleContactSimulator {
public:
    typedef SimulationResult<Configuration> Result;
    // devices empty: devices 0 .. n_devices-1
    MultiGpuParticleContactSimulator(const std::vector<int32_t>& devices, int32_t n_devices, const fks_env_desc& environment,
                                     const fks_robot_desc& robot, const fks_solver_params& solver_config,
                                     double simulation_controller_frequency, uint64_t prng_seed, int32_t debug_level)
        : sim_(nullptr) {
        Check(fks_multi_sim_create(devices.empty() ? nullptr : devices.data(), devices.empty() ? n_devices : (int32_t)devices.size(),
                                   &environment, &robot, &solver_config, simulation_controller_frequency, prng_seed, debug_level, &sim_));
        stride_ = robot.kind == FKS_ROBOT_SE2 ? 3 : (robot.kind == FKS_ROBOT_SE3 ? 12 : robot.n_dof);
        record_ = fks_multi_sim_result_stride(sim_);
    }
    ~MultiGpuParticleContactSimulator() { fks_multi_sim_destroy(sim_); }
    MultiGpuParticleContactSimulator(const MultiGpuParticleContactSimulator&) = delete;
    MultiGpuParticleContactSimulator& operator=(const MultiGpuParticleContactSimulator&) = delete;
    int DeviceCount() const { return fks_multi_sim_device_count(sim_); }

    // spcs.hpp:788 over all devices
    std::vector<Result> ForwardSimulateRobots(const std::vector<Configuration>& starts, const std::vector<Configuration>& targets,
                                              bool allow_contacts) {
        const size_t n = starts.size();
        if (!(targets.size() == 1 || targets.size() == n)) throw std::invalid_argument("fksgpu: need 1 target or one per start");
        std::vector<double> hs(n * (size_t)stride_), ht(targets.size() * (size_t)stride_);
        for (size_t i = 0; i < n; i++) ConfigTraits<Configuration>::Flatten(starts[i], hs.data() + i * (size_t)stride_, stride_);
        for (size_t i = 0; i < targets.size(); i++) ConfigTraits<Configuration>::Flatten(targets[i], ht.data() + i * (size_t)stride_, stride_);
        std::vector<unsigned char> rec(n * record_);
        Check(fks_multi_forward_simulate(sim_, hs.data(), ht.data(), n, targets.size(), allow_contacts ? 1 : 0, FKS_NOISE_PHILOX, nullptr,
                                         next_particle_id_, rec.data()));
        next_particle_id_ += n;
        std::vector<Result> out(n);
        for (size_t i = 0; i < n; i++) out[i] = Unpack(rec.data() + i * record_, targets.size() == 1 ? targets[0] : targets[i]);
        return out;
    }
    // GpuParticleContactSimulator::ForwardSimulateRobotsSequence over all devices
    std::vector<std::vector<Result>> ForwardSimulateRobotsSequence(const std::vector<Configuration>& starts,
                                                                   const std::vector<std::vector<Configuration>>& targets_per_leg,
                                                                   bool allow_contacts) {
        const size_t n = starts.size(), m = targets_per_leg.size();
        std::vector<double> hs, ht;
        const size_t n_targets = FlattenSequence(starts, targets_per_leg, stride_, &hs, &ht);
        std::vector<unsigned char> rec(m * n * record_);
        Check(fks_multi_forward_simulate_sequence(sim_, hs.data(), ht.data(), n, n_targets, m, allow_contacts ? 1 : 0, FKS_NOISE_PHILOX,
                                                  nullptr, next_particle_id_, rec.data()));
        next_particle_id_ += n * m;
        std::vector<std::vector<Result>> out(m, std::vector<Result>(n));
        for (size_t k = 0; k < m; k++)
            for (size_t i = 0; i < n; i++)
                out[k][i] = Unpack(rec.data() + (k * n + i) * record_, n_targets == 1 ? targets_per_leg[k][0] : targets_per_leg[k][i]);
        return out;
    }
    std::vector<uint64_t> GetStatisticCounters() {
        std::vector<uint64_t> s(FKS_NUM_STATS);
        Check(fks_multi_get_statistics(sim_, s.data()));
        return s;
    }
    void ResetStatistics() { Check(fks_multi_reset_statistics(sim_)); }
    void SetNextParticleId(uint64_t id) { next_particle_id_ = id; }

private:
    Result Unpack(const unsigned char* r, const Configuration& target) const {
        Result out;
        fks_result_tail tail;
        std::memcpy(&tail, r + sizeof(double) * (size_t)stride_, sizeof(tail));
        out.result_config = ConfigTraits<Configuration>::Unflatten(reinterpret_cast<const double*>(r), stride_);
        out.actual_target = target;
        out.did_contact = (tail.flags & FKS_FLAG_DID_CONTACT) != 0;
        out.outcome_is_nominal = true;
        out.flags = tail.flags;
        out.n_microsteps = tail.n_microsteps;
        out.n_resolver_iterations = tail.n_resolver_iters;
        out.n_steps = tail.n_steps;
        return out;
    }

    fks_multi_sim* sim_;
    int stride_ = 0;
    size_t record_ = 0;
    uint64_t next_particle_id_ = 0;
};

typedef GpuParticleContactSimulator<std::vector<double>> GpuSimulator;
typedef std::shared_ptr<GpuSimulator> GpuSimulatorPtr;

// fast_kinematic_simulator.hpp:18-22, same argument order (grid + SDF + surface normals = one fks_env_desc)
inline GpuSimulatorPtr MakeGpuSimulator(int kind, const fks_env_desc& environment, const fks_robot_desc& robot,
                                        const fks_solver_params& solver_config, double simulation_controller_frequency,
                                        uint64_t prng_seed, int32_t debug_level) {
    if (robot.kind != kind) throw std::invalid_argument("fksgpu: robot description does not match the factory");
    return GpuSimulatorPtr(new GpuSimulator(environment, robot, solver_config, simulation_controller_frequency, prng_seed, debug_level));
}
inline GpuSimulatorPtr MakeGpuSimulator(int kind, const std::shared_ptr<DeviceEnvironment>& environment, const fks_robot_desc& robot,
                                        const fks_solver_params& solver_config, double simulation_controller_frequency,
                                        uint64_t prng_seed, int32_t debug_level) {
    if (robot.kind != kind) throw std::invalid_argument("fksgpu: robot description does not match the factory");
    return GpuSimulatorPtr(new GpuSimulator(environment, robot, solver_config, simulation_controller_frequency, prng_seed, debug_level));
}
inline GpuSimulatorPtr MakeGpuSE2Simulator(const fks_env_desc& e, const fks_robot_desc& r, const fks_solver_params& p, double f, uint64_t seed, int32_t dbg) {
    return MakeGpuSimulator(FKS_ROBOT_SE2, e, r, p, f, seed, dbg);
}
inline GpuSimulatorPtr MakeGpuSE3Simulator(const fks_env_desc& e, const fks_robot_desc& r, const fks_solver_params& p, double f, uint64_t seed, int32_t dbg) {
    return MakeGpuSimulator(FKS_ROBOT_SE3, e, r, p, f, seed, dbg);
}
inline GpuSimulatorPtr MakeGpuLinkedSimulator(const fks_env_desc& e, const fks_robot_desc& r, const fks_solver_params& p, double f, uint64_t seed, int32_t dbg) {
    return MakeGpuSimulator(FKS_ROBOT_LINKED, e, r, p, f, seed, dbg);
}

}  // namespace fksgpu

#endif  // FKSGPU_SIMULATOR_HPP
