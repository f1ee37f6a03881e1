/*
 * fksgpu.h -- C ABI of the B200-native batched particle contact simulator.
 *
 * This is the drop-in boundary for ONE path of calderpg/fast_kinematic_simulator:
 * the batched forward simulation of uncertain "particles"
 *   SimpleParticleContactSimulator::ForwardSimulateRobots
 *     (include/fast_kinematic_simulator/simple_particle_contact_simulator.hpp:788-804,
 *      alias ReverseSimulateRobots :806-822)
 * and everything it calls per particle (:824-919 step loop, :1546-1816 microstep +
 * resolver loop, :921-981 env check, :983-1275 self collision, :1818-1939 corrections,
 * :1990-1998 stacked-Jacobian solve; robots tnuva_robot_models.hpp, actuator noise
 * simple_uncertainty_models.hpp:48-90, PID simple_pid_controller.hpp:98-135).
 *
 * The reference has no FFI; its boundary is the C++ virtual interface
 * simple_simulator_interface::SimulatorInterface (spcs.hpp:372) created by the factories in
 * fast_kinematic_simulator.hpp:18-22.  A C++ adapter (include/fksgpu_simulator.hpp) mirrors that interface on top of
 * the functions below (include/fksgpu_glue.hpp derives it from the reference's own types); INTEGRATION.md shows the binding.
 *
 * Conventions
 *  - plain C, opaque handles, int status return (0 = FKS_OK), no exceptions cross the boundary;
 *  - rigid transforms are 12 doubles, row-major 3x4 [R | t];
 *  - configurations are flat doubles: SE2 (x,y,theta) = 3, SE3 = 12 (row-major 3x4 [R|t],
 *    never quaternions), linked = one value per ACTIVE joint in joint order;
 *  - all arithmetic on the device is FP64 except SDF storage (float) and cell indices (int64).
 */
#ifndef FKSGPU_H
#define FKSGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FKS_ABI_VERSION 2

/* ---- status codes ------------------------------------------------------------------------ */
enum {
    FKS_OK = 0,
    FKS_ERR_INVALID_ARGUMENT = 1,
    FKS_ERR_CUDA = 2,
    FKS_ERR_NO_DEVICE = 3,
    FKS_ERR_UNSUPPORTED = 4,
    FKS_ERR_OUT_OF_MEMORY = 5
};

/* ---- robot kinds (tnuva_robot_models.hpp:26,201,415) -------------------------------------- */
enum { FKS_ROBOT_SE2 = 0, FKS_ROBOT_SE3 = 1, FKS_ROBOT_LINKED = 2 };

/* ---- joint types (arc_utilities SimpleJointModel; call sites tnuva.hpp:544-559) ----------- */
enum { FKS_JOINT_PRISMATIC = 0, FKS_JOINT_REVOLUTE = 1, FKS_JOINT_CONTINUOUS = 2, FKS_JOINT_FIXED = 3 };

/* ---- noise source ------------------------------------------------------------------------- */
enum {
    FKS_NOISE_PHILOX = 0,   /* counter-based Philox4x32-10 keyed by (seed, particle, step, microstep, dof) */
    FKS_NOISE_INJECTED = 1, /* consume a caller-provided tape of truncated-normal draws (parity mode)      */
    FKS_NOISE_NONE = 2      /* all draws are 0.0 (deterministic debugging)                                  */
};

/* ---- per-particle result flags (bit field in fks_result_tail.flags) ----------------------- */
enum {
    FKS_FLAG_DID_CONTACT        = 1u << 0, /* SimulationResult::did_contact (spcs.hpp:879,918)          */
    FKS_FLAG_RESOLVE_FAILED     = 1u << 1, /* some ResolveForwardSimulation returned failed (:1745)      */
    FKS_FLAG_ENDED_BY_FAILURE   = 1u << 2, /* failed_resolves_end_motion break (:884-887)                */
    FKS_FLAG_ENDED_BY_NOCONTACT = 1u << 3, /* allow_contacts==false stop (:904-909)                      */
    FKS_FLAG_ENDED_BY_SHORTCUT  = 1u << 4, /* simulation_shortcut_distance break (:898-902)              */
    /* conditions on which the reference would abort() (asserts are live, CMakeLists.txt:66);
       the device path records them and keeps going with the documented behaviour instead. */
    FKS_FLAG_WOULD_ASSERT_MICROSTEP = 1u << 8,  /* microstep motion > resolution (:1570-1575)           */
    FKS_FLAG_WOULD_ASSERT_NORMAL    = 1u << 9,  /* zero motion / OOB in normal lookup (:91-92,:1882)     */
    FKS_FLAG_WOULD_ASSERT_NAN       = 1u << 10, /* NaN/Inf control input (unc.hpp:72-73)                 */
    FKS_FLAG_EMPTY_JACOBIAN         = 1u << 11, /* resolver entered with no correcting point             */
    FKS_FLAG_TAPE_EXHAUSTED         = 1u << 12, /* injected tape shorter than the draws consumed         */
    FKS_FLAG_NEAR_RANK_CUT          = 1u << 13, /* a QR pivot came within 1e3x of Eigen's rank threshold
                                                   (result is round-off determined in the reference)    */
    FKS_FLAG_J_SPILLED              = 1u << 14, /* stacked Jacobian exceeded the shared-memory tile     */
    /* parity mode with a decision tape (fks_noise_tape.decisions) only: */
    FKS_FLAG_DECISION_OVERRIDDEN    = 1u << 15, /* the device's own pivot order / rank differed from the
                                                   injected one, or a round-off solution was injected   */
    FKS_FLAG_DECISION_DESYNC        = 1u << 16  /* the tape ran out or its row count did not match the
                                                   device's stacked system: trajectories have diverged  */
};

/* spcs.hpp:345-369 (same field order, defaults :357-368) */
typedef struct fks_solver_params {
    double forward_simulation_time;
    double simulation_shortcut_distance;
    double environment_collision_check_tolerance;
    double resolve_correction_step_scaling_decay_rate;
    double resolve_correction_initial_step_size;
    double resolve_correction_min_step_scaling;
    uint32_t max_resolver_iterations;
    uint32_t resolve_correction_step_scaling_decay_iterations;
    int32_t failed_resolves_end_motion;
    int32_t _pad;
} fks_solver_params;

/* Environment: what SimpleParticleContactSimulator copies at construction (spcs.hpp:420):
 * collision-map METADATA (cells are never read on the hot path), the SDF floats and the
 * SurfaceNormalGrid (spcs.hpp:44-343) flattened to a sparse CSR-like table. */
typedef struct fks_env_desc {
    double origin[12];          /* grid origin transform (VoxelGrid), world <- grid              */
    double inverse_origin[12];  /* grid <- world (GetInverseOriginTransform, spcs.hpp:1176)       */
    double map_resolution;      /* environment_.GetResolution() (spcs.hpp:524-527,1560,1219)      */
    double sdf_resolution;      /* environment_sdf_.GetResolution() (spcs.hpp:923,957)            */
    int64_t nx, ny, nz;         /* cells; linear index = (x*ny + y)*nz + z                        */
    const float* sdf;           /* nx*ny*nz raw SDF cell values (GetImmutable4d, spcs.hpp:941)    */
    float oob_value;            /* value returned out of bounds (+inf, envb.cpp:473)              */
    int32_t _pad;
    /* surface normals: only non-empty cells are listed, sorted by ascending linear index */
    int64_t n_normal_cells;
    const int64_t* normal_cell_index;  /* [n_normal_cells]                                       */
    const uint32_t* normal_cell_start; /* [n_normal_cells+1] offsets into normal_entries         */
    const double* normal_entries;      /* 7 doubles each: entry_direction xyzw, normal xyz
                                          (StoredSurfaceNormal, spcs.hpp:48-83; already SafeNormal'd) */
} fks_env_desc;

/* One actuated axis: SimplePIDController (pid.hpp:53-136) + TruncatedNormalUncertainVelocityActuator
 * (unc.hpp:48-121).  SE2: 3 axes (x,y,zr); SE3: 6 (x,y,z,xr,yr,zr); linked: one per active joint. */
typedef struct fks_axis_params {
    double kp, ki, kd, integral_clamp;
    double velocity_limit;
    double proportional_noise;  /* max_actuator_proportional_noise */
    double minimum_noise;       /* max_actuator_minimum_noise      */
    double noise_sigma;         /* percent_variance, 0.5 in every tnuva ctor (tnuva.hpp:128,318,469) */
} fks_axis_params;

/* arc_utilities RobotJoint (call sites tnuva.hpp:487-500,544-559) */
typedef struct fks_joint_desc {
    int32_t parent_link;
    int32_t child_link;
    int32_t type;          /* FKS_JOINT_* */
    int32_t _pad;
    double transform[12];  /* parent link -> joint frame */
    double axis[3];
    double lower_limit, upper_limit;
    double distance_weight;
} fks_joint_desc;

typedef struct fks_robot_desc {
    int32_t kind;        /* FKS_ROBOT_* */
    int32_t n_links;     /* 1 for SE2/SE3 */
    int32_t n_joints;    /* 0 for SE2/SE3 */
    int32_t n_dof;       /* 3 / 6 / active joints */
    int64_t n_points;    /* total collision points, stored link-major, point-minor (spcs.hpp:925-936) */
    const double* points_xyz;    /* [n_points*3] link-relative */
    const int32_t* point_link;   /* [n_points] non-decreasing */
    const fks_axis_params* axes; /* [n_dof] */
    /* linked only */
    double base_transform[12];
    const fks_joint_desc* joints;           /* [n_joints], kinematic order */
    const uint8_t* allowed_self_collision;  /* [n_links*n_links], 1 = allowed (CheckIfSelfCollisionAllowed) */
    /* configuration distance weights (ComputeConfigurationDistanceTo, spcs.hpp:898) */
    double position_distance_weight;
    double rotation_distance_weight;
} fks_robot_desc;

/* Injected noise: the truncated-normal outputs of noise_distribution_(rng) (unc.hpp:86) in the
 * order the reference draws them, [particle][step][microstep][dof] (SURVEY.md A.6).
 *
 * Optional DECISION TAPE (parity instrumentation, NULL in production): the discrete outcomes of every
 * J.colPivHouseholderQr().solve(c) (spcs.hpp:1990-1998) the reference side took for a particle, in call order.
 * Eigen's rank decision compares a pivot with ~epsilon * the largest column norm; when the stacked Jacobian is
 * structurally rank deficient (a single distal link of a 7-dof arm touching: rank <= 6 in 7 unknowns) the last
 * pivot IS round-off and the reference cuts or keeps it by the last bit.  No other arithmetic reproduces that bit,
 * so in parity mode the device takes the decision from the tape (and reports where its own differed) and everything
 * downstream of it stays comparable.  One record per solve, 2 + n_dof 64-bit words:
 *   word 0: bits 0..7 nonzero_pivots, bits 8..15 FKS_DECISION_* flags, bits 16..47 rows of the stacked system
 *   word 1: pivot order, 4 bits per step: the column picked at step k
 *   words 2..: the reference's solution (bit pattern of n_dof doubles); consumed only with
 *              FKS_DECISION_OVERRIDE_SOLUTION (a round-off pivot was KEPT: the solution itself is round-off) */
enum {
    FKS_DECISION_OVERRIDE_SOLUTION = 1u << 8,
    FKS_DECISION_ROUNDOFF_PIVOT    = 1u << 9,  /* informational: a pivot at round-off level was met */
    FKS_DECISION_PIVOT_TIE         = 1u << 10  /* informational: two pivot candidates within 1e-9 relative */
};
typedef struct fks_noise_tape {
    const double* draws;       /* flat */
    const uint64_t* offsets;   /* [n_particles+1] start of each particle's draws */
    const uint64_t* decisions;        /* flat records of 2 + n_dof words, or NULL */
    const uint64_t* decision_offsets; /* [n_particles+1] first RECORD of each particle, or NULL */
} fks_noise_tape;

/* Tail of every result record; record = cfg_stride doubles followed by this struct. */
typedef struct fks_result_tail {
    uint32_t flags;            /* FKS_FLAG_* */
    uint32_t n_microsteps;     /* executed iterations of the loop at spcs.hpp:1590 */
    uint32_t n_resolver_iters; /* executed iterations of the loop at spcs.hpp:1625 */
    uint32_t n_steps;          /* controller steps executed (spcs.hpp:863)         */
} fks_result_tail;

/* keys of GetStatistics (spcs.hpp:488-500), in this order, then three extra totals */
enum {
    FKS_STAT_SUCCESSFUL_RESOLVES = 0,
    FKS_STAT_UNSUCCESSFUL_RESOLVES = 1,
    FKS_STAT_FREE_RESOLVES = 2,
    FKS_STAT_COLLISION_RESOLVES = 3,
    FKS_STAT_FALLBACK_RESOLVES = 4,
    FKS_STAT_UNSUCCESSFUL_SELF_COLLISION_RESOLVES = 5,
    FKS_STAT_UNSUCCESSFUL_ENV_COLLISION_RESOLVES = 6,
    FKS_STAT_RECOVERED_UNSUCCESSFUL_RESOLVES = 7,
    FKS_STAT_TOTAL_MICROSTEPS = 8,
    FKS_STAT_TOTAL_RESOLVER_ITERATIONS = 9,
    FKS_STAT_TOTAL_CORRECTED_POINTS = 10, /* sum over resolver iterations of the points that got a correction (rows / 3) */
    FKS_NUM_STATS = 11
};

typedef struct fks_env fks_env;
typedef struct fks_robot fks_robot;
typedef struct fks_sim fks_sim;

/* -------------------------------------------------------------------------------------------
 * Library
 * ----------------------------------------------------------------------------------------- */
int fks_abi_version(void);
/* message of the last failing call on this thread */
const char* fks_last_error_string(void);
int fks_device_count(int* count);

/* defaults of SimulatorSolverParameters() (spcs.hpp:357-368); replaces GetDefaultSolverParameters (fks.hpp:13-16) */
void fks_default_solver_params(fks_solver_params* out);

/* -------------------------------------------------------------------------------------------
 * Environment (replaces the by-value copies of grid / SDF / SurfaceNormalGrid, spcs.hpp:420)
 * Uploads to `device`, builds the device normal table, requests an L2 persistence window.
 * ----------------------------------------------------------------------------------------- */
int fks_env_create(int device, const fks_env_desc* desc, fks_env** out);
void fks_env_destroy(fks_env* env);

/* -------------------------------------------------------------------------------------------
 * Robot (replaces the immutable_robot argument of ForwardSimulateRobots, spcs.hpp:788)
 * ----------------------------------------------------------------------------------------- */
int fks_robot_create(int device, const fks_robot_desc* desc, fks_robot** out);
void fks_robot_destroy(fks_robot* robot);
/* doubles per flattened configuration: 3 / 12 / n_dof */
int fks_robot_config_stride(const fks_robot* robot);

/* -------------------------------------------------------------------------------------------
 * Simulator (replaces Make{SE2,SE3,Linked}Simulator, fks.hpp:18-22 / fks.cpp:4-71, and the
 * SimpleParticleContactSimulator ctor, spcs.hpp:420-444)
 * ----------------------------------------------------------------------------------------- */
int fks_sim_create(const fks_env* env, const fks_robot* robot, const fks_solver_params* params,
                   double simulation_controller_frequency, uint64_t prng_seed, int32_t debug_level,
                   fks_sim** out);
void fks_sim_destroy(fks_sim* sim);
/* bytes per result record = 8*cfg_stride + sizeof(fks_result_tail) */
size_t fks_sim_result_stride(const fks_sim* sim);

/* ForwardSimulateRobots (spcs.hpp:788-804) with HOST buffers.
 *  starts:  n_particles * cfg_stride doubles; targets: n_targets (1 or n_particles) * cfg_stride
 *  noise_mode FKS_NOISE_INJECTED requires `tape`; FKS_NOISE_PHILOX uses (prng_seed, first_particle_id + i)
 *  results: n_particles records of fks_sim_result_stride() bytes
 * Host->device copies of starts/targets(/tape), the kernel, and the device->host copy of results
 * all happen inside the call; it returns after the results are on the host. */
int fks_forward_simulate(fks_sim* sim, const double* starts, const double* targets,
                         size_t n_particles, size_t n_targets, int allow_contacts,
                         int noise_mode, const fks_noise_tape* tape, uint64_t first_particle_id,
                         void* results);

/* ReverseSimulateRobots (spcs.hpp:806-822, :838-841): identical computation */
int fks_reverse_simulate(fks_sim* sim, const double* starts, const double* targets,
                         size_t n_particles, size_t n_targets, int allow_contacts,
                         int noise_mode, const fks_noise_tape* tape, uint64_t first_particle_id,
                         void* results);

/* fks_forward_simulate without the final wait: returns once the copies and the kernels are enqueued on the simulator's own
 * stream; `results` (pinned memory makes the copy truly asynchronous) is complete after fks_sim_synchronize. */
int fks_forward_simulate_async(fks_sim* sim, const double* starts, const double* targets,
                               size_t n_particles, size_t n_targets, int allow_contacts,
                               int noise_mode, const fks_noise_tape* tape, uint64_t first_particle_id,
                               void* results);
int fks_sim_synchronize(fks_sim* sim);

/* Same with DEVICE buffers, asynchronous on `cuda_stream` (a cudaStream_t; NULL = default stream).
 * d_tape_draws / d_tape_offsets may be NULL unless noise_mode == FKS_NOISE_INJECTED.
 * Streams: a simulator owns ONE particle counter, context store and scratch, so its batch calls never overlap -- each launch
 * records an event and the next launch of the same simulator, on whatever stream (a caller's or the simulator's own, which
 * the host-buffer calls use), waits for it.  Calls on different streams are therefore safe and ordered by issue; for
 * batches that should run concurrently use one simulator per stream.  Like the reference (spcs.hpp:846-850) a simulator
 * serves one caller thread at a time. */
int fks_forward_simulate_device(fks_sim* sim, const double* d_starts, const double* d_targets,
                                size_t n_particles, size_t n_targets, int allow_contacts,
                                int noise_mode, const double* d_tape_draws,
                                const uint64_t* d_tape_offsets, uint64_t first_particle_id,
                                void* d_results, void* cuda_stream);

/* Sequence call: every particle runs n_legs consecutive legs in ONE kernel launch; leg k is exactly one ForwardSimulateRobot
 * (spcs.hpp:824-829) from where leg k-1 left the particle towards leg k's target.  The records equal, byte for byte, those of
 * the chain of single calls
 *     for k in 0 .. n_legs-1:
 *         fks_forward_simulate(sim, starts_k, targets + k * n_targets * cfg_stride, n, n_targets, allow_contacts, noise_mode,
 *                              tape_k, first_particle_id + k * n, results + k * n * fks_sim_result_stride(sim))
 *         starts_{k+1} = the configurations of those records
 * in every noise mode, and so do the statistics (fks_get_statistics afterwards = the chain's sum).
 *  - noise: leg k of particle i draws Philox noise as particle first_particle_id + k * n_particles + i, controller steps counted
 *    from 0 inside the leg -- the ids a caller that advances first_particle_id by n_particles per call uses;
 *  - each leg restarts like ForwardSimulateRobot: PID state zeroed (ResetPosition), flags and counters cleared.  A leg that
 *    ended by a failed resolve, the shortcut distance or a stop with allow_contacts == 0 still hands its end state on;
 *  - targets: leg-major, [n_legs][n_targets][cfg_stride]; n_targets is 1 or n_particles, the same for every leg;
 *  - results: leg-major, [n_legs][n_particles] records of fks_sim_result_stride() bytes: leg k's records are a batch result
 *    of their own (fks_end_states_* take them at d_results + k * n_particles * stride);
 *  - injected tapes: ONE span per particle (offsets / decision_offsets have n_particles + 1 entries) holding the particle's
 *    per-leg spans of the chain's tapes one after the other.  The tape positions are not reset between legs, so the equality
 *    with the chain holds when every leg consumes exactly its own span -- as when the tapes record the same trajectories.
 *    A leg that consumes fewer draws or decision records than its span (e.g. a particle that desynchronised from the recorded
 *    run) shifts every later leg's draws, and one that consumes more reads the next leg's draws instead of raising
 *    FKS_FLAG_TAPE_EXHAUSTED (only the particle's last leg can run out);
 *  - n_legs == 1 is fks_forward_simulate.
 * n_legs == 0 or above 2^31 - 1, a null `targets` or first_particle_id + n_legs * n_particles beyond 64 bits (the sum itself must
 * not wrap) is FKS_ERR_INVALID_ARGUMENT;
 * n_particles == 0 launches nothing.  The _device flavour takes device buffers and runs asynchronously on `cuda_stream` like
 * fks_forward_simulate_device; the _multi flavour shards the particles over the devices like fks_multi_forward_simulate
 * (records do not depend on the device count). */
int fks_forward_simulate_sequence(fks_sim* sim, const double* starts, const double* targets, size_t n_particles,
                                  size_t n_targets, size_t n_legs, int allow_contacts, int noise_mode,
                                  const fks_noise_tape* tape, uint64_t first_particle_id, void* results);
int fks_forward_simulate_sequence_device(fks_sim* sim, const double* d_starts, const double* d_targets, size_t n_particles,
                                         size_t n_targets, size_t n_legs, int allow_contacts, int noise_mode,
                                         const double* d_tape_draws, const uint64_t* d_tape_offsets,
                                         uint64_t first_particle_id, void* d_results, void* cuda_stream);

/* CheckConfigCollision (spcs.hpp:1398-1416), batched: out_collides[i] = 1 when configuration i collides with the
 * environment inflated by inflation_ratio cells (CheckEnvironmentCollision, spcs.hpp:921-981 with threshold
 * inflation_ratio * resolution) or with itself (CheckSelfCollisions, spcs.hpp:1324-1396, cells of
 * (inflation_ratio + 1) * resolution).  HOST buffers: configs n * cfg_stride doubles, out_collides n bytes. */
int fks_check_config_collision(fks_sim* sim, const double* configs, size_t n_configs, double inflation_ratio,
                               uint8_t* out_collides);

/* ForwardSimulateRobot with enable_tracing == true (spcs.hpp:824-829; ForwardSimulationStepTrace filled at :1583-1617,
 * :1703, :1714, :1778) for ONE particle -- SURVEY.md 8(f)-4.  The nested trace of the reference (controller step ->
 * microstep -> configurations) is returned flat, in the order the reference appends: every record carries its step /
 * microstep / resolver-iteration indices.  HOST buffers; trace_records holds up to trace_capacity records of
 * fks_sim_trace_stride() bytes (fks_trace_header followed by max(cfg_stride, n_dof) doubles); *n_records receives the number
 * the simulation produced (records beyond the capacity are counted but not stored). */
enum {
    FKS_TRACE_CONTROL_INPUT = 0,      /* resolver_steps.back().control_input = real_control_input (:1586), n_dof values   */
    FKS_TRACE_CONTROL_INPUT_STEP = 1, /* .control_input_step (:1587), n_dof values                                         */
    FKS_TRACE_POST_ACTION = 2,        /* contact_resolution_steps.push_back(post_action_configuration) (:1617), cfg_stride */
    FKS_TRACE_RESOLUTION_STEP = 3,    /* ... push_back(active_configuration) after a correction step (:1703)               */
    FKS_TRACE_RETURNED_PREVIOUS = 4   /* ... push_back(previous_configuration): failed resolve (:1714) / no-contact (:1778) */
};
typedef struct fks_trace_header {
    uint32_t kind;      /* FKS_TRACE_* */
    uint32_t step;      /* controller step (index into resolver_steps) */
    uint32_t microstep; /* index into contact_resolver_steps of that step */
    uint32_t iteration; /* resolver iterations completed when the record was made */
} fks_trace_header;
size_t fks_sim_trace_stride(const fks_sim* sim);
int fks_forward_simulate_traced(fks_sim* sim, const double* start, const double* target, int allow_contacts,
                                int noise_mode, const fks_noise_tape* tape, uint64_t particle_id, void* result,
                                void* trace_records, size_t trace_capacity, size_t* n_records);

/* GetStatistics / ResetStatistics (spcs.hpp:488-512); out has FKS_NUM_STATS entries.
 * Synchronises the simulator's stream. */
int fks_get_statistics(fks_sim* sim, uint64_t* out);
int fks_reset_statistics(fks_sim* sim);

/* Measurement aid: fks_sim_enable_kernel_timing records CUDA events around the simulate kernel from now on;
 * fks_sim_kernel_times returns the device milliseconds of the kernel of the LAST batch call in out_ms[0] (and 1 in
 * *n_kernels when it was timed).  It waits for that call. */
int fks_sim_enable_kernel_timing(fks_sim* sim, int enable);
int fks_sim_kernel_times(fks_sim* sim, double* out_ms, int* n_kernels);

/* number of kernel launches issued by this simulator so far (bench "gpu_launches") */
uint64_t fks_sim_launch_count(const fks_sim* sim);
/* kernel attributes of the simulate kernel for this robot kind (regs, smem, occupancy) as a
 * short human-readable string owned by the sim */
const char* fks_sim_kernel_info(fks_sim* sim);

/* -------------------------------------------------------------------------------------------
 * Several GPUs of one box behind the same call (SURVEY.md 8e).  ForwardSimulateRobots is data parallel over particles
 * (spcs.hpp:795-802): the batch is cut into contiguous shards, one per device, environment and robot are replicated per
 * device at creation (what the factories fks.hpp:18-22 + the constructor spcs.hpp:420-444 do once), Philox noise is keyed
 * by the global particle id, so the records do not depend on the device count.
 *   fks_multi_forward_simulate         host buffers; every device copies its records straight into `results`: all N
 *                                      records return to the caller, no collective needed.  Tapes (parity mode) are sharded too.
 *   fks_multi_forward_simulate_device  device buffers: d_starts[d] / d_targets[d] hold device d's SHARD (n / n_devices
 *                                      particles; one target or one per particle of the shard), d_results[d] is a full
 *                                      n-record array on device d; after the call every device holds ALL n records,
 *                                      exchanged by one ncclAllGather over NVLink (libnccl.so.2 bound at run time).  Philox noise.
 *   fks_multi_get_statistics           the counters summed over the devices.
 * devices == NULL selects devices 0 .. n_devices-1.
 * ----------------------------------------------------------------------------------------- */
typedef struct fks_multi_sim fks_multi_sim;
int fks_multi_sim_create(const int32_t* devices, int32_t n_devices, const fks_env_desc* env, const fks_robot_desc* robot,
                         const fks_solver_params* params, double simulation_controller_frequency, uint64_t prng_seed,
                         int32_t debug_level, fks_multi_sim** out);
void fks_multi_sim_destroy(fks_multi_sim* sim);
int fks_multi_sim_device_count(const fks_multi_sim* sim);
size_t fks_multi_sim_result_stride(const fks_multi_sim* sim);
int fks_multi_forward_simulate(fks_multi_sim* sim, const double* starts, const double* targets, size_t n_particles,
                               size_t n_targets, int allow_contacts, int noise_mode, const fks_noise_tape* tape,
                               uint64_t first_particle_id, void* results);
/* fks_forward_simulate_sequence over the devices: host buffers, same layouts, tapes sharded like fks_multi_forward_simulate */
int fks_multi_forward_simulate_sequence(fks_multi_sim* sim, const double* starts, const double* targets, size_t n_particles,
                                        size_t n_targets, size_t n_legs, int allow_contacts, int noise_mode,
                                        const fks_noise_tape* tape, uint64_t first_particle_id, void* results);
int fks_multi_forward_simulate_device(fks_multi_sim* sim, const double* const* d_starts, const double* const* d_targets,
                                      size_t n_particles, size_t n_targets, int allow_contacts, uint64_t first_particle_id,
                                      void* const* d_results);
int fks_multi_get_statistics(fks_multi_sim* sim, uint64_t* out);
int fks_multi_reset_statistics(fks_multi_sim* sim);

/* -------------------------------------------------------------------------------------------
 * Environment builder (host C++; replaces simulator_environment_builder::BuildCompleteEnvironment,
 * simulator_environment_builder.cpp:470-476).  Obstacles are cuboids (OBSTACLE_CONFIG,
 * simulator_environment_builder.hpp:25-49).  The result owns its arrays; `desc` points into it.
 * ----------------------------------------------------------------------------------------- */
typedef struct fks_obstacle {
    double pose[12];
    double extents[3]; /* half extents */
    uint32_t object_id;
    uint32_t _pad;
} fks_obstacle;

typedef struct fks_built_env fks_built_env;
int fks_build_environment(const fks_obstacle* obstacles, size_t n_obstacles, double resolution,
                          fks_built_env** out);
const fks_env_desc* fks_built_env_desc(const fks_built_env* env);
/* occupancy of the collision map (1 byte per cell, 1 = filled); not used on the hot path */
const uint8_t* fks_built_env_occupancy(const fks_built_env* env);
void fks_built_env_destroy(fks_built_env* env);

/* -------------------------------------------------------------------------------------------
 * Environment builder on the device (SURVEY.md 8(f)-1): the same BuildCompleteEnvironment
 * (simulator_environment_builder.cpp:470-476: BuildEnvironment :49-160, ExtractSignedDistanceField :473,
 * BuildSurfaceNormalsGrid :258-468) computed by CUDA kernels straight into a device environment -- occupancy
 * rasterisation, exact Euclidean distance transform, float SDF, surface-normal table and its hash -- with no host
 * copy of the grids.  Results are bit-identical to fks_build_environment + fks_env_create.
 * fks_env_build_timings: out_ms[0] = total device time of the build, [1] rasterise, [2] z pass, [3] y pass,
 * [4] x pass + SDF, [5] surface marking, [6] normal count/scan/emit, [7] distance-field check, [8] the host-side allocation
 * of the table arrays inside phase 6 (their size is known only after the scan; included in [0], not in [6]) -- milliseconds.
 * fks_env_download: copies a device environment back into host arrays (any fks_env; occupancy only when the
 * environment was built on the device, else fks_built_env_occupancy returns NULL).
 * ----------------------------------------------------------------------------------------- */
int fks_env_build_device(int device, const fks_obstacle* obstacles, size_t n_obstacles, double resolution,
                         fks_env** out);
int fks_env_build_timings(const fks_env* env, double* out_ms, int n);
int fks_env_download(const fks_env* env, fks_built_env** out);

/* -------------------------------------------------------------------------------------------
 * First consumer of a batch, on the device (SURVEY.md 8f-3).  The planner that holds the simulator
 * (uncertainty_planning_core.cpp:97-99) splits the returned particles by did_contact and groups them by configuration
 * distance; with these two calls the end-state records of fks_forward_simulate_device stay in HBM for that step.
 *   fks_end_states_partition          d_order[0 .. counts[0]) = ids of the particles WITHOUT contact, ascending;
 *                                     d_order[counts[0] .. n) = ids of the particles WITH contact, ascending
 *                                     (SimulationResult::did_contact, spcs.hpp:918).  counts is a HOST array of 2; the call
 *                                     returns after the stream has finished these kernels.
 *   fks_end_states_pairwise_distance  d_out[a * m + b] = robot.ComputeConfigurationDistanceTo (the call at spcs.hpp:898) from
 *                                     record d_subset[a] to record d_subset[b]; d_subset == NULL takes records 0 .. m-1.
 *                                     SE2 / SE3: position_distance_weight * |dt| + rotation_distance_weight * angle;
 *                                     linked: weighted joint-space norm, continuous joints wrapped.  Asynchronous on the stream.
 * d_results: device records as written by fks_forward_simulate_device (fks_sim_result_stride bytes each).
 * ----------------------------------------------------------------------------------------- */
int fks_end_states_partition(fks_sim* sim, const void* d_results, size_t n_particles, uint32_t* d_order, uint64_t* counts,
                             void* cuda_stream);
int fks_end_states_pairwise_distance(fks_sim* sim, const void* d_results, const uint32_t* d_subset, size_t m, double* d_out,
                                     void* cuda_stream);

/* fks_end_states_cluster: the grouping step itself -- flat agglomerative clustering under a distance cutoff, per segment.
 * Positions 0 .. m-1 name records d_order[p] (d_order == NULL: record p); segment s covers positions
 * [segment_offsets[s], segment_offsets[s+1]) of the HOST array segment_offsets (n_segments + 1 entries, [0] = 0,
 * non-decreasing, last = m; empty segments are allowed).  Typical segments: {0, n_free, n} over the order of
 * fks_end_states_partition, or one per leg of a sequence result (ids k * n + i from the base pointer).
 *  - distance of positions p < q of one segment: d(p, q) = entry [p][q] of fks_end_states_pairwise_distance over the same ids
 *    (same direction, same bits); +inf where that is NaN, and with separate_contact != 0 where the two records'
 *    FKS_FLAG_DID_CONTACT differ;
 *  - every segment starts from singletons; a cluster is named by its smallest position (its representative); the linkage of
 *    clusters A, B is the minimum (FKS_LINKAGE_SINGLE) or maximum (FKS_LINKAGE_COMPLETE) of d over their pairs; while some
 *    pair has a finite linkage <= max_cluster_distance, the pair with the smallest (linkage, smaller rep, larger rep) merges.
 *    Clusters never cross segments and a pair at +inf never merges.  (scipy: linkage + fcluster(t, "distance") up to ties);
 *  - d_labels[p] (device, m entries) = global cluster id: segment s's clusters are base_s .. base_s + cluster_counts[s] - 1
 *    in increasing order of representative, base_s = the sum of the earlier segments' counts; cluster_counts is a HOST
 *    array of n_segments entries.  The call returns after the stream has finished.
 * Segments of up to 160 positions are clustered in shared memory, longer ones (up to 8192 positions) in a device workspace
 * the simulator keeps.  FKS_ERR_INVALID_ARGUMENT: NaN max_cluster_distance, unknown linkage, null buffers when m > 0,
 * malformed offsets, m >= 2^32, or a segment longer than 8192 positions.  m == 0 or n_segments == 0 launches nothing. */
enum { FKS_LINKAGE_SINGLE = 0, FKS_LINKAGE_COMPLETE = 1 };
int fks_end_states_cluster(fks_sim* sim, const void* d_results, const uint32_t* d_order, const uint64_t* segment_offsets,
                           size_t n_segments, int linkage, double max_cluster_distance, int separate_contact, uint32_t* d_labels,
                           uint64_t* cluster_counts, void* cuda_stream);

/* fks_end_states_groups: clusters as particle groups -- the planner's child states.  Positions 0 .. m-1 name records as in
 * fks_end_states_cluster (d_order[p], or p); d_labels[p] < n_clusters is position p's cluster (e.g. that call's output).
 *  - members: d_members[d_group_offsets[c] .. d_group_offsets[c+1]) = the record ids of the positions labelled c, in
 *    increasing order of position (a stable counting sort by label); d_group_offsets[0] = 0, [n_clusters] = m;
 *  - d(p, q), p < q positions of one cluster = entry [p][q] of fks_end_states_pairwise_distance over the same ids (same
 *    direction, same bits), +inf where that is NaN;
 *  - representative: the minimax member, the p that minimises r(p) = max over the other members q of d(min(p,q), max(p,q)),
 *    ties to the smallest position; d_representatives[c] = its record id, d_radius[c] = r(p) (0.0 for a singleton; +inf,
 *    with the smallest position, when every r is +inf);
 *  - group_sizes (HOST, n_clusters entries) = member counts.  The call returns after the stream has finished.
 * Clusters of up to 256 members are searched one CTA each, larger ones (up to 8192) with their rows split over CTAs.
 * FKS_ERR_INVALID_ARGUMENT: a label >= n_clusters, a cluster without members or with more than 8192, n_clusters > m,
 * m >= 2^32, null buffers when m > 0; device outputs are then unspecified.  m == 0 launches nothing. */
int fks_end_states_groups(fks_sim* sim, const void* d_results, const uint32_t* d_order, size_t m, const uint32_t* d_labels,
                          size_t n_clusters, uint32_t* d_group_offsets, uint32_t* d_members, uint32_t* d_representatives,
                          double* d_radius, uint64_t* group_sizes, void* cuda_stream);

/* fks_end_states_gather_starts: the next batch from chosen groups.  For slot s < n_selected (g = selected[s], a HOST array;
 * repeats and any order allowed), k = the size of group g and j < per_group:
 *   d_starts[s * per_group + j]  = the configuration (cfg_stride doubles) of record d_members[d_group_offsets[g] + j mod k];
 *   d_targets[s * per_group + j] = d_group_targets[s] (both NULL: no targets).
 * The outputs are the starts / targets of fks_forward_simulate_device(n = n_targets = n_selected * per_group).  Groups as
 * fks_end_states_groups writes them; a group of 0 members gets NaN starts.  Asynchronous on the stream.
 * FKS_ERR_INVALID_ARGUMENT: per_group == 0, a selected id >= n_clusters, n_selected * per_group >= 2^32, null buffers when
 * the output is not empty, or exactly one of d_targets / d_group_targets.  n_selected == 0 launches nothing. */
int fks_end_states_gather_starts(fks_sim* sim, const void* d_results, const uint32_t* d_group_offsets, const uint32_t* d_members,
                                 size_t n_clusters, const uint32_t* selected, size_t n_selected, size_t per_group,
                                 const double* d_group_targets, double* d_starts, double* d_targets, void* cuda_stream);

/* -------------------------------------------------------------------------------------------
 * Test entry: the device's stacked-Jacobian solver (ComputeResolverCorrectionStepStackedJacobian, spcs.hpp:1990-1998 =
 * J.colPivHouseholderQr().solve(c)) on caller-provided systems, one warp each.  System i has rows[i] rows and `cols`
 * unknowns and is stored at systems + offsets[i] as cols + 1 columns of rows[i] doubles (column major, right-hand side
 * last); offsets has n + 1 entries.  solutions: n * cols doubles; flags: the FKS_FLAG_* bits the solver raised.
 * The solver follows Eigen operation for operation, so on the same system it returns the bits of the CPU oracle.
 * ----------------------------------------------------------------------------------------- */
int fks_debug_qr_solve(int device, const double* systems, const uint64_t* offsets, const int32_t* rows, int32_t cols, size_t n,
                       double* solutions, uint32_t* flags);

/* -------------------------------------------------------------------------------------------
 * Device micro-benchmarks used for the roofline denominators (SURVEY.md 8d): dependent-free DFMA
 * throughput (FLOP/s) and random 4-byte gather rate (gathers/s) over a `bytes`-sized array.
 * ----------------------------------------------------------------------------------------- */
int fks_measure_fp64_peak(int device, double* flops_per_s);
int fks_measure_gather_rate(int device, size_t bytes, double* gathers_per_s);

#ifdef __cplusplus
}
#endif
#endif /* FKSGPU_H */
