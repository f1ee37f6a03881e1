"""Constants and ctypes structures of include/fksgpu.h, field for field -- and NOTHING that loads a library: the CPU
oracle's harness (oracle/, bench.py --impl reference) describes robots and environments with the same structures without
touching the product.  fast_kinematic_simulator_b200.capi re-exports everything here next to the loaded library."""
import ctypes as C

OK, ERR_INVALID_ARGUMENT, ERR_CUDA, ERR_NO_DEVICE, ERR_UNSUPPORTED, ERR_OUT_OF_MEMORY = range(6)
ROBOT_SE2, ROBOT_SE3, ROBOT_LINKED = 0, 1, 2
JOINT_PRISMATIC, JOINT_REVOLUTE, JOINT_CONTINUOUS, JOINT_FIXED = 0, 1, 2, 3
NOISE_PHILOX, NOISE_INJECTED, NOISE_NONE = 0, 1, 2
LINKAGE_SINGLE, LINKAGE_COMPLETE = 0, 1
FLAG_DID_CONTACT = 1 << 0
FLAG_RESOLVE_FAILED = 1 << 1
FLAG_ENDED_BY_FAILURE = 1 << 2
FLAG_ENDED_BY_NOCONTACT = 1 << 3
FLAG_ENDED_BY_SHORTCUT = 1 << 4
FLAG_WOULD_ASSERT_MICROSTEP = 1 << 8
FLAG_WOULD_ASSERT_NORMAL = 1 << 9
FLAG_WOULD_ASSERT_NAN = 1 << 10
FLAG_EMPTY_JACOBIAN = 1 << 11
FLAG_TAPE_EXHAUSTED = 1 << 12
FLAG_NEAR_RANK_CUT = 1 << 13
FLAG_J_SPILLED = 1 << 14
FLAG_DECISION_OVERRIDDEN = 1 << 15
FLAG_DECISION_DESYNC = 1 << 16
TRACE_CONTROL_INPUT, TRACE_CONTROL_INPUT_STEP, TRACE_POST_ACTION, TRACE_RESOLUTION_STEP, TRACE_RETURNED_PREVIOUS = range(5)
NUM_STATS = 11
STAT_NAMES = (
    "successful_resolves",
    "unsuccessful_resolves",
    "free_resolves",
    "collision_resolves",
    "fallback_resolves",
    "unsuccessful_self_collision_resolves",
    "unsuccessful_env_collision_resolves",
    "recovered_unsuccessful_resolves",
    "total_microsteps",
    "total_resolver_iterations",
    "total_corrected_points",
)


class SolverParams(C.Structure):
    _fields_ = [
        ("forward_simulation_time", C.c_double),
        ("simulation_shortcut_distance", C.c_double),
        ("environment_collision_check_tolerance", C.c_double),
        ("resolve_correction_step_scaling_decay_rate", C.c_double),
        ("resolve_correction_initial_step_size", C.c_double),
        ("resolve_correction_min_step_scaling", C.c_double),
        ("max_resolver_iterations", C.c_uint32),
        ("resolve_correction_step_scaling_decay_iterations", C.c_uint32),
        ("failed_resolves_end_motion", C.c_int32),
        ("_pad", C.c_int32),
    ]


class EnvDesc(C.Structure):
    _fields_ = [
        ("origin", C.c_double * 12),
        ("inverse_origin", C.c_double * 12),
        ("map_resolution", C.c_double),
        ("sdf_resolution", C.c_double),
        ("nx", C.c_int64),
        ("ny", C.c_int64),
        ("nz", C.c_int64),
        ("sdf", C.POINTER(C.c_float)),
        ("oob_value", C.c_float),
        ("_pad", C.c_int32),
        ("n_normal_cells", C.c_int64),
        ("normal_cell_index", C.POINTER(C.c_int64)),
        ("normal_cell_start", C.POINTER(C.c_uint32)),
        ("normal_entries", C.POINTER(C.c_double)),
    ]


class AxisParams(C.Structure):
    _fields_ = [
        ("kp", C.c_double),
        ("ki", C.c_double),
        ("kd", C.c_double),
        ("integral_clamp", C.c_double),
        ("velocity_limit", C.c_double),
        ("proportional_noise", C.c_double),
        ("minimum_noise", C.c_double),
        ("noise_sigma", C.c_double),
    ]


class JointDesc(C.Structure):
    _fields_ = [
        ("parent_link", C.c_int32),
        ("child_link", C.c_int32),
        ("type", C.c_int32),
        ("_pad", C.c_int32),
        ("transform", C.c_double * 12),
        ("axis", C.c_double * 3),
        ("lower_limit", C.c_double),
        ("upper_limit", C.c_double),
        ("distance_weight", C.c_double),
    ]


class RobotDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("n_links", C.c_int32),
        ("n_joints", C.c_int32),
        ("n_dof", C.c_int32),
        ("n_points", C.c_int64),
        ("points_xyz", C.POINTER(C.c_double)),
        ("point_link", C.POINTER(C.c_int32)),
        ("axes", C.POINTER(AxisParams)),
        ("base_transform", C.c_double * 12),
        ("joints", C.POINTER(JointDesc)),
        ("allowed_self_collision", C.POINTER(C.c_uint8)),
        ("position_distance_weight", C.c_double),
        ("rotation_distance_weight", C.c_double),
    ]


class NoiseTape(C.Structure):
    _fields_ = [("draws", C.POINTER(C.c_double)), ("offsets", C.POINTER(C.c_uint64)),
                ("decisions", C.POINTER(C.c_uint64)), ("decision_offsets", C.POINTER(C.c_uint64))]


class Obstacle(C.Structure):
    _fields_ = [
        ("pose", C.c_double * 12),
        ("extents", C.c_double * 3),
        ("object_id", C.c_uint32),
        ("_pad", C.c_uint32),
    ]


def default_solver_params():
    """SimulatorSolverParameters() (simple_particle_contact_simulator.hpp:357-368) without loading the library
    (fks_default_solver_params returns the same values; tests/test_capi_symbols.py compares them)."""
    p = SolverParams()
    p.forward_simulation_time = 1.0
    p.simulation_shortcut_distance = 0.0
    p.environment_collision_check_tolerance = 0.001
    p.resolve_correction_step_scaling_decay_rate = 0.5
    p.resolve_correction_initial_step_size = 1.0
    p.resolve_correction_min_step_scaling = 0.03125
    p.max_resolver_iterations = 25
    p.resolve_correction_step_scaling_decay_iterations = 5
    p.failed_resolves_end_motion = 1
    return p


def env_desc_from_arrays(e):
    """fks_env_desc over numpy arrays (keys shape, origin, inverse_origin, resolution, sdf, normal_cell_index, normal_cell_start, normal_entries); returns (desc, keepalive)."""
    import numpy as np

    sdf = np.ascontiguousarray(e["sdf"], dtype=np.float32)
    cells = np.ascontiguousarray(e["normal_cell_index"], dtype=np.int64)
    starts = np.ascontiguousarray(e["normal_cell_start"], dtype=np.uint32)
    entries = np.ascontiguousarray(e["normal_entries"], dtype=np.float64)
    d = EnvDesc()
    d.origin = (C.c_double * 12)(*[float(v) for v in e["origin"]])
    d.inverse_origin = (C.c_double * 12)(*[float(v) for v in e["inverse_origin"]])
    d.map_resolution = float(e["resolution"])
    d.sdf_resolution = float(e["resolution"])
    d.nx, d.ny, d.nz = [int(v) for v in e["shape"]]
    d.sdf = sdf.ctypes.data_as(C.POINTER(C.c_float))
    d.oob_value = float("inf")
    d.n_normal_cells = int(cells.shape[0])
    d.normal_cell_index = cells.ctypes.data_as(C.POINTER(C.c_int64))
    d.normal_cell_start = starts.ctypes.data_as(C.POINTER(C.c_uint32))
    d.normal_entries = entries.ctypes.data_as(C.POINTER(C.c_double))
    return d, (sdf, cells, starts, entries)
