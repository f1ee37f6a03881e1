"""ctypes binding of include/fksgpu.h (the C ABI of libfksgpu.so).  Structures mirror the header
field for field; nothing here computes."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))


def library_path():
    # FKSGPU_LIBRARY: developer override used to A/B kernel builds (always an in-tree libfksgpu*.so)
    return os.environ.get("FKSGPU_LIBRARY", os.path.join(_HERE, "libfksgpu.so"))


class FksError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("fksgpu error %d: %s" % (code, message))
        self.code = code


if not os.path.exists(library_path()):
    raise ImportError(
        "libfksgpu.so is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
        "or `make -C fast_kinematic_simulator_b200/csrc` (there is no CPU fallback)"
    )
lib = C.CDLL(library_path())

from .abi import *  # noqa: F401,F403,E402  (constants and structures of include/fksgpu.h)
from .abi import AxisParams, EnvDesc, JointDesc, NoiseTape, Obstacle, RobotDesc, SolverParams  # noqa: F401,E402

# every symbol include/fksgpu.h declares (tests/test_capi_symbols.py checks the list against the header)
EXPORTS = (
    "fks_abi_version",
    "fks_last_error_string",
    "fks_device_count",
    "fks_default_solver_params",
    "fks_env_create",
    "fks_env_destroy",
    "fks_robot_create",
    "fks_robot_destroy",
    "fks_robot_config_stride",
    "fks_sim_create",
    "fks_sim_destroy",
    "fks_sim_result_stride",
    "fks_forward_simulate",
    "fks_reverse_simulate",
    "fks_forward_simulate_async",
    "fks_sim_synchronize",
    "fks_forward_simulate_device",
    "fks_forward_simulate_sequence",
    "fks_forward_simulate_sequence_device",
    "fks_multi_sim_create",
    "fks_multi_sim_destroy",
    "fks_multi_sim_device_count",
    "fks_multi_sim_result_stride",
    "fks_multi_forward_simulate",
    "fks_multi_forward_simulate_device",
    "fks_multi_forward_simulate_sequence",
    "fks_multi_get_statistics",
    "fks_multi_reset_statistics",
    "fks_check_config_collision",
    "fks_sim_trace_stride",
    "fks_forward_simulate_traced",
    "fks_get_statistics",
    "fks_reset_statistics",
    "fks_sim_enable_kernel_timing",
    "fks_sim_kernel_times",
    "fks_sim_launch_count",
    "fks_sim_kernel_info",
    "fks_build_environment",
    "fks_built_env_desc",
    "fks_built_env_occupancy",
    "fks_built_env_destroy",
    "fks_env_build_device",
    "fks_env_build_timings",
    "fks_env_download",
    "fks_end_states_partition",
    "fks_end_states_pairwise_distance",
    "fks_end_states_cluster",
    "fks_end_states_groups",
    "fks_end_states_gather_starts",
    "fks_debug_qr_solve",
    "fks_measure_fp64_peak",
    "fks_measure_gather_rate",
)

P = C.POINTER
lib.fks_abi_version.restype = C.c_int
lib.fks_last_error_string.restype = C.c_char_p
lib.fks_device_count.argtypes = [P(C.c_int)]
lib.fks_default_solver_params.argtypes = [P(SolverParams)]
lib.fks_default_solver_params.restype = None
lib.fks_env_create.argtypes = [C.c_int, P(EnvDesc), P(C.c_void_p)]
lib.fks_env_destroy.argtypes = [C.c_void_p]
lib.fks_env_destroy.restype = None
lib.fks_robot_create.argtypes = [C.c_int, P(RobotDesc), P(C.c_void_p)]
lib.fks_robot_destroy.argtypes = [C.c_void_p]
lib.fks_robot_destroy.restype = None
lib.fks_robot_config_stride.argtypes = [C.c_void_p]
lib.fks_sim_create.argtypes = [C.c_void_p, C.c_void_p, P(SolverParams), C.c_double, C.c_uint64, C.c_int32, P(C.c_void_p)]
lib.fks_sim_destroy.argtypes = [C.c_void_p]
lib.fks_sim_destroy.restype = None
lib.fks_sim_result_stride.argtypes = [C.c_void_p]
lib.fks_sim_result_stride.restype = C.c_size_t
_sim_args = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, P(NoiseTape), C.c_uint64, C.c_void_p]
lib.fks_forward_simulate.argtypes = _sim_args
lib.fks_reverse_simulate.argtypes = _sim_args
lib.fks_forward_simulate_async.argtypes = _sim_args
lib.fks_sim_synchronize.argtypes = [C.c_void_p]
_seq_args = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, P(NoiseTape), C.c_uint64,
             C.c_void_p]
lib.fks_forward_simulate_sequence.argtypes = _seq_args
lib.fks_multi_forward_simulate_sequence.argtypes = _seq_args
lib.fks_forward_simulate_sequence_device.argtypes = [
    C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
    C.c_uint64, C.c_void_p, C.c_void_p,
]
lib.fks_multi_sim_create.argtypes = [P(C.c_int32), C.c_int32, P(EnvDesc), P(RobotDesc), P(SolverParams), C.c_double, C.c_uint64, C.c_int32,
                                     P(C.c_void_p)]
lib.fks_multi_sim_destroy.argtypes = [C.c_void_p]
lib.fks_multi_sim_destroy.restype = None
lib.fks_multi_sim_device_count.argtypes = [C.c_void_p]
lib.fks_multi_sim_result_stride.argtypes = [C.c_void_p]
lib.fks_multi_sim_result_stride.restype = C.c_size_t
lib.fks_multi_forward_simulate.argtypes = _sim_args
lib.fks_multi_forward_simulate_device.argtypes = [C.c_void_p, P(C.c_void_p), P(C.c_void_p), C.c_size_t, C.c_size_t, C.c_int, C.c_uint64,
                                                  P(C.c_void_p)]
lib.fks_multi_get_statistics.argtypes = [C.c_void_p, P(C.c_uint64)]
lib.fks_multi_reset_statistics.argtypes = [C.c_void_p]
lib.fks_forward_simulate_device.argtypes = [
    C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
    C.c_uint64, C.c_void_p, C.c_void_p,
]
lib.fks_check_config_collision.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_double, C.c_void_p]
lib.fks_sim_trace_stride.argtypes = [C.c_void_p]
lib.fks_sim_trace_stride.restype = C.c_size_t
lib.fks_forward_simulate_traced.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, P(NoiseTape), C.c_uint64, C.c_void_p,
                                            C.c_void_p, C.c_size_t, P(C.c_size_t)]
lib.fks_get_statistics.argtypes = [C.c_void_p, P(C.c_uint64)]
lib.fks_reset_statistics.argtypes = [C.c_void_p]
lib.fks_sim_enable_kernel_timing.argtypes = [C.c_void_p, C.c_int]
lib.fks_sim_kernel_times.argtypes = [C.c_void_p, P(C.c_double), P(C.c_int)]
lib.fks_sim_launch_count.argtypes = [C.c_void_p]
lib.fks_sim_launch_count.restype = C.c_uint64
lib.fks_sim_kernel_info.argtypes = [C.c_void_p]
lib.fks_sim_kernel_info.restype = C.c_char_p
lib.fks_build_environment.argtypes = [P(Obstacle), C.c_size_t, C.c_double, P(C.c_void_p)]
lib.fks_built_env_desc.argtypes = [C.c_void_p]
lib.fks_built_env_desc.restype = P(EnvDesc)
lib.fks_built_env_occupancy.argtypes = [C.c_void_p]
lib.fks_built_env_occupancy.restype = P(C.c_uint8)
lib.fks_built_env_destroy.argtypes = [C.c_void_p]
lib.fks_built_env_destroy.restype = None
lib.fks_env_build_device.argtypes = [C.c_int, P(Obstacle), C.c_size_t, C.c_double, P(C.c_void_p)]
lib.fks_env_build_timings.argtypes = [C.c_void_p, P(C.c_double), C.c_int]
lib.fks_env_download.argtypes = [C.c_void_p, P(C.c_void_p)]
lib.fks_end_states_partition.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, P(C.c_uint64), C.c_void_p]
lib.fks_end_states_pairwise_distance.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
lib.fks_end_states_cluster.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, P(C.c_uint64), C.c_size_t, C.c_int, C.c_double, C.c_int,
                                       C.c_void_p, P(C.c_uint64), C.c_void_p]
lib.fks_end_states_groups.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, P(C.c_uint64), C.c_void_p]
lib.fks_end_states_gather_starts.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, P(C.c_uint32), C.c_size_t,
                                             C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
lib.fks_debug_qr_solve.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_size_t, C.c_void_p, C.c_void_p]
lib.fks_measure_fp64_peak.argtypes = [C.c_int, P(C.c_double)]
lib.fks_measure_gather_rate.argtypes = [C.c_int, C.c_size_t, P(C.c_double)]


def check(code):
    if code != OK:
        msg = lib.fks_last_error_string()
        raise FksError(code, msg.decode() if msg else "")


def default_solver_params():  # noqa: F811  (the library's own defaults replace abi.default_solver_params here)
    """GetDefaultSolverParameters (fast_kinematic_simulator.hpp:13-16)."""
    p = SolverParams()
    lib.fks_default_solver_params(C.byref(p))
    return p
