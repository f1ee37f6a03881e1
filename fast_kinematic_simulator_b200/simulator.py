"""Host-side mirror of the reference's simulator interface for the batched forward-simulate path.

Names follow the reference:

* ``build_complete_environment``  <- simulator_environment_builder::BuildCompleteEnvironment
  (src/fast_kinematic_simulator/simulator_environment_builder.cpp:470-476)
* ``make_{se2,se3,linked}_simulator`` <- fast_kinematic_simulator::Make{SE2,SE3,Linked}Simulator
  (include/fast_kinematic_simulator/fast_kinematic_simulator.hpp:18-22)
* ``GpuParticleContactSimulator.forward_simulate_robots`` <- SimpleParticleContactSimulator::
  ForwardSimulateRobots (simple_particle_contact_simulator.hpp:788-804); ``reverse_simulate_robots``
  (:806-822); ``get_statistics`` / ``reset_statistics`` (:488-512).
* ``forward_simulate_sequence`` runs every particle through several consecutive ForwardSimulateRobot legs in one call
  (fks_forward_simulate_sequence): the records equal those of chained ``forward_simulate_robots`` calls whose
  ``first_particle_id`` advances by n per call.

Everything computes in libfksgpu.so; this module only marshals numpy arrays across the C ABI.
"""
import ctypes as C

import numpy as np

from . import capi
from .capi import lib, check
from .robots import IDENTITY12, RobotDescription, make_transform  # noqa: F401


def _as_f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _dptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


class BuiltEnvironment:
    """Result of BuildCompleteEnvironment: collision-map metadata + SDF + surface-normal table,
    owned by the C library; numpy views are exposed for tests and the oracle."""

    def __init__(self, handle):
        self._h = handle
        self.desc = lib.fks_built_env_desc(handle).contents
        d = self.desc
        self.shape = (int(d.nx), int(d.ny), int(d.nz))
        n = self.shape[0] * self.shape[1] * self.shape[2]
        self.resolution = float(d.sdf_resolution)
        self.sdf = np.ctypeslib.as_array(d.sdf, shape=(n,)).reshape(self.shape)
        occ = lib.fks_built_env_occupancy(handle)
        self.occupancy = np.ctypeslib.as_array(occ, shape=(n,)).reshape(self.shape) if occ else None
        self.origin = np.array(list(d.origin))
        self.inverse_origin = np.array(list(d.inverse_origin))
        nc = int(d.n_normal_cells)
        self.n_normal_cells = nc
        if nc:
            self.normal_cell_index = np.ctypeslib.as_array(d.normal_cell_index, shape=(nc,))
            self.normal_cell_start = np.ctypeslib.as_array(d.normal_cell_start, shape=(nc + 1,))
            ne = int(self.normal_cell_start[-1])
            self.normal_entries = np.ctypeslib.as_array(d.normal_entries, shape=(ne * 7,)).reshape(ne, 7)
        else:
            self.normal_cell_index = np.zeros(0, np.int64)
            self.normal_cell_start = np.zeros(1, np.uint32)
            self.normal_entries = np.zeros((0, 7))

    def close(self):
        if self._h:
            lib.fks_built_env_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def build_complete_environment(obstacles, resolution):
    """obstacles: iterable of (pose12, half_extents3, object_id) -- OBSTACLE_CONFIG
    (simulator_environment_builder.hpp:25-49)."""
    arr, n = _obstacle_array(obstacles)
    h = C.c_void_p()
    check(lib.fks_build_environment(arr, n, float(resolution), C.byref(h)))
    return BuiltEnvironment(h)


def _obstacle_array(obstacles):
    obstacles = list(obstacles)
    arr = (capi.Obstacle * max(len(obstacles), 1))()
    for i, (pose, ext, oid) in enumerate(obstacles):
        arr[i].pose = (C.c_double * 12)(*[float(v) for v in pose])
        arr[i].extents = (C.c_double * 3)(*[float(v) for v in ext])
        arr[i].object_id = int(oid)
    return arr, len(obstacles)


BUILD_PHASES = ("total", "rasterize", "edt_z", "edt_y", "edt_x_sdf", "normals_mark", "normals_emit", "distance_field_check",
                "table_allocation")


def build_complete_environment_on_device(obstacles, resolution, device=0):
    """BuildCompleteEnvironment (simulator_environment_builder.cpp:470-476) computed by CUDA kernels straight into a
    device environment (fks_env_build_device): no host copy of the occupancy grid, SDF or normal table."""
    arr, n = _obstacle_array(obstacles)
    h = C.c_void_p()
    check(lib.fks_env_build_device(int(device), arr, n, float(resolution), C.byref(h)))
    return GpuEnvironment(None, device, _handle=h)


class GpuEnvironment:
    """Device copy of what the simulator copies at construction (spcs.hpp:420): SDF + normals."""

    def __init__(self, built_env, device=0, _handle=None):
        self.built = built_env
        self.device = device
        if _handle is not None:  # built on the device (build_complete_environment_on_device)
            self._h = _handle
            return
        self._h = C.c_void_p()
        desc = built_env.desc if isinstance(built_env, BuiltEnvironment) else built_env
        check(lib.fks_env_create(device, C.byref(desc), C.byref(self._h)))

    def download(self):
        """Host copy of the device environment (fks_env_download) as a BuiltEnvironment."""
        h = C.c_void_p()
        check(lib.fks_env_download(self._h, C.byref(h)))
        return BuiltEnvironment(h)

    @property
    def build_timings_ms(self):
        """Device time of each phase of the device builder (zeros for uploaded environments)."""
        out = (C.c_double * len(BUILD_PHASES))()
        check(lib.fks_env_build_timings(self._h, out, len(BUILD_PHASES)))
        return {k: float(out[i]) for i, k in enumerate(BUILD_PHASES)}

    def close(self):
        if self._h:
            lib.fks_env_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GpuRobot:
    def __init__(self, description, device=0):
        self.description = description
        self.device = device
        self._h = C.c_void_p()
        d = description.to_c()
        check(lib.fks_robot_create(device, C.byref(d), C.byref(self._h)))
        self.config_stride = lib.fks_robot_config_stride(self._h)

    def close(self):
        if self._h:
            lib.fks_robot_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def result_dtype(stride):
    """fks_result record: cfg_stride doubles followed by fks_result_tail."""
    return np.dtype([("cfg", np.float64, (stride,)), ("flags", np.uint32), ("n_microsteps", np.uint32),
                     ("n_resolver_iters", np.uint32), ("n_steps", np.uint32)])


class SimulationResults:
    """vector<SimulationResult> (spcs.hpp:918): result_config, did_contact, plus the per-particle
    counters the parity tests and the metric need."""

    def __init__(self, records):
        self.records = records
        self.configs = records["cfg"]
        self.flags = records["flags"]
        self.n_microsteps = records["n_microsteps"]
        self.n_resolver_iters = records["n_resolver_iters"]
        self.n_steps = records["n_steps"]

    @property
    def did_contact(self):
        return (self.flags & capi.FLAG_DID_CONTACT) != 0

    @property
    def resolve_failed(self):
        return (self.flags & capi.FLAG_RESOLVE_FAILED) != 0

    def __len__(self):
        return len(self.records)


def make_tape(draws, offsets, decisions=None, decision_offsets=None):
    """fks_noise_tape: the injected truncated-normal draws and, optionally, the decision tape (include/fksgpu.h)."""
    draws = _as_f64(draws)
    if not draws.size:
        draws = np.zeros(1)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    t = capi.NoiseTape()
    t.draws = _dptr(draws)
    t.offsets = offsets.ctypes.data_as(C.POINTER(C.c_uint64))
    keep = [draws, offsets]
    if decisions is not None:
        decisions = np.ascontiguousarray(decisions, dtype=np.uint64)
        if not decisions.size:
            decisions = np.zeros(1, dtype=np.uint64)
        decision_offsets = np.ascontiguousarray(decision_offsets, dtype=np.uint64)
        t.decisions = decisions.ctypes.data_as(C.POINTER(C.c_uint64))
        t.decision_offsets = decision_offsets.ctypes.data_as(C.POINTER(C.c_uint64))
        keep += [decisions, decision_offsets]
    return t, keep


def sequence_inputs(starts, targets, stride):
    """Checked arrays of a sequence call: starts (n, stride); targets (M, n_targets, stride), (M, stride) meaning one
    target per leg."""
    starts = _as_f64(starts).reshape(-1, stride)
    targets = _as_f64(targets)
    if targets.ndim == 2:
        targets = targets.reshape(targets.shape[0], 1, targets.shape[1])
    if targets.ndim != 3 or targets.shape[2] != stride:
        raise ValueError("sequence targets must have shape (legs, n_targets, %d) or (legs, %d), not %s" % (stride, stride, targets.shape))
    return starts, np.ascontiguousarray(targets)


def _dev_ptr(x):
    if x is None:
        return None
    return x.data_ptr() if hasattr(x, "data_ptr") else int(x)


class GpuParticleContactSimulator:
    """The GPU sibling of SimpleParticleContactSimulator for the batch calls."""

    def __init__(self, env, robot, solver_params=None, simulation_controller_frequency=25.0, prng_seed=42, debug_level=0):
        self.env = env
        self.robot = robot
        self.params = solver_params if solver_params is not None else capi.default_solver_params()
        self._h = C.c_void_p()
        check(lib.fks_sim_create(env._h, robot._h, C.byref(self.params), float(simulation_controller_frequency),
                                 int(prng_seed), int(debug_level), C.byref(self._h)))
        self.config_stride = robot.config_stride
        self.result_stride = lib.fks_sim_result_stride(self._h)
        self.dtype = result_dtype(self.config_stride)
        assert self.dtype.itemsize == self.result_stride

    # -- ForwardSimulateRobots / ReverseSimulateRobots (host buffers; H2D + kernel + D2H inside) --
    def _simulate(self, fn, starts, targets, allow_contacts, noise_mode, tape, first_particle_id, out):
        starts = _as_f64(starts).reshape(-1, self.config_stride)
        targets = _as_f64(targets).reshape(-1, self.config_stride)
        n = starts.shape[0]
        if out is None:
            out = np.empty(n, dtype=self.dtype)
        ctape, keep = (None, None)
        if tape is not None:
            ctape, keep = make_tape(*tape)
        check(fn(self._h, starts.ctypes.data, targets.ctypes.data, n, targets.shape[0], int(bool(allow_contacts)),
                 int(noise_mode), C.byref(ctape) if ctape is not None else None, int(first_particle_id), out.ctypes.data))
        return SimulationResults(out)

    def forward_simulate_robots(self, starts, targets, allow_contacts=True, noise_mode=capi.NOISE_PHILOX, tape=None,
                                first_particle_id=0, out=None):
        return self._simulate(lib.fks_forward_simulate, starts, targets, allow_contacts, noise_mode, tape, first_particle_id, out)

    def reverse_simulate_robots(self, starts, targets, allow_contacts=True, noise_mode=capi.NOISE_PHILOX, tape=None,
                                first_particle_id=0, out=None):
        return self._simulate(lib.fks_reverse_simulate, starts, targets, allow_contacts, noise_mode, tape, first_particle_id, out)

    def forward_simulate_sequence(self, starts, targets, allow_contacts=True, noise_mode=capi.NOISE_PHILOX, tape=None,
                                  first_particle_id=0, out=None):
        """Every particle through M consecutive legs in one kernel launch (fks_forward_simulate_sequence): leg k drives it from
        where leg k-1 left it to targets[k].  targets: (M, n_targets, stride) or (M, stride).  Returns SimulationResults over
        records of shape (M, n), equal to M chained forward_simulate_robots calls with first_particle_id + k * n.  An injected
        tape holds one span per particle covering all its legs."""
        starts, targets = sequence_inputs(starts, targets, self.config_stride)
        n, (m, n_targets) = starts.shape[0], targets.shape[:2]
        if out is None:
            out = np.empty((m, n), dtype=self.dtype)
        ctape, keep = (None, None)
        if tape is not None:
            ctape, keep = make_tape(*tape)
        check(lib.fks_forward_simulate_sequence(self._h, starts.ctypes.data, targets.ctypes.data, n, n_targets, m, int(bool(allow_contacts)),
                                                int(noise_mode), C.byref(ctape) if ctape is not None else None, int(first_particle_id),
                                                out.ctypes.data))
        return SimulationResults(out)

    # -- device-resident variant (torch tensors or raw pointers), asynchronous on `stream` --------
    def forward_simulate_sequence_device(self, d_starts, d_targets, n, n_targets, n_legs, d_results, allow_contacts=True,
                                         noise_mode=capi.NOISE_PHILOX, d_tape=None, d_tape_offsets=None, first_particle_id=0, stream=0):
        """forward_simulate_sequence on device buffers: d_targets [n_legs][n_targets][stride], d_results [n_legs][n] records."""
        check(lib.fks_forward_simulate_sequence_device(self._h, _dev_ptr(d_starts), _dev_ptr(d_targets), int(n), int(n_targets), int(n_legs),
                                                       int(bool(allow_contacts)), int(noise_mode), _dev_ptr(d_tape), _dev_ptr(d_tape_offsets),
                                                       int(first_particle_id), _dev_ptr(d_results), int(stream) if stream else None))

    def forward_simulate_device(self, d_starts, d_targets, n, n_targets, d_results, allow_contacts=True,
                                noise_mode=capi.NOISE_PHILOX, d_tape=None, d_tape_offsets=None, first_particle_id=0, stream=0):
        def ptr(x):
            if x is None:
                return None
            return x.data_ptr() if hasattr(x, "data_ptr") else int(x)

        check(lib.fks_forward_simulate_device(self._h, ptr(d_starts), ptr(d_targets), int(n), int(n_targets),
                                              int(bool(allow_contacts)), int(noise_mode), ptr(d_tape), ptr(d_tape_offsets),
                                              int(first_particle_id), ptr(d_results), int(stream) if stream else None))

    # -- first consumer of a batch on the device (SURVEY 8f-3; the planner's use of the results, uncertainty_planning_core.cpp:97-99)
    def end_states_partition(self, d_results, n, d_order, stream=0):
        """d_order (n x uint32 on the device) = ids without contact (ascending), then ids with contact (ascending);
        returns (n_without_contact, n_with_contact)."""
        counts = (C.c_uint64 * 2)()
        check(lib.fks_end_states_partition(self._h, _dev_ptr(d_results), int(n), _dev_ptr(d_order), counts, int(stream) if stream else None))
        return int(counts[0]), int(counts[1])

    def end_states_pairwise_distance(self, d_results, m, d_out, d_subset=None, stream=0):
        """d_out[a * m + b] = ComputeConfigurationDistanceTo (spcs.hpp:898) between records d_subset[a] and d_subset[b]."""
        check(lib.fks_end_states_pairwise_distance(self._h, _dev_ptr(d_results), _dev_ptr(d_subset), int(m), _dev_ptr(d_out),
                                                   int(stream) if stream else None))

    def end_states_cluster(self, d_results, segment_offsets, d_labels, max_cluster_distance, linkage=capi.LINKAGE_COMPLETE, d_order=None,
                           separate_contact=False, stream=0):
        """Flat single / complete-linkage clustering under max_cluster_distance inside every segment [offsets[s], offsets[s+1])
        of the positions (record d_order[p], or p), on the device (fks_end_states_cluster).  d_labels (m x uint32 on the device)
        receives global cluster ids, segment by segment in increasing order of each cluster's smallest position; returns the
        clusters per segment (numpy uint64)."""
        offsets = np.ascontiguousarray(segment_offsets, dtype=np.uint64)
        n_segments = max(len(offsets) - 1, 0)
        counts = np.zeros(max(n_segments, 1), np.uint64)
        check(lib.fks_end_states_cluster(self._h, _dev_ptr(d_results), _dev_ptr(d_order), offsets.ctypes.data_as(C.POINTER(C.c_uint64)),
                                         n_segments, int(linkage), float(max_cluster_distance), int(bool(separate_contact)),
                                         _dev_ptr(d_labels), counts.ctypes.data_as(C.POINTER(C.c_uint64)), int(stream) if stream else None))
        return counts[:n_segments]

    def end_states_groups(self, d_results, m, d_labels, n_clusters, d_group_offsets, d_members, d_representatives, d_radius, d_order=None,
                          stream=0):
        """The clusters of positions 0 .. m-1 (record d_order[p], or p; cluster d_labels[p]) as groups, on the device
        (fks_end_states_groups): d_members[d_group_offsets[c] .. d_group_offsets[c+1]) = group c's record ids in position
        order, d_representatives[c] / d_radius[c] = its minimax member and that member's largest distance to the others.
        Device buffers (uint32 / float64) of n_clusters + 1, m, n_clusters, n_clusters entries; returns the group sizes
        (numpy uint64)."""
        sizes = np.zeros(max(int(n_clusters), 1), np.uint64)
        check(lib.fks_end_states_groups(self._h, _dev_ptr(d_results), _dev_ptr(d_order), int(m), _dev_ptr(d_labels), int(n_clusters),
                                        _dev_ptr(d_group_offsets), _dev_ptr(d_members), _dev_ptr(d_representatives), _dev_ptr(d_radius),
                                        sizes.ctypes.data_as(C.POINTER(C.c_uint64)), int(stream) if stream else None))
        return sizes[:int(n_clusters)]

    def end_states_gather_starts(self, d_results, d_group_offsets, d_members, n_clusters, selected, per_group, d_starts,
                                 d_group_targets=None, d_targets=None, stream=0):
        """The next batch from groups (fks_end_states_gather_starts): slot s takes group selected[s] (host ids, repeats
        allowed) and fills per_group starts with its members' configurations, cyclically; with d_group_targets
        ([len(selected)][stride]), d_targets gets slot s's target per_group times.  Asynchronous on `stream`."""
        sel = np.asarray(selected).reshape(-1)
        if sel.size and (sel.min() < 0 or sel.max() > 0xFFFFFFFF):
            raise capi.FksError(capi.ERR_INVALID_ARGUMENT, "end_states_gather_starts: a selected group id is not a uint32")
        sel = np.ascontiguousarray(sel, dtype=np.uint32)
        check(lib.fks_end_states_gather_starts(self._h, _dev_ptr(d_results), _dev_ptr(d_group_offsets), _dev_ptr(d_members), int(n_clusters),
                                               sel.ctypes.data_as(C.POINTER(C.c_uint32)), sel.size, int(per_group), _dev_ptr(d_group_targets),
                                               _dev_ptr(d_starts), _dev_ptr(d_targets), int(stream) if stream else None))

    def trace_dtype(self):
        width = (lib.fks_sim_trace_stride(self._h) - 16) // 8
        return np.dtype([("kind", np.uint32), ("step", np.uint32), ("microstep", np.uint32), ("iteration", np.uint32),
                         ("values", np.float64, (width,))])

    def forward_simulate_robot_traced(self, start, target, allow_contacts=True, noise_mode=capi.NOISE_PHILOX, tape=None,
                                      particle_id=0, capacity=65536):
        """ForwardSimulateRobot with enable_tracing (spcs.hpp:824-829): (SimulationResults of one particle, trace records).
        The flat records follow the order in which the reference fills ForwardSimulationStepTrace (spcs.hpp:1583-1617,
        :1703, :1714, :1778); `values` holds n_dof control values or cfg_stride configuration values."""
        start = _as_f64(start).reshape(1, self.config_stride)
        target = _as_f64(target).reshape(1, self.config_stride)
        out = np.empty(1, dtype=self.dtype)
        rec = np.zeros(capacity, dtype=self.trace_dtype())
        ctape, keep = (None, None)
        if tape is not None:
            ctape, keep = make_tape(*tape)
        n = C.c_size_t(0)
        check(lib.fks_forward_simulate_traced(self._h, start.ctypes.data, target.ctypes.data, int(bool(allow_contacts)), int(noise_mode),
                                              C.byref(ctape) if ctape is not None else None, int(particle_id), out.ctypes.data,
                                              rec.ctypes.data, capacity, C.byref(n)))
        if n.value > capacity:
            raise capi.FksError(capi.ERR_INVALID_ARGUMENT, "trace capacity %d too small for %d records" % (capacity, n.value))
        return SimulationResults(out), rec[: n.value]

    def check_config_collision(self, configs, inflation_ratio=0.0):
        """CheckConfigCollision (spcs.hpp:1398-1416) for a batch of configurations -> bool array."""
        configs = _as_f64(configs).reshape(-1, self.config_stride)
        out = np.zeros(configs.shape[0], dtype=np.uint8)
        check(lib.fks_check_config_collision(self._h, configs.ctypes.data, configs.shape[0], float(inflation_ratio), out.ctypes.data))
        return out.astype(bool)

    def get_statistics(self):
        out = (C.c_uint64 * capi.NUM_STATS)()
        check(lib.fks_get_statistics(self._h, out))
        return {k: int(out[i]) for i, k in enumerate(capi.STAT_NAMES)}

    def reset_statistics(self):
        check(lib.fks_reset_statistics(self._h))

    def enable_kernel_timing(self, enable=True):
        check(lib.fks_sim_enable_kernel_timing(self._h, int(bool(enable))))

    def kernel_times_ms(self):
        """Device time of the simulate kernel of the last batch call (a one-element list once timing is enabled)."""
        out = (C.c_double * 4)()
        n = C.c_int(0)
        check(lib.fks_sim_kernel_times(self._h, out, C.byref(n)))
        return [float(out[i]) for i in range(n.value)]

    @property
    def launch_count(self):
        return int(lib.fks_sim_launch_count(self._h))

    @property
    def kernel_info(self):
        return lib.fks_sim_kernel_info(self._h).decode()

    def close(self):
        if self._h:
            lib.fks_sim_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _make(kind, built_env, robot_description, solver_params, simulation_controller_frequency, prng_seed, debug_level, device):
    if robot_description.kind != kind:
        raise ValueError("robot description kind does not match the factory")
    env = built_env if isinstance(built_env, GpuEnvironment) else GpuEnvironment(built_env, device)
    robot = GpuRobot(robot_description, device)
    return GpuParticleContactSimulator(env, robot, solver_params, simulation_controller_frequency, prng_seed, debug_level)


def make_se2_simulator(built_env, robot_description, solver_params=None, simulation_controller_frequency=25.0, prng_seed=42,
                       debug_level=0, device=0):
    """MakeSE2Simulator (fast_kinematic_simulator.cpp:4-25)."""
    return _make(capi.ROBOT_SE2, built_env, robot_description, solver_params, simulation_controller_frequency, prng_seed, debug_level, device)


def make_se3_simulator(built_env, robot_description, solver_params=None, simulation_controller_frequency=25.0, prng_seed=42,
                       debug_level=0, device=0):
    """MakeSE3Simulator (fast_kinematic_simulator.cpp:27-48)."""
    return _make(capi.ROBOT_SE3, built_env, robot_description, solver_params, simulation_controller_frequency, prng_seed, debug_level, device)


def make_linked_simulator(built_env, robot_description, solver_params=None, simulation_controller_frequency=25.0, prng_seed=42,
                          debug_level=0, device=0):
    """MakeLinkedSimulator (fast_kinematic_simulator.cpp:50-71)."""
    return _make(capi.ROBOT_LINKED, built_env, robot_description, solver_params, simulation_controller_frequency, prng_seed, debug_level, device)


def debug_qr_solve(systems, device=0):
    """fks_debug_qr_solve: the device's stacked-Jacobian solver on a list of (A rows x cols, b) systems sharing `cols`.
    Returns (solutions n x cols, flags n)."""
    n = len(systems)
    cols = int(systems[0][0].shape[1])
    rows = np.array([A.shape[0] for A, _ in systems], dtype=np.int32)
    offsets = np.zeros(n + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(rows.astype(np.uint64) * np.uint64(cols + 1))
    flat = np.empty(int(offsets[-1]), dtype=np.float64)
    for i, (A, b) in enumerate(systems):
        o = int(offsets[i])
        r = int(rows[i])
        flat[o:o + r * cols] = np.asarray(A, dtype=np.float64).T.reshape(-1)  # column major
        flat[o + r * cols:o + r * (cols + 1)] = b
    x = np.zeros((n, cols))
    flags = np.zeros(n, dtype=np.uint32)
    check(lib.fks_debug_qr_solve(int(device), flat.ctypes.data, offsets.ctypes.data, rows.ctypes.data, cols, n, x.ctypes.data,
                                 flags.ctypes.data))
    return x, flags


class MultiGpuParticleContactSimulator:
    """ForwardSimulateRobots over several GPUs of one box behind one call (fks_multi_*, SURVEY 8e): contiguous particle shards,
    environment and robot replicated per device, records independent of the device count."""

    def __init__(self, built_env, robot_description, devices, solver_params=None, simulation_controller_frequency=25.0,
                 prng_seed=42, debug_level=0):
        self.params = solver_params if solver_params is not None else capi.default_solver_params()
        self.robot_description = robot_description
        desc = built_env.desc if isinstance(built_env, BuiltEnvironment) else built_env
        devices = list(range(devices)) if isinstance(devices, int) else list(devices)
        dev = (C.c_int32 * len(devices))(*devices)
        rd = robot_description.to_c()
        self._h = C.c_void_p()
        check(lib.fks_multi_sim_create(dev, len(devices), C.byref(desc), C.byref(rd), C.byref(self.params),
                                       float(simulation_controller_frequency), int(prng_seed), int(debug_level), C.byref(self._h)))
        self.devices = devices
        self.config_stride = robot_description.config_stride
        self.result_stride = lib.fks_multi_sim_result_stride(self._h)
        self.dtype = result_dtype(self.config_stride)

    def forward_simulate_robots(self, starts, targets, allow_contacts=True, noise_mode=capi.NOISE_PHILOX, tape=None,
                                first_particle_id=0, out=None):
        starts = _as_f64(starts).reshape(-1, self.config_stride)
        targets = _as_f64(targets).reshape(-1, self.config_stride)
        n = starts.shape[0]
        if out is None:
            out = np.empty(n, dtype=self.dtype)
        ctape, keep = (None, None)
        if tape is not None:
            ctape, keep = make_tape(*tape)
        check(lib.fks_multi_forward_simulate(self._h, starts.ctypes.data, targets.ctypes.data, n, targets.shape[0],
                                             int(bool(allow_contacts)), int(noise_mode), C.byref(ctape) if ctape is not None else None,
                                             int(first_particle_id), out.ctypes.data))
        return SimulationResults(out)

    def forward_simulate_sequence(self, starts, targets, allow_contacts=True, noise_mode=capi.NOISE_PHILOX, tape=None,
                                  first_particle_id=0, out=None):
        """GpuParticleContactSimulator.forward_simulate_sequence over the devices (fks_multi_forward_simulate_sequence)."""
        starts, targets = sequence_inputs(starts, targets, self.config_stride)
        n, (m, n_targets) = starts.shape[0], targets.shape[:2]
        if out is None:
            out = np.empty((m, n), dtype=self.dtype)
        ctape, keep = (None, None)
        if tape is not None:
            ctape, keep = make_tape(*tape)
        check(lib.fks_multi_forward_simulate_sequence(self._h, starts.ctypes.data, targets.ctypes.data, n, n_targets, m,
                                                      int(bool(allow_contacts)), int(noise_mode),
                                                      C.byref(ctape) if ctape is not None else None, int(first_particle_id),
                                                      out.ctypes.data))
        return SimulationResults(out)

    def forward_simulate_device(self, d_starts, d_targets, n, n_targets, d_results, allow_contacts=True, first_particle_id=0):
        """d_starts / d_targets / d_results: one device pointer (or torch tensor) per device; every d_results[d] ends up
        holding all n records (ncclAllGather)."""
        def arr(xs):
            return (C.c_void_p * len(xs))(*[x.data_ptr() if hasattr(x, "data_ptr") else int(x) for x in xs])

        check(lib.fks_multi_forward_simulate_device(self._h, arr(d_starts), arr(d_targets), int(n), int(n_targets),
                                                    int(bool(allow_contacts)), int(first_particle_id), arr(d_results)))

    def get_statistics(self):
        out = (C.c_uint64 * capi.NUM_STATS)()
        check(lib.fks_multi_get_statistics(self._h, out))
        return {k: int(out[i]) for i, k in enumerate(capi.STAT_NAMES)}

    def reset_statistics(self):
        check(lib.fks_multi_reset_statistics(self._h))

    def close(self):
        if self._h:
            lib.fks_multi_sim_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
