"""ctypes binding of libstomp_b200.so (include/stomp_b200.h) for the test and benchmark harness.

The product is the C-ABI library and the C++ StompPlanner above it (include/wrapper/stomp/StompPlanner.hpp);
this module only marshals numpy arrays into those calls.  There is no Python or CPU fallback: if the
shared library is missing, or there is no CUDA device, the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libstomp_b200.so")
MAX_DIMS = 32
COMM_ID_BYTES = 128

OK = 0
ERR_NO_DEVICE = -2
ERR_UNSUPPORTED = -5

TENSORS = dict(rollouts=0, noise=1, state_costs=2, verdicts=3, control_costs=4, cumulative_costs=5, full_costs=6,
               total_cost=7, probabilities=8, full_probabilities=9, updates=10, parameters=11, parameters_all=12,
               stddevs=13, noiseless_state_costs=14, noiseless_control_costs=15, unit_noise=16, epsilon=17,
               rollout_validity=18, noise_projected=19, rollouts_projected=20)
KERNELS = dict(sample=0, cost=1, weights=2, update=3, apply=4, reuse=5, rows=6)

# every symbol include/stomp_b200.h declares (tests/test_cabi_symbols.py checks the library exports them)
SYMBOLS = [
    "stomp_b200_default_config", "stomp_b200_abi_version", "stomp_b200_status_string", "stomp_b200_last_error",
    "stomp_b200_create", "stomp_b200_destroy", "stomp_b200_set_chain", "stomp_b200_set_spheres", "stomp_b200_set_sdf",
    "stomp_b200_set_control_cost_matrices", "stomp_b200_set_policy", "stomp_b200_set_policies", "stomp_b200_host_policy",
    "stomp_b200_host_initial_trajectory", "stomp_b200_begin_solve", "stomp_b200_iterate",
    "stomp_b200_next_num_generated", "stomp_b200_run", "stomp_b200_solve", "stomp_b200_finish_solve", "stomp_b200_num_rollouts",
    "stomp_b200_get_tensor", "stomp_b200_evaluate_states", "stomp_b200_sphere_centres", "stomp_b200_comm_unique_id",
    "stomp_b200_comm_init", "stomp_b200_exchange_kind", "stomp_b200_set_profiling", "stomp_b200_kernel_stats", "stomp_b200_reset_kernel_stats",
    "stomp_b200_set_timeline", "stomp_b200_get_timeline", "stomp_b200_launch_count", "stomp_b200_graph_replays", "stomp_b200_timer_begin", "stomp_b200_timer_end", "stomp_b200_synchronize",
    "stomp_b200_state_kernel_kind", "stomp_b200_state_kernel_source", "stomp_b200_codegen_selftest",
    "stomp_b200_set_cost_cumulation", "stomp_b200_set_self_collision", "stomp_b200_set_cost_extras",
    "stomp_b200_build_sdf_primitives", "stomp_b200_build_sdf_occupancy", "stomp_b200_build_sdf_scene", "stomp_b200_get_sdf",
    "stomp_b200_select_scene", "stomp_b200_set_query_scenes",
]


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("num_time_steps", C.c_int32), ("num_dimensions", C.c_int32),
        ("min_rollouts", C.c_int32), ("max_rollouts", C.c_int32), ("num_rollouts_per_iteration", C.c_int32),
        ("num_queries", C.c_int32),
        ("movement_duration", C.c_double), ("control_cost_weight", C.c_double), ("min_cost_improvement", C.c_double),
        ("noise_stddev", C.c_double * MAX_DIMS), ("noise_decay", C.c_double * MAX_DIMS),
        ("noise_min_stddev", C.c_double * MAX_DIMS), ("derivative_weights", C.c_double * 4),
        ("cost_scaling_h", C.c_double),
        ("use_noise_adaptation", C.c_int32), ("use_cumulative_costs", C.c_int32), ("use_projection", C.c_int32),
        ("per_timestep_minmax", C.c_int32), ("device", C.c_int32), ("world_size", C.c_int32), ("rank", C.c_int32),
        ("shard_mode", C.c_int32), ("keep_debug_tensors", C.c_int32), ("seed", C.c_uint64),
    ]


def codegen_selftest():
    """Generates the specialised state kernel for a structure that uses every branch and compiles it with NVRTC
    for sm_100a (no device needed).  Returns (status, log)."""
    log = C.create_string_buffer(1 << 16)
    rc = lib().stomp_b200_codegen_selftest(log, len(log))
    return rc, log.value.decode()


class StompB200Error(RuntimeError):
    def __init__(self, code, where, detail=""):
        self.code = code
        super().__init__(f"{where}: status {code} ({detail})")


_lib = None


def lib():
    """Load the C-ABI library; raises if it has not been built (python -c 'import __graft_entry__ as g; g.build()')."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(f"{LIB_PATH} is missing: the CUDA extension has not been built and there is no fallback")
        L = C.CDLL(LIB_PATH)
        dp, ip, u8p, vp = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint8), C.c_void_p
        L.stomp_b200_default_config.argtypes = [C.POINTER(Config)]
        L.stomp_b200_default_config.restype = None
        L.stomp_b200_abi_version.restype = C.c_int
        L.stomp_b200_status_string.restype = C.c_char_p
        L.stomp_b200_status_string.argtypes = [C.c_int]
        L.stomp_b200_last_error.restype = C.c_char_p
        L.stomp_b200_last_error.argtypes = [vp]
        L.stomp_b200_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
        L.stomp_b200_destroy.argtypes = [vp]
        L.stomp_b200_set_chain.argtypes = [vp, C.c_int32, dp, dp, dp, ip, ip, dp, dp]
        L.stomp_b200_set_spheres.argtypes = [vp, C.c_int32, ip, dp, dp]
        L.stomp_b200_set_sdf.argtypes = [vp, ip, dp, C.c_double, C.POINTER(C.c_float)]
        L.stomp_b200_set_self_collision.argtypes = [vp, C.c_int32, ip]
        L.stomp_b200_build_sdf_primitives.argtypes = [vp, ip, dp, C.c_double, C.c_int32, ip, dp, dp]
        L.stomp_b200_build_sdf_occupancy.argtypes = [vp, ip, dp, C.c_double, u8p]
        L.stomp_b200_build_sdf_scene.argtypes = [vp, ip, dp, C.c_double, C.c_int32, dp, C.c_int32, C.c_int32, dp, dp, u8p]
        L.stomp_b200_get_sdf.argtypes = [vp, C.POINTER(C.c_float), C.c_size_t, ip, dp, dp]
        L.stomp_b200_select_scene.argtypes = [vp, C.c_int32]
        L.stomp_b200_set_query_scenes.argtypes = [vp, C.c_int32, C.c_int32, ip]
        L.stomp_b200_set_control_cost_matrices.argtypes = [vp, dp, dp, dp]
        L.stomp_b200_set_policy.argtypes = [vp, C.c_int32, dp, dp]
        L.stomp_b200_set_policies.argtypes = [vp, C.c_int32, C.c_int32, dp, dp]
        L.stomp_b200_host_policy.argtypes = [C.c_int32, C.c_int32, C.c_double, dp, dp, C.c_int32, dp, dp, dp, dp, dp]
        L.stomp_b200_host_initial_trajectory.argtypes = [C.c_int32, C.c_int32, dp, dp, dp]
        L.stomp_b200_begin_solve.argtypes = [vp]
        L.stomp_b200_iterate.argtypes = [vp, C.c_int32, dp, dp, dp, u8p, ip]
        L.stomp_b200_next_num_generated.argtypes = [vp]
        L.stomp_b200_next_num_generated.restype = C.c_int32
        L.stomp_b200_run.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32]
        L.stomp_b200_solve.argtypes = [vp, C.c_int32, C.c_int32, ip]
        L.stomp_b200_finish_solve.argtypes = [vp, dp, ip, ip, dp]
        L.stomp_b200_num_rollouts.argtypes = [vp, ip, ip]
        L.stomp_b200_get_tensor.argtypes = [vp, C.c_int32, vp, C.c_size_t]
        L.stomp_b200_evaluate_states.argtypes = [vp, dp, C.c_int32, C.c_int32, dp, u8p, u8p]
        L.stomp_b200_sphere_centres.argtypes = [vp, dp, C.c_int32, dp]
        L.stomp_b200_comm_unique_id.argtypes = [vp]
        L.stomp_b200_comm_init.argtypes = [vp, vp]
        L.stomp_b200_set_profiling.argtypes = [vp, C.c_int32]
        L.stomp_b200_kernel_stats.argtypes = [vp, C.c_int32, dp, C.POINTER(C.c_int64)]
        L.stomp_b200_reset_kernel_stats.argtypes = [vp]
        L.stomp_b200_set_timeline.argtypes = [vp, C.c_int32]
        L.stomp_b200_get_timeline.argtypes = [vp, C.c_int32, dp, ip]
        L.stomp_b200_launch_count.argtypes = [vp]
        L.stomp_b200_graph_replays.argtypes = [vp]
        L.stomp_b200_graph_replays.restype = C.c_int64
        L.stomp_b200_state_kernel_kind.argtypes = [vp, C.c_char_p, C.c_size_t]
        L.stomp_b200_state_kernel_kind.restype = C.c_int32
        L.stomp_b200_set_cost_extras.argtypes = [vp, C.c_int32, C.c_double, C.c_double, C.c_int32, dp, dp, C.c_double]
        L.stomp_b200_exchange_kind.argtypes = [vp, C.c_char_p, C.c_size_t]
        L.stomp_b200_exchange_kind.restype = C.c_int32
        L.stomp_b200_state_kernel_source.argtypes = [vp, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.stomp_b200_codegen_selftest.argtypes = [C.c_char_p, C.c_size_t]
        L.stomp_b200_set_cost_cumulation.argtypes = [vp, C.c_int32]
        L.stomp_b200_launch_count.restype = C.c_int64
        L.stomp_b200_timer_begin.argtypes = [vp]
        L.stomp_b200_timer_end.argtypes = [vp, dp]
        L.stomp_b200_synchronize.argtypes = [vp]
        _lib = L
    return _lib


def _dp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_int32))


def _c64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def default_config() -> Config:
    cfg = Config()
    lib().stomp_b200_default_config(C.byref(cfg))
    return cfg


def host_initial_trajectory(start, goal, T):
    """OptimizationTask::updateTrajectory on the host (no device needed)."""
    s, g = _c64(start), _c64(goal)
    D = s.shape[0]
    out = np.empty((D, T + 12))
    rc = lib().stomp_b200_host_initial_trajectory(T, D, _dp(s), _dp(g), _dp(out))
    if rc:
        raise StompB200Error(rc, "stomp_b200_host_initial_trajectory")
    return out


def host_policy(initial_all, duration, weights=(0.0, 0.0, 1.0, 0.0), set_to_min_control_cost=True):
    """CovariantMovementPrimitive::initialize (+ setToMinControlCost) on the host (no device needed)."""
    init = _c64(initial_all)
    D, N = init.shape
    T = N - 12
    w = _c64(weights)
    out = dict(R=np.empty((T, T)), Rinv=np.empty((T, T)), L=np.empty((T, T)), params_all=np.empty((D, N)),
               mincc=np.empty((D, T)))
    rc = lib().stomp_b200_host_policy(T, D, float(duration), _dp(w), _dp(init), int(set_to_min_control_cost),
                                      _dp(out["R"]), _dp(out["Rinv"]), _dp(out["L"]), _dp(out["params_all"]), _dp(out["mincc"]))
    if rc:
        raise StompB200Error(rc, "stomp_b200_host_policy")
    return out


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(COMM_ID_BYTES)
    rc = lib().stomp_b200_comm_unique_id(buf)
    if rc:
        raise StompB200Error(rc, "stomp_b200_comm_unique_id")
    return buf.raw


class Engine:
    """One stomp_b200_engine (one GPU)."""

    def __init__(self, *, num_time_steps, num_dimensions, min_rollouts, max_rollouts, num_rollouts_per_iteration,
                 num_queries=1, movement_duration=5.0, control_cost_weight=0.001, min_cost_improvement=0.01,
                 noise_stddev=None, noise_decay=None, noise_min_stddev=None, derivative_weights=(0.0, 0.0, 1.0, 0.0),
                 use_noise_adaptation=True, use_cumulative_costs=True, use_projection=False, per_timestep_minmax=False,
                 device=0, world_size=1, rank=0, shard_mode=0, keep_debug_tensors=False, seed=2024):
        cfg = default_config()
        cfg.num_time_steps, cfg.num_dimensions = num_time_steps, num_dimensions
        cfg.min_rollouts, cfg.max_rollouts = min_rollouts, max_rollouts
        cfg.num_rollouts_per_iteration, cfg.num_queries = num_rollouts_per_iteration, num_queries
        cfg.movement_duration, cfg.control_cost_weight = movement_duration, control_cost_weight
        cfg.min_cost_improvement = min_cost_improvement
        for i in range(num_dimensions):
            if noise_stddev is not None:
                cfg.noise_stddev[i] = float(noise_stddev[i])
            if noise_decay is not None:
                cfg.noise_decay[i] = float(noise_decay[i])
            if noise_min_stddev is not None:
                cfg.noise_min_stddev[i] = float(noise_min_stddev[i])
        for i in range(4):
            cfg.derivative_weights[i] = float(derivative_weights[i])
        cfg.use_noise_adaptation, cfg.use_cumulative_costs = int(use_noise_adaptation), int(use_cumulative_costs)
        cfg.use_projection, cfg.per_timestep_minmax = int(use_projection), int(per_timestep_minmax)
        cfg.device, cfg.world_size, cfg.rank, cfg.shard_mode = device, world_size, rank, shard_mode
        cfg.keep_debug_tensors, cfg.seed = int(keep_debug_tensors), seed
        self.cfg = cfg
        self.T, self.D, self.N = num_time_steps, num_dimensions, num_time_steps + 12
        self.S = 0
        self.h = C.c_void_p()
        rc = lib().stomp_b200_create(C.byref(cfg), C.byref(self.h))
        if rc:
            self.h = None
            raise StompB200Error(rc, "stomp_b200_create", lib().stomp_b200_status_string(rc).decode())
        if world_size > 1 and shard_mode == 1:
            from . import sharding
            self.query_offset, self.Q = sharding.query_shard(num_queries, world_size, rank)   # as stomp_b200_create
        else:
            self.query_offset, self.Q = 0, num_queries

    def close(self):
        if getattr(self, "h", None):
            lib().stomp_b200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, where):
        if rc:
            raise StompB200Error(rc, where, lib().stomp_b200_last_error(self.h).decode())

    # ---- scene -----------------------------------------------------------------------------------
    def set_chain(self, chain):
        xyz, rpy, ax = _c64(chain.origin_xyz), _c64(chain.origin_rpy), _c64(chain.axis)
        par = np.ascontiguousarray(chain.parent, dtype=np.int32)
        pri = np.ascontiguousarray(chain.prismatic, dtype=np.int32)
        lo, up = _c64(chain.lower), _c64(chain.upper)
        self._check(lib().stomp_b200_set_chain(self.h, self.D, _dp(xyz), _dp(rpy), _dp(ax), _ip(par), _ip(pri), _dp(lo), _dp(up)),
                    "stomp_b200_set_chain")

    def set_spheres(self, spheres):
        link = np.ascontiguousarray(spheres.link, dtype=np.int32)
        xyz, rad = _c64(spheres.xyz), _c64(spheres.radius)
        self._check(lib().stomp_b200_set_spheres(self.h, len(link), _ip(link), _dp(xyz), _dp(rad)), "stomp_b200_set_spheres")
        self.S = len(link)

    def set_self_collision(self, pairs):
        """pairs [n][2]: sphere indices checked against each other (problems.self_collision_pairs); empty = off.
        Call after set_spheres / set_problem (which clear the list)."""
        pr = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        self._check(lib().stomp_b200_set_self_collision(self.h, len(pr), _ip(pr)), "stomp_b200_set_self_collision")

    def set_sdf(self, sdf):
        """A host grid is uploaded; a lazy Sdf (grid None, primitives listed) is built on the device."""
        if sdf.grid is None:
            return self.build_sdf_primitives(sdf.dims, sdf.origin, sdf.voxel, *sdf.primitive_arrays())
        grid = np.ascontiguousarray(sdf.grid, dtype=np.float32)
        dims = np.ascontiguousarray(sdf.dims, dtype=np.int32)
        org = _c64(sdf.origin)
        self._check(lib().stomp_b200_set_sdf(self.h, _ip(dims), _dp(org), float(sdf.voxel),
                                             grid.ctypes.data_as(C.POINTER(C.c_float))), "stomp_b200_set_sdf")

    def build_sdf_primitives(self, dims, origin, voxel, kind, centre, size):
        """Distance field of a union of spheres / boxes, built on the device."""
        dims = np.ascontiguousarray(dims, dtype=np.int32)
        org, kind = _c64(origin), np.ascontiguousarray(kind, dtype=np.int32)
        centre, size = _c64(centre).reshape(-1, 3), _c64(size).reshape(-1, 3)
        self._check(lib().stomp_b200_build_sdf_primitives(self.h, _ip(dims), _dp(org), float(voxel), len(kind), _ip(kind),
                                                          _dp(centre), _dp(size)), "stomp_b200_build_sdf_primitives")

    def build_sdf_occupancy(self, occupied, origin, voxel):
        """Signed Euclidean distance transform of an occupancy grid [nz][ny][nx] (uint8), built on the device."""
        occ = np.ascontiguousarray(occupied, dtype=np.uint8)
        dims = np.array(occ.shape[::-1], dtype=np.int32)
        org = _c64(origin)
        self._check(lib().stomp_b200_build_sdf_occupancy(self.h, _ip(dims), _dp(org), float(voxel),
                                                         occ.ctypes.data_as(C.POINTER(C.c_uint8))), "stomp_b200_build_sdf_occupancy")

    def build_sdf_scene(self, dims, origin, voxel, triangles=None, solid=False, leaf_centres=None, leaf_sizes=None, occupied=None):
        """Mesh (triangles [n][3][3]) + octomap leaves (centres [m][3], edge lengths [m]) + occupancy grid -> signed distance
        field, voxelised and transformed on the device (stomp_b200_build_sdf_scene)."""
        dims = np.ascontiguousarray(dims, dtype=np.int32)
        org = _c64(origin)
        tri = _c64(triangles).reshape(-1, 9) if triangles is not None else np.zeros((0, 9))
        lc = _c64(leaf_centres).reshape(-1, 3) if leaf_centres is not None else np.zeros((0, 3))
        ls = _c64(leaf_sizes).reshape(-1) if leaf_sizes is not None else np.zeros(0)
        occ = np.ascontiguousarray(occupied, dtype=np.uint8) if occupied is not None else None
        u8 = C.POINTER(C.c_uint8)
        self._check(lib().stomp_b200_build_sdf_scene(self.h, _ip(dims), _dp(org), float(voxel), len(tri), _dp(tri) if len(tri) else None,
                                                     int(solid), len(ls), _dp(lc) if len(ls) else None, _dp(ls) if len(ls) else None,
                                                     occ.ctypes.data_as(u8) if occ is not None else None), "stomp_b200_build_sdf_scene")

    def get_sdf(self):
        """(grid float32 [nz][ny][nx], origin[3], voxel) of the field the engine holds."""
        dims = np.zeros(3, dtype=np.int32)
        org = np.zeros(3)
        vox = C.c_double(0)
        self._check(lib().stomp_b200_get_sdf(self.h, None, 0, _ip(dims), _dp(org), C.byref(vox)), "stomp_b200_get_sdf")
        out = np.empty((int(dims[2]), int(dims[1]), int(dims[0])), dtype=np.float32)
        self._check(lib().stomp_b200_get_sdf(self.h, out.ctypes.data_as(C.POINTER(C.c_float)), out.size, None, None, None),
                    "stomp_b200_get_sdf")
        return out, org, vox.value

    def select_scene(self, scene):
        """The scene the SDF setters, builders, get_sdf and evaluate_states act on from now on; selecting the current
        number of scenes creates an empty one (stomp_b200_select_scene)."""
        self._check(lib().stomp_b200_select_scene(self.h, int(scene)), "stomp_b200_select_scene")

    def set_query_scenes(self, first_query, scenes):
        """scenes[i]: the scene local query first_query + i plans in (stomp_b200_set_query_scenes)."""
        sc = np.ascontiguousarray(scenes, dtype=np.int32).reshape(-1)
        self._check(lib().stomp_b200_set_query_scenes(self.h, int(first_query), len(sc), _ip(sc)), "stomp_b200_set_query_scenes")

    def set_matrices(self, R, Rinv, L):
        R, L = _c64(R), _c64(L)
        Rinv = None if Rinv is None else _c64(Rinv)
        self._check(lib().stomp_b200_set_control_cost_matrices(self.h, _dp(R), _dp(Rinv), _dp(L)),
                    "stomp_b200_set_control_cost_matrices")

    def set_policy(self, query, params_all, mincc):
        pa, mc = _c64(params_all), _c64(mincc)
        assert pa.shape == (self.D, self.N) and mc.shape == (self.D, self.T)
        self._check(lib().stomp_b200_set_policy(self.h, query, _dp(pa), _dp(mc)), "stomp_b200_set_policy")

    def set_policies(self, first_query, params_all, mincc):
        """a batch of consecutive queries in one call: params_all [count][D][N], mincc [count][D][T]"""
        pa, mc = _c64(params_all), _c64(mincc)
        assert pa.ndim == 3 and pa.shape[1:] == (self.D, self.N) and mc.shape == (pa.shape[0], self.D, self.T)
        self._check(lib().stomp_b200_set_policies(self.h, first_query, pa.shape[0], _dp(pa), _dp(mc)), "stomp_b200_set_policies")

    def set_problem(self, problem, policy=None):
        """Scene + StompPlanner::setStartGoalTrajectory for every local query.  `policy`, when given, is a
        dict (R, Rinv, L, params_all, mincc) shared with the oracle in parity tests.  A problem with a list of scenes
        (problems.batch_problem_scenes) gets one field per scene and each query the scene of its query_scene entry."""
        self.set_chain(problem.chain)
        self.set_spheres(problem.spheres)
        if problem.scenes:
            for i, sdf in enumerate(problem.scenes):
                self.select_scene(i)
                self.set_sdf(sdf)
            self.select_scene(0)
            self.set_query_scenes(0, np.asarray(problem.query_scene)[self.query_offset:self.query_offset + self.Q])
        else:
            self.set_sdf(problem.sdf)
        starts = np.atleast_2d(problem.start)
        goals = np.atleast_2d(problem.goal)
        pol = policy
        for ql in range(self.Q):
            qg = self.query_offset + ql
            if policy is None:
                init = host_initial_trajectory(starts[qg], goals[qg], self.T)
                pol = host_policy(init, self.cfg.movement_duration, tuple(self.cfg.derivative_weights))
            if ql == 0:
                self.set_matrices(pol["R"], pol.get("Rinv"), pol["L"])
            self.set_policy(ql, pol["params_all"], pol["mincc"])
        return pol

    # ---- loop ------------------------------------------------------------------------------------
    def begin_solve(self):
        self._check(lib().stomp_b200_begin_solve(self.h), "stomp_b200_begin_solve")

    def next_num_generated(self):
        return lib().stomp_b200_next_num_generated(self.h)

    def iterate(self, iteration, noise=None, epsilon=None):
        n = None if noise is None else _c64(noise)
        ep = None if epsilon is None else _c64(epsilon)
        cost = np.empty(self.Q)
        valid = np.empty(self.Q, dtype=np.uint8)
        stop = np.empty(self.Q, dtype=np.int32)
        self._check(lib().stomp_b200_iterate(self.h, iteration, _dp(n), _dp(ep), _dp(cost),
                                             valid.ctypes.data_as(C.POINTER(C.c_uint8)), _ip(stop)), "stomp_b200_iterate")
        return cost, valid.astype(bool), stop.astype(bool)

    def run(self, first_iteration, num_iterations, honour_stop=False):
        self._check(lib().stomp_b200_run(self.h, first_iteration, num_iterations, int(honour_stop)), "stomp_b200_run")

    def solve(self, max_iterations, poll_every=0):
        """The StompPlanner::solve loop on the device (stop rule honoured, stop flags polled every `poll_every` iterations);
        returns the iterations queued."""
        n = C.c_int32(0)
        self._check(lib().stomp_b200_solve(self.h, int(max_iterations), int(poll_every), C.byref(n)), "stomp_b200_solve")
        return n.value

    def finish_solve(self):
        sol = np.empty((self.Q, self.D, self.T))
        status = np.empty(self.Q, dtype=np.int32)
        iters = np.empty(self.Q, dtype=np.int32)
        cost = np.empty(self.Q)
        self._check(lib().stomp_b200_finish_solve(self.h, _dp(sol), _ip(status), _ip(iters), _dp(cost)), "stomp_b200_finish_solve")
        return dict(solution=sol, found=status.astype(bool), iterations=iters, cost=cost)

    def num_rollouts(self):
        a, b = C.c_int32(0), C.c_int32(0)
        self._check(lib().stomp_b200_num_rollouts(self.h, C.byref(a), C.byref(b)), "stomp_b200_num_rollouts")
        return a.value, b.value

    def tensor(self, name):
        n, g = self.num_rollouts()
        world = self.cfg.world_size if self.cfg.shard_mode == 0 else 1
        nl = n if world == 1 else g + (1 if n > g * world else 0)   # local rollouts
        Q, D, T, N = self.Q, self.D, self.T, self.N
        shapes = {
            "rollouts": (Q, nl, D, T), "noise": (Q, nl, D, T), "state_costs": (Q, nl, T), "verdicts": (Q, nl, T),
            "control_costs": (Q, nl, D, T), "cumulative_costs": (Q, n, D), "full_costs": (Q, n, D),
            "total_cost": (Q, n), "probabilities": (Q, n, D, T), "full_probabilities": (Q, n, D),
            "updates": (Q, D, T), "parameters": (Q, D, T), "parameters_all": (Q, D, N), "stddevs": (Q, D),
            "noiseless_state_costs": (Q, T), "noiseless_control_costs": (Q, D, T), "unit_noise": (Q, g, D, T),
            "epsilon": (Q, g, D, T), "rollout_validity": (Q, g), "noise_projected": (Q, nl, D, T),
            "rollouts_projected": (Q, nl, D, T),
        }
        dtype = np.uint8 if name in ("verdicts", "rollout_validity") else np.float64
        out = np.empty(shapes[name], dtype=dtype)
        self._check(lib().stomp_b200_get_tensor(self.h, TENSORS[name], out.ctypes.data_as(C.c_void_p), out.nbytes),
                    f"stomp_b200_get_tensor({name})")
        return out

    # ---- kernel-level ----------------------------------------------------------------------------
    def evaluate_states(self, theta):
        th = _c64(theta)
        K, D, Tq = th.shape
        assert D == self.D
        costs = np.empty((K, Tq))
        verdicts = np.empty((K, Tq), dtype=np.uint8)
        validity = np.empty(K, dtype=np.uint8)
        u8 = C.POINTER(C.c_uint8)
        self._check(lib().stomp_b200_evaluate_states(self.h, _dp(th), K, Tq, _dp(costs), verdicts.ctypes.data_as(u8),
                                                     validity.ctypes.data_as(u8)), "stomp_b200_evaluate_states")
        return costs, verdicts, validity

    def sphere_centres(self, q):
        qc = np.atleast_2d(_c64(q))
        out = np.empty((qc.shape[0], self.S, 3))
        self._check(lib().stomp_b200_sphere_centres(self.h, _dp(qc), qc.shape[0], _dp(out)), "stomp_b200_sphere_centres")
        return out

    # ---- multi-GPU / measurement -----------------------------------------------------------------
    def comm_init(self, unique_id: bytes):
        buf = C.create_string_buffer(unique_id, COMM_ID_BYTES)
        self._check(lib().stomp_b200_comm_init(self.h, buf), "stomp_b200_comm_init")

    def set_cost_extras(self, smooth=None, joint_constraint=None):
        """smooth: (margin, weight) or None; joint_constraint: (value [D], tolerance [D], weight) or None."""
        sm = smooth or (0.0, 1.0)
        if joint_constraint is not None:
            v, tol, w = _c64(joint_constraint[0]), _c64(joint_constraint[1]), float(joint_constraint[2])
            rc = lib().stomp_b200_set_cost_extras(self.h, int(smooth is not None), float(sm[0]), float(sm[1]), 1, _dp(v), _dp(tol), w)
        else:
            rc = lib().stomp_b200_set_cost_extras(self.h, int(smooth is not None), float(sm[0]), float(sm[1]), 0, None, None, 1.0)
        self._check(rc, "stomp_b200_set_cost_extras")

    def exchange_kind(self):
        """("peer" | "nccl" | "none", note): how a rollout-sharded engine exchanges its per-iteration scalars."""
        note = C.create_string_buffer(1024)
        rc = lib().stomp_b200_exchange_kind(self.h, note, len(note))
        if rc < 0:
            self._check(rc, "stomp_b200_exchange_kind")
        return {2: "peer", 1: "nccl"}.get(rc, "none"), note.value.decode()

    def set_profiling(self, on):
        self._check(lib().stomp_b200_set_profiling(self.h, int(on)), "stomp_b200_set_profiling")

    def kernel_stats(self):
        out = {}
        for name, kid in KERNELS.items():
            ms, n = C.c_double(0), C.c_int64(0)
            self._check(lib().stomp_b200_kernel_stats(self.h, kid, C.byref(ms), C.byref(n)), "stomp_b200_kernel_stats")
            out[name] = (ms.value, n.value)
        return out

    def reset_kernel_stats(self):
        self._check(lib().stomp_b200_reset_kernel_stats(self.h), "stomp_b200_reset_kernel_stats")

    def set_timeline(self, on):
        self._check(lib().stomp_b200_set_timeline(self.h, int(on)), "stomp_b200_set_timeline")

    def timeline(self, max_iterations=64):
        """[iterations][8 kernels][begin, end] in microseconds (oldest first; -1 where a kernel did not run)."""
        out = np.empty((max_iterations, 8, 2))
        n = C.c_int32(0)
        self._check(lib().stomp_b200_get_timeline(self.h, max_iterations, _dp(out), C.byref(n)), "stomp_b200_get_timeline")
        return out[:n.value]

    def launch_count(self):
        return lib().stomp_b200_launch_count(self.h)

    def graph_replays(self):
        return lib().stomp_b200_graph_replays(self.h)

    def set_cost_cumulation(self, use_cumulative_costs: bool):
        """stomp::Stomp::setCostCumulation."""
        self._check(lib().stomp_b200_set_cost_cumulation(self.h, int(use_cumulative_costs)), "stomp_b200_set_cost_cumulation")

    def state_kernel_kind(self):
        """("specialised" | "generic" | "self-collision", note): which state kernel the engine launches for its robot (state_codegen.hpp)."""
        note = C.create_string_buffer(4096)
        rc = lib().stomp_b200_state_kernel_kind(self.h, note, len(note))
        if rc < 0:
            self._check(rc, "stomp_b200_state_kernel_kind")
        return {1: "specialised", 2: "self-collision"}.get(rc, "generic"), note.value.decode()

    def state_kernel_source(self):
        need = C.c_size_t(0)
        self._check(lib().stomp_b200_state_kernel_source(self.h, None, 0, C.byref(need)), "stomp_b200_state_kernel_source")
        buf = C.create_string_buffer(need.value)
        self._check(lib().stomp_b200_state_kernel_source(self.h, buf, need.value, None), "stomp_b200_state_kernel_source")
        return buf.value.decode()

    def timer_begin(self):
        self._check(lib().stomp_b200_timer_begin(self.h), "stomp_b200_timer_begin")

    def timer_end(self):
        ms = C.c_double(0)
        self._check(lib().stomp_b200_timer_end(self.h, C.byref(ms)), "stomp_b200_timer_end")
        return ms.value

    def synchronize(self):
        self._check(lib().stomp_b200_synchronize(self.h), "stomp_b200_synchronize")


def engine_for_problem(problem, *, min_rollouts=None, max_rollouts=None, per_iteration=None, policy=None, **kw) -> Engine:
    """Engine configured like the reference's StompPlanner for `problem` (K = min = max = per-iteration by default)."""
    K = problem.num_rollouts
    e = Engine(num_time_steps=problem.num_time_steps, num_dimensions=problem.chain.num_dimensions,
               min_rollouts=min_rollouts or K, max_rollouts=max_rollouts or K,
               num_rollouts_per_iteration=per_iteration or K, num_queries=problem.num_queries,
               movement_duration=problem.movement_duration, control_cost_weight=problem.control_cost_weight,
               noise_stddev=problem.noise_stddev, **kw)
    e.policy = e.set_problem(problem, policy)
    return e
