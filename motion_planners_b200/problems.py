"""Synthetic planning problems of the shapes BASELINE.json names (SURVEY.md §8d).

Pure data generation (numpy): the 7-DoF KUKA LBR iiwa 14 R820 chain of the reference's test fixture
(values read from reference test/data/kuka_iiwa.urdf:162-210), link spheres fitted by hand to the
collision-mesh bounding boxes listed in SURVEY.md §8c, a synthetic signed-distance field, and the
start / goal of reference test/test_motion_planners.cpp:212-215.  Nothing here is on the hot path.
"""
from __future__ import annotations

import dataclasses
import hashlib
import os
import tempfile

import numpy as np

TRAJECTORY_PADDING = 6

# reference test/test_motion_planners.cpp:212-215
IIWA_START = np.array([0.5, 0.5, 0.5, -1.5, 0.5, 0.5, 0.5])
IIWA_GOAL = np.array([-1.5, -1.5, -1.5, 1.5, -1.5, -1.5, -0.5])
# reference test/config/stomp.yml:16-21
IIWA_NOISE_STDDEV = np.array([0.1, 0.2, 0.5, 0.4, 0.3, 0.3, 0.1])


@dataclasses.dataclass
class Chain:
    origin_xyz: np.ndarray   # [D,3]
    origin_rpy: np.ndarray   # [D,3]
    axis: np.ndarray         # [D,3]
    parent: np.ndarray       # [D] int32, -1 = hangs off the base frame, else d-1
    prismatic: np.ndarray    # [D] int32
    lower: np.ndarray        # [D]
    upper: np.ndarray        # [D]
    names: list

    @property
    def num_dimensions(self) -> int:
        return int(self.axis.shape[0])


@dataclasses.dataclass
class Spheres:
    link: np.ndarray   # [S] int32, sorted ascending
    xyz: np.ndarray    # [S,3] centre in the link frame
    radius: np.ndarray  # [S]


@dataclasses.dataclass
class Sdf:
    dims: np.ndarray    # [3] int32 (nx, ny, nz), x fastest in `grid`
    origin: np.ndarray  # [3] world position of the min corner
    voxel: float
    grid: np.ndarray    # float32 [nz, ny, nx]; None = not materialised on the host: the engine builds the field on the
                        # device from `obstacles` (stomp_b200_build_sdf_primitives), the oracle with its own builder
    obstacles: list = None   # [(kind, centre[3], size[3])]: kind 0 sphere (size[0] = radius), 1 box (half extents)

    def primitive_arrays(self):
        """(kind int32[n], centre float64[n,3], size float64[n,3]) of `obstacles`, as the C ABI takes them."""
        obs = self.obstacles or []
        kind = np.array([int(k) for k, _, _ in obs], dtype=np.int32).reshape(-1)
        centre = np.array([np.asarray(c, dtype=np.float64) for _, c, _ in obs], dtype=np.float64).reshape(-1, 3)
        size = np.array([np.asarray(s, dtype=np.float64) for _, _, s in obs], dtype=np.float64).reshape(-1, 3)
        return kind, centre, size


def iiwa_chain(base_xyz=(0.0, 0.0, 0.0)) -> Chain:
    """joint_a1..joint_a7 of kuka_iiwa.urdf:162-210 (all rpy = 0)."""
    xyz = np.array([
        [0.0, 0.0, 0.0],
        [-0.00043624, 0.0, 0.36],
        [0.0, 0.0, 0.0],
        [0.00043624, 0.0, 0.42],
        [0.0, 0.0, 0.0],
        [0.0, 0.0, 0.4],
        [0.0, 0.0, 0.0],
    ])
    xyz[0] += np.asarray(base_xyz, dtype=np.float64)
    axis = np.array([
        [0, 0, 1], [0, 1, 0], [0, 0, 1], [0, -1, 0], [0, 0, 1], [0, 1, 0], [0, 0, 1],
    ], dtype=np.float64)
    lim = np.array([2.9668, 2.0942, 2.9668, 2.0942, 2.9668, 2.0942, 3.0541])
    return Chain(origin_xyz=xyz, origin_rpy=np.zeros((7, 3)), axis=axis,
                 parent=np.array([-1, 0, 1, 2, 3, 4, 5], dtype=np.int32),
                 prismatic=np.zeros(7, dtype=np.int32), lower=-lim, upper=lim.copy(),
                 names=[f"joint_a{i}" for i in range(1, 8)])


def iiwa_spheres() -> Spheres:
    """20 spheres, ~3 per moving link, radii 0.05-0.10 m (SURVEY.md §8d)."""
    rows = [
        (0, (0.0, 0.0, 0.18), 0.10), (0, (0.0, 0.0, 0.28), 0.10), (0, (0.0, 0.0, 0.38), 0.10),
        (1, (0.0, 0.0, 0.0), 0.10), (1, (0.0, 0.05, 0.10), 0.09), (1, (0.0, 0.03, 0.20), 0.09),
        (2, (0.0, 0.0, 0.25), 0.09), (2, (0.0, 0.0, 0.34), 0.09), (2, (0.0, 0.0, 0.42), 0.09),
        (3, (0.0, 0.0, 0.0), 0.09), (3, (0.0, -0.04, 0.09), 0.08), (3, (0.0, -0.02, 0.18), 0.08),
        (4, (0.0, 0.0, 0.22), 0.08), (4, (0.0, 0.0, 0.31), 0.08), (4, (0.0, 0.0, 0.40), 0.08),
        (5, (0.0, 0.0, 0.0), 0.08), (5, (0.0, 0.0, 0.06), 0.07),
        (6, (0.0, 0.0, 0.09), 0.06), (6, (0.0, 0.0, 0.13), 0.05), (6, (0.0, 0.0, 0.16), 0.05),
    ]
    return Spheres(link=np.array([r[0] for r in rows], dtype=np.int32),
                   xyz=np.array([r[1] for r in rows], dtype=np.float64),
                   radius=np.array([r[2] for r in rows], dtype=np.float64))


def dual_arm_chain(separation=0.8) -> Chain:
    """Config 5: two iiwa arms, bases at y = +-separation/2, D = 14."""
    a = iiwa_chain((0.0, -separation / 2, 0.0))
    b = iiwa_chain((0.0, +separation / 2, 0.0))
    pb = b.parent.copy()
    pb[1:] += 7
    return Chain(origin_xyz=np.vstack([a.origin_xyz, b.origin_xyz]), origin_rpy=np.zeros((14, 3)),
                 axis=np.vstack([a.axis, b.axis]), parent=np.concatenate([a.parent, pb]).astype(np.int32),
                 prismatic=np.zeros(14, dtype=np.int32), lower=np.concatenate([a.lower, b.lower]),
                 upper=np.concatenate([a.upper, b.upper]),
                 names=[f"left_{n}" for n in a.names] + [f"right_{n}" for n in b.names])


def dual_arm_spheres() -> Spheres:
    """2 x 20 link spheres + 8 grasped-object spheres on the tip link of arm 1 = 48."""
    s = iiwa_spheres()
    obj = [(6, (0.06 * (i % 2) - 0.03, 0.06 * ((i // 2) % 2) - 0.03, 0.22 + 0.06 * (i // 4)), 0.04) for i in range(8)]
    link = np.concatenate([s.link, np.full(8, 6, dtype=np.int32), s.link + 7]).astype(np.int32)
    xyz = np.vstack([s.xyz, np.array([o[1] for o in obj]), s.xyz])
    rad = np.concatenate([s.radius, np.array([o[2] for o in obj]), s.radius])
    return Spheres(link=link, xyz=xyz, radius=rad)


def self_collision_pairs(chain: Chain, spheres: Spheres, disabled_links=(), skip_adjacent=True) -> np.ndarray:
    """Sphere pairs [n][2] to check against each other: all pairs on different links, minus links joined by one
    joint (skip_adjacent) and minus the link pairs listed in `disabled_links` (what an SRDF's disable_collisions
    entries say; reference test/data/kuka_iiwa.srdf:46-70).  Links are named by the index of the joint they hang on."""
    off = {(min(a, b), max(a, b)) for a, b in disabled_links}
    out = []
    link = spheres.link
    for i in range(len(link)):
        for j in range(i + 1, len(link)):
            a, b = int(link[i]), int(link[j])
            if a == b or (a, b) in off:
                continue
            if skip_adjacent and chain.parent[b] == a:
                continue
            out.append((i, j))
    return np.asarray(out, dtype=np.int32).reshape(-1, 2)


def _rot(axis, q):
    a = np.asarray(axis, dtype=np.float64)
    a = a / np.linalg.norm(a)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(q) * K + (1 - np.cos(q)) * (K @ K)


def _rpy(rpy):
    r, p, y = rpy
    Rx = _rot([1, 0, 0], r); Ry = _rot([0, 1, 0], p); Rz = _rot([0, 0, 1], y)
    return Rz @ Ry @ Rx


def sphere_centres_numpy(chain: Chain, spheres: Spheres, q) -> np.ndarray:
    """Plain textbook FK (libm sin/cos) used for obstacle rejection when a scene is generated."""
    q = np.asarray(q, dtype=np.float64)
    out = np.zeros((len(spheres.link), 3))
    R = np.eye(3); p = np.zeros(3)
    for d in range(chain.num_dimensions):
        if chain.parent[d] < 0:
            R = np.eye(3); p = np.zeros(3)
        p = p + R @ chain.origin_xyz[d]
        R = R @ _rpy(chain.origin_rpy[d])
        if chain.prismatic[d]:
            p = p + q[d] * (R @ chain.axis[d])
        else:
            R = R @ _rot(chain.axis[d], q[d])
        for s in np.nonzero(spheres.link == d)[0]:
            out[s] = p + R @ spheres.xyz[s]
    return out


def _obstacle_distance(pts, kind, centre, size):
    d = pts - centre
    if kind == 0:      # sphere, size[0] = radius
        return np.sqrt((d * d).sum(-1)) - size[0]
    qd = np.abs(d) - size   # box, size = half extents
    outside = np.sqrt((np.maximum(qd, 0.0) ** 2).sum(-1))
    inside = np.minimum(qd.max(-1), 0.0)
    return outside + inside


# a sphere obstacle on the straight joint-space line from IIWA_START to IIWA_GOAL (where the tool
# sphere is at 40 % of the way), so that the initial trajectory is in collision and STOMP has work to do
IIWA_BLOCKER = (0, np.array([-0.17, 0.03, 1.31]), np.array([0.15, 0.15, 0.15]))


def make_obstacles(seed=1234, count=16, keep_clear=None, clear_margin=0.05, blockers=(), urdf_box=True):
    """`count` random spheres / boxes in [-1.5,1.5]^3 + the URDF's box_1 (kuka_iiwa.urdf:29-56).

    Rejected if within 0.35 m of the base column or (keep_clear = [(centres[S,3], radii[S]), ...])
    touching the robot at the given configurations."""
    rng = np.random.default_rng(seed)
    obstacles = ([(1, np.array([0.5, 0.0, 0.5]), np.array([0.1, 0.1, 0.3]))] if urdf_box else []) + list(blockers)
    fixed = len(obstacles)
    while len(obstacles) < count + fixed:
        kind = int(rng.integers(0, 2))
        centre = rng.uniform(-1.3, 1.3, 3)
        size = rng.uniform(0.05, 0.25, 3)
        if np.hypot(centre[0], centre[1]) < 0.35 + size.max() * (1.0 if kind == 0 else np.sqrt(3.0)):
            continue
        ok = True
        for centres, radii in (keep_clear or []):
            if np.any(_obstacle_distance(centres, kind, centre, size) < radii + clear_margin):
                ok = False
                break
        if ok:
            obstacles.append((kind, centre, size))
    return obstacles


def make_sdf(n=128, obstacles=None, lo=-1.5, hi=1.5, slab=16, lazy=None) -> Sdf:
    """float32 grid [nz,ny,nx]; value = signed distance from the voxel centre to the obstacle union.

    lazy (default: n >= 256, or STOMP_B200_SDF_LAZY=0/1): no host grid — only the geometry and the primitive list; the
    engine then builds the field on the device (milliseconds instead of minutes of NumPy for 512^3)."""
    if obstacles is None:
        obstacles = make_obstacles()
    h = (hi - lo) / n
    if lazy is None:
        env = os.environ.get("STOMP_B200_SDF_LAZY")
        lazy = (n >= 256) if env is None else env != "0"
    if lazy:
        return Sdf(dims=np.array([n, n, n], dtype=np.int32), origin=np.array([lo, lo, lo], dtype=np.float64),
                   voxel=float(h), grid=None, obstacles=list(obstacles))
    # The exact field of a 256^3 scene takes half a minute of NumPy (512^3: four minutes) and every rank of a benchmark
    # builds the same one: large grids are kept on disk, keyed by everything they depend on.
    cache_path = None
    if n >= 128 and os.environ.get("STOMP_B200_SDF_CACHE", "1") != "0":
        key = hashlib.sha256(repr((n, lo, hi, [(k, np.asarray(c, dtype=np.float64).tolist(), np.asarray(sz, dtype=np.float64).tolist())
                                               for k, c, sz in obstacles])).encode()).hexdigest()[:24]
        cache_dir = os.environ.get("STOMP_B200_CACHE_DIR", os.path.join(tempfile.gettempdir(), "stomp_b200_cache"))
        cache_path = os.path.join(cache_dir, f"sdf_{n}_{key}.npy")
        try:
            grid = np.load(cache_path)
            if grid.shape == (n, n, n) and grid.dtype == np.float32:
                return Sdf(dims=np.array([n, n, n], dtype=np.int32), origin=np.array([lo, lo, lo], dtype=np.float64),
                           voxel=float(h), grid=grid, obstacles=list(obstacles))
        except (OSError, ValueError):
            pass
    c = lo + (np.arange(n, dtype=np.float64) + 0.5) * h
    grid = np.empty((n, n, n), dtype=np.float32)
    for z0 in range(0, n, slab):
        z1 = min(n, z0 + slab)
        Z, Y, X = np.meshgrid(c[z0:z1], c, c, indexing="ij")
        pts = np.stack([X, Y, Z], axis=-1)
        dist = np.full(pts.shape[:-1], np.inf)
        for kind, centre, size in obstacles:
            dist = np.minimum(dist, _obstacle_distance(pts, kind, centre, size))
        grid[z0:z1] = dist.astype(np.float32)
    if cache_path is not None:
        try:
            os.makedirs(os.path.dirname(cache_path), exist_ok=True)
            tmp = f"{cache_path}.{os.getpid()}.tmp"
            with open(tmp, "wb") as f:
                np.save(f, grid)
            os.replace(tmp, cache_path)
        except OSError:
            pass
    return Sdf(dims=np.array([n, n, n], dtype=np.int32), origin=np.array([lo, lo, lo], dtype=np.float64),
               voxel=float(h), grid=grid, obstacles=list(obstacles))


@dataclasses.dataclass
class Problem:
    chain: Chain
    spheres: Spheres
    sdf: Sdf
    start: np.ndarray          # [Q,D] or [D]
    goal: np.ndarray
    noise_stddev: np.ndarray   # [D]
    num_time_steps: int
    num_rollouts: int
    num_queries: int = 1
    movement_duration: float = 5.0
    control_cost_weight: float = 0.001
    name: str = ""
    scenes: list = None        # [Sdf] one field per scene (sdf is scenes[0]), or None: every query plans in `sdf`
    query_scene: np.ndarray = None   # [Q] int32 scene of each query


def _scene(chain, spheres, configs, n, seed, blockers=(), urdf_box=True):
    keep = [(sphere_centres_numpy(chain, spheres, q), spheres.radius) for q in configs]
    return make_sdf(n, make_obstacles(seed=seed, keep_clear=keep, blockers=blockers, urdf_box=urdf_box))


def single_arm_problem(K=128, T=100, sdf_n=128, seed=1234, name="") -> Problem:
    """Configs 2 / 3: iiwa, K rollouts (min = max = per-iteration = K), T steps, sdf_n^3 SDF."""
    chain, spheres = iiwa_chain(), iiwa_spheres()
    sdf = _scene(chain, spheres, [IIWA_START, IIWA_GOAL], sdf_n, seed, blockers=(IIWA_BLOCKER,))
    return Problem(chain, spheres, sdf, IIWA_START.copy(), IIWA_GOAL.copy(), IIWA_NOISE_STDDEV.copy(),
                   T, K, name=name or f"iiwa7_K{K}_T{T}_sdf{sdf_n}")


def dual_arm_problem(K=2048, T=150, sdf_n=512, seed=1234) -> Problem:
    """Config 5: 14-DoF dual arm with grasped-object spheres."""
    chain, spheres = dual_arm_chain(), dual_arm_spheres()
    start = np.concatenate([IIWA_START, IIWA_START * np.array([-1, 1, -1, 1, -1, 1, -1])])
    goal = np.concatenate([IIWA_GOAL, IIWA_GOAL * np.array([-1, 1, -1, 1, -1, 1, -1])])
    # the URDF's box_1 stands where the two mirrored arms start; the dual-arm scene leaves it out
    sdf = _scene(chain, spheres, [start, goal], sdf_n, seed, urdf_box=False)
    return Problem(chain, spheres, sdf, start, goal, np.concatenate([IIWA_NOISE_STDDEV, IIWA_NOISE_STDDEV]),
                   T, K, name=f"dual14_K{K}_T{T}_sdf{sdf_n}")


def batch_problem(Q=1024, K=64, T=200, sdf_n=128, seed=1234, query_seed=4321) -> Problem:
    """Config 4: Q independent start/goal pairs drawn within the joint limits, collision-free."""
    chain, spheres = iiwa_chain(), iiwa_spheres()
    sdf = _scene(chain, spheres, [IIWA_START, IIWA_GOAL], sdf_n, seed)
    rng = np.random.default_rng(query_seed)

    def free(q):
        c = sphere_centres_numpy(chain, spheres, q)
        idx = np.clip(np.floor((c - sdf.origin) / sdf.voxel).astype(np.int64), 0, sdf.dims - 1)
        return np.all(sdf.grid[idx[:, 2], idx[:, 1], idx[:, 0]] - spheres.radius >= 0.0)

    def draw():
        while True:
            q = rng.uniform(0.9 * chain.lower, 0.9 * chain.upper)
            if free(q):
                return q

    start = np.stack([draw() for _ in range(Q)])
    goal = np.stack([draw() for _ in range(Q)])
    return Problem(chain, spheres, sdf, start, goal, IIWA_NOISE_STDDEV.copy(), T, K, num_queries=Q,
                   name=f"batch_Q{Q}_K{K}_T{T}_sdf{sdf_n}")


def batch_problem_scenes(Q=1024, K=64, T=200, sdf_n=128, num_scenes=16, seed=1234, query_seed=4321) -> Problem:
    """Config 4 over `num_scenes` worlds: scene s is the obstacle set of seed + s as a primitive list (the engine builds the
    fields on the device), query q plans in scene q mod num_scenes, and its start and goal are drawn within the joint limits,
    free in its own scene: every sphere at least its radius plus one voxel from every obstacle (exact primitive distances,
    no host grid)."""
    chain, spheres = iiwa_chain(), iiwa_spheres()
    keep = [(sphere_centres_numpy(chain, spheres, q), spheres.radius) for q in (IIWA_START, IIWA_GOAL)]
    scenes = [make_sdf(sdf_n, make_obstacles(seed=seed + s, keep_clear=keep), lazy=True) for s in range(num_scenes)]
    query_scene = (np.arange(Q) % num_scenes).astype(np.int32)
    rng = np.random.default_rng(query_seed)

    def free(q, sdf):
        c = sphere_centres_numpy(chain, spheres, q)
        return all(np.all(_obstacle_distance(c, kind, centre, size) >= spheres.radius + sdf.voxel)
                   for kind, centre, size in sdf.obstacles)

    def draw(sdf):
        while True:
            q = rng.uniform(0.9 * chain.lower, 0.9 * chain.upper)
            if free(q, sdf):
                return q

    start = np.stack([draw(scenes[s]) for s in query_scene])
    goal = np.stack([draw(scenes[s]) for s in query_scene])
    return Problem(chain, spheres, scenes[0], start, goal, IIWA_NOISE_STDDEV.copy(), T, K, num_queries=Q,
                   name=f"batch_Q{Q}_K{K}_T{T}_sdf{sdf_n}_scenes{num_scenes}", scenes=scenes, query_scene=query_scene)
