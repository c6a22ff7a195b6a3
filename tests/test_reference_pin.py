"""The CPU restatement (oracle/stomp_oracle.cpp) against the REFERENCE'S OWN CODE: the reference project's
src/planners/stomp/src/{Stomp,PolicyImprovement,CovariantMovementPrimitive,StompUtils}.cpp compiled unmodified against the Eigen / Boost
stand-ins of oracle/ref/shim (oracle/ref/Makefile -> oracle/_ref/libstomp_ref.so).  Both sides are fed the same
standard normals; every field of every rollout, the update, the parameters, the adapted noise and the noise-less
rollout must agree to 1e-12 relative over whole solves — in practice they agree bit for bit.

Where the reference's sources are absent, the reference's side is replayed from tests/golden/reference_pin/<test>.npz,
which tests/golden/make_pin_golden.py records from the reference build: every value the test takes from it, including
the unit noise L·eps the reference formed, which the oracle is then fed.  Arrays of more than FULL elements are kept as
their shape, 64 elements at fixed positions, and their plain, position-weighted and absolute sums.  A test with neither
the reference build nor its recording skips."""
import os

import numpy as np
import pytest

from motion_planners_b200 import problems as P
from oracle.binding import Oracle
from oracle import ref_binding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RECORDINGS = os.path.join(ROOT, "tests", "golden", "reference_pin")
LIVE = ref_binding.available()
FULL = 256
_RECORD = None      # {key: array} while tests/golden/make_pin_golden.py records the running test
_CURRENT = [""]     # name of the running test


@pytest.fixture(autouse=True)
def _test_name(request):
    _CURRENT[0] = request.node.name


def _recording():
    return os.path.join(RECORDINGS, _CURRENT[0] + ".npz")


class _Print:
    """What the recording keeps of a large array."""

    def __init__(self, shape, sums, sample):
        self.shape, self.sums, self.sample = tuple(int(n) for n in shape), np.asarray(sums, dtype=np.float64), sample


def _print(a):
    flat = a.reshape(-1)
    rng = np.random.default_rng(flat.size)
    weights = np.arange(1, flat.size + 1, dtype=np.float64) / flat.size
    sums = [np.abs(flat).sum(), flat.sum(), (weights * flat).sum()]      # the absolute sum bounds the others' rounding
    return _Print(a.shape, sums, flat[np.sort(rng.choice(flat.size, 64, replace=False))])


def _store(key, v, out):
    if v is None:
        out[key + "~"] = np.zeros(0)
    elif isinstance(v, dict):
        for k, x in v.items():
            _store(f"{key}.{k}", x, out)
    elif isinstance(v, tuple):
        for i, x in enumerate(v):
            _store(f"{key}.{i}", x, out)
        out[key + "()"] = np.array(len(v))
    elif isinstance(v, np.ndarray) and v.size > FULL:
        p = _print(v)
        out[key + "#"] = np.concatenate([[len(p.shape)], p.shape, p.sums, p.sample])     # one entry: ndim, shape, sums, sample
    else:
        out[key] = np.array(v)


def _load(key, g):
    if key + "~" in g:
        return None
    if key in g:
        return g[key][()] if g[key].ndim == 0 else g[key]
    if key + "()" in g:
        return tuple(_load(f"{key}.{i}", g) for i in range(int(g[key + "()"])))
    if key + "#" in g:
        p = g[key + "#"]
        nd = int(p[0])
        return _Print(p[1:1 + nd], p[1 + nd:4 + nd], p[4 + nd:])
    names = sorted({k[len(key) + 1:].split(".")[0].rstrip("#~") for k in g.files if k.startswith(key + ".")})
    assert names, f"{key} is not in {_recording()}: record it again with tests/golden/make_pin_golden.py"
    return {n: _load(f"{key}.{n}", g) for n in names}


class _Recorded:
    """Answers the reference's calls in the order the test makes them: recorded from the reference build while
    make_pin_golden.py runs, else replayed from the test's recording.  iterate's unit noise is kept whole: it is the
    oracle's input."""

    def __init__(self, reference=None, stored=None):
        self.reference, self.stored, self.n = reference, stored, 0

    def _call(self, name, *args):
        key = f"{self.n:03d}.{name}"
        self.n += 1
        if self.stored is None:
            v = getattr(self.reference, name)(*args)
            if name == "iterate":
                _RECORD[key + ".stop"], _RECORD[key + ".unit"] = np.array(v[0]), v[1]
            else:
                _store(key, v, _RECORD)
            return v
        if name == "iterate":
            return bool(self.stored[key + ".stop"]), self.stored[key + ".unit"]
        return _load(key, self.stored)

    def __getattr__(self, name):
        return lambda *args: self._call(name, *args)


def _as_print(a, like):
    return _print(a) if isinstance(like, _Print) and isinstance(a, np.ndarray) else a


def _same(a, b, what):
    if isinstance(a, _Print) or isinstance(b, _Print):
        a, b = _as_print(a, b), _as_print(b, a)
        assert a.shape == b.shape, what
        np.testing.assert_allclose(a.sample, b.sample, rtol=RTOL, atol=0.0, err_msg=what)
        np.testing.assert_allclose(a.sums, b.sums, rtol=0.0, atol=RTOL * 4 * max(a.sums[0], b.sums[0]), err_msg=what)
        return
    assert a.shape == b.shape, what
    np.testing.assert_allclose(a, b, rtol=RTOL, atol=0.0, err_msg=what)


def _equal(a, b):
    if isinstance(a, _Print) or isinstance(b, _Print):
        a, b = _as_print(a, b), _as_print(b, a)
        return a.shape == b.shape and np.array_equal(a.sample, b.sample) and np.array_equal(a.sums, b.sums)
    return np.array_equal(a, b)


FIELDS = ["parameters_noise", "noise", "noise_projected", "parameters_noise_projected", "state_costs", "control_costs",
          "total_costs", "cumulative_costs", "probabilities", "full_probabilities", "full_costs", "total_cost"]
RTOL = 1e-12


def _pair(pb, min_r, max_r, per_it, **kw):
    T, D = pb.num_time_steps, pb.chain.num_dimensions
    o = Oracle(num_time_steps=T, num_dimensions=D, min_rollouts=min_r, max_rollouts=max_r, num_rollouts_per_iteration=per_it,
               noise_stddev=pb.noise_stddev, **kw)
    o.set_problem(pb)
    if _RECORD is not None:
        r = _Recorded(reference=ref_binding.Reference(o))
    elif LIVE:
        r = ref_binding.Reference(o)
    elif os.path.exists(_recording()):
        r = _Recorded(stored=np.load(_recording()))
    else:
        pytest.skip("needs the reference's sources (oracle/ref/Makefile) or this test's recording of them "
                    "(tests/golden/make_pin_golden.py)")
    r.set_start_goal(pb.start, pb.goal)
    return o, r


def _run(o, r, iterations, seed, scale_at=None, cumulative=True, projection=False):
    rng = np.random.default_rng(seed)
    T, D = o.T, o.D
    o.begin_solve(); r.begin_solve()
    if projection:
        r.set_projection(True)               # the oracle takes the switch at construction (use_projection=True)
    if not cumulative:
        r.set_cost_cumulation(False)         # the oracle takes the switch at construction (use_cumulative_costs=False)
    counts, exact = [], True
    for it in range(iterations):
        G = r.next_num_generated()
        eps = rng.standard_normal((G, D, T))
        if scale_at is not None and it == scale_at:
            eps *= 8.0          # pushes samples onto the joint limits: the filter / setRollouts / computeNoise path
        stop_r, unit = r.iterate(it, eps)
        stop_o = o.iterate(it, noise=unit)
        assert r.num_rollouts() == o.num_rollouts()
        for f in FIELDS:
            a, b = r.field(f), o.field(f)
            _same(a, b, f"iteration {it}: {f}")
            exact = exact and _equal(a, b)
        if not cumulative:
            p = o.field("probabilities")
            assert not np.all(p == p[:, :, :1]), "per-time-step mode must give time-varying probabilities"
        _same(r.updates(), o.updates(), "updates")
        _same(r.parameters(), o.parameters(), "parameters")
        _same(r.stddevs(), o.stddevs(), "stddevs")
        nr, no = r.noiseless(), o.noiseless()
        assert nr["valid"] == no["valid"]
        np.testing.assert_allclose(nr["total_cost"], no["total_cost"], rtol=RTOL)
        np.testing.assert_allclose(nr["best_cost"], no["best_cost"], rtol=RTOL)
        assert _equal(nr["state_costs"], no["state_costs"]), "noise-less state costs"
        _same(nr["control_costs"], no["control_costs"], "noise-less control costs")
        assert _equal(r.rollout_validity(), o.rollout_validity()), "rollout validity"
        assert bool(stop_r) == bool(stop_o)
        counts.append(r.num_rollouts()[0])
    fr = r.finish_solve()
    found_o, solution_o, iterations_o = o.finish_solve()
    _same(fr["solution"], solution_o, "solution")
    assert fr["iterations"] == iterations_o and fr["found"] == found_o
    return counts, exact


def test_policy_products_match_the_reference():
    pb = P.single_arm_problem(K=8, T=100, sdf_n=64)
    o, r = _pair(pb, 8, 8, 8)
    po, pr = o.policy(), r.policy()
    for k in ("R", "Rinv", "L", "params_all", "mincc", "linear"):
        _same(pr[k], po[k], k)


def test_whole_solve_without_reuse_matches_the_reference():
    pb = P.single_arm_problem(K=24, T=60, sdf_n=64)
    o, r = _pair(pb, 24, 24, 24)
    counts, exact = _run(o, r, 6, seed=1, scale_at=2)
    assert counts == [24, 25, 25, 25, 25, 25]
    assert exact, "the restatement no longer matches the reference bit for bit (still within 1e-12)"


def test_shipped_yml_shape_with_rollout_reuse_matches_the_reference():
    # reference test/config/stomp.yml: min 5, max 50, 10 per iteration, T = 20
    pb = P.single_arm_problem(K=10, T=20, sdf_n=64)
    o, r = _pair(pb, 5, 50, 10)
    counts, _ = _run(o, r, 9, seed=2)
    assert counts == [10, 21, 32, 43, 51, 51, 51, 51, 51]


def test_min_rollouts_above_per_iteration_matches_the_reference():
    pb = P.single_arm_problem(K=10, T=20, sdf_n=64)
    o, r = _pair(pb, 12, 20, 4)
    counts, _ = _run(o, r, 6, seed=3)
    assert counts[0] == 12


def test_no_adaptation_and_noise_decay_matches_the_reference():
    pb = P.single_arm_problem(K=16, T=20, sdf_n=64)
    o, r = _pair(pb, 16, 16, 16, use_noise_adaptation=False, noise_decay=np.full(7, 0.9))
    _run(o, r, 4, seed=4)


def test_dual_arm_matches_the_reference():
    pb = P.dual_arm_problem(K=12, T=30, sdf_n=64)
    o, r = _pair(pb, 12, 12, 12)
    _run(o, r, 3, seed=5)


def test_warm_start_matches_the_reference():
    # StompPlanner::updateInitialTrajectory -> updatePolicy / updateMinControlCostParameters (StompPlanner.cpp:186-208)
    pb = P.single_arm_problem(K=12, T=30, sdf_n=64)
    o, r = _pair(pb, 12, 12, 12)
    _run(o, r, 2, seed=6)
    warm = o.parameters() + 0.01
    o.set_initial_trajectory(warm); r.set_initial_trajectory(warm)
    for k in ("params_all", "mincc"):
        _same(r.policy()[k], o.policy()[k], k)
    _run(o, r, 3, seed=7)


def test_per_timestep_costs_match_the_reference():
    # Stomp::setCostCumulation(false): cumulative_costs_[d] = total_costs_[d], probabilities vary with the time step
    # (PolicyImprovement.cpp:473-481,497-582).  Not what StompPlanner ships; it pins the restatement's other branch, which the
    # GPU's per-time-step kernels are compared with in tests/test_gpu_parity.py (SURVEY 8f rank 4).
    pb = P.single_arm_problem(K=12, T=30, sdf_n=64)
    o, r = _pair(pb, 12, 12, 12, use_cumulative_costs=False)
    _run(o, r, 4, seed=8, cumulative=False)


def test_projection_branch_matches_the_reference():
    # use_projection_ = true (PolicyImprovement.cpp:421-440,706,750-801): M = R^-1 with columns scaled by 1 / (T R^-1[p,p]),
    # noise_projected = M noise, update row = M (sum_r P noise).  Disabled in the reference (no setter) and not built
    # on the GPU; pinned here so that the restatement's branch is ready when it is (SURVEY 8f rank 4).
    pb = P.single_arm_problem(K=12, T=30, sdf_n=64)
    o, r = _pair(pb, 12, 12, 12, use_projection=True)
    _run(o, r, 3, seed=9, projection=True)
