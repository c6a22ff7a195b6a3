"""Parity of the CUDA path (through the C ABI) with the CPU oracle on the same seeded inputs.

Bars (BASELINE.json north_star): costs, probabilities and updated trajectories within 1e-9 relative
in FP64; the collision / no-collision verdict per timestep bit-exact."""
import numpy as np
import pytest

from motion_planners_b200 import binding, problems as P
from oracle.binding import Oracle

pytestmark = pytest.mark.gpu

RTOL = 1e-9


def _pair(pb, min_r=None, max_r=None, per_it=None, **kw):
    K = pb.num_rollouts
    min_r, max_r, per_it = min_r or K, max_r or K, per_it or K
    T, D = pb.num_time_steps, pb.chain.num_dimensions
    okw = {k: v for k, v in kw.items() if k in ("use_noise_adaptation", "noise_decay")}
    o = Oracle(num_time_steps=T, num_dimensions=D, min_rollouts=min_r, max_rollouts=max_r,
               num_rollouts_per_iteration=per_it, noise_stddev=pb.noise_stddev, **okw)
    o.set_problem(pb)
    pol = o.policy()
    ekw = {k: v for k, v in kw.items() if k in ("use_noise_adaptation", "noise_decay")}
    e = binding.engine_for_problem(pb, min_rollouts=min_r, max_rollouts=max_r, per_iteration=per_it, policy=pol,
                                   keep_debug_tensors=True, **ekw)
    return o, e, pol


def _assert_control_costs(got, ref):
    """Per-timestep control costs are squared finite differences, dt*w*(sum_j c_j x_j)^2 with |c_j x_j| ~ 1e3:
    an element that is 1e-7 of its row's scale has a condition number of ~1e5 with respect to x, so the
    ulp-level differences in theta that the update's summation order leaves (covered by the `parameters`
    check at 1e-9) show as ~1e-9 relative there.  Bar: 1e-9 relative, plus 1e-12 of the tensor's scale for
    the cancelled elements; the row sums (full / cumulative / total costs) are held to the pure 1e-9."""
    np.testing.assert_allclose(got, ref, rtol=RTOL, atol=1e-12 * float(np.max(np.abs(ref))) + 1e-18)


def _compare_iteration(o, e, cost, valid):
    num, gen = o.num_rollouts()
    assert e.num_rollouts() == (num, gen)
    np.testing.assert_allclose(e.tensor("rollouts")[0][:gen], o.field("parameters_noise")[:gen], rtol=RTOL, atol=1e-12)
    np.testing.assert_allclose(e.tensor("noise")[0], o.field("noise"), rtol=RTOL, atol=1e-12)
    # verdicts: bit-exact
    np.testing.assert_array_equal(e.tensor("verdicts")[0].astype(bool), o.field("state_costs") > 0.5)
    np.testing.assert_array_equal(e.tensor("state_costs")[0], o.field("state_costs"))
    np.testing.assert_array_equal(e.tensor("rollout_validity")[0], o.rollout_validity())
    _assert_control_costs(e.tensor("control_costs")[0], o.field("control_costs"))
    np.testing.assert_allclose(e.tensor("cumulative_costs")[0], o.field("cumulative_costs")[:, :, 0], rtol=RTOL)
    np.testing.assert_allclose(e.tensor("full_costs")[0], o.field("full_costs"), rtol=RTOL)
    np.testing.assert_allclose(e.tensor("total_cost")[0], o.field("total_cost"), rtol=RTOL)
    np.testing.assert_allclose(e.tensor("probabilities")[0], o.field("probabilities"), rtol=RTOL, atol=1e-300)
    np.testing.assert_allclose(e.tensor("full_probabilities")[0], o.field("full_probabilities"), rtol=RTOL, atol=1e-300)
    np.testing.assert_allclose(e.tensor("updates")[0], o.updates(), rtol=RTOL, atol=1e-13)
    np.testing.assert_allclose(e.tensor("parameters")[0], o.parameters(), rtol=RTOL, atol=1e-12)
    np.testing.assert_allclose(e.tensor("stddevs")[0], o.stddevs(), rtol=RTOL)
    nl = o.noiseless()
    np.testing.assert_allclose(cost[0], nl["total_cost"], rtol=RTOL)
    assert bool(valid[0]) == nl["valid"]
    np.testing.assert_array_equal(e.tensor("noiseless_state_costs")[0], nl["state_costs"])
    _assert_control_costs(e.tensor("noiseless_control_costs")[0], nl["control_costs"])


def test_sphere_centres_are_bit_identical():
    chain, spheres = P.dual_arm_chain(), P.dual_arm_spheres()
    chain.axis[2] = np.array([1.0, 2.0, 2.0]) / 3.0      # general axis
    chain.origin_rpy[4] = [0.3, -0.2, 0.7]               # fixed rotation
    chain.axis[9] = [-1.0, 0.0, 0.0]                     # negated axis
    chain.prismatic[12] = 1
    o = Oracle(num_time_steps=10, num_dimensions=14, min_rollouts=2, max_rollouts=2, num_rollouts_per_iteration=2,
               noise_stddev=np.ones(14))
    o.set_chain(chain)
    o.set_spheres(spheres)
    e = binding.Engine(num_time_steps=10, num_dimensions=14, min_rollouts=2, max_rollouts=2, num_rollouts_per_iteration=2)
    e.set_chain(chain)
    e.set_spheres(spheres)
    rng = np.random.default_rng(5)
    q = rng.uniform(-3.1, 3.1, (512, 14))
    q[0] = 0.0
    q[1] = 1e4 * rng.standard_normal(14)                 # far outside the joint range: reduction still agrees
    got = e.sphere_centres(q)
    ref = np.stack([o.sphere_centres(x) for x in q])
    assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))


@pytest.mark.parametrize("shape", ["iiwa", "dual_arm"])
def test_state_verdicts_are_bit_exact(shape, medium_problem):
    pb = medium_problem if shape == "iiwa" else P.dual_arm_problem(K=8, T=30, sdf_n=96)
    o, e, _ = _pair(pb)
    D = pb.chain.num_dimensions
    rng = np.random.default_rng(3)
    theta = rng.uniform(pb.chain.lower[None, :, None], pb.chain.upper[None, :, None], (64, D, pb.num_time_steps))
    costs, verdicts, validity = e.evaluate_states(theta)
    rc, rv, rval = o.state_costs(theta, threads=4)
    np.testing.assert_array_equal(verdicts, rv)
    np.testing.assert_array_equal(costs, rc)
    np.testing.assert_array_equal(validity, rval)
    assert 0.02 < costs.mean() < 0.98
    # K = 1, T = 1: the start / goal validity query of MotionPlanners::checkStartState
    for q, free in ((pb.start, True), (pb.goal, True)):
        c1, v1, val1 = e.evaluate_states(q[None, :, None])
        assert c1.shape == (1, 1) and bool(val1[0]) == free and bool(v1[0, 0]) != free


def test_iterations_with_injected_noise(medium_problem):
    pb = medium_problem
    T, D, K = pb.num_time_steps, pb.chain.num_dimensions, pb.num_rollouts
    o, e, pol = _pair(pb)
    o.begin_solve(); e.begin_solve()
    rng = np.random.default_rng(11)
    for it in range(5):
        unit = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((K, D, T)))
        if it == 2:
            unit *= 8.0      # push many samples onto the joint limits (filter / clamp path)
        o.iterate(it, noise=unit)
        cost, valid, stop = e.iterate(it, noise=unit[None])
        _compare_iteration(o, e, cost, valid)
    assert e.num_rollouts() == (K + 1, K)


def test_shipped_yml_shape_with_rollout_reuse(small_problem):
    # reference test/config/stomp.yml:3-5: min 5, max 50, 10 per iteration -> 10, 21, 32, 43, 51, 51 rollouts
    pb = small_problem
    T, D = pb.num_time_steps, pb.chain.num_dimensions
    o, e, pol = _pair(pb, 5, 50, 10)
    o.begin_solve(); e.begin_solve()
    rng = np.random.default_rng(7)
    counts = []
    for it in range(8):
        assert e.next_num_generated() == 10
        unit = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((10, D, T)))
        o.iterate(it, noise=unit)
        cost, valid, stop = e.iterate(it, noise=unit[None])
        _compare_iteration(o, e, cost, valid)
        counts.append(e.num_rollouts()[0])
    assert counts == [10, 21, 32, 43, 51, 51, 51, 51]


def test_min_rollouts_above_per_iteration(small_problem):
    # first iteration generates min_rollouts (PolicyImprovement.cpp:175-180)
    pb = small_problem
    T, D = pb.num_time_steps, pb.chain.num_dimensions
    o, e, pol = _pair(pb, 12, 20, 4)
    o.begin_solve(); e.begin_solve()
    rng = np.random.default_rng(8)
    for it in range(5):
        g = e.next_num_generated()
        assert g == (12 if it == 0 else 4)
        unit = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((g, D, T)))
        o.iterate(it, noise=unit)
        cost, valid, _ = e.iterate(it, noise=unit[None])
        _compare_iteration(o, e, cost, valid)


def test_no_adaptation_and_noise_decay(small_problem):
    pb = small_problem
    T, D = pb.num_time_steps, pb.chain.num_dimensions
    o, e, pol = _pair(P.single_arm_problem(K=16, T=20, sdf_n=64), use_noise_adaptation=False, noise_decay=np.full(7, 0.9))
    o.begin_solve(); e.begin_solve()
    rng = np.random.default_rng(9)
    for it in range(4):
        unit = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((16, D, T)))
        o.iterate(it, noise=unit)
        cost, valid, _ = e.iterate(it, noise=unit[None])
        _compare_iteration(o, e, cost, valid)
    np.testing.assert_allclose(e.tensor("stddevs")[0], pb.noise_stddev * 0.9 ** 2, rtol=1e-15)


def test_epsilon_goes_through_the_cholesky_factor_on_the_device(medium_problem):
    pb = medium_problem
    T, D, K = pb.num_time_steps, pb.chain.num_dimensions, pb.num_rollouts
    o, e, pol = _pair(pb)
    o.begin_solve(); e.begin_solve()
    rng = np.random.default_rng(13)
    for it in range(2):
        eps = rng.standard_normal((K, D, T))
        cost, valid, _ = e.iterate(it, epsilon=eps[None])
        unit = e.tensor("unit_noise")[0]
        ref = np.einsum("tu,kdu->kdt", pol["L"], eps)
        np.testing.assert_allclose(unit, ref, rtol=1e-12, atol=1e-14 * abs(ref).max())
        o.iterate(it, noise=unit)           # downstream of the contraction the loop is compared as usual
        _compare_iteration(o, e, cost, valid)


def test_on_device_sampler(medium_problem):
    pb = medium_problem
    T, D, K = pb.num_time_steps, pb.chain.num_dimensions, pb.num_rollouts
    o, e, pol = _pair(pb)
    o.begin_solve(); e.begin_solve()
    all_eps = []
    for it in range(3):
        cost, valid, _ = e.iterate(it)
        eps = e.tensor("epsilon")[0]
        unit = e.tensor("unit_noise")[0]
        ref = np.einsum("tu,kdu->kdt", pol["L"], eps)
        # the on-device sampler applies L through its banded inverse (test_recurrence_sampler_is_the_same_map_as_the_contraction):
        # agreement with the product by the reference's L is limited by the accuracy of that L, cond(R) * eps
        assert abs(unit - ref).max() <= 4e-9 * abs(ref).max()
        o.iterate(it, noise=unit)
        _compare_iteration(o, e, cost, valid)
        all_eps.append(eps)
    z = np.concatenate([a.ravel() for a in all_eps])
    n = z.size
    assert abs(z.mean()) < 5.0 / np.sqrt(n)
    assert abs(z.var() - 1.0) < 5.0 * np.sqrt(2.0 / n)
    assert abs((z ** 4).mean() - 3.0) < 0.2
    assert not np.array_equal(all_eps[0], all_eps[1])          # the iteration is part of the counter
    # same seed, same numbers; another seed, other numbers
    e2 = binding.engine_for_problem(pb, policy=pol, keep_debug_tensors=True)
    e2.begin_solve(); e2.iterate(0)
    np.testing.assert_array_equal(e2.tensor("epsilon")[0], all_eps[0])
    e3 = binding.engine_for_problem(pb, policy=pol, keep_debug_tensors=True, seed=7)
    e3.begin_solve(); e3.iterate(0)
    assert not np.array_equal(e3.tensor("epsilon")[0], all_eps[0])


def test_run_equals_iterate_and_stop_rule_freezes_the_query(small_problem):
    pb = P.single_arm_problem(K=32, T=20, sdf_n=64)
    pol = None
    a = binding.engine_for_problem(pb, keep_debug_tensors=True)
    b = binding.engine_for_problem(pb, keep_debug_tensors=True)
    a.begin_solve(); b.begin_solve()
    stops = []
    for it in range(12):
        cost, valid, stop = a.iterate(it)
        stops.append(bool(stop[0]))
    b.run(0, 12, honour_stop=False)
    np.testing.assert_array_equal(a.tensor("parameters"), b.tensor("parameters"))
    ra, rb = a.finish_solve(), b.finish_solve()
    np.testing.assert_array_equal(ra["solution"], rb["solution"])
    assert ra["iterations"][0] == 12
    # with the stop rule honoured the query freezes at the first iteration that satisfied it
    c = binding.engine_for_problem(pb)
    c.begin_solve()
    c.run(0, 12, honour_stop=True)
    rc = c.finish_solve()
    if any(stops):
        first = stops.index(True)
        assert rc["iterations"][0] == first + 1
        assert rc["found"][0]
    else:
        assert rc["iterations"][0] == 12


def test_batch_of_queries_equals_separate_engines():
    Q, K, T = 6, 16, 40
    pb = P.batch_problem(Q=Q, K=K, T=T, sdf_n=64)
    batch = binding.engine_for_problem(pb, keep_debug_tensors=True)
    batch.begin_solve()
    units = []
    for it in range(4):
        batch.iterate(it)
        units.append(batch.tensor("unit_noise"))
    got = batch.finish_solve()
    assert got["solution"].shape == (Q, 7, T)
    for q in range(Q):
        single = P.Problem(pb.chain, pb.spheres, pb.sdf, pb.start[q], pb.goal[q], pb.noise_stddev, T, K)
        # the same query alone, fed the unit noise the batch engine drew for it: the same trajectory — to rounding, not
        # bit for bit: the batch engine's sampler leaves the control-cost sums itself (FMA form), the injected-noise path
        # takes them from the row kernel (the reference's operation order)
        e = binding.engine_for_problem(single)
        e.begin_solve()
        for it in range(4):
            e.iterate(it, noise=units[it][q][None])
        np.testing.assert_allclose(e.finish_solve()["solution"][0], got["solution"][q], rtol=1e-12, atol=1e-13)
        # and the oracle (its own policy products: agreement limited by the conditioning of R)
        o = Oracle(num_time_steps=T, num_dimensions=7, min_rollouts=K, max_rollouts=K, num_rollouts_per_iteration=K,
                   noise_stddev=pb.noise_stddev)
        o.set_problem(single)
        o.begin_solve()
        for it in range(4):
            o.iterate(it, noise=units[it][q])
        np.testing.assert_allclose(got["solution"][q], o.parameters(), rtol=0, atol=1e-7)


def test_batched_policy_upload_equals_the_per_query_calls():
    """stomp_b200_set_policies (one pair of stream-ordered copies for a batch of requests) against stomp_b200_set_policy per
    query: the same solves bit for bit, also when the policies are uploaded again right after a solve (re-planning), and
    ranges beyond the engine's queries are refused."""
    Q, K, T = 5, 16, 40
    pb = P.batch_problem(Q=Q, K=K, T=T, sdf_n=64)
    a = binding.engine_for_problem(pb)
    b = binding.engine_for_problem(pb)
    pols = [binding.host_policy(binding.host_initial_trajectory(pb.start[q], pb.goal[q], T), a.cfg.movement_duration,
                                tuple(a.cfg.derivative_weights)) for q in range(Q)]
    pa = np.stack([p_["params_all"] for p_ in pols]); mc = np.stack([p_["mincc"] for p_ in pols])
    for round_ in range(2):
        for q in range(Q):
            a.set_policy(q, pa[q], mc[q])
        b.set_policies(0, pa[:2], mc[:2])
        b.set_policies(2, pa[2:], mc[2:])
        a.begin_solve(); b.begin_solve()
        a.solve(12); b.solve(12)
        ra, rb = a.finish_solve(), b.finish_solve()
        np.testing.assert_array_equal(ra["solution"], rb["solution"])
        np.testing.assert_array_equal(ra["iterations"], rb["iterations"])
        np.testing.assert_array_equal(ra["cost"], rb["cost"])
    with pytest.raises(Exception):
        b.set_policies(Q - 1, pa[:2], mc[:2])
    bad = pa.copy(); bad[1, 0, 3] = np.nan
    with pytest.raises(Exception):
        b.set_policies(0, bad, mc)


def test_full_size_properties_config3():
    # BASELINE config 3 shape: K=4096, T=100, 7-DoF, 256^3 SDF — size-independent properties
    pb = P.single_arm_problem(K=4096, T=100, sdf_n=256)
    e = binding.engine_for_problem(pb)
    e.begin_solve()
    for it in range(3):
        cost, valid, stop = e.iterate(it)
        p = e.tensor("probabilities")[0]
        np.testing.assert_allclose(p.sum(0), 1.0, rtol=1e-11)
        np.testing.assert_allclose(e.tensor("full_probabilities")[0].sum(0), 1.0, rtol=1e-11)
        assert np.all(p == p[:, :, :1])
        np.testing.assert_allclose(p.min(0)[:, 0] / p.max(0)[:, 0], np.exp(-10.0), rtol=1e-9)
        sc = e.tensor("state_costs")[0]
        assert set(np.unique(sc)) <= {0.0, 1.0}
        np.testing.assert_array_equal(sc > 0.5, e.tensor("verdicts")[0].astype(bool))
        rl = e.tensor("rollouts")[0]
        assert np.all(rl >= pb.chain.lower[None, :, None]) and np.all(rl <= pb.chain.upper[None, :, None])
        # the verdict kernel on its own agrees with the loop's verdicts (idempotence of the cost path)
        _, v2, _ = e.evaluate_states(rl[:256])
        np.testing.assert_array_equal(v2, e.tensor("verdicts")[0][:256])
    n, g = e.num_rollouts()
    assert (n, g) == (4097, 4096)
    # a sample of the full-size rollouts against the oracle's verdicts
    o = Oracle(num_time_steps=100, num_dimensions=7, min_rollouts=4, max_rollouts=4, num_rollouts_per_iteration=4,
               noise_stddev=pb.noise_stddev)
    o.set_problem(pb)
    _, rv, _ = o.state_costs(rl[::64], threads=4)
    np.testing.assert_array_equal(rv, e.tensor("verdicts")[0][::64][: rv.shape[0]])


def _general_dual_arm_problem():
    """14-DoF dual arm with every structural branch of the FK: general axis, fixed rpy rotation, negated axis,
    prismatic joint, chain restart (second arm)."""
    pb = P.dual_arm_problem(K=24, T=30, sdf_n=96)
    pb.chain.axis[2] = np.array([1.0, 2.0, 2.0]) / 3.0
    pb.chain.origin_rpy[4] = [0.3, -0.2, 0.7]
    pb.chain.axis[9] = [-1.0, 0.0, 0.0]
    pb.chain.prismatic[12] = 1
    return pb


@pytest.mark.parametrize("shape", ["iiwa", "general_dual_arm"])
def test_specialised_state_kernel_equals_generic_kernel_and_oracle(shape, medium_problem, monkeypatch):
    """The loop's state kernel is compiled at run time for the robot's structure (state_codegen.hpp); the generic
    kernel (STOMP_B200_STATES=generic) and the oracle must give the same verdicts bit for bit."""
    pb = medium_problem if shape == "iiwa" else _general_dual_arm_problem()
    D, T, K = pb.chain.num_dimensions, pb.num_time_steps, pb.num_rollouts
    spec = binding.engine_for_problem(pb, keep_debug_tensors=True)
    kind, note = spec.state_kernel_kind()
    assert kind == "specialised", note
    src = spec.state_kernel_source()
    # one sine / cosine evaluation per revolute joint and one gather per sphere, however the chain walk is emitted
    revolute = D - int(np.count_nonzero(pb.chain.prismatic))
    assert src.count("det_sincos(q") == revolute
    assert src.count("voxel_of_centre<") == pb.spheres.link.size
    monkeypatch.setenv("STOMP_B200_STATES", "generic")
    gen = binding.engine_for_problem(pb, keep_debug_tensors=True)
    assert gen.state_kernel_kind()[0] == "generic"
    monkeypatch.delenv("STOMP_B200_STATES")
    o = Oracle(num_time_steps=T, num_dimensions=D, min_rollouts=K, max_rollouts=K, num_rollouts_per_iteration=K,
               noise_stddev=pb.noise_stddev)
    o.set_problem(pb)
    spec.begin_solve(); gen.begin_solve()
    hits = 0
    for it in range(3):
        spec.iterate(it); gen.iterate(it)
        vs, vg = spec.tensor("verdicts")[0], gen.tensor("verdicts")[0]
        np.testing.assert_array_equal(vs, vg)
        np.testing.assert_array_equal(spec.tensor("state_costs")[0], gen.tensor("state_costs")[0])
        np.testing.assert_array_equal(spec.tensor("rollout_validity")[0], gen.tensor("rollout_validity")[0])
        np.testing.assert_array_equal(spec.tensor("parameters")[0], gen.tensor("parameters")[0])
        # the noise-less states: the tail of the specialised kernel against a generic state pass over the policy rows
        np.testing.assert_array_equal(spec.tensor("noiseless_state_costs")[0], gen.tensor("noiseless_state_costs")[0])
        _, rv, _ = o.state_costs(spec.tensor("rollouts")[0][:K], threads=4)
        np.testing.assert_array_equal(vs[:K], rv)
        hits += int(vs.sum())
    assert hits > 0


def test_evaluate_states_beyond_the_specialised_kernels_range(medium_problem):
    """Joint values the specialised kernel cannot vouch for (|q| > 1e6) send stomp_b200_evaluate_states to the generic
    kernel even where the specialised one is in use: its verdicts must still be the oracle's, bit for bit.  A NaN in one
    state must not fail the call nor change any other state's verdict."""
    pb = medium_problem
    o, e, _ = _pair(pb)
    assert e.state_kernel_kind()[0] == "specialised"
    D, T = pb.chain.num_dimensions, pb.num_time_steps
    rng = np.random.default_rng(17)
    theta = rng.uniform(pb.chain.lower[None, :, None], pb.chain.upper[None, :, None], (32, D, T))
    far = rng.random(theta.shape) < 0.3
    theta[far] += rng.choice([-1.0, 1.0], far.sum()) * rng.uniform(2e6, 1e7, far.sum())
    assert np.abs(theta).max() > 1e6
    costs, verdicts, validity = e.evaluate_states(theta)
    rc, rv, rval = o.state_costs(theta, threads=4)
    np.testing.assert_array_equal(verdicts, rv)
    np.testing.assert_array_equal(costs, rc)
    np.testing.assert_array_equal(validity, rval)
    assert 0.0 < costs.mean() < 1.0
    bad = theta.copy()
    bad[5, 3, 40] = np.nan
    c2, v2, val2 = e.evaluate_states(bad)
    keep = np.ones((32, T), dtype=bool)
    keep[5, 40] = False
    np.testing.assert_array_equal(v2[keep], verdicts[keep])
    np.testing.assert_array_equal(c2[keep], costs[keep])
    np.testing.assert_array_equal(val2, validity)


def test_static_spheres_are_walked_once_per_scene_and_follow_scene_changes(monkeypatch):
    """Spheres on the axis of a chain's first joint do not move with the state; the generated module evaluates them in
    stomp_b200_static_spheres, once per robot / scene, and the walk starts from that verdict.  The verdicts must stay those
    of the kernel that walks every sphere per state (STOMP_B200_STATES_STATIC=0), of the generic kernel and of the oracle —
    also when the scene changes under a live engine: an obstacle put on the base column condemns every state, and taking it
    away again clears them."""
    import copy
    pb = P.single_arm_problem(K=16, T=40, sdf_n=64)
    D, T, K = pb.chain.num_dimensions, pb.num_time_steps, pb.num_rollouts
    e = binding.engine_for_problem(pb, keep_debug_tensors=True)
    assert e.state_kernel_kind()[0] == "specialised"
    src = e.state_kernel_source()
    assert "stomp_b200_static_spheres" in src and "static_spheres_hit" in src
    import re
    n_static = int(re.search(r"// (\d+) static spheres", src).group(1))
    assert n_static >= 1
    # the walk gathers for every sphere but the static ones
    walk = src.split("bool state_hit(", 1)[1]
    assert walk.count("voxel_of_centre<") == pb.spheres.link.size - n_static
    monkeypatch.setenv("STOMP_B200_STATES_STATIC", "0")
    full = binding.engine_for_problem(pb, keep_debug_tensors=True)
    assert full.state_kernel_kind()[0] == "specialised"                       # the kernel is resolved here, under the switch
    assert "stomp_b200_static_spheres" not in full.state_kernel_source()
    monkeypatch.delenv("STOMP_B200_STATES_STATIC")
    monkeypatch.setenv("STOMP_B200_STATES", "generic")
    gen = binding.engine_for_problem(pb, keep_debug_tensors=True)
    assert gen.state_kernel_kind()[0] == "generic"
    monkeypatch.delenv("STOMP_B200_STATES")
    o = Oracle(num_time_steps=T, num_dimensions=D, min_rollouts=K, max_rollouts=K, num_rollouts_per_iteration=K,
               noise_stddev=pb.noise_stddev)
    o.set_problem(pb)
    rng = np.random.default_rng(5)
    theta = rng.uniform(-1.5, 1.5, size=(K, D, T))
    centre0 = e.sphere_centres(np.zeros(D))[0, 0]          # a static sphere: the same for every q
    np.testing.assert_array_equal(e.sphere_centres(theta[:, :, 0])[:, 0], np.broadcast_to(centre0, (K, 3)))

    def scene(blocked):
        sdf = copy.copy(pb.sdf)
        grid = np.array(pb.sdf.grid, dtype=np.float32, copy=True)
        if blocked:     # a small obstacle where the first sphere sits: distance 0 in its voxel and the ones around it
            ix, iy, iz = np.floor((centre0 - pb.sdf.origin) / pb.sdf.voxel).astype(int)
            grid[iz - 1:iz + 2, iy - 1:iy + 2, ix - 1:ix + 2] = 0.0
        sdf.grid = grid
        return sdf

    import contextlib

    @contextlib.contextmanager
    def switch(name, value):       # the state kernel is resolved again after every scene change, under the switches of that moment
        if name:
            monkeypatch.setenv(name, value)
        try:
            yield
        finally:
            if name:
                monkeypatch.delenv(name)

    seen = []
    for blocked in (False, True, False):
        sdf = scene(blocked)
        o.set_sdf(sdf)
        _, vo, _ = o.state_costs(theta, threads=4)
        v = {}
        for tag, eng, name, value in (("hoisted", e, None, None), ("full", full, "STOMP_B200_STATES_STATIC", "0"), ("generic", gen, "STOMP_B200_STATES", "generic")):
            with switch(name, value):
                eng.set_sdf(sdf)
                _, v[tag], _ = eng.evaluate_states(theta)
                assert (eng.state_kernel_kind()[0] == "generic") == (tag == "generic")
                if tag != "generic":
                    assert ("stomp_b200_static_spheres" in eng.state_kernel_source()) == (tag == "hoisted")
                if tag != "generic":     # and through the loop (graph replays included): the flag reaches the rollouts and the noise-less tail
                    eng.begin_solve()
                    for it in range(3):
                        eng.iterate(it)
                    v[tag + " loop"] = (eng.tensor("verdicts")[0], eng.tensor("parameters")[0], eng.tensor("rollouts")[0])
        np.testing.assert_array_equal(v["hoisted"], v["full"])
        np.testing.assert_array_equal(v["hoisted"], v["generic"])
        np.testing.assert_array_equal(v["hoisted"], vo)
        for a, b in zip(v["hoisted loop"], v["full loop"]):
            np.testing.assert_array_equal(a, b)
        if blocked:
            assert v["hoisted loop"][0][:K].all()
        seen.append(int(v["hoisted"].sum()))
    assert seen[1] == K * T and seen[0] < K * T and seen[2] == seen[0]


@pytest.mark.parametrize("T", [20, 25, 40, 60, 100, 150, 200])
def test_trajectory_lengths_cover_every_kernel_variant(T):
    """T selects the kernel instantiations: tiles per slab of the DMMA sampler (4 / 7 / 10 / 13, one or two slabs), groups
    per lane of the control-cost tile kernel (2 / 4 / 7 / 11 / 14), and — for odd T — the scalar epilogue and the generic
    control-cost kernel.  Standard normals go through the on-device Cholesky contraction; everything downstream is
    compared with the oracle as usual.  K = 9 leaves the last 8-row / 8-column tiles ragged."""
    pb = P.single_arm_problem(K=9, T=T, sdf_n=64)
    D, K = pb.chain.num_dimensions, pb.num_rollouts
    o, e, pol = _pair(pb)
    o.begin_solve(); e.begin_solve()
    rng = np.random.default_rng(100 + T)
    for it in range(3):
        eps = rng.standard_normal((K, D, T))
        cost, valid, _ = e.iterate(it, epsilon=eps[None])
        unit = e.tensor("unit_noise")[0]
        ref = np.einsum("tu,kdu->kdt", pol["L"], eps)
        np.testing.assert_allclose(unit, ref, rtol=1e-12, atol=1e-14 * abs(ref).max())
        o.iterate(it, noise=unit)
        _compare_iteration(o, e, cost, valid)
    # and the on-device sampler of the same shape: replayed through the oracle
    cost, valid, _ = e.iterate(3)
    unit = e.tensor("unit_noise")[0]
    ref = np.einsum("tu,kdu->kdt", pol["L"], e.tensor("epsilon")[0])
    assert abs(unit - ref).max() <= 4e-9 * abs(ref).max()      # recurrence sampler: limited by the accuracy of L itself
    o.iterate(3, noise=unit)
    _compare_iteration(o, e, cost, valid)


def test_unfused_weights_and_update_kernels_match_the_fused_kernel(monkeypatch):
    """Single-GPU runs use weights_update_kernel (K7-K9 in one launch); multi-GPU, rollout reuse and the per-kernel
    profiling pass use rollout_weights_kernel -> weighted_update_kernel -> apply_update_kernel.  K' = 1101 makes the
    unfused weights kernel run three CTAs per joint (partial sums in wpart) and the update 35 chunks of 32 rollouts
    (the chunk stomp_b200_create picks for 1101 slots, 7 joints and one query on a 148-SM B200).  With
    STOMP_B200_FUSE_WEIGHTS=0 the apply step rides on weighted_update_kernel's last chunk CTA; profiling splits it off
    into apply_update_kernel, which adds the same partials in the same chunk order: bit-identical."""
    pb = P.single_arm_problem(K=1100, T=40, sdf_n=64)
    fused = binding.engine_for_problem(pb, keep_debug_tensors=True)
    monkeypatch.setenv("STOMP_B200_FUSE_WEIGHTS", "0")
    unfused = binding.engine_for_problem(pb, keep_debug_tensors=True)
    monkeypatch.delenv("STOMP_B200_FUSE_WEIGHTS")
    profiled = binding.engine_for_problem(pb, keep_debug_tensors=True)
    profiled.set_profiling(True)
    fused.begin_solve(); unfused.begin_solve(); profiled.begin_solve()
    for it in range(4):
        c1, v1, s1 = fused.iterate(it)
        c2, v2, s2 = unfused.iterate(it)
        c3, v3, s3 = profiled.iterate(it)
        for name in ("epsilon", "verdicts", "total_cost", "probabilities", "full_probabilities", "updates", "parameters", "stddevs"):
            np.testing.assert_array_equal(profiled.tensor(name)[0], unfused.tensor(name)[0], err_msg=name)
        np.testing.assert_array_equal(c3, c2)
        np.testing.assert_array_equal(fused.tensor("epsilon")[0], unfused.tensor("epsilon")[0])
        np.testing.assert_array_equal(fused.tensor("verdicts")[0], unfused.tensor("verdicts")[0])
        for name in ("total_cost", "probabilities", "full_probabilities", "updates", "parameters", "stddevs"):
            np.testing.assert_allclose(fused.tensor(name)[0], unfused.tensor(name)[0], rtol=1e-9, atol=1e-13, err_msg=name)
        np.testing.assert_allclose(c1, c2, rtol=1e-9)
        p = fused.tensor("probabilities")[0]
        np.testing.assert_allclose(p.sum(0), 1.0, rtol=1e-11)


def test_per_timestep_costs_mode():
    """Stomp::setCostCumulation(false) (PolicyImprovement.cpp:473-481): costs and probabilities per time step.  Not what
    StompPlanner ships; the oracle's branch is pinned against the reference's own code (tests/test_reference_pin.py)."""
    pb = P.single_arm_problem(K=24, T=40, sdf_n=64)
    T, D, K = pb.num_time_steps, pb.chain.num_dimensions, pb.num_rollouts
    o = Oracle(num_time_steps=T, num_dimensions=D, min_rollouts=K, max_rollouts=K, num_rollouts_per_iteration=K,
               noise_stddev=pb.noise_stddev, use_cumulative_costs=False)
    o.set_problem(pb)
    pol = o.policy()
    e = binding.engine_for_problem(pb, policy=pol, keep_debug_tensors=True, use_cumulative_costs=False)
    o.begin_solve(); e.begin_solve()
    rng = np.random.default_rng(21)
    for it in range(4):
        unit = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((K, D, T)))
        o.iterate(it, noise=unit)
        cost, valid, _ = e.iterate(it, noise=unit[None])
        p_ref = o.field("probabilities")
        assert not np.all(p_ref == p_ref[:, :, :1])
        np.testing.assert_array_equal(e.tensor("verdicts")[0].astype(bool), o.field("state_costs") > 0.5)
        _assert_control_costs(e.tensor("control_costs")[0], o.field("control_costs"))
        np.testing.assert_allclose(e.tensor("probabilities")[0], p_ref, rtol=RTOL, atol=1e-300)
        np.testing.assert_allclose(e.tensor("probabilities")[0].sum(0), 1.0, rtol=1e-11)
        np.testing.assert_allclose(e.tensor("full_probabilities")[0], o.field("full_probabilities"), rtol=RTOL, atol=1e-300)
        np.testing.assert_allclose(e.tensor("updates")[0], o.updates(), rtol=RTOL, atol=1e-13)
        np.testing.assert_allclose(e.tensor("parameters")[0], o.parameters(), rtol=RTOL, atol=1e-12)
        np.testing.assert_allclose(e.tensor("stddevs")[0], o.stddevs(), rtol=RTOL)
        np.testing.assert_allclose(cost[0], o.noiseless()["total_cost"], rtol=RTOL)
    # the same switch at run time (Stomp::setCostCumulation after initialize), on an engine created in the default mode
    o2 = Oracle(num_time_steps=T, num_dimensions=D, min_rollouts=K, max_rollouts=K, num_rollouts_per_iteration=K,
                noise_stddev=pb.noise_stddev, use_cumulative_costs=False)
    o2.set_problem(pb)
    e2 = binding.engine_for_problem(pb, policy=pol)
    o2.begin_solve(); e2.begin_solve()
    e2.set_cost_cumulation(False)
    for it in range(2):
        unit = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((K, D, T)))
        o2.iterate(it, noise=unit)
        e2.iterate(it, noise=unit[None])
        np.testing.assert_allclose(e2.tensor("probabilities")[0], o2.field("probabilities"), rtol=RTOL, atol=1e-300)
        np.testing.assert_allclose(e2.tensor("parameters")[0], o2.parameters(), rtol=RTOL, atol=1e-12)
    # the combinations that are not built say so
    with pytest.raises(binding.StompB200Error) as err:
        binding.Engine(num_time_steps=T, num_dimensions=D, min_rollouts=5, max_rollouts=50, num_rollouts_per_iteration=10,
                       use_cumulative_costs=False)
    assert err.value.code == binding.ERR_UNSUPPORTED


@pytest.mark.parametrize("K,T", [(1, 4), (2, 10), (5, 2)])
def test_smallest_shapes(K, T):
    """One rollout, two time steps: the ragged ends of every kernel (single tiles, windows that are mostly padding)."""
    pb = P.single_arm_problem(K=K, T=T, sdf_n=64)
    D = pb.chain.num_dimensions
    o, e, pol = _pair(pb)
    o.begin_solve(); e.begin_solve()
    rng = np.random.default_rng(300 + 10 * K + T)
    for it in range(3):
        eps = rng.standard_normal((K, D, T))
        cost, valid, _ = e.iterate(it, epsilon=eps[None])
        unit = e.tensor("unit_noise")[0]
        ref = np.einsum("tu,kdu->kdt", pol["L"], eps)
        np.testing.assert_allclose(unit, ref, rtol=1e-12, atol=1e-14 * max(abs(ref).max(), 1e-300))
        o.iterate(it, noise=unit)
        _compare_iteration(o, e, cost, valid)


def test_longest_trajectory_and_the_fallback_kernels(monkeypatch):
    """T = STOMP_B200_MAX_TIME_STEPS = 256: three slabs in the DMMA sampler, and N = 268 is past the control-cost tile
    kernel's instantiations, so control_rows_fast_kernel runs.  Then T = 100 with the generic state kernel
    (STOMP_B200_STATES=generic): the fallback agrees with the oracle like the default kernel does."""
    def check(pb, iterations):
        D, K, T = pb.chain.num_dimensions, pb.num_rollouts, pb.num_time_steps
        o, e, pol = _pair(pb)
        o.begin_solve(); e.begin_solve()
        rng = np.random.default_rng(500 + T)
        for it in range(iterations):
            eps = rng.standard_normal((K, D, T))
            cost, valid, _ = e.iterate(it, epsilon=eps[None])
            unit = e.tensor("unit_noise")[0]
            ref = np.einsum("tu,kdu->kdt", pol["L"], eps)
            np.testing.assert_allclose(unit, ref, rtol=1e-12, atol=1e-14 * abs(ref).max())
            o.iterate(it, noise=unit)
            _compare_iteration(o, e, cost, valid)
        return e
    check(P.single_arm_problem(K=3, T=256, sdf_n=64), 2)
    monkeypatch.setenv("STOMP_B200_STATES", "generic")
    e = check(P.single_arm_problem(K=10, T=100, sdf_n=64), 2)
    assert e.state_kernel_kind()[0] == "generic"


def test_largest_robot():
    """STOMP_B200_MAX_DIMS = 32 joints, STOMP_B200_MAX_SPHERES = 128 spheres: the generated state kernel at its largest,
    against the generic kernel's sphere centres (bit-identical) and the oracle's loop."""
    D, S = 32, 128
    rng = np.random.default_rng(77)
    axes = np.array([[0, 0, 1], [0, 1, 0], [1, 0, 0], [0, -1, 0]], dtype=np.float64)
    chain = P.Chain(origin_xyz=np.concatenate([[[0.0, 0.0, 0.1]], np.tile([[0.0, 0.01, 0.04]], (D - 1, 1))]),
                    origin_rpy=np.zeros((D, 3)), axis=np.stack([axes[d % 4] for d in range(D)]),
                    parent=np.arange(-1, D - 1, dtype=np.int32), prismatic=np.zeros(D, dtype=np.int32),
                    lower=np.full(D, -1.0), upper=np.full(D, 1.0), names=[f"j{d}" for d in range(D)])
    spheres = P.Spheres(link=np.repeat(np.arange(D, dtype=np.int32), S // D),
                        xyz=rng.uniform(-0.02, 0.02, (S, 3)) * np.array([1.0, 0.0, 1.0]), radius=np.full(S, 0.03))
    base = P.single_arm_problem(K=6, T=20, sdf_n=64)
    pb = P.Problem(chain, spheres, base.sdf, np.full(D, -0.3), np.full(D, 0.4), np.full(D, 0.3), 20, 6)
    o, e, pol = _pair(pb)
    assert e.state_kernel_kind()[0] == "specialised"
    q = rng.uniform(-1.0, 1.0, (16, D))
    assert np.array_equal(e.sphere_centres(q).view(np.uint64), np.stack([o.sphere_centres(x) for x in q]).view(np.uint64))
    o.begin_solve(); e.begin_solve()
    for it in range(3):
        unit = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((6, D, 20)))
        o.iterate(it, noise=unit)
        cost, valid, _ = e.iterate(it, noise=unit[None])
        _compare_iteration(o, e, cost, valid)


def _projection_pair(pb, min_r=None, max_r=None, per_it=None, **okw):
    K = pb.num_rollouts
    min_r, max_r, per_it = min_r or K, max_r or K, per_it or K
    T, D = pb.num_time_steps, pb.chain.num_dimensions
    o = Oracle(num_time_steps=T, num_dimensions=D, min_rollouts=min_r, max_rollouts=max_r,
               num_rollouts_per_iteration=per_it, noise_stddev=pb.noise_stddev, **okw)
    o.set_problem(pb)
    pol = o.policy()
    e = binding.engine_for_problem(pb, min_rollouts=min_r, max_rollouts=max_r, per_iteration=per_it, policy=pol,
                                   keep_debug_tensors=True, **okw)
    return o, e, pol


@pytest.mark.parametrize("T", [20, 100, 150])
def test_m_matrix_projection(T):
    """PolicyImprovement::use_projection_ (PolicyImprovement.cpp:421-440,706,750-801): noise_projected_ = M * noise_ feeds the
    control costs, the update row is multiplied by M.  The oracle's branch is pinned against the reference's own code
    (tests/test_reference_pin.py); here the CUDA path against the oracle.  T = 150 leaves ragged tiles in the DMMA
    projection kernel (64-wide time tiles, 32-column tiles with K * D = 63)."""
    pb = P.single_arm_problem(K=9, T=T, sdf_n=64)
    D, K = pb.chain.num_dimensions, pb.num_rollouts
    o, e, pol = _projection_pair(pb, use_projection=True)
    o.begin_solve(); e.begin_solve()
    rng = np.random.default_rng(40 + T)
    for it in range(4):
        unit = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((K, D, T)))
        if it == 1:
            unit *= 6.0          # clamped samples: the projection sees the noise AFTER the joint-limit filter
        o.iterate(it, noise=unit)
        cost, valid, _ = e.iterate(it, noise=unit[None])
        ref = o.field("noise_projected")
        assert not np.allclose(ref, o.field("noise"))          # M really is not the identity
        np.testing.assert_allclose(e.tensor("noise_projected")[0], ref, rtol=RTOL, atol=1e-13 * abs(ref).max())
        _compare_iteration(o, e, cost, valid)
    # without the switch the same inputs give another trajectory
    o2, e2, _ = _projection_pair(pb)
    o2.begin_solve(); o2.iterate(0, noise=unit)
    assert not np.allclose(o2.parameters(), o.parameters())


def test_m_matrix_projection_with_rollout_reuse(small_problem):
    """Reused rollouts under projection: noise_ = M^-1 (parameters_noise_projected_ - parameters_) (PolicyImprovement.cpp:
    201-204), shipped yml rollout counts."""
    pb = small_problem
    T, D = pb.num_time_steps, pb.chain.num_dimensions
    o, e, pol = _projection_pair(pb, 5, 50, 10, use_projection=True)
    o.begin_solve(); e.begin_solve()
    rng = np.random.default_rng(17)
    for it in range(7):
        unit = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((10, D, T)))
        o.iterate(it, noise=unit)
        cost, valid, _ = e.iterate(it, noise=unit[None])
        n, g = o.num_rollouts()
        ref = o.field("noise_projected")
        np.testing.assert_allclose(e.tensor("noise_projected")[0], ref, rtol=1e-8, atol=1e-11 * abs(ref).max())
        np.testing.assert_allclose(e.tensor("rollouts_projected")[0], o.field("parameters_noise_projected"), rtol=1e-8, atol=1e-11)
        # M^-1 is ill conditioned (M ~ R^-1): the reused rollouts' noise_ carries that into everything downstream, so the
        # whole-iteration comparison of this case is held to 1e-6 of the tensor scale, not 1e-9
        np.testing.assert_allclose(e.tensor("noise")[0], o.field("noise"), rtol=1e-6, atol=1e-6 * abs(o.field("noise")).max())
        np.testing.assert_array_equal(e.tensor("verdicts")[0].astype(bool), o.field("state_costs") > 0.5)
        np.testing.assert_allclose(e.tensor("total_cost")[0], o.field("total_cost"), rtol=1e-6)
        np.testing.assert_allclose(e.tensor("parameters")[0], o.parameters(), rtol=1e-6, atol=1e-9)
    assert e.num_rollouts()[0] == 51


def test_per_timestep_minmax_variant():
    """The min / max variant the reference keeps commented out (PolicyImprovement.cpp:518-528), in per-time-step cost mode
    (in cumulative mode it coincides with the shipped rule): min and max over the rollouts of each time step."""
    pb = P.single_arm_problem(K=24, T=40, sdf_n=64)
    T, D, K = pb.num_time_steps, pb.chain.num_dimensions, pb.num_rollouts
    o, e, pol = _projection_pair(pb, use_cumulative_costs=False, per_timestep_minmax=True)
    o_plain, _, _ = _projection_pair(pb, use_cumulative_costs=False)
    o.begin_solve(); e.begin_solve(); o_plain.begin_solve()
    rng = np.random.default_rng(23)
    for it in range(3):
        unit = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((K, D, T)))
        o.iterate(it, noise=unit)
        cost, valid, _ = e.iterate(it, noise=unit[None])
        np.testing.assert_allclose(e.tensor("probabilities")[0], o.field("probabilities"), rtol=RTOL, atol=1e-300)
        np.testing.assert_allclose(e.tensor("updates")[0], o.updates(), rtol=RTOL, atol=1e-13)
        np.testing.assert_allclose(e.tensor("parameters")[0], o.parameters(), rtol=RTOL, atol=1e-12)
        np.testing.assert_allclose(e.tensor("stddevs")[0], o.stddevs(), rtol=RTOL)
        np.testing.assert_allclose(cost[0], o.noiseless()["total_cost"], rtol=RTOL)
    o_plain.iterate(0, noise=unit)
    assert not np.allclose(o_plain.parameters(), o.parameters())      # the variant is a different rule
    # in cumulative mode the switch changes nothing (cumulative_costs_ is constant over t)
    o3, e3, pol3 = _projection_pair(pb, per_timestep_minmax=True)
    o3.begin_solve(); e3.begin_solve()
    for it in range(2):
        unit = np.einsum("tu,kdu->kdt", pol3["L"], rng.standard_normal((K, D, T)))
        o3.iterate(it, noise=unit)
        cost, valid, _ = e3.iterate(it, noise=unit[None])
        _compare_iteration(o3, e3, cost, valid)


def test_projection_in_per_timestep_mode():
    pb = P.single_arm_problem(K=12, T=40, sdf_n=64)
    T, D, K = pb.num_time_steps, pb.chain.num_dimensions, pb.num_rollouts
    o, e, pol = _projection_pair(pb, use_cumulative_costs=False, use_projection=True)
    o.begin_solve(); e.begin_solve()
    rng = np.random.default_rng(29)
    for it in range(3):
        unit = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((K, D, T)))
        o.iterate(it, noise=unit)
        cost, valid, _ = e.iterate(it, noise=unit[None])
        _assert_control_costs(e.tensor("control_costs")[0], o.field("control_costs"))
        np.testing.assert_allclose(e.tensor("probabilities")[0], o.field("probabilities"), rtol=RTOL, atol=1e-300)
        np.testing.assert_allclose(e.tensor("updates")[0], o.updates(), rtol=RTOL, atol=1e-13)
        np.testing.assert_allclose(e.tensor("parameters")[0], o.parameters(), rtol=RTOL, atol=1e-12)
        np.testing.assert_allclose(cost[0], o.noiseless()["total_cost"], rtol=RTOL)


@pytest.mark.parametrize("poll_every,ahead", [(0, 1), (0, 3), (0, 0), (1, 0), (5, 0)])
def test_device_solve_loop_equals_the_host_driven_loop(poll_every, ahead, monkeypatch):
    """stomp_b200_solve (the loop StompPlanner::solve queues on the device, stop rule evaluated there) against the
    reference's control flow driven from the host: iterate, read the noise-less cost, break when it is below 1 and the
    improvement below min_cost_improvement (StompPlanner.cpp:96-118).  Same iteration count, same final trajectory bit
    for bit, whether the host paces its queue by the device's progress words (ahead > 0, the default) or synchronises
    every poll_every iterations (iterations queued past the stop are no-ops)."""
    pb = P.single_arm_problem(K=32, T=20, sdf_n=64)
    monkeypatch.setenv("STOMP_B200_SOLVE_AHEAD", str(ahead))
    a = binding.engine_for_problem(pb)
    b = binding.engine_for_problem(pb)
    a.begin_solve(); b.begin_solve()
    old, used = 0.0, 0
    for it in range(40):
        cost, valid, stop = a.iterate(it)
        used += 1
        improvement = cost[0] - old
        old = cost[0]
        if cost[0] < 1 and abs(improvement) < a.cfg.min_cost_improvement:
            assert bool(stop[0])
            break
        assert not bool(stop[0])
    queued = b.solve(40, poll_every)
    ra, rb = a.finish_solve(), b.finish_solve()
    assert rb["iterations"][0] == used == ra["iterations"][0]
    if ahead > 0:
        assert used <= queued <= used + ahead + 1  # the record of iteration i rides on iteration i + 1; `ahead` more may be queued behind it
    else:
        assert queued >= used and (poll_every != 1 or queued == used)
    np.testing.assert_array_equal(ra["solution"], rb["solution"])
    assert ra["cost"][0] == rb["cost"][0] and bool(ra["found"][0]) == bool(rb["found"][0])
    assert used < 40 and rb["found"][0]


def test_on_device_sampler_covariance():
    """The Philox path's distribution (the parity tests inject their noise): standard normals with the right moments, and
    unit noise L * eps whose sample covariance is R^-1 = L L^T — the covariance MultivariateGaussian is constructed with
    (PolicyImprovement.cpp:95-99).  Normals are FP32 Box-Muller from 24-bit uniforms (|z| <= 5.9): documented in DESIGN.md."""
    pb = P.single_arm_problem(K=4096, T=40, sdf_n=64)
    e = binding.engine_for_problem(pb, keep_debug_tensors=True)
    pol = e.policy
    e.begin_solve()
    eps_all, unit_all = [], []
    for it in range(3):
        e.iterate(it)
        eps_all.append(e.tensor("epsilon")[0].reshape(-1, 40))
        unit_all.append(e.tensor("unit_noise")[0].reshape(-1, 40))
    z = np.concatenate(eps_all)                # [3 * 4096 * 7][40]
    u = np.concatenate(unit_all)
    n = z.shape[0]
    assert abs(z.mean()) < 5 / np.sqrt(z.size) and abs(z.var() - 1) < 5 * np.sqrt(2 / z.size)
    assert abs((z ** 3).mean()) < 5 * np.sqrt(15 / z.size) and abs((z ** 4).mean() - 3) < 5 * np.sqrt(96 / z.size)
    assert 4.0 < np.abs(z).max() <= 5.95
    # identity covariance of eps: every entry within 6 standard errors
    ce = z.T @ z / n
    assert np.abs(ce - np.eye(40)).max() < 6 / np.sqrt(n) * np.sqrt(2)
    # covariance of the unit noise against R^-1, entry-wise within 6 standard errors sqrt((S_ii S_jj + S_ij^2) / n)
    S = pol["L"] @ pol["L"].T
    np.testing.assert_allclose(S, pol["Rinv"], rtol=1e-6, atol=1e-9 * np.abs(pol["Rinv"]).max())
    cu = u.T @ u / n
    se = np.sqrt((np.outer(np.diag(S), np.diag(S)) + S ** 2) / n)
    assert (np.abs(cu - S) / se).max() < 6.0
    # columns (rollout, joint) are independent draws: neighbouring columns are uncorrelated
    r = np.corrcoef(z[:-1].ravel(), z[1:].ravel())[0, 1]
    assert abs(r) < 5 / np.sqrt(z.size)


def _exact_unit_noise(R, eps):
    """n with U^T n = eps for the upper-triangular U of R = U U^T, in long double: the exact statement of n = L eps."""
    T = R.shape[0]
    J = np.eye(T)[::-1]
    Rl = R.astype(np.longdouble)
    # Cholesky of the flipped matrix in long double (plain loops: numpy has no long-double factorisations)
    A = (J @ R @ J).astype(np.longdouble)
    C = np.zeros_like(A)
    for j in range(T):
        C[j, j] = np.sqrt(A[j, j] - (C[j, :j] ** 2).sum())
        for i in range(j + 1, min(T, j + 8)):
            C[i, j] = (A[i, j] - (C[i, :j] * C[j, :j]).sum()) / C[j, j]
    B = (J.astype(np.longdouble) @ C @ J.astype(np.longdouble)).T       # lower, B n = eps
    n = np.zeros(eps.shape, dtype=np.longdouble)
    e = eps.astype(np.longdouble)
    for t in range(T):
        lo = max(0, t - 7)
        n[..., t] = (e[..., t] - (n[..., lo:t] * B[t, lo:t]).sum(-1)) / B[t, t]
    return n.astype(np.float64)


@pytest.mark.parametrize("T", [20, 50, 100, 150, 200, 256])
def test_recurrence_sampler_is_the_same_map_as_the_contraction(T, monkeypatch):
    """The on-device sampler does not multiply by the dense L: L^-1 is banded, so n = L eps is a 4-term recurrence
    (kernels.cuh: sample_rollouts_banded_kernel).  Same epsilon (same Philox counters) through both kernels: the unit noise
    agrees to the accuracy of the reference's own L (cond(R) * eps: 1e-10 at T = 100, 1e-9 at T = 256, relative to the
    tensor's scale), the recurrence agrees with an exact long-double solve to 1e-13, and everything downstream of the unit
    noise is compared with the oracle as usual.  K = 70 leaves a ragged third warp of rollouts; odd strides via T = 50 / 150."""
    pb = P.single_arm_problem(K=70, T=T, sdf_n=64)
    D, K = pb.chain.num_dimensions, pb.num_rollouts
    o, e, pol = _pair(pb)
    monkeypatch.setenv("STOMP_B200_SAMPLER", "dmma")
    e_dmma = binding.engine_for_problem(pb, policy=pol, keep_debug_tensors=True)
    monkeypatch.delenv("STOMP_B200_SAMPLER")
    o.begin_solve(); e.begin_solve(); e_dmma.begin_solve()
    for it in range(3):
        cost, valid, _ = e.iterate(it)
        e_dmma.iterate(it)
        eps, unit = e.tensor("epsilon")[0], e.tensor("unit_noise")[0]
        if it == 0:
            np.testing.assert_array_equal(eps, e_dmma.tensor("epsilon")[0])           # same counters, same normals
            ref = e_dmma.tensor("unit_noise")[0]
            scale = abs(ref).max()
            assert abs(unit - ref).max() <= 4e-9 * scale
            np.testing.assert_allclose(ref, np.einsum("tu,kdu->kdt", pol["L"], eps), rtol=1e-12, atol=1e-14 * scale)
        exact = _exact_unit_noise(pol["R"], eps)
        assert abs(unit - exact).max() <= 1e-12 * abs(exact).max()
        o.iterate(it, noise=unit)
        _compare_iteration(o, e, cost, valid)


def test_fused_control_cost_sums_of_the_recurrence_sampler(monkeypatch):
    """Without debug tensors the recurrence sampler leaves the control-cost sums and n^T R n itself (FMA form, in registers);
    with them the row kernel also runs to store the per-time-step costs.  The three ways to get the sums — fused, the row
    kernels behind the recurrence sampler (T odd: generic kernel), the row kernels behind the contraction — agree with the
    oracle to 1e-9 (replayed from the unit noise of a debug engine with the same seed)."""
    for T in (40, 100):
        pb = P.single_arm_problem(K=200, T=T, sdf_n=64)
        D, K = pb.chain.num_dimensions, pb.num_rollouts
        o, dbg, pol = _pair(pb)
        lean = binding.engine_for_problem(pb, policy=pol)                    # fused sums only
        monkeypatch.setenv("STOMP_B200_SAMPLER", "dmma")
        old = binding.engine_for_problem(pb, policy=pol)                     # contraction + row kernel
        monkeypatch.delenv("STOMP_B200_SAMPLER")
        for eng in (dbg, lean, old):
            eng.begin_solve()
        o.begin_solve()
        for it in range(4):
            cost, valid, _ = dbg.iterate(it)
            c2, v2, _ = lean.iterate(it)
            c3, v3, _ = old.iterate(it)
            o.iterate(it, noise=dbg.tensor("unit_noise")[0])
            _compare_iteration(o, dbg, cost, valid)
            for eng, c in ((lean, c2), (old, c3)):
                np.testing.assert_allclose(eng.tensor("total_cost")[0], o.field("total_cost"), rtol=1e-8 if eng is old else RTOL)
                np.testing.assert_allclose(eng.tensor("full_costs")[0], o.field("full_costs"), rtol=1e-8 if eng is old else RTOL)
                if eng is lean:
                    np.testing.assert_array_equal(eng.tensor("verdicts")[0], dbg.tensor("verdicts")[0])
                    np.testing.assert_allclose(eng.tensor("probabilities")[0], o.field("probabilities"), rtol=RTOL, atol=1e-300)
                    np.testing.assert_allclose(eng.tensor("parameters")[0], o.parameters(), rtol=RTOL, atol=1e-12)
                    np.testing.assert_allclose(eng.tensor("stddevs")[0], o.stddevs(), rtol=RTOL)
                    np.testing.assert_allclose(c, cost, rtol=RTOL)


# The shapes of the generate stage (engine.cu: generate_shape): noise source, STOMP_B200_SAMPLER, T (odd: the row kernels
# cannot be fused into the recurrence sampler), debug tensors (the fused sampler then leaves the per-time-step store to the
# row kernel), use_projection; and launch_count() added by each of three iterate() calls, the owed noise-less rollout that
# the call's read-back launches included.  The counts pin what the stage launches in each shape (bench.py reports them
# per step).
_GENERATE_SHAPES = {
    "philox-recurrence-fused-lean": ("philox", None, 40, False, False, (7, 4, 4)),
    "philox-recurrence-fused-store": ("philox", None, 40, True, False, (8, 5, 5)),
    "philox-recurrence-unfused": ("philox", None, 41, True, False, (8, 5, 5)),
    "philox-contraction": ("philox", "dmma", 40, False, False, (8, 5, 5)),
    "epsilon-contraction": ("epsilon", None, 40, True, False, (8, 5, 5)),
    "epsilon-recurrence": ("epsilon", "banded", 40, True, False, (8, 5, 5)),
    "unit-noise-shift": ("unit", None, 40, True, False, (8, 5, 5)),
    "philox-projection": ("philox", None, 40, True, True, (10, 7, 7)),
}


def _generate_shape_iterations(case, monkeypatch):
    """Three iterations of one generate shape; returns the launch_count() each added.  The two shapes no other test holds
    to the oracle, injected epsilon through the recurrence sampler and on-device noise under the M-projection, are
    compared with it here, replayed from the engine's unit noise."""
    noise, sampler, T, debug, projection = _GENERATE_SHAPES[case][:5]
    pb = P.single_arm_problem(K=24, T=T, sdf_n=64)
    D, K = pb.chain.num_dimensions, pb.num_rollouts
    compare = case in ("epsilon-recurrence", "philox-projection")
    okw = {"use_projection": True} if projection else {}
    if sampler:
        monkeypatch.setenv("STOMP_B200_SAMPLER", sampler)
    if compare:
        o, e, pol = _projection_pair(pb, **okw)
        o.begin_solve()
    else:
        e = binding.engine_for_problem(pb, keep_debug_tensors=debug, **okw)
        pol = e.policy
    monkeypatch.delenv("STOMP_B200_SAMPLER", raising=False)
    e.begin_solve()
    rng = np.random.default_rng(600 + T)
    added = []
    for it in range(3):
        kw = {}
        if noise == "epsilon":
            kw["epsilon"] = rng.standard_normal((1, K, D, T))
        elif noise == "unit":
            kw["noise"] = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((K, D, T)))[None]
        before = e.launch_count()
        cost, valid, _ = e.iterate(it, **kw)
        added.append(e.launch_count() - before)
        if compare:
            unit = e.tensor("unit_noise")[0]
            ref = np.einsum("tu,kdu->kdt", pol["L"], e.tensor("epsilon")[0])
            assert abs(unit - ref).max() <= 4e-9 * abs(ref).max()      # recurrence sampler: limited by the accuracy of L itself
            o.iterate(it, noise=unit)
            if projection:
                ref = o.field("noise_projected")
                np.testing.assert_allclose(e.tensor("noise_projected")[0], ref, rtol=RTOL, atol=1e-13 * abs(ref).max())
            _compare_iteration(o, e, cost, valid)
    return added


@pytest.mark.parametrize("case", list(_GENERATE_SHAPES))
def test_each_generate_shape_keeps_its_launch_count(case, monkeypatch):
    assert _generate_shape_iterations(case, monkeypatch) == list(_GENERATE_SHAPES[case][5])


def test_forward_cumulation_variant():
    """cumulative_costs_(t) = sum_{t' >= t} total_costs_(t'): the "forward cumulation" the reference keeps commented out at
    PolicyImprovement.cpp:473-477, selected with use_cumulative_costs = 2.  Cost-to-go differs per time step, so the
    per-time-step probability machinery runs; against the oracle's statement of the three commented lines."""
    pb = P.single_arm_problem(K=24, T=40, sdf_n=64)
    T, D, K = pb.num_time_steps, pb.chain.num_dimensions, pb.num_rollouts
    o, e, pol = _projection_pair(pb, use_cumulative_costs=2)
    o_total, _, _ = _projection_pair(pb)
    o.begin_solve(); e.begin_solve(); o_total.begin_solve()
    rng = np.random.default_rng(31)
    for it in range(4):
        unit = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((K, D, T)))
        o.iterate(it, noise=unit)
        cost, valid, _ = e.iterate(it, noise=unit[None])
        p_ref = o.field("probabilities")
        assert not np.all(p_ref == p_ref[:, :, :1])           # the probabilities do depend on the time step
        cum = o.field("cumulative_costs")
        assert np.all(np.diff(cum, axis=2) <= 1e-12)           # cost-to-go falls along the trajectory
        np.testing.assert_allclose(e.tensor("probabilities")[0], p_ref, rtol=RTOL, atol=1e-300)
        np.testing.assert_allclose(e.tensor("full_probabilities")[0], o.field("full_probabilities"), rtol=RTOL, atol=1e-300)
        np.testing.assert_allclose(e.tensor("updates")[0], o.updates(), rtol=RTOL, atol=1e-13)
        np.testing.assert_allclose(e.tensor("parameters")[0], o.parameters(), rtol=RTOL, atol=1e-12)
        np.testing.assert_allclose(e.tensor("stddevs")[0], o.stddevs(), rtol=RTOL)
        np.testing.assert_allclose(cost[0], o.noiseless()["total_cost"], rtol=RTOL)
    o_total.iterate(0, noise=unit)
    assert not np.allclose(o_total.parameters(), o.parameters())


@pytest.mark.parametrize("mode", ["smooth", "joint_constraint", "both"])
def test_alternative_state_costs(mode, medium_problem):
    """SURVEY 8f rank 4: the smooth obstacle cost (penetration of the link spheres into the clearance band, the non-boolean
    obstacle shape of stomp_2d_test.cpp:337-363) and the joint-constraint cost of OptimizationTask::computeJointsConstraintCost
    (OptimizationTask.cpp:206-237, call commented out in the reference).  State costs are no longer 0 / 1: the whole
    iteration against the oracle, the verdicts still bit-exact."""
    pb = medium_problem
    T, D, K = pb.num_time_steps, pb.chain.num_dimensions, pb.num_rollouts
    o, e, pol = _pair(pb)
    smooth = (0.05, 3.0) if mode in ("smooth", "both") else None
    jc = None
    if mode in ("joint_constraint", "both"):
        mid = 0.5 * (np.asarray(pb.start).reshape(-1)[:D] + np.asarray(pb.goal).reshape(-1)[:D])
        jc = (mid, np.full(D, 0.3), 0.7)
    o.set_cost_extras(smooth=smooth, joint_constraint=jc)
    e.set_cost_extras(smooth=smooth, joint_constraint=jc)
    o.begin_solve(); e.begin_solve()
    rng = np.random.default_rng(37)
    seen_fraction = False
    for it in range(3):
        unit = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((K, D, T)))
        o.iterate(it, noise=unit)
        cost, valid, _ = e.iterate(it, noise=unit[None])
        sc_ref = o.field("state_costs")
        seen_fraction = seen_fraction or bool(np.any((sc_ref > 0) & (sc_ref != 1.0)))
        np.testing.assert_allclose(e.tensor("state_costs")[0], sc_ref, rtol=RTOL, atol=1e-15)
        np.testing.assert_array_equal(e.tensor("rollout_validity")[0], o.rollout_validity())
        np.testing.assert_allclose(e.tensor("total_cost")[0], o.field("total_cost"), rtol=RTOL)
        np.testing.assert_allclose(e.tensor("probabilities")[0], o.field("probabilities"), rtol=RTOL, atol=1e-300)
        np.testing.assert_allclose(e.tensor("updates")[0], o.updates(), rtol=RTOL, atol=1e-13)
        np.testing.assert_allclose(e.tensor("parameters")[0], o.parameters(), rtol=RTOL, atol=1e-12)
        np.testing.assert_allclose(e.tensor("stddevs")[0], o.stddevs(), rtol=RTOL)
        nl = o.noiseless()
        np.testing.assert_allclose(cost[0], nl["total_cost"], rtol=RTOL)
        np.testing.assert_allclose(e.tensor("noiseless_state_costs")[0], nl["state_costs"], rtol=RTOL, atol=1e-15)
        assert bool(valid[0]) == nl["valid"]
    assert seen_fraction, "the problem never produced a non-binary state cost"
    # the stand-alone cost call carries the same costs
    theta = e.tensor("rollouts")[0][:4]
    costs, verdicts, validity = e.evaluate_states(theta)
    rc, rv, _ = o.state_costs(theta, threads=1)
    np.testing.assert_array_equal(verdicts.astype(bool), rv.astype(bool))
    np.testing.assert_allclose(costs, rc, rtol=RTOL, atol=1e-15)
    # switching the extras off restores the 0 / 1 cost
    e.set_cost_extras()
    costs01, _, _ = e.evaluate_states(theta)
    np.testing.assert_array_equal(costs01, verdicts.astype(np.float64))
    assert not np.array_equal(costs01, costs)


def test_sampler_that_draws_before_it_waits_changes_nothing(monkeypatch):
    """With enough rollouts to fill the GPU the sampler is a programmatic dependent of the previous iteration's update kernel and
    draws and shapes its noise (phases 1 and 2) before it waits for it (LoopParams::early_sampler); such loops are launched
    plainly, because a graph boundary would serialise the two kernels again.  Whatever the combination — early or late wait,
    plain launches or graph replays (which take the sampler's own iteration counter and its ticket) — the kernels see the same
    data: parameters, costs and standard deviations are bit for bit the same."""
    pb = P.single_arm_problem(K=4096, T=100, sdf_n=64)
    results, replays = [], []
    for graph, early in (("1", "1"), ("2", "1"), ("0", "0"), ("2", "0"), ("0", "1")):
        monkeypatch.setenv("STOMP_B200_GRAPH", graph)
        monkeypatch.setenv("STOMP_B200_SAMPLER_EARLY", early)
        e = binding.engine_for_problem(pb)
        e.begin_solve()
        e.run(0, 9)
        e.run(9, 1)
        e.run(10, 5, honour_stop=True)
        replays.append(e.graph_replays())
        r = e.finish_solve()
        results.append((e.tensor("parameters").copy(), r["solution"].copy(), r["cost"].copy(), r["iterations"].copy(), e.tensor("stddevs").copy()))
        e.close()
    # default (graphs allowed): this loop overlaps, so it is not replayed; STOMP_B200_GRAPH=2 insists on the graph
    assert replays[0] == 0 and replays[1] > 0 and replays[2] == 0 and replays[3] > 0 and replays[4] == 0
    for other in results[1:]:
        for a, b in zip(results[0], other):
            np.testing.assert_array_equal(a, b)


# launch_count() added by the run sequence of the test below and graph_replays() after it, per (STOMP_B200_GRAPH,
# STOMP_B200_PDL), as measured on an NVIDIA B200 (1000 W): a replay counts the kernels of the iteration it captured, and
# each time the device-side iteration counter is set from the host, set_counters_kernel adds one launch
_REPLAY_SEQUENCE_COUNTS = {("1", "13"): (50, 9), ("0", "0"): (48, 0), ("1", "0"): (50, 9), ("0", "13"): (48, 0)}


def _last_iteration_record(e):
    """What the engine reports of its last iteration: the rollout counts and the read-backs that follow the host's record of
    it (noise: the array, or the error when the loop did not materialise it)."""
    record = [e.num_rollouts(), e.next_num_generated()]
    record += [e.tensor(name).copy() for name in ("rollouts", "total_cost", "probabilities", "rollout_validity", "noiseless_state_costs")]
    try:
        record.append(e.tensor("noise").copy())
    except binding.StompB200Error as err:
        record.append(str(err))
    return record


def test_graph_replay_and_dependent_launch_change_nothing(medium_problem, monkeypatch):
    """Steady iterations replay from CUDA graphs (device-side iteration counter, double-buffered noise-less record) and the
    sampler / update kernels are launched as programmatic dependents: the same kernels on the same data, so the whole solve
    is bit for bit the one plain launches give — parameters, noise-less cost, iteration count, stop behaviour — and a replay
    leaves the host's record of the iteration as the iteration itself would: rollout counts and read-backs."""
    pb = medium_problem
    results, records = [], []
    for graph, pdl in _REPLAY_SEQUENCE_COUNTS:
        monkeypatch.setenv("STOMP_B200_GRAPH", graph)
        monkeypatch.setenv("STOMP_B200_PDL", pdl)
        e = binding.engine_for_problem(pb)
        e.begin_solve()
        before = e.launch_count()
        e.run(0, 7)                      # queued back to back: graphs from the fourth iteration on
        e.run(7, 1)                      # a lone iteration: plain launches, the noise-less tail launched alone at the join
        e.run(8, 6, honour_stop=True)
        counts = (e.launch_count() - before, e.graph_replays())
        assert counts == _REPLAY_SEQUENCE_COUNTS[(graph, pdl)]
        r = e.finish_solve()
        results.append((r["solution"].copy(), r["cost"].copy(), r["iterations"].copy(), e.tensor("stddevs").copy()))
        records.append(_last_iteration_record(e))
        e.close()
    for other in results[1:]:
        for a, b in zip(results[0], other):
            np.testing.assert_array_equal(a, b)
    for other in records[1:]:
        assert len(other) == len(records[0])
        for a, b in zip(records[0], other):
            np.testing.assert_array_equal(a, b)
    # and the device-side solve loop on top of graphs: same answer as the host-paced loop without them
    monkeypatch.setenv("STOMP_B200_GRAPH", "1"); monkeypatch.setenv("STOMP_B200_PDL", "13")
    e1 = binding.engine_for_problem(pb); e1.begin_solve(); e1.solve(25, 4); r1 = e1.finish_solve(); n1 = e1.graph_replays(); e1.close()
    # ... and the host pacing its queue by the device's progress words (the default) instead of synchronising every poll
    monkeypatch.setenv("STOMP_B200_GRAPH", "0"); monkeypatch.setenv("STOMP_B200_PDL", "0"); monkeypatch.setenv("STOMP_B200_SOLVE_AHEAD", "0")
    e2 = binding.engine_for_problem(pb); e2.begin_solve(); e2.solve(25, 1); r2 = e2.finish_solve(); e2.close()
    assert n1 > 0
    np.testing.assert_array_equal(r1["solution"], r2["solution"])
    np.testing.assert_array_equal(r1["iterations"], r2["iterations"])
    np.testing.assert_array_equal(r1["cost"], r2["cost"])
