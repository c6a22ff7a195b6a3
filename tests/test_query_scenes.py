"""A batch whose queries plan in different worlds: one distance field per scene, each query reading the field of its scene
(stomp_b200_select_scene / stomp_b200_set_query_scenes).

The Philox noise of a query depends on its global index only, so query q of a batch spread over several scenes must be, bit
for bit, query q of the same batch with every query in q's scene.  That is the yardstick of the GPU tests below, for every
state kernel that reads the field; the oracle and the sharded engine are held to the same batch."""
import copy

import numpy as np
import pytest

from motion_planners_b200 import binding, problems as P

ERR_INVALID_ARGUMENT, ERR_NOT_READY = -1, -4


def _mixed(Q=8, K=32, T=40):
    """Q queries over 3 scenes (round robin); scene 2 has its own dims, origin and voxel size."""
    pb = P.batch_problem_scenes(Q=Q, K=K, T=T, sdf_n=48, num_scenes=3, seed=77, query_seed=11)
    s2 = pb.scenes[2]
    pb.scenes[2] = P.make_sdf(40, s2.obstacles, lo=-1.6, hi=1.7, lazy=True)
    assert tuple(pb.scenes[2].dims) != tuple(pb.scenes[0].dims) and pb.scenes[2].voxel != pb.scenes[0].voxel
    return pb


def _uniform(pb, s):
    """The same queries, every one of them in scene s, as a one-scene problem."""
    u = copy.copy(pb)
    u.sdf, u.scenes, u.query_scene = pb.scenes[s], None, None
    return u


def _pairs(pb):
    """Sphere pairs on links at least three joints apart: with closer links the iiwa's spheres overlap in every state, and
    every verdict would be a hit whatever the scene."""
    pr = P.self_collision_pairs(pb.chain, pb.spheres)
    link = pb.spheres.link
    return pr[np.abs(link[pr[:, 0]] - link[pr[:, 1]]) >= 3]


def _engine(pb, flavour=None, **kw):
    e = binding.engine_for_problem(pb, **kw)
    if flavour in ("pairs", "pairs_generic"):
        e.set_self_collision(_pairs(pb))
    if flavour == "extras":
        D = pb.chain.num_dimensions
        e.set_cost_extras(smooth=(0.05, 2.0), joint_constraint=(np.zeros(D), np.full(D, 1.2), 0.5))
    return e


def _reset_policies(e, pb):
    for ql in range(e.Q):
        qg = e.query_offset + ql
        init = binding.host_initial_trajectory(pb.start[qg], pb.goal[qg], pb.num_time_steps)
        pol = binding.host_policy(init, e.cfg.movement_duration, tuple(e.cfg.derivative_weights))
        e.set_policy(ql, pol["params_all"], pol["mincc"])


def _solve(e, iterations=12):
    e.begin_solve()
    e.solve(iterations)
    return e.finish_solve()


def _iterations(e, n=3):
    e.begin_solve()
    out = []
    for it in range(n):
        cost, valid, stop = e.iterate(it)
        out.append(dict(cost=cost, valid=valid, stop=stop, verdicts=e.tensor("verdicts"), state_costs=e.tensor("state_costs"),
                        parameters=e.tensor("parameters")))
    return out


def _assert_query_equal(a, qa, b, qb):
    for key in a:
        np.testing.assert_array_equal(a[key][qa], b[key][qb], err_msg=key)


# ---------------------------------------------------------------------------------------------------------------------
# no GPU needed
# ---------------------------------------------------------------------------------------------------------------------
def test_batch_problem_scenes_is_deterministic_and_every_query_starts_and_ends_free_in_its_own_scene():
    a = P.batch_problem_scenes(Q=24, K=8, T=20, sdf_n=32, num_scenes=5, seed=3, query_seed=9)
    b = P.batch_problem_scenes(Q=24, K=8, T=20, sdf_n=32, num_scenes=5, seed=3, query_seed=9)
    np.testing.assert_array_equal(a.start, b.start)
    np.testing.assert_array_equal(a.goal, b.goal)
    np.testing.assert_array_equal(a.query_scene, np.arange(24) % 5)
    assert len(a.scenes) == 5 and all(s.grid is None and s.obstacles for s in a.scenes)     # built on the device
    assert repr(a.scenes[1].obstacles) != repr(a.scenes[2].obstacles)
    for s_a, s_b in zip(a.scenes, b.scenes):
        assert repr(s_a.obstacles) == repr(s_b.obstacles)
    for q in range(24):
        sdf = a.scenes[a.query_scene[q]]
        for conf in (a.start[q], a.goal[q]):
            c = P.sphere_centres_numpy(a.chain, a.spheres, conf)
            for kind, centre, size in sdf.obstacles:
                assert np.all(P._obstacle_distance(c, kind, centre, size) >= a.spheres.radius + sdf.voxel)


def test_codegen_selftest_compiles_the_per_query_field_branch():
    rc, log = binding.codegen_selftest()
    assert rc == 0, log
    assert log.count("field per query") == 2, log      # the wide-index world-only walk and the walk with the pair rule


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
FLAVOURS = ["generated", "generic", "pairs", "pairs_generic", "extras"]


def _flavour_env(monkeypatch, flavour):
    if flavour == "generic":
        monkeypatch.setenv("STOMP_B200_STATES", "generic")
    if flavour == "pairs_generic":
        monkeypatch.setenv("STOMP_B200_SELF", "generic")


@pytest.mark.gpu
@pytest.mark.parametrize("flavour", FLAVOURS)
def test_mixed_batch_equals_the_uniform_batch_of_each_query_scene(monkeypatch, flavour):
    _flavour_env(monkeypatch, flavour)
    pb = _mixed()
    mixed = _engine(pb, flavour)
    kind = mixed.state_kernel_kind()
    if flavour == "generated":
        assert kind[0] == "specialised" and "query_sdf" in mixed.state_kernel_source()
    if flavour == "generic":
        assert kind[0] == "generic"
    if flavour == "pairs":
        assert kind[0] == "self-collision" and "pair rule inside" in kind[1]
    if flavour == "pairs_generic":
        assert kind[0] == "self-collision" and "generic FK" in kind[1]
    got = _solve(mixed)
    steps = _iterations(mixed)
    wants = []
    for s in range(3):
        uni = _engine(_uniform(pb, s), flavour)
        assert "query_sdf" not in uni.state_kernel_source()        # one scene: the kernel of an engine without scenes
        want = _solve(uni)
        want_steps = _iterations(uni)
        for q in np.nonzero(pb.query_scene == s)[0]:
            for key in ("solution", "found", "iterations", "cost"):
                np.testing.assert_array_equal(got[key][q], want[key][q], err_msg=f"{flavour} scene {s} query {q} {key}")
            for a, b in zip(steps, want_steps):
                _assert_query_equal(a, q, b, q)
        wants.append(want)
        uni.close()
    # the scenes matter: some query plans differently in another scene than in its own
    assert any(not np.array_equal(wants[pb.query_scene[q]]["solution"][q], wants[(pb.query_scene[q] + 1) % 3]["solution"][q])
               for q in range(pb.num_queries))


@pytest.mark.gpu
def test_two_queries_of_a_mixed_batch_match_the_oracle_in_their_scenes():
    from oracle.binding import Oracle
    pb = _mixed()
    T, D, K, Q = pb.num_time_steps, pb.chain.num_dimensions, pb.num_rollouts, pb.num_queries
    e = _engine(pb, keep_debug_tensors=True)
    oracles = {}
    for q in (1, 2):                                     # scene 1, and scene 2 with its own geometry
        o = Oracle(num_time_steps=T, num_dimensions=D, min_rollouts=K, max_rollouts=K, num_rollouts_per_iteration=K,
                   noise_stddev=pb.noise_stddev)
        o.set_problem(_uniform(pb, int(pb.query_scene[q])), query=q)
        pol = o.policy()
        if not oracles:
            e.set_matrices(pol["R"], pol["Rinv"], pol["L"])
        e.set_policy(q, pol["params_all"], pol["mincc"])
        oracles[q] = o
    e.begin_solve()
    for o in oracles.values():
        o.begin_solve()
    rng = np.random.default_rng(8)
    hits = 0
    for it in range(3):
        eps = rng.standard_normal((Q, e.next_num_generated(), D, T))
        cost, valid, _ = e.iterate(it, epsilon=eps)
        verdicts, probs, params = e.tensor("verdicts"), e.tensor("probabilities"), e.tensor("parameters")
        total = e.tensor("total_cost")
        for q, o in oracles.items():
            o.iterate(it, epsilon=eps[q])
            np.testing.assert_array_equal(verdicts[q].astype(bool), o.field("state_costs") > 0.5)
            hits += int(verdicts[q].sum())
            np.testing.assert_allclose(total[q], o.field("total_cost"), rtol=1e-9)
            np.testing.assert_allclose(probs[q], o.field("probabilities"), rtol=1e-9, atol=1e-300)
            np.testing.assert_allclose(params[q], o.parameters(), rtol=1e-9, atol=1e-12)
            nl = o.noiseless()
            np.testing.assert_allclose(cost[q], nl["total_cost"], rtol=1e-9)
            assert bool(valid[q]) == nl["valid"]
    assert hits > 0         # the verdicts compared include collisions


@pytest.mark.gpu
def test_static_spheres_follow_their_scene():
    pb = _mixed()
    D = pb.chain.num_dimensions
    probe = binding.engine_for_problem(_uniform(pb, 0))
    centre0 = probe.sphere_centres(np.zeros(D))[0, 0]          # a sphere on the first joint's axis: static
    probe.close()
    blocker = (0, np.asarray(centre0, dtype=np.float64), np.array([0.05, 0.0, 0.0]))

    def with_blocker(sdf):
        out = copy.copy(sdf)
        out.obstacles = list(sdf.obstacles) + [blocker]
        return out

    clean = list(pb.scenes)
    blocked = copy.copy(pb)
    blocked.scenes = [clean[0], with_blocker(clean[1]), clean[2]]
    e = _engine(blocked)
    assert "stomp_b200_static_spheres" in e.state_kernel_source()

    def all_hit():
        e.begin_solve()
        e.iterate(0)
        v = e.tensor("verdicts")
        return np.array([bool(v[q].all()) for q in range(pb.num_queries)])

    np.testing.assert_array_equal(all_hit(), pb.query_scene == 1)
    # move the obstacle to scene 2: the effect moves with it
    e.select_scene(1)
    e.set_sdf(clean[1])
    e.select_scene(2)
    e.set_sdf(with_blocker(clean[2]))
    _reset_policies(e, pb)
    np.testing.assert_array_equal(all_hit(), pb.query_scene == 2)


@pytest.mark.gpu
@pytest.mark.parametrize("graph", ["2", "0"])
def test_scene_rebuilds_and_reassignments_between_solves_equal_a_fresh_engine(monkeypatch, graph):
    monkeypatch.setenv("STOMP_B200_GRAPH", graph)
    pb = _mixed()
    e = _engine(pb)
    _solve(e)
    # rebuild scene 1 with other obstacles
    rebuilt = copy.copy(pb)
    rebuilt.scenes = list(pb.scenes)
    rebuilt.scenes[1] = P.make_sdf(48, P.make_obstacles(seed=901), lazy=True)
    e.select_scene(1)
    e.set_sdf(rebuilt.scenes[1])
    _reset_policies(e, pb)
    got = _solve(e)
    fresh = _engine(rebuilt)
    want = _solve(fresh)
    for key in want:
        np.testing.assert_array_equal(got[key], want[key], err_msg=f"rebuild {key}")
    # reassign the queries
    moved = copy.copy(rebuilt)
    moved.query_scene = ((np.arange(pb.num_queries) + 1) % 3).astype(np.int32)
    e.set_query_scenes(0, moved.query_scene)
    _reset_policies(e, pb)
    got = _solve(e)
    want = _solve(_engine(moved))
    for key in want:
        np.testing.assert_array_equal(got[key], want[key], err_msg=f"reassign {key}")
    if graph == "2":
        assert e.graph_replays() > 0


@pytest.mark.gpu
def test_query_shards_on_one_device_equal_the_unsharded_mixed_batch():
    pb = _mixed(Q=9)
    want = _solve(_engine(pb))
    parts = []
    for rank in range(2):
        e = _engine(pb, world_size=2, rank=rank, shard_mode=1)
        assert e.Q < pb.num_queries
        parts.append(_solve(e))
        e.close()
    for key in want:
        np.testing.assert_array_equal(np.concatenate([p[key] for p in parts]), want[key], err_msg=key)


@pytest.mark.gpu
def test_missing_fields_and_bad_arguments_are_reported():
    pb = _mixed()
    e = _engine(pb)
    Q = e.Q

    def code(fn, *args):
        with pytest.raises(binding.StompB200Error) as err:
            fn(*args)
        return err.value.code, str(err.value)

    assert code(e.set_query_scenes, Q - 1, [0, 0])[0] == ERR_INVALID_ARGUMENT      # past the last query
    assert code(e.set_query_scenes, -1, [0])[0] == ERR_INVALID_ARGUMENT
    assert code(e.set_query_scenes, 0, [-1])[0] == ERR_INVALID_ARGUMENT            # negative scene
    assert code(e.set_query_scenes, 0, [3])[0] == ERR_INVALID_ARGUMENT             # a scene that does not exist
    assert code(e.select_scene, 5)[0] == ERR_INVALID_ARGUMENT                      # sparse index
    assert code(e.select_scene, -1)[0] == ERR_INVALID_ARGUMENT
    e.select_scene(3)                                                              # a new, empty scene
    e.set_query_scenes(5, [3])
    rc, text = code(e.begin_solve)
    assert rc == ERR_NOT_READY and "query 5" in text and "scene 3" in text
    e.set_query_scenes(5, [pb.query_scene[5]])
    e.begin_solve()
    e.set_query_scenes(2, [3])                                                     # after begin_solve: solve refuses
    rc, text = code(e.solve, 4)
    assert rc == ERR_NOT_READY and "query 2" in text and "scene 3" in text
    assert code(e.run, 0, 1)[0] == ERR_NOT_READY
    assert code(e.iterate, 0)[0] == ERR_NOT_READY
    assert code(e.evaluate_states, np.zeros((1, pb.chain.num_dimensions, 4)))[0] == ERR_NOT_READY   # scene 3 is selected
    # evaluate_states reads the selected scene: the states of a one-scene engine with that field
    rng = np.random.default_rng(2)
    theta = rng.uniform(-2.0, 2.0, size=(16, pb.chain.num_dimensions, 30))
    for s in (2, 0, 1):
        e.select_scene(s)
        one = binding.engine_for_problem(_uniform(pb, s))
        got, want = e.evaluate_states(theta), one.evaluate_states(theta)
        for a, b in zip(got, want):
            np.testing.assert_array_equal(a, b)
        grid, origin, voxel = e.get_sdf()
        np.testing.assert_array_equal(grid, one.get_sdf()[0])
        assert voxel == one.get_sdf()[2]
        one.close()
