"""The control-cost operator (K5 / K6: computeControlCosts, the per-rollout sums C_d and the n^T R n of the noise adaptation)
on every row kernel and every caller, for derivative weights beyond the acceleration rule, against oracle/numpy_ref.py's
Policy(...).control_costs, which takes any derivative weights.

Each case states the row kernel and the generate shape it is meant to reach, restated from the weights, T and N the way
engine.cu's rows_shape / generate_shape decide, and asserts that the restatement agrees.  Then, per iteration:
  - the per-time-step control costs (padding rows folded in) against NumPy at the bar of _assert_control_costs;
  - the sums C_d (cumulative costs minus the state-cost row sum) at 1e-9;
  - the noise-less control costs (the updated parameters, zero noise);
  - with noise adaptation, sigma after the iteration, which carries n^T R n, within test_update_stage.py's bound."""
import numpy as np
import pytest

from motion_planners_b200 import binding, problems as P
from oracle import numpy_ref
from test_gpu_parity import RTOL, _assert_control_costs
from test_update_stage import _banded, _excess, _sms, host_chunk, reference, sigma_bound, weight_blocks

pytestmark = pytest.mark.gpu

ACC, VEL, JERK, MIXED = (0.0, 0.0, 1.0, 0.0), (0.0, 1.0, 0.0, 0.0), (0.0, 0.0, 0.0, 1.0), (0.0, 1.0, 0.5, 0.1)


def rows_kernel(weights, T, R, adapt=True):
    """engine.cu rows_shape + launch_rows: which row kernel serves the operator."""
    N = T + 2 * numpy_ref.PAD
    active = [r for r in range(4) if weights[r] != 0.0]
    bw = max(abs(i - j) for i, j in zip(*np.nonzero(R)))
    toeplitz = all(np.all(np.diag(R, o) == R[0, o]) for o in range(bw + 1))
    if not (len(active) == 1 and (toeplitz or not adapt) and T % 2 == 0 and N >= 12):
        return "generic"
    taps = numpy_ref.RULES[active[0]]
    if taps[0] != 0.0 or taps[6] != 0.0 or bw > 4:
        return "window"
    return "tile" if -(-N // 16) <= 14 else "fast<true,true>"


def generate_shape(noise, kernel, debug, projection):
    """engine.cu generate_shape: (sampler, the row work after it)."""
    sampler = {"unit": "shift", "epsilon": "contraction", "philox": "recurrence"}[noise]
    if projection:
        return sampler, "projection"
    if sampler == "recurrence" and kernel == "tile":
        return sampler, "store" if debug else "none"
    return sampler, "rows"


class Case:
    def __init__(self, name, weights, T, kernel, shape, *, noise="philox", debug=True, projection=False, reuse=False,
                 cumulative=True, K=24):
        self.name, self.weights, self.T, self.kernel, self.shape = name, weights, T, kernel, shape
        self.noise, self.debug, self.projection, self.reuse, self.cumulative, self.K = noise, debug, projection, reuse, cumulative, K


CASES = [
    Case("acc-T40-philox-fused-store", ACC, 40, "tile", ("recurrence", "store")),
    Case("acc-T40-unit-shift-tile", ACC, 40, "tile", ("shift", "rows"), noise="unit"),
    Case("acc-T256-eps-contraction-fast17", ACC, 256, "fast<true,true>", ("contraction", "rows"), noise="epsilon"),
    Case("acc-T41-generic", ACC, 41, "generic", ("recurrence", "rows")),
    Case("velocity-T40-unit-tile", VEL, 40, "tile", ("shift", "rows"), noise="unit"),
    Case("jerk-T40-window", JERK, 40, "window", ("recurrence", "rows")),
    Case("mixed-T40-generic", MIXED, 40, "generic", ("recurrence", "rows")),
    Case("acc-T40-projection", ACC, 40, "tile", ("recurrence", "projection"), projection=True),
    Case("acc-T40-reuse", ACC, 40, "tile", ("recurrence", "store"), reuse=True),
    Case("mixed-T40-reuse", MIXED, 40, "generic", ("recurrence", "rows"), reuse=True),
    Case("mixed-T40-lean", MIXED, 40, "generic", ("recurrence", "rows"), debug=False),
    Case("mixed-T40-lean-generic-states", MIXED, 40, "generic", ("recurrence", "rows"), debug=False),
    Case("jerk-T40-per-time-step", JERK, 40, "window", ("recurrence", "rows"), cumulative=False),
]


def _run(case, sms):
    T, K = case.T, case.K
    pb = P.single_arm_problem(K=K, T=T, sdf_n=64)
    D = pb.chain.num_dimensions
    kw = dict(min_rollouts=(2 * K) // 3, max_rollouts=K, per_iteration=(2 * K) // 3) if case.reuse else {}
    e = binding.engine_for_problem(pb, derivative_weights=case.weights, keep_debug_tensors=case.debug,
                                   use_projection=case.projection, use_cumulative_costs=case.cumulative, **kw)
    pol = e.policy
    assert rows_kernel(case.weights, T, pol["R"]) == case.kernel, case.name
    assert generate_shape(case.noise, case.kernel, case.debug, case.projection) == case.shape, case.name
    pad = numpy_ref.PAD
    ref_pol = numpy_ref.Policy(T, D, pb.movement_duration, e.tensor("parameters_all")[0], case.weights)
    weight = e.cfg.control_cost_weight
    band, bw = _banded(pol["R"])
    S = e.cfg.max_rollouts + 1
    chunk = host_chunk(S, D, 1, sms)
    sigma_min = np.asarray([e.cfg.noise_min_stddev[d] for d in range(D)])
    rng = np.random.default_rng(700 + T)
    e.begin_solve()
    nl_state = None
    for it in range(3):
        theta_all = e.tensor("parameters_all")[0]
        theta = theta_all[:, pad:pad + T]
        if it == 0:
            sigma_before = np.asarray([e.cfg.noise_stddev[d] * e.cfg.noise_decay[d] ** (it - 1) for d in range(D)])
        else:
            sigma_before = e.tensor("stddevs")[0]
        gen = e.next_num_generated()
        nkw = {}
        if case.noise == "unit":
            nkw["noise"] = np.einsum("tu,kdu->kdt", pol["L"], rng.standard_normal((gen, D, T)))[None]
        elif case.noise == "epsilon":
            nkw["epsilon"] = rng.standard_normal((1, gen, D, T))
        e.iterate(it, **nkw)
        kp, _ = e.num_rollouts()
        nl_slot = kp - 1 if it > 0 else -1          # the noise-less rollout of theta joins as the last slot from iteration 1 on
        live = kp - (1 if nl_slot >= 0 else 0)
        if case.debug:
            noise = e.tensor("noise")[0]
        else:
            noise = e.tensor("rollouts")[0] - theta[None]
            if nl_slot >= 0:
                noise[nl_slot] = 0.0
        cc_noise = e.tensor("noise_projected")[0] if case.projection else noise    # the control costs see parameters + M noise
        want = ref_pol.control_costs(theta[None] + cc_noise[:live], weight)
        if case.debug:
            _assert_control_costs(e.tensor("control_costs")[0][:live], want)
        if case.cumulative:
            # C_d = cumulative - sum_t state; the subtraction itself may round by an ulp of the cumulative cost
            cum = e.tensor("cumulative_costs")[0]
            st = e.tensor("state_costs")[0][:kp].sum(-1)
            C_want = want.sum(-1)
            if nl_slot >= 0:
                st[nl_slot] = nl_state.sum()
                C_want = np.concatenate([C_want, ref_pol.control_costs(theta[None], weight).sum(-1)])
            got = cum - st[:, None]
            np.testing.assert_allclose(got, C_want, rtol=RTOL, atol=4 * np.finfo(float).eps * np.abs(cum).max())
            if e.cfg.use_noise_adaptation:
                c = e.tensor("full_costs")[0]
                ref = reference(c, noise[:kp], band, theta, sigma_before, sigma_min, True)
                parts = -(-kp // chunk) + weight_blocks(kp)
                r = _excess(e.tensor("stddevs")[0], ref["sigma"], sigma_bound(ref, parts, T, bw))
                assert r <= 1, f"{case.name} iteration {it}: stddevs {r:.3g}x over the bound"
        nl_state = e.tensor("noiseless_state_costs")[0]
        if case.debug or case.kernel == "generic":      # the lean loop with one rule keeps the noise-less sums only
            params = e.tensor("parameters")[0]
            _assert_control_costs(e.tensor("noiseless_control_costs")[0], ref_pol.control_costs(params, weight))
    e.close()


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_control_cost_rows_match_numpy(case, monkeypatch):
    if case.name.endswith("generic-states"):
        # the noise-less rollout as a state pass + noiseless_rollout_kernel instead of the update kernel's last CTA
        monkeypatch.setenv("STOMP_B200_STATES", "generic")
    _run(case, _sms())
