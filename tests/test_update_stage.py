"""The weights/update stage (K7-K9: min / max cost normalisation, exponential weights, the probability-weighted noise sum,
noise adaptation and the parameter step; PolicyImprovement.cpp:497-711, CovariantMovementPrimitive.cpp:476-479) against
a plain extended-precision restatement of the same operation, fed with the engine's own per-iteration read-backs.

The inputs the stage consumes are read back and taken as exact: the full costs c[k, d], the noise n[k, d, t] (the `noise`
tensor where the engine keeps it, else rollouts - theta in double: the subtraction the update kernel does itself on the
shipped path), theta and sigma before the iteration, and R of the policy.  The outputs (probabilities, updates,
parameters, stddevs) must lie within rounding-error bounds derived below, not within a flat tolerance: dropping one
rollout of K' shifts an update by about 1 / K' of its scale, far above any of these bounds.

Every case states the chunk size the host picks (rollouts per CTA of the update kernels), the rows of the last chunk, the
update shape (fused lean, fused with debug tensors, separate kernels, profiled, rollout reuse, per-time-step costs) and
the cost-spread regime it is meant to reach, and asserts that it reaches them."""
import dataclasses
import os

import numpy as np
import pytest

from motion_planners_b200 import binding, problems as P

pytestmark = pytest.mark.gpu

U = 2.0 ** -53            # unit roundoff of FP64
H = 10.0                  # cost_scaling_h (PolicyImprovement.cpp:55, the engine's default)
CLAMP = 1e-8              # den = max(max - min, 1e-8) (PolicyImprovement.cpp:514-516)

# Timeline slots (kernels.cuh: TimelineScope) of the update stage's kernels: rollout_weights_kernel, the update kernel
# (weights_update_kernel or weighted_update_kernel), apply_update_kernel.
TL_WEIGHTS, TL_UPDATE, TL_APPLY = 2, 3, 4


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def host_chunk(S, D, Q, sms):
    """Rollouts per CTA of the update kernels, as stomp_b200_create picks it (engine.cu, "rollouts per CTA of the
    weights / update kernels"): halve 128 while the grid of the halved chunk still fits three CTAs per SM.  S = slots =
    max_rollouts + 1."""
    chunk = 128
    while chunk > 32 and -(-S // (chunk // 2)) * D * Q <= 3 * sms:
        chunk //= 2
    return chunk


def slots_for(chunk, nk, D, Q, sms, min_chunks=3):
    """The smallest S = K' with at least min_chunks chunks for which the host picks `chunk` and the last chunk has nk rows."""
    m = min_chunks
    while True:
        S = (m - 1) * chunk + nk
        if host_chunk(S, D, Q, sms) == chunk:
            return S
        if S > 1 << 16:
            raise AssertionError(f"no K' lands in chunk {chunk} on {sms} SMs")
        m += 1


def weight_blocks(n):
    """rollout_weights_kernel's CTAs per joint (engine.cu launch_update_stage: kWeightThreads = 512, at most 8)."""
    return max(1, min(8, -(-n // 512)))


# ---- the reference ---------------------------------------------------------------------------------------------------
def _banded(R):
    """The diagonals of the banded R: {offset: R[i, i + offset]}."""
    T = R.shape[0]
    bw = max(abs(i - j) for i, j in zip(*np.nonzero(R)))
    return {o: np.array([R[i, i + o] for i in range(max(0, -o), T - max(0, o))], dtype=np.longdouble)
            for o in range(-bw, bw + 1)}, bw


def _quad(n, band):
    """q = n^T R n and its cancellation companion |n|^T |R| |n| per row, in long double; n [..., T]."""
    T = n.shape[-1]
    Rn = np.zeros_like(n)
    aRn = np.zeros_like(n)
    an = np.abs(n)
    for o, dg in band.items():
        lo, hi = max(0, -o), T - max(0, o)
        Rn[..., lo:hi] += dg * n[..., lo + o:hi + o]
        aRn[..., lo:hi] += np.abs(dg) * an[..., lo + o:hi + o]
    return (n * Rn).sum(-1), (an * aRn).sum(-1)


def _weights(c, axis):
    """exp(-h (c - min) / den) with den = max(max - min, 1e-8); min / max over `axis`; long double."""
    mn = c.min(axis=axis, keepdims=True)
    mx = c.max(axis=axis, keepdims=True)
    den = np.maximum(mx - mn, np.longdouble(CLAMP))
    return np.exp(-np.longdouble(H) * (c - mn) / den), (mx - mn)


def reference(c, n, band, theta, sigma, sigma_min, adapt, pt_costs=None):
    """oracle/numpy_ref.py:238-253 in long double.  c [K', D] full costs, n [K', D, T] noise, theta [D, T], sigma [D].
    pt_costs [K', D, T]: per-time-step costs (setCostCumulation(false)); the update then weighs per time step."""
    ld = np.longdouble
    T = n.shape[-1]
    cl, nl_ = c.astype(ld), n.astype(ld)
    w, spread = _weights(cl, axis=0)
    Pf = w / w.sum(0)                                         # full_probabilities_ [K', D]
    if pt_costs is None:
        Pu = Pf[:, :, None]
    else:
        wt, _ = _weights(pt_costs.astype(ld), axis=(0, 2))
        Pu = wt / wt.sum(0)                                   # probabilities_ per time step [K', D, T]
    u = (Pu * nl_).sum(0)
    scale = (Pu * np.abs(nl_)).sum(0)                         # sum_k P |n|: the scale of the update's rounding
    out = dict(P=Pf, Pt=None if pt_costs is None else Pu, u=u, scale=scale, spread=spread[0].astype(np.float64),
               theta=theta.astype(ld) + u)
    if adapt:
        q, comp = _quad(nl_, band)
        numer = (Pf * q).sum(0)
        frob = np.sqrt(numer / (Pf.sum(0) * T))
        raw = ld(0.8) * sigma.astype(ld) + ld(0.2) * frob
        out.update(q=q, comp=comp, numer=numer, frob=frob, sigma_raw=raw,
                   sigma=np.maximum(raw, sigma_min.astype(ld)))
    else:
        out["sigma"] = sigma.astype(ld)
    return out


# ---- the bounds ------------------------------------------------------------------------------------------------------
# A weight is exp(a) with a = -h (c - mn) / den, |a| <= h, formed with four roundings of a value <= h: 4 h u absolute in
# a, i.e. relative in exp(a); exp itself adds <= 1 ulp.  The sum of the weights is a positive sum: a tree inside the
# CTA, then `parts` partials (chunks or weight blocks) in order, each step <= u relative.  P = w / sum w doubles the
# weight's share and adds the division:
def prob_bound(parts):
    return 2 * (4 * H + 16 + parts) * U                      # |dP| <= this * P


# The update row adds P n over the rows: at most `rows` of them in sequence per thread (a chunk's rows, or all K' in the
# per-time-step kernel), then the partials of `parts` chunks; each rounding is <= u of the running sum of |P n|, and P
# carries its own relative error:
def update_bound(rows, parts):
    return 2 * (4 * H + 16 + rows + parts) * U               # |du| <= this * sum_k P |n|


# n^T R n on the device is an FMA form of the banded operator summed over T time steps (bandwidth bw): its error is bounded
# by the sum of the magnitudes of its terms, |n|^T |R| |n|, not by q, which cancels.
def quad_bound(T, bw):
    return (T + 2 * bw + 8) * U                               # |dq| <= this * |n|^T |R| |n|


def sigma_bound(ref, parts, T, bw):
    """|d sigma'|: the numerator sum_k P q carries P's relative error and each row's |dq|; the denominator sum_k P is 1 up
    to P's error; the sqrt halves relative errors; 0.8 sigma + 0.2 frob adds a few roundings of sigma'."""
    gP = prob_bound(parts)
    numer = np.asarray(ref["numer"], dtype=np.float64)
    dnumer = gP * numer + np.asarray((ref["P"] * ref["comp"]).sum(0), dtype=np.float64) * quad_bound(T, bw)
    with np.errstate(divide="ignore", invalid="ignore"):
        rel = np.where(numer > 0, dnumer / numer, 0.0)
    frob = np.asarray(ref["frob"], dtype=np.float64)
    rel_frob = 0.5 * (rel + gP + 4 * U) + 2 * U
    return 0.2 * frob * rel_frob + 4 * U * np.asarray(ref["sigma"], dtype=np.float64)


def _excess(got, want, bound):
    """max of |got - want| / bound (<= 1 passes); long double difference."""
    err = np.abs(got.astype(np.longdouble) - want)
    b = np.asarray(bound, dtype=np.longdouble)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0, 0.0, err / b)
    return float(np.max(r)) if r.size else 0.0


def check_iteration(tag, ref, got, *, rows, parts, T, bw, adapt):
    """Every output of the stage against the reference within its bound."""
    fails = []
    r = _excess(got["P"], ref["P"], prob_bound(parts) * ref["P"])
    if r > 1: fails.append(f"full probabilities {r:.3g}x over the bound")
    if ref["Pt"] is not None:
        r = _excess(got["Pt"], ref["Pt"], prob_bound(parts) * ref["Pt"])
        if r > 1: fails.append(f"per-time-step probabilities {r:.3g}x over the bound")
    ub = update_bound(rows, parts) * ref["scale"]
    r = _excess(got["u"], ref["u"], ub)
    if r > 1: fails.append(f"updates {r:.3g}x over the bound")
    r = _excess(got["theta"], ref["theta"], ub + U * np.abs(ref["theta"]))
    if r > 1: fails.append(f"parameters {r:.3g}x over the bound")
    if adapt:
        r = _excess(got["sigma"], ref["sigma"], sigma_bound(ref, parts, T, bw))
        if r > 1: fails.append(f"stddevs {r:.3g}x over the bound")
    else:
        if not np.array_equal(got["sigma"], np.asarray(ref["sigma"], dtype=np.float64)):
            fails.append("stddevs changed without noise adaptation")
    assert not fails, f"{tag}: " + "; ".join(fails)


# ---- driving the engine ----------------------------------------------------------------------------------------------
class Case:
    def __init__(self, name, *, chunk, nk, T, shape, K=None, inject=None, adapt=True, min_stddev=None, reuse=False,
                 wblocks=None, regime=None, Q=1):
        self.name, self.chunk, self.nk, self.T, self.shape = name, chunk, nk, T, shape
        self.K, self.inject, self.adapt, self.min_stddev, self.reuse = K, inject, adapt, min_stddev, reuse
        self.wblocks, self.regime, self.Q = wblocks, regime, Q


# shape: "lean" (weights_update_kernel, no debug tensors, on-device sampler: the kernel forms noise = rollout - theta),
# "debug" (weights_update_kernel, debug tensors), "unfused" (STOMP_B200_FUSE_WEIGHTS=0: rollout_weights_kernel ->
# weighted_update_kernel, apply on its last chunk CTA), "profiled" (the same with apply_update_kernel split off),
# "reuse" (separate kernels with reused rollouts), "pertimestep" (setCostCumulation(false)).
# nk: rows of the last chunk at K' = K + 1 (the noise-less rollout joins from the second iteration on): 1, 30, 31, 32, 33,
# chunk - 1 and chunk are the edges of stream_chunk's 16-load body (its two halves start at rows 0 and 1).
# inject: None (on-device sampler), "gauss" (L eps), "zero" (spread exactly 0), "clamp" / "narrow" (spread < 1e-8 /
# in [1e-8, 1e-6], with duplicated rows tied at the minimum).
CASES = [
    Case("lean-c32-nk1-T40", chunk=32, nk=1, T=40, shape="lean"),
    Case("lean-c32-nk30-T128", chunk=32, nk=30, T=128, shape="lean"),
    Case("lean-c32-nk31-T130", chunk=32, nk=31, T=130, shape="lean"),
    Case("lean-c32-nk32-T256", chunk=32, nk=32, T=256, shape="lean"),
    Case("lean-c64-nk33-T40", chunk=64, nk=33, T=40, shape="lean"),
    Case("lean-c64-nk63-T130", chunk=64, nk=63, T=130, shape="lean"),
    Case("lean-c64-nk64-T128", chunk=64, nk=64, T=128, shape="lean"),
    Case("lean-c128-nk1-T40", chunk=128, nk=1, T=40, shape="lean"),
    Case("lean-c128-nk127-T256", chunk=128, nk=127, T=256, shape="lean"),
    Case("lean-c128-nk128-T40-noadapt", chunk=128, nk=128, T=40, shape="lean", adapt=False),
    Case("lean-c32-nk32-T128-minstd", chunk=32, nk=32, T=128, shape="lean", min_stddev="split"),
    Case("debug-c32-nk31-T40-gauss", chunk=32, nk=31, T=40, shape="debug", inject="gauss"),
    Case("debug-c64-nk32-T256-gauss", chunk=64, nk=32, T=256, shape="debug", inject="gauss"),
    Case("debug-c32-nk30-T40-zero", chunk=32, nk=30, T=40, shape="debug", inject="zero", regime="zero"),
    Case("debug-c64-nk33-T40-clamp", chunk=64, nk=33, T=40, shape="debug", inject="clamp", regime="clamp"),
    Case("injected-c64-nk31-T40-narrow", chunk=64, nk=31, T=40, shape="injected", inject="narrow", regime="narrow"),
    Case("unfused-c32-nk1-T40-w1", chunk=32, nk=1, T=40, shape="unfused", K=480, wblocks=1),
    Case("unfused-c32-nk31-T130-w3", chunk=32, nk=31, T=130, shape="unfused", K=1054, wblocks=3),
    Case("unfused-c128-nk33-T40-w8", chunk=128, nk=33, T=40, shape="unfused", wblocks=8),
    Case("profiled-c64-nk63-T40", chunk=64, nk=63, T=40, shape="profiled"),
    Case("reuse-c32-nk32-T40", chunk=32, nk=32, T=40, shape="reuse", reuse=True),
    Case("pertimestep-c128-nk1-T40", chunk=128, nk=1, T=40, shape="pertimestep", inject="gauss"),
]


def _make_engine(case, K, sms, extra_env=None, **kw):
    T = case.T
    pb = P.single_arm_problem(K=K, T=T, sdf_n=64)
    D = pb.chain.num_dimensions
    ekw = dict(use_noise_adaptation=case.adapt, keep_debug_tensors=case.shape in ("debug", "pertimestep"))
    if case.shape == "pertimestep":
        ekw["use_cumulative_costs"] = False
    if case.min_stddev == "split":      # binds on the even joints (above any sigma' this scene reaches), not on the odd ones
        ekw["noise_min_stddev"] = [0.6 if d % 2 == 0 else 1e-6 for d in range(D)]
    ekw.update(kw)
    old = os.environ.get("STOMP_B200_FUSE_WEIGHTS")
    if case.shape == "unfused":
        os.environ["STOMP_B200_FUSE_WEIGHTS"] = "0"
    try:
        e = binding.engine_for_problem(pb, **ekw)
    finally:
        if old is None:
            os.environ.pop("STOMP_B200_FUSE_WEIGHTS", None)
        else:
            os.environ["STOMP_B200_FUSE_WEIGHTS"] = old
    if case.shape == "profiled":
        e.set_profiling(True)
    e.set_timeline(True)
    return e, pb


def _expected_timeline(shape):
    """Which of (rollout_weights_kernel, update kernel, apply_update_kernel) run in each update shape."""
    return {"lean": (False, True, False), "debug": (False, True, False), "injected": (False, True, False),
            "unfused": (True, True, False), "reuse": (True, True, False), "profiled": (True, True, True),
            "pertimestep": (True, False, True)}[shape]


def _readback(e, lean):
    """What the stage consumed and produced in the last iteration, as the engine reports it."""
    out = dict(c=e.tensor("full_costs"), P=e.tensor("full_probabilities"), u=e.tensor("updates"),
               theta=e.tensor("parameters"), sigma=e.tensor("stddevs"))
    if lean:
        with pytest.raises(binding.StompB200Error) as err:      # the shipped path does not materialise noise_
            e.tensor("noise")
        assert err.value.code != binding.OK
        out["rollouts"] = e.tensor("rollouts")
    else:
        out["noise"] = e.tensor("noise")
    return out


def _noise_of(rb, theta_before, noiseless_slot, lean):
    """n [Q, K', D, T]: the noise tensor, or rollouts - theta (the subtraction weights_update_kernel does) with the
    noise-less slot's zero noise."""
    if not lean:
        return rb["noise"]
    n = rb["rollouts"] - theta_before[:, None]
    if noiseless_slot >= 0:
        n[:, noiseless_slot] = 0.0
    return n


def _unit_noise(pol, K, D, T, rng, kind, scale):
    """Injected unit noise [1, K, D, T]: scale[d] L eps, with rows 0..3 zero and rows 9..12 copies of row 8 (exact ties)."""
    eps = rng.standard_normal((K, D, T))
    unit = np.einsum("tu,kdu->kdt", pol["L"], eps) * np.asarray(scale)[None, :, None]
    if kind == "zero":
        unit[:] = 0.0
    elif kind in ("clamp", "narrow"):
        unit[:4] = 0.0
        unit[9:13] = unit[8]
    return unit[None]


def _scales_for(case, K, sms, pol, D, T, target):
    """Per-joint noise scales that put the spread of the full costs near `target`: the control cost is quadratic in the
    noise about the minimum-control-cost start, so one trial run at scale s0 gives s = s0 sqrt(target / spread)."""
    s = np.full(D, 1e-3)
    for _ in range(2):      # a second round absorbs what is not quadratic
        e, _ = _make_engine(case, K, sms)
        e.begin_solve()
        e.iterate(0, noise=_unit_noise(pol, K, D, T, np.random.default_rng(5), case.inject, s))
        c = e.tensor("full_costs")[0]
        e.close()
        spread = c.max(0) - c.min(0)
        assert np.all(spread > 0)
        s = s * np.sqrt(target / spread)
    return s


def _regime(spread):
    if np.all(spread == 0):
        return "zero"
    if np.all((spread > 0) & (spread < CLAMP)):
        return "clamp"
    if np.all((spread >= CLAMP) & (spread <= 1e-6)):
        return "narrow"
    return "wide"


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_update_stage_within_rounding_bounds(case):
    assert np.finfo(np.longdouble).nmant >= 63, "the reference needs an extended-precision long double"
    sms = _sms()
    D, Q = 7, 1
    if case.reuse:
        # rollout reuse (min < max): 2/3 of the slots generated per iteration, the rest reused from the last one
        S = slots_for(case.chunk, case.nk, D, Q, sms)
        K = S - 1
        per_it = (2 * K) // 3
        kw = dict(min_rollouts=per_it, max_rollouts=K, per_iteration=per_it)
    else:
        S = case.K + 1 if case.K else slots_for(case.chunk, case.nk, D, Q, sms)
        K = S - 1
        kw = {}
    chunk = host_chunk(S, D, Q, sms)
    assert chunk == case.chunk, f"K' = {S} gives chunk {chunk}, not {case.chunk} on {sms} SMs"
    nk = S - (-(-S // chunk) - 1) * chunk
    assert nk == case.nk, f"K' = {S} leaves {nk} rows in the last chunk, not {case.nk}"
    T = case.T
    lean = case.shape == "lean"

    def build():
        if not case.reuse:
            return _make_engine(case, K, sms)
        pb = P.single_arm_problem(K=K, T=T, sdf_n=64)
        e = binding.engine_for_problem(pb, use_noise_adaptation=case.adapt, **kw)
        e.set_timeline(True)
        return e, pb

    e, pb = build()
    pol = e.policy
    band, bw = _banded(pol["R"])
    gen = kw.get("per_iteration", K)
    scale = np.ones(D)
    if case.inject in ("clamp", "narrow"):
        scale = _scales_for(case, K, sms, pol, D, T, 1e-9 if case.inject == "clamp" else 1e-7)
    sigma_min = np.asarray([e.cfg.noise_min_stddev[d] for d in range(D)])
    rng = np.random.default_rng(11)
    e.begin_solve()
    regimes = []
    for it in range(2):
        theta_before = e.tensor("parameters")
        if it == 0 or not case.adapt:      # set by value at the start of the iteration (Stomp.cpp:179)
            sigma_before = np.asarray([e.cfg.noise_stddev[d] * e.cfg.noise_decay[d] ** (it - 1) for d in range(D)])[None]
        else:
            sigma_before = e.tensor("stddevs")
        noise = None if case.inject is None else _unit_noise(pol, gen, D, T, rng, case.inject, scale)
        e.iterate(it, noise=noise)
        kp, _ = e.num_rollouts()                      # K'
        nl_slot = kp - 1 if it > 0 else -1            # the noise-less rollout joins as the last slot from iteration 1 on
        if it == 1:
            assert kp == S
        # the update shape, from the kernels that ran
        tl = e.timeline(4)[-1]
        ran = tuple(bool(tl[k, 1] >= 0) for k in (TL_WEIGHTS, TL_UPDATE, TL_APPLY))
        assert ran == _expected_timeline(case.shape), f"{case.name}: kernels that ran {ran}"
        wblocks = weight_blocks(kp) if ran[0] else 1
        if case.wblocks is not None and it == 1:
            assert wblocks == case.wblocks
        nchunks = -(-kp // chunk)
        rb = _readback(e, lean)
        n = _noise_of(rb, theta_before, nl_slot, lean)[0]
        c = rb["c"][0]
        pt = None
        got_pt = None
        if case.shape == "pertimestep":
            pt = e.tensor("state_costs")[0][:, None, :] + e.tensor("control_costs")[0]     # 1.0 * (st + cc), FP64
            got_pt = e.tensor("probabilities")[0]
        ref = reference(c, n, band, theta_before[0], sigma_before[0], sigma_min, case.adapt, pt_costs=pt)
        regimes.append(_regime(ref["spread"]))
        if it == 0 and case.regime is not None:
            assert regimes[0] == case.regime, f"{case.name}: spread {ref['spread']} is not in the {case.regime} regime"
        if case.min_stddev == "split" and it == 0:
            binds = np.asarray(ref["sigma_raw"] < sigma_min)
            assert binds.any() and not binds.all(), f"the sigma clamp binds on joints {binds}"
        got = dict(P=rb["P"][0], Pt=got_pt, u=rb["u"][0], theta=rb["theta"][0], sigma=rb["sigma"][0])
        if case.shape == "pertimestep":
            rows, parts = kp, kp + wblocks                 # sequential sums over all K' rollouts per time step
        else:
            rows, parts = chunk, nchunks + wblocks
        check_iteration(f"{case.name} iteration {it}", ref, got, rows=rows, parts=parts, T=T, bw=bw, adapt=case.adapt)
        # exact checks where the arithmetic allows them
        if case.inject == "zero" and it == 0:
            assert np.all(got["P"] == 1.0 / kp)
        if case.inject in ("clamp", "narrow"):
            gen_rows = slice(0, gen)
            Pg = got["P"][gen_rows]
            for group in (range(0, 4), range(8, 13)):
                g0 = group[0]
                assert np.all(c[list(group)] == c[g0]), "identical noise rows must cost the same"
                assert np.all(Pg[list(group)] == Pg[g0]), "identical noise rows must weigh the same"
            if it == 0:
                assert np.all(c[0] == c.min(0)), "the zero-noise rows tie at the minimum"
    e.close()
    print(f"{case.name}: K'={S} chunk={chunk} last chunk={nk} wblocks={wblocks} shape={case.shape} T={T} "
          f"spread regimes={regimes}")


def test_batch_with_a_frozen_query():
    """Q = 4 queries at a K' that reaches chunk 128; query 0 starts at its goal, so the stop rule freezes it after its
    first iteration, while the other three cross the blocker of the single-arm scene and stay live.  A frozen query keeps
    its parameters and stddevs bit for bit; the other queries meet the bounds on the following iterations, which shows
    the per-(query, joint) tickets were left at zero by the frozen query's CTAs."""
    assert np.finfo(np.longdouble).nmant >= 63
    sms = _sms()
    D, Q, T = 7, 4, 40
    S = next(s for s in range(600, 1 << 16) if host_chunk(s, D, Q, sms) == 128)
    K = S - 1
    one = P.single_arm_problem(K=K, T=T, sdf_n=64)
    pb = dataclasses.replace(one, start=np.stack([one.start] * Q), goal=np.stack([one.start] + [one.goal] * (Q - 1)),
                             num_queries=Q)
    e = binding.engine_for_problem(pb)
    pol = e.policy
    band, bw = _banded(pol["R"])
    sigma_min = np.asarray([e.cfg.noise_min_stddev[d] for d in range(D)])
    e.begin_solve()
    warm = 2
    e.run(0, warm, honour_stop=True)
    records = []
    for it in range(warm, warm + 2):
        theta_before, sigma_before = e.tensor("parameters"), e.tensor("stddevs")
        e.run(it, 1, honour_stop=True)
        n_all, _ = e.num_rollouts()
        assert n_all == S
        rb = _readback(e, lean=True)
        records.append((theta_before, sigma_before, rb, _noise_of(rb, theta_before, S - 1, True)))
    done = e.finish_solve()
    e.close()
    # iterations[q] counts the iterations query q ran: iteration `it` updated it iff it < iterations[q]
    live = done["iterations"]
    assert live[0] <= warm and done["found"][0], f"query 0 was not frozen before iteration {warm}: {live}"
    assert (live == warm + 2).any()
    chunk = host_chunk(S, D, Q, sms)
    for i, (theta_before, sigma_before, rb, n) in enumerate(records):
        for q in range(Q):
            if warm + i >= live[q]:
                np.testing.assert_array_equal(rb["theta"][q], theta_before[q])
                np.testing.assert_array_equal(rb["sigma"][q], sigma_before[q])
                continue
            ref = reference(rb["c"][q], n[q], band, theta_before[q], sigma_before[q], sigma_min, True)
            got = dict(P=rb["P"][q], Pt=None, u=rb["u"][q], theta=rb["theta"][q], sigma=rb["sigma"][q])
            check_iteration(f"batch query {q} iteration {warm + i}", ref, got, rows=chunk, parts=-(-S // chunk) + 1,
                            T=T, bw=bw, adapt=True)
    print(f"batch: Q={Q} K'={S} chunk={chunk} iterations per query={live.tolist()}")
