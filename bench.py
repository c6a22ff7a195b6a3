#!/usr/bin/env python
"""Benchmark of the STOMP rollout loop (BASELINE.json metric: rollout-timesteps/s and ms/iteration,
K=4096, T=100, 7-DoF, 256^3 SDF, at 1/2/4/8 GPUs).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path through the C ABI
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results as DIR/*.npy

A "step" is one STOMP iteration (Stomp::runSingleIteration): generate K rollouts, cost them, weight them,
update the trajectory, cost the noise-less rollout.  One JSON line is printed by rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "stomp_rollout_timesteps_per_sec"
UNIT = "rollout-timesteps/s"

WORKLOADS = {
    # BASELINE.json configs[2]: the configuration the metric is quoted on; fits one GPU
    "c3": dict(kind="single", K=4096, T=100, sdf_n=256, label="STOMP 7-DoF iiwa, K=4096 rollouts, T=100, 256^3 SDF"),
    "c2": dict(kind="single", K=128, T=100, sdf_n=128, label="STOMP 7-DoF iiwa, K=128 rollouts, T=100, 128^3 SDF"),
    "c4": dict(kind="batch", Q=1024, K=64, T=200, sdf_n=128, label="1024 independent 7-DoF queries, K=64, T=200"),
    "c5": dict(kind="dual", K=2048, T=150, sdf_n=512, label="dual-arm 14-DoF, K=2048, T=150, 512^3 SDF"),
}


def make_problem(name):
    from motion_planners_b200 import problems as P
    w = WORKLOADS[name]
    if w["kind"] == "single":
        return P.single_arm_problem(K=w["K"], T=w["T"], sdf_n=w["sdf_n"])
    if w["kind"] == "batch":
        return P.batch_problem(Q=w["Q"], K=w["K"], T=w["T"], sdf_n=w["sdf_n"])
    return P.dual_arm_problem(K=w["K"], T=w["T"], sdf_n=w["sdf_n"])


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            sm, mx, reasons = [], [], set()
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            if sm:
                out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        finally:
            try:
                os.unlink(self.path)
            except OSError:
                pass
        return out


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local)
        dist_mod.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
        dist = dist_mod
    return rank, world, local, dist


def dist_max(dist, value, local):
    if dist is None:
        return value
    import torch
    t = torch.tensor([value], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def dist_barrier(dist, local):
    if dist is not None:
        import torch
        dist.barrier(device_ids=[local])
        torch.cuda.synchronize(local)


def broadcast_bytes(dist, payload, local):
    if dist is None:
        return payload
    from motion_planners_b200 import sharding
    return sharding.broadcast_bytes(dist, payload, 128, f"cuda:{local}")


# what a caller of stomp_b200_run reads back after a step: the trajectory, its update and noise levels, the noise-less
# rollout's costs, and the rollout-indexed tables of the step (probabilities as full_probabilities: with cumulative costs
# the per-time-step table repeats that value along T)
DUMP_TENSORS = ("parameters", "updates", "stddevs", "noiseless_state_costs", "noiseless_control_costs", "total_cost",
                "cumulative_costs", "full_probabilities", "state_costs", "verdicts", "rollouts")
DUMP_LIMIT_BYTES = 60 << 20          # array data; with the .npy headers the directory stays below 64 MB (64e6 bytes)


def read_outputs(eng):
    """The engine's DUMP_TENSORS as numpy arrays.  In rollout sharding a read-back is collective: every rank calls this,
    and rollouts / state_costs / verdicts are the calling rank's share of the rollouts (their shapes depend on N)."""
    return {name: eng.tensor(name) for name in DUMP_TENSORS}


def dump_outputs(outputs, out_dir):
    """Writes every array as out_dir/<name>.npy (float64; the 0 / 1 verdicts as float32), within DUMP_LIMIT_BYTES in all.
    Smallest first, each array may use an equal share of what the ones before it left; one larger than that keeps a fixed
    sample of its rows (leading two axes flattened, rows drawn with seed 0 and kept in order), so that two builds given
    the same arguments store the same elements.  Returns {name: {"shape", "stored"}}."""
    os.makedirs(out_dir, exist_ok=True)
    left, info = DUMP_LIMIT_BYTES, {}
    for i, name in enumerate(sorted(outputs, key=lambda k: outputs[k].size)):
        a = outputs[name].astype(np.float32 if outputs[name].dtype == np.uint8 else np.float64)
        share = left // (len(outputs) - i)
        full_shape = list(a.shape)
        if a.nbytes > share:
            lead = 2 if a.ndim > 2 else 1
            rows = a.reshape((-1,) + a.shape[lead:])
            keep = max(1, share // (rows[0].nbytes or 1))
            pick = np.sort(np.random.default_rng(0).choice(rows.shape[0], size=min(keep, rows.shape[0]), replace=False))
            a = rows[pick]
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a))
        left -= a.nbytes
        info[name] = {"shape": full_shape, "stored": list(a.shape)}
    return {name: info[name] for name in outputs}


class L2Flusher:
    """Writes a buffer larger than the 126 MB L2 between timed iterations."""

    def __init__(self, local, nbytes=256 << 20):
        import torch
        self.torch = torch
        self.buf = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{local}")
        self.val = 0

    def flush(self):
        self.val = (self.val + 1) % 251
        self.buf.fill_(self.val)
        self.torch.cuda.synchronize()


def reference_kind():
    """"reference": oracle/_ref/libstomp_ref.so is here — the reference's own STOMP core (Stomp.cpp, PolicyImprovement.cpp,
    CovariantMovementPrimitive.cpp, StompUtils.cpp, unmodified) compiled against the Eigen / Boost stand-ins of
    oracle/ref/shim; "port": only the oracle restatement is available."""
    try:
        from oracle import ref_binding
        return "reference" if os.path.exists(ref_binding._LIB_PATH) else "port"
    except Exception:
        return "port"


def cpu_baseline(problem, workload, threads, sample_rollouts, iterations, dense=True):
    """The reference's CPU path on a bounded sample of the workload: same T, D, spheres and SDF, `sample_rollouts`
    rollouts per iteration.  The reference's own code when oracle/_ref is present (state verdicts from the oracle's
    sphere / SDF task in place of the FCL query), else the oracle port.  Timed around the iteration loop, where the
    reference times (MotionPlanners.cpp:506-512); one-time policy setup excluded."""
    from oracle.binding import Oracle
    T, D = problem.num_time_steps, problem.chain.num_dimensions
    o = Oracle(num_time_steps=T, num_dimensions=D, min_rollouts=sample_rollouts, max_rollouts=sample_rollouts,
               num_rollouts_per_iteration=sample_rollouts, noise_stddev=problem.noise_stddev,
               use_openmp=threads > 1, dense_control_costs=dense, seed=42)
    from oracle import binding as ob_
    ob_.set_num_threads(max(1, threads))     # explicit: torchrun exports OMP_NUM_THREADS=1 to its workers
    o.set_problem(problem, query=0)
    states = sample_rollouts * T * iterations
    if reference_kind() == "reference":
        from oracle import ref_binding
        r = ref_binding.Reference(o)
        s, g = problem.start, problem.goal
        if s.ndim == 2:
            s, g = s[0], g[0]
        r.set_start_goal(s, g)
        res = r.solve(iterations, honour_stop=False)
        return states / res["seconds"], res["seconds"]
    res = o.solve(iterations, honour_stop=False)
    return states / res["seconds"], res["seconds"]


def run_reference(args):
    # under torchrun rank 0 alone runs the CPU arm; no process group is needed (or created) for it
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import binding as ob
    problem = make_problem(args.workload)
    w = WORKLOADS[args.workload]
    threads = ob.set_num_threads(ob.host_cores())
    T = problem.num_time_steps
    sample = min(w["K"], args.reference_sample)
    # warm-up + timed steps; every step is one iteration over the bounded sample
    cpu_baseline(problem, args.workload, threads, sample, max(1, args.warmup))
    rate, seconds = cpu_baseline(problem, args.workload, threads, sample, args.steps)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * seconds / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": w["label"], "name": args.workload},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": reference_kind(),
                         "sample": f"{sample} of {w['K']} rollouts per iteration, same T / D / spheres / SDF; "
                                   f"OpenMP over rollouts in Task::execute as the reference (Stomp.cpp:210); dense "
                                   f"O(N^2) control-cost and n^T R n forms kept"},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": ("the reference's own STOMP core (src/planners/stomp/src/*.cpp, unmodified) compiled against Eigen / Boost "
                 "stand-ins (oracle/ref); the FCL state query, whose libraries are not in this image, is replaced by the "
                 "same sphere-vs-SDF task the CUDA path evaluates; the Eigen stand-in is an unvectorised eager "
                 "implementation, so a build against real Eigen would be faster" if reference_kind() == "reference" else
                 "oracle port of the reference's algorithm (oracle/_ref was not built: /root/reference absent at build time)"),
    }
    print(json.dumps(line), flush=True)


def sharded_parity_check(problem, shard_mode, world, rank, local, dist, iterations=3):
    """N > 1 only: the sharded run against a single-GPU run of the same problem on this rank's GPU, before anything is
    timed.  Rollout sharding: same Philox samples by construction (the counters use the global rollout index), so the
    local verdicts / rollouts are the matching slice of the single-GPU ones and the rollout-indexed tables, the update
    and the parameters agree within 1e-9.  Query sharding: bit for bit.  Returns (ok, detail); all ranks agree on ok."""
    import numpy as np
    from motion_planners_b200 import binding, problems as P, sharding
    ok, detail = True, ""
    try:
        if shard_mode == 0:
            single = binding.engine_for_problem(problem, device=local, keep_debug_tensors=False)
            shard = binding.engine_for_problem(problem, device=local, world_size=world, rank=rank, shard_mode=0)
            uid = binding.comm_unique_id() if rank == 0 else bytes(128)
            shard.comm_init(broadcast_bytes(dist, uid, local))
            K = problem.num_rollouts
            off, cnt = sharding.rollout_shard(K, world, rank)
            single.begin_solve(); shard.begin_solve()
            for it in range(iterations):
                c1, v1, _ = single.iterate(it)
                c2, v2, _ = shard.iterate(it)
                np.testing.assert_array_equal(shard.tensor("verdicts")[0][:cnt], single.tensor("verdicts")[0][off:off + cnt])
                np.testing.assert_allclose(shard.tensor("rollouts")[0][:cnt], single.tensor("rollouts")[0][off:off + cnt], rtol=1e-9, atol=1e-12)
                np.testing.assert_allclose(shard.tensor("total_cost")[0], single.tensor("total_cost")[0], rtol=1e-9)
                np.testing.assert_allclose(shard.tensor("probabilities")[0][:, :, 0], single.tensor("probabilities")[0][:, :, 0], rtol=1e-9, atol=1e-300)
                np.testing.assert_allclose(shard.tensor("updates")[0], single.tensor("updates")[0], rtol=1e-9, atol=1e-13)
                np.testing.assert_allclose(shard.tensor("parameters")[0], single.tensor("parameters")[0], rtol=1e-9, atol=1e-12)
                np.testing.assert_allclose(shard.tensor("stddevs")[0], single.tensor("stddevs")[0], rtol=1e-9)
                np.testing.assert_allclose(c2, c1, rtol=1e-9)
                assert bool(v1[0]) == bool(v2[0])
            single.close(); shard.close()
            detail = f"rollout sharding: {iterations} iterations at K={K}, verdicts identical, costs / probabilities / update / parameters within 1e-9 of the single-GPU run"
        else:
            Qs = 4 * world + 1
            sub = P.Problem(problem.chain, problem.spheres, problem.sdf, problem.start[:Qs], problem.goal[:Qs], problem.noise_stddev,
                            problem.num_time_steps, problem.num_rollouts, num_queries=Qs)
            whole = binding.engine_for_problem(sub, device=local)
            part = binding.engine_for_problem(sub, device=local, world_size=world, rank=rank, shard_mode=1)
            whole.begin_solve(); part.begin_solve()
            whole.run(0, iterations); part.run(0, iterations)
            a, b = whole.finish_solve(), part.finish_solve()
            np.testing.assert_array_equal(b["solution"], a["solution"][part.query_offset:part.query_offset + part.Q])
            np.testing.assert_array_equal(b["cost"], a["cost"][part.query_offset:part.query_offset + part.Q])
            whole.close(); part.close()
            detail = f"query sharding: {Qs} queries x {iterations} iterations, solutions bit for bit those of one engine"
    except Exception as exc:      # a failed comparison must not hide the timing; it is reported in the line
        ok, detail = False, f"{type(exc).__name__}: {str(exc)[:300]}"
    # every rank must have passed
    import torch
    t = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    all_ok = bool(t.item() > 0.5)
    if ok and not all_ok:
        detail = "another rank failed: " + detail
    return all_ok, detail


def query_sharded_c4(args, rank, world, local, dist, steps):
    """BASELINE configs[3] — 1024 independent queries (K=64, T=200), queries sharded over the ranks, no collective —
    measured next to the main workload so that its scaling is in the driver's own lines.  Device time, max over ranks,
    L2 not flushed (the working set of one rank's share, 0.73 GB at N=1, is beyond L2 anyway)."""
    from motion_planners_b200 import binding
    w = WORKLOADS["c4"]
    problem = make_problem("c4")
    eng = binding.engine_for_problem(problem, device=local, world_size=world, rank=rank, shard_mode=1)
    eng.begin_solve()
    eng.run(0, 3)
    dist_barrier(dist, local)
    eng.timer_begin()
    eng.run(3, steps)
    ms = dist_max(dist, eng.timer_end(), local)
    eng.finish_solve()
    eng.close()
    states = w["Q"] * w["K"] * w["T"]
    return {"workload": w["label"], "value": states * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps,
            "steps": steps, "n_gpus": world, "sharding": "queries" if world > 1 else "none", "scaling": "strong (1024 queries in total)",
            "l2": "not flushed: the working set is beyond L2"}


def run_ours(args):
    from motion_planners_b200 import binding
    rank, world, local, dist = dist_setup(args.gpus)
    w = WORKLOADS[args.workload]
    problem = make_problem(args.workload)
    T, D, K = problem.num_time_steps, problem.chain.num_dimensions, problem.num_rollouts
    S = len(problem.spheres.link)
    Q = problem.num_queries
    shard_mode = 1 if w["kind"] == "batch" else 0
    parity_ok, parity_detail = (None, "single GPU: nothing is sharded")
    if world > 1:
        parity_ok, parity_detail = sharded_parity_check(problem, shard_mode, world, rank, local, dist)
    eng = binding.engine_for_problem(problem, device=local, world_size=world, rank=rank, shard_mode=shard_mode)
    if world > 1 and shard_mode == 0:
        uid = binding.comm_unique_id() if rank == 0 else bytes(128)
        eng.comm_init(broadcast_bytes(dist, uid, local))
    states_per_step = Q * K * T                       # whole job, all ranks
    flusher = L2Flusher(local) if args.l2 == "flush" else None

    eng_kind = eng.state_kernel_kind()
    exchange = eng.exchange_kind()

    # clocks / throttle reasons are sampled from before the warm-up to the end of the last measured pass: the timed
    # region itself lasts a few milliseconds, less than one nvidia-smi sampling period
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)

    # ---- warm-up ----
    eng.begin_solve()
    eng.run(0, args.warmup)
    it = args.warmup

    # ---- timed region: device-side (value) ----
    dist_barrier(dist, local)
    launches0 = eng.launch_count()
    total_ms = 0.0
    if flusher is None:
        eng.timer_begin()
        eng.run(it, args.steps)
        total_ms = eng.timer_end()
        it += args.steps
    else:
        for _ in range(args.steps):
            flusher.flush()
            eng.timer_begin()
            eng.run(it, 1)
            total_ms += eng.timer_end()
            it += 1
    launches = eng.launch_count() - launches0
    outputs = read_outputs(eng) if args.dump_outputs else None       # the last timed step's results, before anything else runs
    replays0 = eng.graph_replays()
    dist_barrier(dist, local)
    total_ms = dist_max(dist, total_ms, local)
    value = states_per_step * args.steps / (total_ms * 1e-3)

    # ---- steady state (no flush, iterations queued back to back: how solve() runs) ----
    dist_barrier(dist, local)
    eng.timer_begin()
    eng.run(it, args.steps)
    steady_ms = dist_max(dist, eng.timer_end(), local)
    it += args.steps
    graph_replays = eng.graph_replays() - replays0      # of the steady-state pass: one cudaGraphLaunch per iteration when the loop is captured

    # ---- per-kernel pass for the roofline of the dominant kernel (rollout cost) ----
    eng.set_profiling(True)
    # the per-kernel pass launches the unfused kernels (rollout_weights / weighted_update / apply_update), which the
    # timed passes above never ran: two untimed steps take their first-launch module loading out of the statistics
    eng.run(it, 2)
    it += 2
    eng.reset_kernel_stats()
    for _ in range(args.steps):
        if flusher is not None:
            flusher.flush()
        eng.run(it, 1)
        it += 1
    stats = eng.kernel_stats()
    eng.set_profiling(False)
    # ---- the same kernel's true span inside the shipped (fused, overlapped) loop: first-CTA-start to last-CTA-end
    # %globaltimer stamps on isolated, L2-flushed iterations — no launch latency, no event-record overhead in the figure
    span_ms = None
    try:
        eng.set_timeline(True)
        for _ in range(args.steps):
            if flusher is not None:
                flusher.flush()
            eng.run(it, 1)
            it += 1
        tl = eng.timeline(min(args.steps, 64))
        spans = tl[:, 1, 1] - tl[:, 1, 0]
        span_ms = float(np.median(spans[spans > 0])) * 1e-3 if np.any(spans > 0) else None
        eng.set_timeline(False)
    except Exception:
        span_ms = None
    eng.finish_solve()

    # ---- end to end: the call sequence StompPlanner::solve makes, host buffers in and out ----
    # What StompPlanner::solve does (motion_planners_b200/host/StompPlanner.cpp -> stomp::Stomp::solveOnDevice): policy up,
    # stomp_b200_solve — the loop queued on the device, the stop rule evaluated there, the host queueing one iteration ahead of the
    # progress words the device writes into pinned host memory (rollout sharding: a synchronising poll every 8 iterations) —
    # solution and scalars down in one read-back.  Iterations past a query's stop are no-ops, so the rate counts the iterations
    # the queries really ran (finish_solve's iterations_used).
    e2e_iters = args.steps
    poll_every = 8
    pol = eng.policy
    h2d = (pol["params_all"].nbytes + pol["mincc"].nbytes) * eng.Q
    paced = not (world > 1 and shard_mode == 0)
    polls = 1 if paced else (e2e_iters + poll_every - 1) // poll_every + 1
    # per query: the solution + per poll the scalar block (and the solution again when polling) + 8 bytes of progress words per iteration
    d2h = polls * (eng.Q * (D * T * 8 + 25) + 12) + (eng.Q * 8 * 6 if paced else 0)
    # the host buffers of the requests: one policy per local query (the same synthetic request for all of them)
    host_params = np.ascontiguousarray(np.broadcast_to(pol["params_all"], (eng.Q,) + pol["params_all"].shape))
    host_mincc = np.ascontiguousarray(np.broadcast_to(pol["mincc"], (eng.Q,) + pol["mincc"].shape))
    dist_barrier(dist, local)
    t0 = time.perf_counter()
    e2e_ran, e2e_solves = 0.0, 0
    while e2e_ran < e2e_iters and e2e_solves < 64:                   # whole planning queries until `steps` iterations have really run
        eng.set_policies(0, host_params, host_mincc)                 # H2D
        eng.begin_solve()
        eng.solve(e2e_iters, poll_every)                             # D2H per poll: noise-less cost, improvement, stop flag, iteration count, validity
        e2e_result = eng.finish_solve()                              # D2H: solution
        e2e_ran += float(np.mean(e2e_result["iterations"]))          # iterations per query that did work (the stop rule ends a solve early)
        e2e_solves += 1
    e2e_s = dist_max(dist, time.perf_counter() - t0, local)
    h2d, d2h = h2d * e2e_solves, d2h * e2e_solves
    dist_barrier(dist, local)
    if rank == 0 and world == 1:
        # keep the GPU under the same load until nvidia-smi has had a few sampling periods
        t_end = time.perf_counter() + 0.6
        while time.perf_counter() < t_end:
            eng.begin_solve()
            eng.run(0, 50)
    clocks = sampler.stop() if rank == 0 else None
    c4 = None
    if args.workload != "c4" and not args.skip_c4:
        try:
            c4 = query_sharded_c4(args, rank, world, local, dist, max(5, min(args.steps, 20)))
        except Exception as exc:
            c4 = {"error": f"{type(exc).__name__}: {str(exc)[:200]}"}

    if rank != 0:
        eng.close()
        return

    peaks, peak_kind = measured_peaks()
    # the dominant kernel of the cost path: the state kernel (FK + sphere / SDF verdicts), one launch per step
    cost_ms, cost_n = stats["cost"]
    rows_ms, rows_n = stats["rows"]
    states_per_launch = (eng.Q * K * T) // (world if shard_mode == 0 else 1)
    alg_bytes = (8 * D + 4 * S + 9) * states_per_launch
    avg_cost_ms = cost_ms / max(cost_n, 1)
    avg_rows_ms = rows_ms / max(rows_n, args.steps)      # no launch in the bracket when the sampler computes the rows: per step
    achieved = alg_bytes / (avg_cost_ms * 1e-3) / 1e9 if cost_ms > 0 else None
    # SURVEY 8(d) counts K4 + K5 + K6 (state costs + control-cost rows) as one 8D+4S+9 B/state pass: the same bytes
    # over the sum of the two kernels' launch times
    achieved_path = alg_bytes / ((avg_cost_ms + avg_rows_ms) * 1e-3) / 1e9 if cost_ms > 0 else None
    kind, kind_note = eng_kind
    # FP64 arithmetic of the state kernel (DESIGN.md 4): FP64-pipe warp instructions per state from the kernel's SASS
    # FP64-pipe instructions of the generated kernel, counted in its SASS (tools/spec_sass.cu): iiwa 224 DFMA + 63 DADD +
    # 48 DMUL of 749 executed; dual arm with the grasped object (DUAL=1) 574 + 152 + 110
    fp64_ops = {(7, 20): 335, (14, 48): 836}.get((D, S))
    fp64_peak = 18.43e12          # profiles/r1_fp64_peak_b200.json: DFMA / DADD / DMUL issue rate, thread-ops/s
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(args.workload, {}).get("rollout_cost_kernel_dram_bytes_per_launch")
        except Exception:
            traffic = None
    base_rate, base_s = (None, None)
    cb = None
    if not args.skip_cpu_baseline:
        from oracle import binding as ob
        threads = ob.set_num_threads(ob.host_cores())
        sample = min(K, args.cpu_sample)
        base_rate, base_s = cpu_baseline(problem, args.workload, threads, sample, 5)
        one_rate, _ = cpu_baseline(problem, args.workload, 1, max(8, sample // 8), 2)
        cb = {"value": base_rate, "unit": UNIT, "cores": threads, "kind": reference_kind(),
              "sample": f"{sample} of {K} rollouts x 5 iterations, same T / D / spheres / SDF, OpenMP over rollouts",
              "single_thread_value": one_rate}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "weak" if shard_mode == 1 else "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": w["label"], "name": args.workload, "K": K, "T": T, "D": D, "S": S, "Q": Q,
                   "sdf": list(map(int, problem.sdf.dims)), "sharding": ("queries" if shard_mode == 1 else "rollouts") if world > 1 else "none",
                   "l2": "flushed (256 MiB write) between timed iterations" if flusher else "not flushed",
                   "noise": "on-device Philox4x32-10", "exchange": exchange[0] + (": " + exchange[1] if world > 1 else ""),
                   "timed": "CUDA events on the engine's stream, per step: one stomp_b200_run records on the idle stream at its entry, one "
                            "it records behind the last kernel it queues (before its closing host wait); max over ranks, summed over the steps"},
        "clocks": clocks,
        "e2e": {"value": states_per_step * e2e_ran / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d / max(e2e_ran, 1.0),
                "d2h_bytes_per_step": d2h / max(e2e_ran, 1.0), "iterations_run": e2e_ran, "solves": e2e_solves,
                "what": "whole planning queries, the call sequence of StompPlanner::solve — set_policy (H2D) + begin_solve + stomp_b200_solve "
                        "(loop queued on the device, stop rule there, the host one iteration ahead of the device's progress words in pinned memory; "
                        "one read-back of solution + scalars) + finish_solve — repeated until `steps` iterations have really run; host wall clock over the iterations that did work"},
        "gpu_launches": int(launches),
        "graph_replays": int(graph_replays),
        "parity_ok": parity_ok, "parity": parity_detail,
        "query_sharded_c4": c4,
        "steady_state": {"value": states_per_step * args.steps / (steady_ms * 1e-3), "ms_per_step": steady_ms / args.steps,
                         "what": "same steps queued back to back without L2 flushes, as solve() runs them"},
        "roofline": {"kernel": "stomp_b200_states_specialised" if kind == "specialised" else "rollout_states_kernel",
                     "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"],
                     "unit": "GB/s", "frac": (achieved / peaks["hbm_gbs"]) if achieved else None, "traffic": traffic,
                     "peak_kind": peak_kind, "algorithmic_bytes_per_state": 8 * D + 4 * S + 9,
                     "states_per_launch": states_per_launch, "avg_launch_ms": avg_cost_ms,
                     "how": "achieved / frac: CUDA events bracketing every launch of the kernel in a serialised, L2-flushed pass "
                            "(the bracket contains the launch gap and the event records, ~5 us around a ~16 us kernel); "
                            "kernel_span: the kernel's own first-CTA-start to last-CTA-end %globaltimer span on isolated L2-flushed "
                            "iterations of the shipped loop",
                     "kernel_span": ({"ms": span_ms, "achieved": alg_bytes / (span_ms * 1e-3) / 1e9,
                                      "frac": alg_bytes / (span_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]} if span_ms else None),
                     "state_kernel": kind + (": " + kind_note if kind_note else ""),
                     "with_control_rows": {"kernels": "state kernel + control-cost rows (SURVEY 8d: K4+K5+K6, same 8D+4S+9 B/state); in the shipped "
                                                      "loop K5 / K6 are computed inside the sampler from values in registers (no pass over noise): "
                                                      "the second bracket is then empty and measures what an event pair itself costs",
                                           "achieved": achieved_path, "frac": (achieved_path / peaks["hbm_gbs"]) if achieved_path else None,
                                           "avg_launch_ms": avg_cost_ms + avg_rows_ms, "rows_bracket_ms": avg_rows_ms},
                     "whole_iteration": {"algorithmic_bytes_per_state": 24 * D + 4 * S + 9,
                                         "achieved": (24 * D + 4 * S + 9) * states_per_step / (total_ms / args.steps * 1e-3) / 1e9,
                                         "frac": (24 * D + 4 * S + 9) * states_per_step / (total_ms / args.steps * 1e-3) / 1e9 / (peaks["hbm_gbs"] * world),
                                         "steady_state_frac": (24 * D + 4 * S + 9) * states_per_step / (steady_ms / args.steps * 1e-3) / 1e9 / (peaks["hbm_gbs"] * world)},
                     "fp64_pipe": ({"ops_per_state": fp64_ops, "achieved_tops": fp64_ops * states_per_launch / (avg_cost_ms * 1e-3) / 1e12,
                                    "peak_tops": fp64_peak / 1e12,
                                    "frac": fp64_ops * states_per_launch / (avg_cost_ms * 1e-3) / fp64_peak,
                                    "what": "the arithmetic is FP64 by contract: this pipe, not HBM, is the kernel's real ceiling"}
                                   if fp64_ops and cost_ms > 0 and kind == "specialised" else None)},
        "kernel_ms_per_step": {k: v[0] / args.steps for k, v in stats.items()},
        "cpu_baseline": cb,
    }
    if outputs is not None:
        line["dump_outputs"] = {"dir": args.dump_outputs, "what": "results of the last timed step, read from rank 0's engine",
                                "arrays": dump_outputs(outputs, args.dump_outputs)}
    print(json.dumps(line), flush=True)
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--l2", default="flush", choices=["flush", "keep"])
    ap.add_argument("--cpu-sample", type=int, default=2048, dest="cpu_sample")
    ap.add_argument("--reference-sample", type=int, default=1024, dest="reference_sample")
    ap.add_argument("--skip-cpu-baseline", action="store_true", dest="skip_cpu_baseline")
    ap.add_argument("--skip-c4", action="store_true", dest="skip_c4")
    ap.add_argument("--dump-outputs", default=None, dest="dump_outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (64 MB at most); with "
                         "rollout sharding (--gpus N > 1) rollouts, state_costs and verdicts hold rank 0's share of the "
                         "rollouts, so their shapes depend on N")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the CUDA path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
