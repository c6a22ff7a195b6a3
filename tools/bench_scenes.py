"""One GPU, the C4 batch (Q=1024 queries, K=64, T=200, 128^3 fields) spread over 1, 16 and 1024 scenes: rollout-timesteps/s and
ms per iteration of the on-device loop, timed like bench.py (the engine's own timer around stomp_b200_run, after warm-up
iterations; L2 not flushed).  One scene is the shipped one-field engine; with more, every query reads the field of its scene.
At 1024 scenes the fields total 8.6 GB, far beyond the 126 MB of L2.  Engines are measured in interleaved rounds.

    python tools/bench_scenes.py [--steps 20] [--warmup 3] [--rounds 3] [--scenes 1,16,1024] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from motion_planners_b200 import binding, problems as P  # noqa: E402

Q, K, T, SDF_N = 1024, 64, 200, 128


def card():
    out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return out.stdout.strip() if out.returncode == 0 else f"nvidia-smi failed: {out.stderr.strip()}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--scenes", default="1,16,1024")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = [{"card": card(), "workload": f"C4 shape: Q={Q}, K={K}, T={T}, {SDF_N}^3 fields", "unit": "rollout-timesteps/s",
              "steps": args.steps, "warmup": args.warmup, "l2": "not flushed"}]
    engines = {}
    for n in [int(s) for s in args.scenes.split(",")]:
        pb = P.batch_problem_scenes(Q=Q, K=K, T=T, sdf_n=SDF_N, num_scenes=n)
        t0 = time.perf_counter()
        e = binding.engine_for_problem(pb)
        e.synchronize()
        setup_s = time.perf_counter() - t0
        e.begin_solve()
        e.run(0, args.warmup)
        engines[n] = (e, {"num_scenes": n, "setup_s": setup_s, "field_bytes": n * SDF_N ** 3 * 4,
                          "state_kernel": e.state_kernel_kind()[1], "ms_per_step": [], "value": []})
    states = Q * K * T
    for _ in range(args.rounds):
        for n, (e, rec) in engines.items():
            e.timer_begin()
            e.run(args.warmup, args.steps)
            ms = e.timer_end()
            rec["ms_per_step"].append(ms / args.steps)
            rec["value"].append(states * args.steps / (ms * 1e-3))
    for n, (e, rec) in engines.items():
        e.finish_solve()
        e.close()
        rec["median_value"] = sorted(rec["value"])[len(rec["value"]) // 2]
        rec["median_ms_per_step"] = sorted(rec["ms_per_step"])[len(rec["ms_per_step"]) // 2]
        lines.append(rec)
    text = "\n".join(json.dumps(line) for line in lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
