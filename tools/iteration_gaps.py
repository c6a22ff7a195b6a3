"""Where the time of an isolated, L2-flushed iteration goes (what bench.py's `value` times), kernel by kernel and between them:
    python tools/iteration_gaps.py [workload] [iterations] [rounds] [pdl_mask ...]
One engine per programmatic-dependent-launch mask (STOMP_B200_PDL at creation; no mask: the engine's default), the engines
taking turns round by round.  Every iteration is its own stomp_b200_run between the timer's entry and end events, with the
in-pipeline timeline on: %globaltimer stamps of the sampler, the state kernel, the weights / update kernel and the noise-less
tail launched alone at the join.  The event bracket minus the device span (sampler start to tail end) is the time from the
entry event to the sampler's first CTA plus the time from the tail's last CTA to the end event: the two clocks cannot be
aligned, so that sum is one figure."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from motion_planners_b200 import binding  # noqa: E402

name = sys.argv[1] if len(sys.argv) > 1 else "c3"
iters = min(int(sys.argv[2]) if len(sys.argv) > 2 else 40, 64)      # the timeline ring holds 64 iterations
rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 3
masks = [int(m) for m in sys.argv[4:]] or [None]
SAMPLE, STATE, UPDATE, TAIL = 0, 1, 3, 5

pb = bench.make_problem(name)
engines = []
for m in masks:
    if m is None:
        os.environ.pop("STOMP_B200_PDL", None)
    else:
        os.environ["STOMP_B200_PDL"] = str(m)
    e = binding.engine_for_problem(pb)
    e.begin_solve()
    e.run(0, 5)
    engines.append(e)
os.environ.pop("STOMP_B200_PDL", None)
flusher = bench.L2Flusher(0)
rows = {i: [] for i in range(len(masks))}
it = 5
for r in range(rounds):
    for i, e in enumerate(engines):
        e.set_timeline(True)
        ms = []
        for _ in range(iters):
            flusher.flush()
            e.timer_begin()
            e.run(it, 1)
            ms.append(e.timer_end())
            it += 1
        tl = e.timeline(iters)
        e.set_timeline(False)
        rows[i].append((np.array(ms) * 1e3, tl))


def span(tl, k):
    return tl[:, k, 1] - tl[:, k, 0]


def gap(tl, a, b):
    return tl[:, b, 0] - tl[:, a, 1]


print(f"workload {name}: isolated L2-flushed iterations, {iters} per round, {rounds} rounds; medians over all iterations (us)")
for i, m in enumerate(masks):
    ev = np.concatenate([x[0] for x in rows[i]])
    tl = np.concatenate([x[1] for x in rows[i]])
    tail = not np.all(tl[:, TAIL, 0] < 0)
    end = TAIL if tail else UPDATE
    device = tl[:, end, 1] - tl[:, SAMPLE, 0]
    parts = [("event bracket (value)", ev),
             ("sampler", span(tl, SAMPLE)), ("sampler -> state", gap(tl, SAMPLE, STATE)),
             ("state kernel", span(tl, STATE)), ("state -> update", gap(tl, STATE, UPDATE)),
             ("update kernel", span(tl, UPDATE))]
    if tail:
        parts += [("update -> tail", gap(tl, UPDATE, TAIL)), ("tail", span(tl, TAIL))]
    parts += [("device span", device), ("entry -> sampler + " + ("tail" if tail else "update") + " -> end", ev - device)]
    per_round = [float(np.median(x[0])) for x in rows[i]]
    print(f"  STOMP_B200_PDL={'default' if m is None else m}: event bracket per round " + ", ".join(f"{v:.1f}" for v in per_round))
    for label, v in parts:
        print(f"    {label:34s} median {np.median(v):7.1f}   p10 {np.percentile(v, 10):7.1f}   p90 {np.percentile(v, 90):7.1f}")
for e in engines:
    e.finish_solve()
    e.close()
