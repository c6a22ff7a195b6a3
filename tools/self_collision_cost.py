"""Cost of the self-collision state kernel on the dual-arm workload (C5 shape, smaller SDF so that the scene builds in
seconds): per-kernel times of the loop with the pair list off (specialised state kernel) and on (self-collision kernel).
Run on the GPU box:  python tools/self_collision_cost.py [K] [T] [sdf_n]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from motion_planners_b200 import binding, problems as P


def main():
    K = int(sys.argv[1]) if len(sys.argv) > 1 else 2048
    T = int(sys.argv[2]) if len(sys.argv) > 2 else 150
    n = int(sys.argv[3]) if len(sys.argv) > 3 else 128
    pb = P.dual_arm_problem(K=K, T=T, sdf_n=n)
    inside = [(a, b) for base in (0, 7) for a in range(base, base + 7) for b in range(a + 1, base + 7)]
    pairs = P.self_collision_pairs(pb.chain, pb.spheres, disabled_links=inside)
    out = {"workload": f"dual arm K={K} T={T} D=14 S=48 sdf={n}^3", "pairs": int(len(pairs))}
    none = np.zeros((0, 2), dtype=np.int32)
    variants = [("world_only", none, {}), ("list_walk_generic_fk", pairs, {"STOMP_B200_SELF": "generic"}),
                ("pair_rule_in_specialised_kernel", pairs, {"STOMP_B200_SELF": "spec"})]
    for label, pr, env in variants:
        os.environ.update(env)
        e = binding.engine_for_problem(pb)
        e.set_self_collision(pr)
        e.begin_solve()
        e.run(0, 5)
        e.timer_begin(); e.run(5, 30); ms = e.timer_end()
        e.set_profiling(True)
        e.reset_kernel_stats()
        e.run(35, 10)
        stats = {k: round(1e3 * v[0] / max(v[1], 1), 2) for k, v in e.kernel_stats().items() if v[1]}
        out[label] = {"kind": e.state_kernel_kind()[1], "us_per_iteration": round(1e3 * ms / 30, 1), "kernel_us": stats}
        e.close()
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
