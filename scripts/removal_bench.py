#!/usr/bin/env python
"""Scale-down simulation: the planner's candidate loop (SimulateNodeRemoval per unneeded-node candidate, persisted) on a
seeded object-model cluster, today's per-candidate path vs the batched call, with parity against the CPU oracle loop.

    python scripts/removal_bench.py [--nodes 2000] [--cands 100 1000] [--loop-cands 100] [--out removal_bench.json]

* per candidate: SimulateNodeRemoval on the engine = encode without the node, cae_load, cae_filter_schedulable.  Timed on the
  first --loop-cands candidates (the per-candidate cost does not depend on K); `loop_ms_per_cand` x K is the loop's cost.
* batch: SimulateNodeRemovals = one encode, one cae_load, one cae_simulate_removals; wall time and the device time of the
  call (cae_stats.estimate_ms).
* parity: the batch's first 50 answers against the sequential loop on the CPU oracle."""
import argparse
import copy
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def make_cluster(n_nodes, seed):
    from kubernetes_autoscaler_b200.objects import BuildTestNode, BuildTestPod, LabelSelector, NodeInfo, TopologySpreadConstraint
    rng = random.Random(seed)
    cluster = []
    k = 0
    for i in range(n_nodes):
        n = BuildTestNode("node-%d" % i, 4000, 16 << 30)
        n.labels = {"kubernetes.io/hostname": n.name, "topology.kubernetes.io/zone": "z%d" % (i % 3)}
        pods = []
        for _ in range(rng.choice([1, 1, 2, 3, 4, 6, 8, 10])):
            app = "app%d" % rng.randrange(20)
            p = BuildTestPod("pod-%d" % k, rng.choice([100, 200, 250, 500]), rng.choice([1 << 28, 1 << 29]))
            k += 1
            p.labels = {"app": app}
            p.owner_uid, p.owner_kind = "rs-" + app, "ReplicaSet"
            if rng.random() < 0.2:
                p.topology_spread = [TopologySpreadConstraint(rng.choice([1, 2, 3]), "topology.kubernetes.io/zone", LabelSelector({"app": app}),
                                                              when_unsatisfiable=rng.choice(["DoNotSchedule", "ScheduleAnyway"]))]
            pods.append(p)
        ds = BuildTestPod("ds-%d" % i, 50, 1 << 26)
        ds.owner_uid, ds.owner_kind = "ds", "DaemonSet"
        pods.append(ds)
        cluster.append(NodeInfo(n, pods))
    return cluster


def gpu_info():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True).strip()
    except Exception as ex:   # reported, never guessed
        return "unavailable: %s" % ex


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=2000)
    ap.add_argument("--cands", type=int, nargs="+", default=[100, 1000])
    ap.add_argument("--loop-cands", type=int, default=100)
    ap.add_argument("--parity", type=int, default=50)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import __graft_entry__ as ge
    ge.build()
    from kubernetes_autoscaler_b200 import podlistprocessor as plp
    from kubernetes_autoscaler_b200.engine import Engine
    from kubernetes_autoscaler_b200.removal import RemovalSimulator
    from test_removal_batch import reference_loop, summary
    eng = Engine(device=0)
    base = make_cluster(args.nodes, args.seed)
    used = {ni.node.name: sum(p.requests.get("cpu", 0) for p in ni.pods) for ni in base}
    order = sorted((ni.node.name for ni in base), key=lambda n: (used[n], n))   # least utilised first
    dest = {ni.node.name: True for ni in base}
    out = {"gpu": gpu_info(), "nodes": args.nodes, "pods": sum(len(ni.pods) for ni in base), "seed": args.seed, "runs": []}
    for K in args.cands:
        cands = order[:K]
        row = {"K": K}
        # today's path: one encode + load + filter pass per candidate
        lc = min(args.loop_cands, K)
        cl = copy.deepcopy(base)
        r = RemovalSimulator(cl, True, schedulingSimulator=plp.HintingSimulator(eng))
        t0 = time.perf_counter()
        for name in cands[:lc]:
            r.SimulateNodeRemoval(name, dest)
        dt = time.perf_counter() - t0
        row["loop_cands_timed"] = lc
        row["loop_ms_per_cand"] = 1e3 * dt / lc
        row["loop_ms_for_K"] = 1e3 * dt / lc * K
        # the batch
        best = None
        for _ in range(args.reps):
            cl = copy.deepcopy(base)
            r = RemovalSimulator(cl, True, engine=eng)
            t0 = time.perf_counter()
            got = r.SimulateNodeRemovals(cands, dest)
            wall = time.perf_counter() - t0
            dev = eng.stats().estimate_ms
            if best is None or wall < best[0]:
                best = (wall, dev, got)
        row["batch_wall_ms"] = 1e3 * best[0]
        row["batch_device_ms"] = best[1]
        row["removable"] = sum(a is not None for a, _ in best[2])
        row["speedup_vs_loop"] = row["loop_ms_for_K"] / row["batch_wall_ms"]
        # parity: the first candidates against the oracle loop
        m = min(args.parity, K)
        _, want = reference_loop(copy.deepcopy(base), True, cands[:m], dest)
        row["parity_cands"] = m
        row["parity"] = summary(best[2][:m]) == summary(want)
        out["runs"].append(row)
        print(json.dumps(row), flush=True)
    eng.close()
    out["gpu_after"] = gpu_info()
    text = json.dumps(out)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
