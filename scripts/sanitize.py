#!/usr/bin/env python
"""Small end-to-end workload for compute-sanitizer (SURVEY §5: memcheck / racecheck evidence for the kernels that use
self-cleaning accumulators, last-block election, shared-memory state and block-wide barriers):

    compute-sanitizer --tool memcheck  python scripts/sanitize.py
    compute-sanitizer --tool racecheck python scripts/sanitize.py

Dense pass (K1, both variants), Estimate() of every template (K0 + K3: plain closed form, capacity form with the cluster
fallback, per-pod loop), expander scores, the filter-out-schedulable pass — on miniatures of C2, C3 and C4 — and the batched
scale-down loop (cae_simulate_removals), each checked against the CPU oracle so that a "clean" run also means "correct results
under the tool"."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402


def main():
    import __graft_entry__ as ge
    ge.build()
    from kubernetes_autoscaler_b200 import synth
    from kubernetes_autoscaler_b200.engine import Engine, unpack_bits
    from oracle import pyoracle
    eng = Engine(device=0, want_reasons=True)
    for cfg, kw in ((2, dict(pods=3000, templates=40)), (3, dict(pods=2500, templates=24, cluster_nodes=48)),
                    (4, dict(pods=3000, templates=20, cluster_nodes=40))):
        enc = synth.generate(cfg, **kw)
        eng.load(enc)
        bits, reasons, count = eng.feasibility()
        want, _ = pyoracle.feasibility_dense(enc)
        assert np.array_equal(reasons, want) and np.array_equal(unpack_bits(bits, enc.P), want == 0)
        for cap in (30, 0):
            caps = np.full(enc.T, cap, np.int32)
            nc, pc, sched, order = eng.estimate_all(caps)
            onc, opc, osched, oorder, _ = pyoracle.estimate_all(enc, caps)
            assert np.array_equal(nc, onc) and np.array_equal(pc, opc) and np.array_equal(sched, osched) and np.array_equal(order, oorder)
        mask, waste = eng.expander_best([0, 1, 2], nc, pc)
        assert eng.load_pending(enc)
        eng.feasibility()
        if enc.struct.num_cluster_nodes:
            order_p = np.arange(min(enc.P, 600), dtype=np.int32)
            got = eng.filter_schedulable(order_p)
            ref = pyoracle.filter_schedulable(enc, order_p)
            assert np.array_equal(got[0], ref[0]) and got[1:] == ref[1:]
        print("config", cfg, "ok: nodes", int(nc.sum()), "pods", int(pc.sum()), flush=True)
    removal_batch(eng)
    eng.close()
    print("sanitize workload ok")


def removal_batch(eng):
    """The batched scale-down loop (cae_simulate_removals: candidate loop, undo, persisted removals, pods moved again) on a
    small cluster with topology spread and anti-affinity, checked against the sequential SimulateNodeRemoval loop."""
    import copy
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
    from test_removal_batch import _rand_scenario, check_batch
    for seed in range(6):
        cluster, cands, dest, persist, max_removable, hints, li = _rand_scenario(90_000 + seed)
        check_batch(eng, copy.deepcopy(cluster), cands, dest, persist, max_removable, hints, li)
    print("removal batch ok", flush=True)


if __name__ == "__main__":
    main()
