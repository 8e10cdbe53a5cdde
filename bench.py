#!/usr/bin/env python
"""bench.py — pod x node predicate evaluations/sec of the dense feasibility pass (BASELINE.json
metric 1, SURVEY.md §8d) on config C2: 100 000 pods x 1 000 templates, resources + taints/tolerations,
and the scale-up decision latency (metric 2) beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 2] [--dump-outputs DIR]

One "step" = one dense pass of the scale-up predicate path over the whole pending-pod batch:
every pod (not only group exemplars) against every template through the Filter chain.
  value            : whole-job evals/s with the snapshot already resident in HBM (device time, CUDA events)
  e2e              : the same through the C-ABI with HOST buffers: cae_load (intern + H2D + class
                     matrices) + cae_feasibility (kernel + D2H of the bit matrix and counts) per step
  roofline         : the dense kernel's algorithmic bytes / its CUDA-event time vs the measured HBM peak
  cpu_baseline     : the CPU oracle (port of the Go reference) on the box's host cores, same workload
                     (rows for 1 thread, 4 threads = the reference's default parallelism, and all cores)
  parity_checked   : the numbers timed were compared with the oracle (and, N > 1, with an NCCL all-reduce
                     of the per-rank histograms) before the line was printed
  decision_latency : load -> exemplar feasibility -> order -> Estimate() of every template -> expander
                     (C3 on one GPU = the headline of metric 2; C4 template-sharded at every N, C5 at N = 8),
                     with the estimator kernel's roofline and an oracle check of a template slice
N > 1 (torchrun): weak scaling of the dense pass — every rank owns (and uploads) 100 000 pods of an
N x 100 000-pod snapshot, the per-template fit-count histogram int32[T] is exchanged once per step.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


_CLOCK_QUERY = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
               "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"


def _clock_sampler_start(devs):
    """ONE looping nvidia-smi for the whole timed region (the profiling recipe's clocks line), started by rank 0
    only: spawning nvidia-smi per sample from every rank stalls kernel launches on a multi-GPU box for milliseconds."""
    try:
        return subprocess.Popen(["nvidia-smi", "-i", ",".join(str(d) for d in devs), "--query-gpu=" + _CLOCK_QUERY,
                                 "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return None


def _clock_sampler_stop(proc):
    if proc is None:
        return []
    try:
        proc.terminate()
        out, _ = proc.communicate(timeout=5)
    except Exception:
        proc.kill()
        return []
    return [[x.strip() for x in line.split(",")] for line in out.strip().splitlines() if line.count(",") >= 5]


def _clocks_summary(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
    sm = sorted(int(s[0]) for s in samples if s[0].isdigit())
    mx = max(int(s[1]) for s in samples if s[1].isdigit())
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in samples)]
    return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons}


def _peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _host_cores():
    """Threads this process can really use: the affinity mask, cut by a cgroup CPU quota if one is set."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = int(q) / int(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(quota)))
    return n


def _config_dict(cfg, P1, T, world):
    """The SAME dict in the engine's line and the reference arm's line."""
    return {"workload": "%s; %d pods/GPU x %d templates, splitmix64 seed 0xCA5CA1E0+%d" % (cfg.name, P1, T, cfg.index),
            "global_pods": P1 * world, "templates": T, "parallelism": "pods sharded x%d" % world,
            "l2": "flushed between timed iterations (512 MiB memset on the engine's stream)",
            "timing": "CUDA events on the engine's stream, queued behind the flush + a spin kernel (no host launch latency in the window)"}


_W = {}


def _worker_init(config, pods, templates):
    from kubernetes_autoscaler_b200 import synth
    from oracle import pyoracle
    _W["enc"] = synth.generate(config, pods=pods, templates=templates)
    _W["oracle"] = pyoracle
    pyoracle.lib()


def _worker_run(job):
    p_range, t_range = job
    t0 = time.perf_counter()
    ev = _W["oracle"].feasibility_dense(_W["enc"], p_range=p_range, t_range=t_range)[1]
    return ev, time.perf_counter() - t0


def _worker_counts(job):
    p_range, t_range = job
    reasons = _W["oracle"].feasibility_dense(_W["enc"], p_range=p_range, t_range=t_range)[0]
    return t_range[0], (reasons == 0).sum(axis=1).astype(np.int64).tolist()


def _worker_decide(job):
    t, cap = job
    enc = _W["enc"]
    caps = np.full(enc.T, cap, np.int32)
    t0 = time.perf_counter()
    nc, pc, _, _, ev = _W["oracle"].estimate_all(enc, caps, t_range=(t, t + 1))
    return {"t": t, "nodes": int(nc[0]), "pods": int(pc[0]), "filter_evals": int(ev), "secs": time.perf_counter() - t0}


def _worker_pid(_):
    time.sleep(0.02)
    return os.getpid()


def _wait_workers(pool, procs):
    """Block until every pool worker has finished its initializer (generated its snapshot copy)."""
    for _ in range(200):
        if len(set(pool.map(_worker_pid, range(4 * procs), chunksize=1))) >= procs:
            return


def _cpu_dense(pool, procs, p_range, t_range):
    """Oracle dense feasibility on `procs` host processes (templates split across them).
    Returns (evals, wall seconds)."""
    tb, te = t_range
    cuts = [tb + (te - tb) * i // procs for i in range(procs + 1)]
    jobs = [(p_range, (cuts[i], cuts[i + 1])) for i in range(procs) if cuts[i + 1] > cuts[i]]
    t0 = time.perf_counter()
    res = pool.map(_worker_run, jobs)
    return int(sum(r[0] for r in res)), time.perf_counter() - t0


def _spread(n, k):
    return sorted({int(round(i * (n - 1) / max(k - 1, 1))) for i in range(k)})


DUMP_BYTES = 64_000_000


def dump_outputs(path, fit_bits, P, fit_count):
    """Writes what a caller of the dense pass receives, within DUMP_BYTES in all:
      fit.npy       float32 [T][n]  1.0 = pod fit_pods[j] fits template t, else 0.0 (unpacked from fit_bits [T][ceil(P/32)]),
                                    so one wrong verdict is an absolute difference of 1 under any tolerance
      fit_pods.npy  float64 [n]     the pods kept: all P, or above the budget a fixed seeded sample, in ascending order
      fit_count.npy float64 [T]     the fit histogram
    With several ranks, fit covers rank 0's pod shard only (pods 0 .. P-1 of the snapshot) while fit_count counts the pods
    of every rank, so fit_count is not the row sum of fit."""
    T = fit_bits.shape[0]
    room = (DUMP_BYTES - 4096 - 8 * T) // (4 * T + 8) if T else P       # 4096: the three .npy headers
    if P and room < 1:
        raise ValueError("--dump-outputs: one pod column of %d templates exceeds %d bytes" % (T, DUMP_BYTES))
    pods = np.arange(P) if P <= room else np.sort(np.random.default_rng(0).choice(P, room, replace=False))
    fit = (fit_bits[:, pods >> 5] >> (pods & 31).astype(np.uint32)) & 1
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "fit.npy"), fit.astype(np.float32))
    np.save(os.path.join(path, "fit_pods.npy"), pods.astype(np.float64))
    np.save(os.path.join(path, "fit_count.npy"), np.asarray(fit_count, np.float64))


def reference_arm(args, cfg, P1, T, metric):
    """The reference's own CPU implementation of the path (the C++ port of the Go code: no Go toolchain here)."""
    import multiprocessing as mp
    from oracle import pyoracle
    pyoracle.build()
    cores = _host_cores()
    if args.threads:
        cores = max(1, min(cores, args.threads))
    ctx = mp.get_context("fork")
    if args.decision_templates is not None:
        # metric 2 (SURVEY §8d): SchedulablePodGroups + Estimate per template, one template per job
        templates = [int(x) for x in args.decision_templates.split(",") if x != ""]
        with ctx.Pool(min(cores, max(len(templates), 1)), initializer=_worker_init, initargs=(args.config, P1, T)) as pool:
            t0 = time.perf_counter()
            rows = pool.map(_worker_decide, [(t, args.cap) for t in templates], chunksize=1)
            wall = time.perf_counter() - t0
        per = [r["secs"] for r in rows]
        print(json.dumps({"impl": "reference", "decision": True, "templates": rows, "wall_s": wall,
                          "cpu_seconds_per_template": float(np.mean(per)) if per else None, "cores": cores,
                          "extrapolated_s_all_templates_on_these_cores": float(np.mean(per)) * T / max(min(cores, len(templates)), 1) if per else None,
                          "kind": "port"}))
        return
    if args.counts_slice is not None:
        # parity leg: per-template fit counts of a template slice over the pods [p_begin, p_end)
        pb, pe, ts = args.counts_slice.split(":")
        templates = [int(x) for x in ts.split(",")]
        with ctx.Pool(min(cores, len(templates)), initializer=_worker_init, initargs=(args.config, P1, T)) as pool:
            res = dict(pool.map(_worker_counts, [((int(pb), int(pe)), (t, t + 1)) for t in templates], chunksize=1))
        print(json.dumps({"impl": "reference", "counts": {str(k): v[0] for k, v in res.items()}}))
        return
    P = P1
    t_slice = min(T, 8 * cores)   # bounded sample per step: all pods x a template slice (~0.2 s of work per core)
    with ctx.Pool(cores, initializer=_worker_init, initargs=(args.config, P1, T)) as pool:
        _wait_workers(pool, cores)
        for _ in range(2):
            _cpu_dense(pool, cores, (0, P), (0, min(T, t_slice)))
        evals = 0
        secs = 0.0
        for s in range(args.steps):
            tb = (s * t_slice) % max(T - t_slice + 1, 1)
            ev, dt = _cpu_dense(pool, cores, (0, P), (tb, tb + t_slice))
            evals += ev
            secs += dt
    v = evals / secs
    sample = "%d pods x %d templates per step (template slice of the full workload), %d steps" % (P, t_slice, args.steps)
    print(json.dumps({
        "impl": "reference", "metric": metric, "value": v, "unit": "evals/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": _config_dict(cfg, P1, T, max(args.gpus, 1)),
        "note": "CPU oracle = C++ port of the Go reference (no Go toolchain in the image); the `l2` / `timing` keys of config describe the engine's arm",
        "cpu_baseline": {"value": v, "unit": "evals/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def _reference_subprocess(extra, timeout=900):
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "LOCAL_WORLD_SIZE")}
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference"] + extra,
                         capture_output=True, text=True, timeout=timeout, env=env)
    return json.loads(out.stdout.strip().splitlines()[-1])


def decision_run(torch, dist, Engine, synth, config, rank, world, local_rank, reps=4, cap=1000, check_templates=8):
    """One full scale-up decision per rep on `config`: load (intern + H2D + class / counter tables), exemplar feasibility,
    order, Estimate() of every template (templates sharded over the ranks), one all-reduce of int32[2T] + float64[T],
    expander chain on the assembled vectors.  Wall time, max over ranks."""
    enc = synth.generate(config)
    eng = Engine(device=local_rank, rank=rank, world_size=world)
    caps = np.full(enc.T, cap, np.int32)
    counts_t = None
    rows = []
    nc = pc = mask = None
    for rep in range(reps):
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        eng.load(enc)
        t1 = time.perf_counter()
        nc, pc, _, _ = eng.estimate_all(caps, want_sched=False, copy=False)
        t2 = time.perf_counter()
        if dist is not None:
            from kubernetes_autoscaler_b200.engine import expander_chain
            ptr, _ = eng.device_buffer(1)          # node_count | pod_count of this load, on the device

            class _Wrap:
                __cuda_array_interface__ = {"shape": (2 * enc.T,), "typestr": "<i4", "data": (ptr, False), "version": 3}
            counts_t = torch.as_tensor(_Wrap(), device="cuda")
            waste_t = torch.from_numpy(eng.waste_scores()).cuda()   # own rows, 0.0 elsewhere
            dist.all_reduce(counts_t)                                # int32[2T]: node_count | pod_count
            dist.all_reduce(waste_t)                                 # float64[T]: one non-zero contribution per row
            both = counts_t.cpu().numpy()
            nc, pc = both[:enc.T].copy(), both[enc.T:].copy()
            mask = expander_chain([0, 1, 2], nc, pc, waste_t.cpu().numpy())
        else:
            mask, _ = eng.expander_best([0, 1, 2], nc, pc)         # least-waste, most-pods, least-nodes
        t3 = time.perf_counter()
        st = eng.stats()
        row = [1e3 * (t3 - t0), 1e3 * (t1 - t0), 1e3 * (t2 - t1), st.estimate_ms, 1e3 * (t3 - t2)]
        if dist is not None:
            tt = torch.tensor(row, device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            row = [float(x) for x in tt]
        if rep:
            rows.append(row)
    # the same decision when only the pending-pod rows changed since the last tick (cae_load_pending instead of cae_load)
    delta_ms = []
    for rep in range(3):
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        assert eng.load_pending(enc)
        nc2, pc2, _, _ = eng.estimate_all(caps, want_sched=False, copy=False)
        if dist is not None:
            ptr, _ = eng.device_buffer(1)

            class _Wrap2:
                __cuda_array_interface__ = {"shape": (2 * enc.T,), "typestr": "<i4", "data": (ptr, False), "version": 3}
            c2 = torch.as_tensor(_Wrap2(), device="cuda")
            w2 = torch.from_numpy(eng.waste_scores()).cuda()
            dist.all_reduce(c2)
            dist.all_reduce(w2)
            both2 = c2.cpu().numpy()
            expander_chain([0, 1, 2], both2[:enc.T], both2[enc.T:], w2.cpu().numpy())
        else:
            eng.expander_best([0, 1, 2], nc2, pc2)
        dt = 1e3 * (time.perf_counter() - t0)
        if dist is not None:
            tt = torch.tensor([dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt[0])
        delta_ms.append(dt)
    steps = int(eng.stats().estimate_group_steps)
    if dist is not None:
        tt = torch.tensor([steps], device="cuda", dtype=torch.int64)
        dist.all_reduce(tt)
        steps = int(tt[0])
    nc, pc = np.array(nc), np.array(pc)
    eng.close()
    med = np.median(np.asarray(rows), axis=0)
    out = {"workload": synth.CONFIGS[config].name + ", node cap %d per template" % cap, "config": config, "n_gpus": world,
           "ms": float(med[0]), "load_ms": float(med[1]), "estimate_wall_ms": float(med[2]), "estimate_device_ms": float(med[3]),
           "reduce_and_expander_ms": float(med[4]), "templates_sharded": world > 1,
           "ms_with_pending_delta": float(np.median(delta_ms)),
           "nodes_total": int(nc.sum()), "pods_scheduled_total": int(pc.sum()), "options_surviving_chain": int(mask.sum()),
           "group_steps": steps}
    if rank != 0:
        return out
    # ---- estimator kernel roofline: the engine's compulsory HBM traffic (order rows in, per-group records in, per-group
    #      scheduled counts + two counters out; the node state lives in shared memory) vs the §8(d) model of the per-pod scans
    E = enc.E
    alg = enc.T * E * 4 + steps * 144 + enc.T * E * 4 + enc.T * 8
    peak, peak_src = _peak_hbm()
    ach = alg / (out["estimate_device_ms"] * 1e-3) / 1e9 * (1.0 if world == 1 else 1.0)
    out["roofline"] = {"kernel": "binpack_kernel (+ order_kernel, group_reason_kernel in the same window)", "bound": "hbm",
                       "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                       "algorithmic_bytes": int(alg), "peak_source": peak_src,
                       "note": "node state is shared-memory resident: the kernel is bound by issue slots / barrier latency per "
                               "(template, group) step, not by HBM; see profiles/r02_summary.md for the ncu page"}
    # ---- oracle on a template slice: parity of the timed result + the CPU arm of metric 2 + the §8(d) byte model
    try:
        tsel = _spread(enc.T, check_templates)
        ref = _reference_subprocess(["--config", str(config), "--decision-templates", ",".join(str(t) for t in tsel), "--cap", str(cap)])
        ok = all(int(nc[r["t"]]) == r["nodes"] and int(pc[r["t"]]) == r["pods"] for r in ref["templates"])
        out["parity_checked"] = bool(ok)
        out["parity_templates"] = tsel
        out["cpu_baseline"] = {k: ref[k] for k in ("cpu_seconds_per_template", "cores", "wall_s", "kind",
                                                   "extrapolated_s_all_templates_on_these_cores")}
        ev = float(np.mean([r["filter_evals"] for r in ref["templates"]]))
        model = enc.T * (E * 320 + ev * 128)
        out["roofline"]["model_8d"] = {"bytes": model, "definition": "sum_t (E_t x 320 B + filter evaluations of the reference's per-pod "
                                       "any-node scans x 128 B), evaluations from the oracle's trace on the slice, extrapolated to T templates",
                                       "effective_GBps": model / (out["estimate_device_ms"] * 1e-3) / 1e9,
                                       "note": "above the HBM peak = the closed forms never perform those scans"}
        if not ok:
            out["parity_error"] = [(r["t"], int(nc[r["t"]]), r["nodes"], int(pc[r["t"]]), r["pods"]) for r in ref["templates"]]
    except Exception as ex:
        out["parity_checked"] = False
        out["parity_error"] = repr(ex)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine")
    ap.add_argument("--config", type=int, default=2)
    ap.add_argument("--pods", type=int, default=None)
    ap.add_argument("--templates", type=int, default=None)
    ap.add_argument("--threads", type=int, default=0, help="reference arm: cap the host processes (0 = all usable cores)")
    ap.add_argument("--decision-templates", default=None, help="reference arm: time / report full Estimate() of these templates (oracle)")
    ap.add_argument("--counts-slice", default=None, help="reference arm: pb:pe:t0,t1,.. per-template fit counts (parity leg)")
    ap.add_argument("--cap", type=int, default=1000)
    ap.add_argument("--no-decision", action="store_true", help="engine arm: skip the decision-latency figures")
    ap.add_argument("--collective", default="peer", choices=["peer", "nccl"],
                    help="N>1: how the int32[T] fit histogram is reduced: fused P2P exchange in the kernel's last block, or NCCL")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="engine arm: write the results of the last timed step (rank 0's fit verdicts, the fit histogram over all "
                         "ranks) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    args.warmup = max(args.warmup, 3)

    from kubernetes_autoscaler_b200 import synth
    cfg = synth.CONFIGS[args.config]
    P1 = args.pods or cfg.pods
    T = args.templates or cfg.templates
    metric = "pod x node predicate evals/sec"

    # ------------------------------------------------------------------ reference arm (CPU oracle)
    if args.impl == "reference":
        if rank != 0:
            return
        reference_arm(args, cfg, P1, T, metric)
        return

    # ------------------------------------------------------------------ engine arm
    import torch
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    torch.cuda.set_device(local_rank)
    from kubernetes_autoscaler_b200.engine import Engine, shard_pods, unpack_bits

    enc_all = synth.generate(args.config, pods=P1 * world, templates=T)   # weak scaling: P1 pods per rank
    pb, pe = shard_pods(enc_all.P, rank, world)
    enc = enc_all.slice_pods(pb, pe) if world > 1 else enc_all           # a rank uploads ITS pods only
    eng = Engine(device=local_rank, rank=rank, world_size=world, want_reasons=False, pods_presharded=world > 1)
    eng.load(enc)
    Pl = pe - pb
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    count_t = None
    fused = False
    if world > 1 and args.collective == "peer":
        try:
            handles = [None] * world
            dist.all_gather_object(handles, eng.peer_handle())
            eng.peer_attach(handles)
            dist.barrier()
            fused = True
        except Exception as ex:   # no P2P between these devices: fall back to the NCCL all-reduce
            if rank == 0:
                print("peer exchange unavailable (%r); using NCCL" % (ex,), file=sys.stderr)
    if world > 1 and not fused:
        ptr, nbytes = eng.device_buffer(0)

        class _Wrap:
            __cuda_array_interface__ = {"shape": (T,), "typestr": "<i4", "data": (ptr, False), "version": 3}
        count_t = torch.as_tensor(_Wrap(), device="cuda")

    ar0 = torch.cuda.Event(enable_timing=True)
    ar1 = torch.cuda.Event(enable_timing=True)
    # The pass is a single ~10 us kernel: timed right after a host synchronize, the event window would mostly hold
    # the HOST's launch latency (the GPU idles between the first event and the kernel's arrival: ~12 us for an
    # empty kernel on this box, scripts/k1_floor.py).  So the L2 flush and a short spin kernel are queued on the
    # engine's own stream first; event, kernel and event are then enqueued while the GPU is still busy and the
    # window measures device time only.  wall_ms_per_step keeps the host view.
    estream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", local_rank))

    sync_t = torch.zeros(1, device="cuda")

    def flush_l2():
        with torch.cuda.stream(estream):
            flush.zero_()                                      # > L2: evicts everything the previous step left
            torch.cuda._sleep(2_000_000)                       # ~1 ms spin: covers the host's enqueue of the step on every rank
            if dist is not None:
                dist.all_reduce(sync_t)                        # device-side barrier on the engine's stream: the ranks' timed
                                                               # windows open together (a host barrier cannot align queued work)

    def step_resident(to_host=False):
        if to_host:                                            # the same launch; the copies of its results to the host
            out = eng.feasibility()                            # are queued after its timing events
        else:
            eng.lib.cae_feasibility(eng.h, None, None, None)   # kernel only; results stay in HBM
            out = None
        if count_t is not None:
            ar0.record()
            dist.all_reduce(count_t)                           # int32[T] histogram over NVLink
            ar1.record()
        return out

    sampler = _clock_sampler_start([local_rank]) if rank == 0 else None   # rank 0's GPU only: NVML queries delay launches
    first_sample = None
    if sampler is not None:
        # nvidia-smi initialises NVML on EVERY GPU of the box (seconds on an 8-GPU host) and that stalls kernel launches:
        # wait for its first sample line, so that the initialisation is over before the timed steps start
        import select
        r, _, _ = select.select([sampler.stdout], [], [], 20.0)
        if r:
            first_sample = sampler.stdout.readline()
        time.sleep(0.1)
    if dist is not None:
        dist.barrier()
    for _ in range(args.warmup):   # warm-up AFTER the wait above: the GPUs idled while nvidia-smi initialised
        flush_l2()
        step_resident(to_host=bool(args.dump_outputs))        # allocates the pinned result buffers the dumped step reuses
    torch.cuda.synchronize()
    launches0 = eng.stats().kernel_launches
    dev_ms, wall_ms, ar_ms = [], [], []
    for s in range(args.steps):
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        flush_l2()                                             # L2 flush between timed iterations (untimed, same stream)
        out = step_resident(to_host=bool(args.dump_outputs) and s == args.steps - 1)
        torch.cuda.synchronize()
        dev_ms.append(eng.stats().feasibility_ms)
        if count_t is not None:
            ar_ms.append(ar0.elapsed_time(ar1))
    launches = eng.stats().kernel_launches - launches0
    if args.dump_outputs and rank == 0:
        bits, _, cnt = out
        dump_outputs(args.dump_outputs, bits, Pl, count_t.cpu().numpy() if count_t is not None else cnt)
    for _ in range(10):                                        # host view of a step: launch + device + synchronize
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        step_resident()
        torch.cuda.synchronize()
        wall_ms.append(1e3 * (time.perf_counter() - t0))
    kern_ms = float(np.mean(dev_ms))
    # device time of a step: the pass (CUDA events on the engine's stream) + for N>1 the NCCL all-reduce of
    # the histogram (CUDA events on torch's stream), max over ranks
    allreduce_ms = float(np.mean(ar_ms)) if ar_ms else 0.0
    step_ms = kern_ms + allreduce_ms
    step_stats = [float(np.min(dev_ms)), float(np.median(dev_ms)), float(np.percentile(dev_ms, 99)), float(np.max(dev_ms))]
    if dist is not None:
        tt = torch.tensor([step_ms, kern_ms] + step_stats, device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        step_ms, kern_ms = float(tt[0]), float(tt[1])
        step_stats = [float(x) for x in tt[2:]]
    value = (P1 * world) * T / (step_ms * 1e-3)

    # ---- parity of what was just timed -------------------------------------------------------------------
    # the result of one more resident step: the fused (or all-reduced) histogram must equal the sum over ranks of the
    # popcounts of each rank's bit rows; rank 0's rows and counts are compared with the oracle on a template slice
    parity = {"checked": False}
    try:
        step_resident()
        torch.cuda.synchronize()
        bits, _, cnt = eng.feasibility()
        if count_t is not None:
            dist.all_reduce(count_t)
            torch.cuda.synchronize()
            cnt = count_t.cpu().numpy()
        local = unpack_bits(bits, Pl).sum(axis=1).astype(np.int64)
        total = local.copy()
        if dist is not None:
            tt = torch.from_numpy(local).cuda()
            dist.all_reduce(tt)                                # NCCL sum of the per-rank histograms
            total = tt.cpu().numpy()
        ok_hist = bool(np.array_equal(np.asarray(cnt, np.int64), total))
        ok_oracle = True
        tsel = _spread(T, 32)
        if rank == 0:
            ref = _reference_subprocess(["--config", str(args.config), "--pods", str(P1 * world), "--templates", str(T),
                                         "--counts-slice", "%d:%d:%s" % (pb, pe, ",".join(str(t) for t in tsel))], timeout=600)
            ok_oracle = all(int(local[t]) == int(ref["counts"][str(t)]) for t in tsel)
        parity = {"checked": bool(ok_hist and ok_oracle), "histogram_equals_sum_of_rank_popcounts": ok_hist,
                  "rank0_counts_equal_oracle_on_templates": tsel if ok_oracle else False,
                  "how": "popcount of every rank's bit rows, NCCL all_reduce(sum) across ranks vs the %s histogram; oracle dense pass on rank 0's pods x 32 templates"
                         % ("fused peer-exchange" if fused else ("NCCL" if world > 1 else "kernel's"))}
        if dist is not None:
            tt = torch.tensor([1.0 if parity["checked"] else 0.0], device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MIN)
            parity["checked"] = bool(tt[0] > 0.5)
    except Exception as ex:
        parity = {"checked": False, "error": repr(ex)}

    # ---- e2e through the C ABI with host buffers --------------------------------------------------------
    # a tick = the pending-pod rows of this step travel H2D (cae_load_pending: the per-tick delta against the resident
    # snapshot), the dense pass runs, the bit matrix + counts travel D2H.  Also reported: the same with a FULL cae_load per
    # step (interning + every table + class matrices: round 1's definition) and the counts-only answer (no bit matrix).
    def e2e_loop(mode):
        nonlocal h2d, d2h
        ms = []
        for i in range(max(3, min(args.steps, 10)) + 1):
            torch.cuda.synchronize()
            if dist is not None:
                dist.barrier()
            t0 = time.perf_counter()
            if mode == "full":
                eng.load(enc)
            else:
                assert eng.load_pending(enc)
            up = eng.stats().h2d_bytes
            if mode == "counts":
                eng.feasibility(want_bits=False)
            else:
                eng.feasibility()
            if count_t is not None:
                dist.all_reduce(count_t)
                torch.cuda.synchronize()
            dt = 1e3 * (time.perf_counter() - t0)
            if i > 0:
                ms.append(dt)
            if mode == "delta":
                h2d, d2h = up, eng.stats().d2h_bytes
        v = float(np.mean(ms))
        if dist is not None:
            tt = torch.tensor([v], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            v = float(tt[0])
        return v

    h2d = d2h = 0
    eng.load(enc)
    e2e_full = e2e_loop("full")
    e2e_step = e2e_loop("delta")
    e2e_counts = e2e_loop("counts")
    samples = _clock_sampler_stop(sampler)
    if first_sample and first_sample.count(",") >= 5:
        samples.insert(0, [x.strip() for x in first_sample.split(",")])

    # ---- the dense pass where it is not a launch-latency test: C3 (5 x 10^8 cells) on one GPU ------------
    dense_large = None
    if world == 1 and not args.no_decision:
        try:
            enc3 = synth.generate(3)
            eng.load(enc3)
            ms3 = []
            for i in range(6):
                flush_l2()
                eng.lib.cae_feasibility(eng.h, None, None, None)
                torch.cuda.synchronize()
                if i:
                    ms3.append(eng.stats().feasibility_ms)
            m3 = float(np.median(ms3))
            alg3 = enc3.P * 12 + enc3.T * 4 + enc3.P * enc3.T // 8 + 4 * enc3.T     # W = 1 packed-rank word: same formula as `roofline`
            pk3, _ = _peak_hbm()
            dense_large = {"workload": synth.CONFIGS[3].name, "cells": enc3.P * enc3.T, "ms": m3,
                           "evals_per_s": enc3.P * enc3.T / (m3 * 1e-3),
                           "roofline": {"bound": "hbm", "algorithmic_bytes": alg3, "achieved": alg3 / (m3 * 1e-3) / 1e9, "peak": pk3,
                                        "unit": "GB/s", "frac": alg3 / (m3 * 1e-3) / 1e9 / pk3}}
            eng.load(enc)
        except Exception as ex:
            dense_large = {"error": repr(ex)}
    eng.close()

    # ---- metric 2: scale-up decision latency ------------------------------------------------------------
    decisions = []
    if not args.no_decision:
        plan = [3, 4] if world == 1 else ([4, 5] if world >= 8 else [4])
        for c in plan:
            try:
                d = decision_run(torch, dist, Engine, synth, c, rank, world, local_rank)
            except Exception as ex:
                d = {"config": c, "error": repr(ex)}
            decisions.append(d)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (feasibility_lut_kernel) -----------------------------------------
    # algorithmic bytes of the dense kernel (DESIGN.md §4): per pod W packed-rank words + 2 class ids,
    # per template W words, the bit matrix, the fit histogram
    req = enc.arrays["ps_req"][np.unique(enc.arrays["pend_spec"])]
    nbits = 0
    for a in range(req.shape[1]):
        dv = len(np.unique(req[:, a][req[:, a] > 0]))
        if dv:
            nbits += int(dv).bit_length() + 1
    Wd = max(1, (nbits + 31) // 32)
    alg_bytes = Pl * (4 * Wd + 8) + T * 4 * Wd + Pl * T // 8 + 4 * T
    peak, peak_src = _peak_hbm()
    achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
    traffic = None
    traffic_src = None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of this kernel on this workload, one `ncu --set full` capture
        tj = json.load(open(os.path.join(ROOT, "profiles", "r01_k1_traffic.json")))
        if args.config == 2 and P1 == 100_000 and T == 1000:
            traffic = int(tj["dram__bytes_read.sum"]) + int(tj["dram__bytes_write.sum"])
            traffic_src = "profiles/r01_k1_traffic.json (one `ncu --set full` capture of this kernel on this workload; not re-measured in this run)"
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "kernel": "feasibility_lut_kernel", "algorithmic_bytes": alg_bytes,
                "peak_source": peak_src,
                "note": "the contract's HBM fraction; the kernel needs ~1 bit of DRAM traffic per evaluation and is bound by "
                        "shared-memory wavefronts + fixed launch latency (see roofline_secondary and DESIGN.md)"}
    # the kernel's own stated bound: shared-memory wavefronts (ncu l1tex__data_pipe_lsu_wavefronts_mem_shared of the capture above,
    # 1.356 M per launch on C2) at one wavefront per SM per cycle
    sm_mhz = None
    cs = _clocks_summary(samples)
    if cs.get("sm_mhz"):
        sm_mhz = cs["sm_mhz"]
    roofline2 = None
    if args.config == 2 and P1 == 100_000 and T == 1000 and sm_mhz:
        wf = 1.356e6
        floor_us = wf / 148.0 / (sm_mhz * 1e6) * 1e6
        roofline2 = {"bound": "shared-memory wavefronts", "wavefronts_per_launch": wf, "floor_us": floor_us,
                     "measured_us": kern_ms * 1e3, "frac": floor_us / (kern_ms * 1e3)}

    # ---- CPU baseline: the oracle on this box's cores, bounded sample of the same workload ---------------
    # (fresh processes: the oracle's worker pool must fork before any CUDA context exists)
    cpu = {"value": None, "unit": "evals/s", "cores": 0, "kind": "port", "sample": "failed"}
    try:
        base = ["--steps", "4", "--config", str(args.config), "--pods", str(P1), "--templates", str(T)]
        cpu = _reference_subprocess(base, timeout=600)["cpu_baseline"]
        rows = []
        for th in (1, 4):
            r = _reference_subprocess(base + ["--threads", str(th), "--steps", "2"], timeout=600)["cpu_baseline"]
            rows.append({"threads": r["cores"], "value": r["value"]})
        rows.append({"threads": cpu["cores"], "value": cpu["value"]})
        cpu["rows"] = rows
        cpu["note"] = "1 thread = --predicate-parallelism=1 (every reference test), 4 = the reference's default (config/flags/flags.go:234), " \
                      "all = every core the cgroup grants, templates split across processes"
    except Exception as ex:  # the bench line must still be printed
        cpu["sample"] = "failed: %r" % (ex,)

    headline_decision = decisions[0] if decisions else None
    print(json.dumps({
        "metric": metric, "value": value, "unit": "evals/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": _config_dict(cfg, P1, T, world),
        "kernel_ms": kern_ms, "allreduce_ms": allreduce_ms,
        "step_ms_max_over_ranks": {"min": step_stats[0], "median": step_stats[1], "p99": step_stats[2], "max": step_stats[3]},
        "step_ms_rank0": [round(float(x), 5) for x in dev_ms],
        "collective": ("none" if world == 1 else ("fused exchange over NVLink peer memory inside the kernel" if fused else "NCCL all_reduce int32[T]")),
        "wall_ms_per_step": float(np.mean(wall_ms)), "clocks": cs,
        "e2e": {"value": (P1 * world) * T / (e2e_step * 1e-3), "unit": "evals/s", "ms_per_step": e2e_step,
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "what": "per step: cae_load_pending (this step's pending-pod rows, host -> device, per-pod rows re-derived) + dense pass + "
                        "device -> host of the bit matrix and the counts; nodes / templates / pod-spec tables stay resident between ticks",
                "ms_per_step_full_load": e2e_full, "value_full_load": (P1 * world) * T / (e2e_full * 1e-3),
                "ms_per_step_counts_only": e2e_counts, "value_counts_only": (P1 * world) * T / (e2e_counts * 1e-3)},
        "gpu_launches": int(launches), "parity_checked": bool(parity.get("checked")), "parity": parity,
        "roofline": roofline, "roofline_secondary": roofline2, "cpu_baseline": cpu,
        "dense_pass_large": dense_large, "decision_latency": headline_decision, "decisions": decisions}))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
