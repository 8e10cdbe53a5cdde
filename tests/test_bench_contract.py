"""bench.py's reference arm runs without a GPU: its JSON line must carry the benchmark's keys, the SAME config dict the engine
arm prints (both lines describe one workload), and the parity / decision legs must answer through the oracle.  The engine
arm's --dump-outputs writes what its last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args, timeout=300):
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True,
                          timeout=timeout, env=env)


def _ref(*extra):
    out = _bench("--impl", "reference", "--pods", "3000", "--templates", "24", *extra)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_steps_must_be_positive():
    out = _bench("--impl", "reference", "--steps", "0")
    assert out.returncode == 2 and "--steps" in out.stderr


def test_dump_outputs_unpacks_and_samples_pods_above_the_budget(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    from kubernetes_autoscaler_b200.engine import unpack_bits
    rng = np.random.default_rng(1)
    small = rng.integers(0, 2 ** 32, (24, 94), dtype=np.uint32)
    bench.dump_outputs(str(tmp_path / "small"), small, 3000, np.arange(24, dtype=np.int32))
    fit = np.load(tmp_path / "small" / "fit.npy")
    assert fit.dtype == np.float32 and np.array_equal(fit, unpack_bits(small, 3000))
    assert np.array_equal(np.load(tmp_path / "small" / "fit_pods.npy"), np.arange(3000))
    big = rng.integers(0, 2 ** 32, (200, 3125), dtype=np.uint32)           # 200 x 100 000 verdicts = 80 MB as float32
    bench.dump_outputs(str(tmp_path / "big"), big, 100_000, np.arange(200, dtype=np.int32))
    assert sum(f.stat().st_size for f in (tmp_path / "big").iterdir()) <= bench.DUMP_BYTES
    pods = np.load(tmp_path / "big" / "fit_pods.npy").astype(np.int64)
    assert len(pods) > 79_000 and np.all(np.diff(pods) > 0) and pods[-1] < 100_000
    assert np.array_equal(np.load(tmp_path / "big" / "fit.npy"), unpack_bits(big, 100_000)[:, pods])
    assert np.array_equal(np.load(tmp_path / "big" / "fit_count.npy"), np.arange(200))
    with pytest.raises(ValueError):                                       # not even one pod column of every template fits
        bench.dump_outputs(str(tmp_path / "huge"), np.broadcast_to(np.uint32(0), (20_000_000, 1)), 32, np.zeros(1))


@pytest.mark.gpu
def test_engine_arm_dumps_its_last_step(tmp_path, oracle):
    from kubernetes_autoscaler_b200 import synth
    out = _bench("--pods", "3000", "--templates", "24", "--steps", "3", "--warmup", "3", "--no-decision",
                 "--dump-outputs", str(tmp_path), timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["steps"] == 3 and len(d["step_ms_rank0"]) == 3 and d["parity_checked"]
    want, _ = oracle.feasibility_dense(synth.generate(2, pods=3000, templates=24))
    fit = np.load(tmp_path / "fit.npy")
    assert fit.dtype == np.float32 and np.array_equal(fit, want == 0)
    assert np.array_equal(np.load(tmp_path / "fit_count.npy"), (want == 0).sum(axis=1))
    assert np.array_equal(np.load(tmp_path / "fit_pods.npy"), np.arange(3000))


def test_reference_arm_line():
    d = _ref("--steps", "2", "--threads", "2")
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "evals/s" and d["higher_is_better"] is True and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] <= 2 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    sys.path.insert(0, ROOT)
    import bench
    from kubernetes_autoscaler_b200 import synth
    assert d["config"] == bench._config_dict(synth.CONFIGS[2], 3000, 24, 1)      # identical to the engine arm's dict


def test_reference_arm_parity_and_decision_legs(oracle):
    from kubernetes_autoscaler_b200 import synth
    enc = synth.generate(2, pods=3000, templates=24)
    want, _ = oracle.feasibility_dense(enc, p_range=(64, 2048), t_range=(0, 24))
    d = _ref("--counts-slice", "64:2048:0,5,23")
    assert {int(k): v for k, v in d["counts"].items()} == {t: int((want[t] == 0).sum()) for t in (0, 5, 23)}
    d = _ref("--decision-templates", "1,7", "--cap", "40")
    onc, opc, _, _, _ = oracle.estimate_all(enc, np.full(enc.T, 40, np.int32))
    assert [(r["t"], r["nodes"], r["pods"]) for r in d["templates"]] == [(1, int(onc[1]), int(opc[1])), (7, int(onc[7]), int(opc[7]))]
    assert all(r["filter_evals"] > 0 for r in d["templates"])


def test_slice_pods_is_the_dense_pass_of_the_shard(oracle):
    """EncodedObjects.slice_pods (what a rank uploads with CAE_CFG_PODS_PRESHARDED): the dense verdicts of the slice are the
    columns of the full pass; group offsets are clipped to the range."""
    from kubernetes_autoscaler_b200 import synth
    enc = synth.generate(3, pods=1200, templates=10, cluster_nodes=20)
    full, _ = oracle.feasibility_dense(enc)
    for pb, pe in ((0, 1200), (96, 640), (640, 1200), (500, 500)):
        sub = enc.slice_pods(pb, pe)
        assert sub.P == pe - pb and sub.E == enc.E and sub.T == enc.T
        go = sub.arrays["group_off"]
        assert go[0] == 0 and go[-1] == pe - pb and np.all(np.diff(go) >= 0)
        got, _ = oracle.feasibility_dense(sub)
        assert np.array_equal(got, full[:, pb:pe])
    assert enc.P == 1200 and enc.arrays["group_off"][-1] == 1200     # the parent is untouched
