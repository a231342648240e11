"""bench.py's contract on the CPU side: the reference arm (`--impl reference`: the oracle port on the host
cores) prints exactly ONE JSON line with the keys the driver reads, and under a multi-rank launch only rank 0
prints.  `--dump-outputs` writes what the timed path returned in its last step, identically on every run with
the same arguments (the engine arm needs a B200: marked gpu)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE_ARGS = ["--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample", "24", "--n-in", "200"]


def _run(env_extra=None, args=REFERENCE_ARGS, one_cpu=False):
    """one_cpu: pin bench.py to one CPU, so that the reference arm's sample, which grows with the physical
    core count, is --cpu-sample services on every host."""
    env = dict(os.environ)
    env.update(env_extra or {})
    cpu = {min(os.sched_getaffinity(0))}
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args,
                         capture_output=True, text=True, env=env, timeout=300,
                         preexec_fn=(lambda: os.sched_setaffinity(0, cpu)) if one_cpu else None)
    assert res.returncode == 0, res.stderr[-2000:]
    return res.stdout.strip()


def _dumped(d):
    return {p.name[:-4]: np.load(p) for p in sorted(d.iterdir())}


def test_reference_arm_prints_one_json_line():
    out = _run()
    assert len(out.splitlines()) == 1
    d = json.loads(out)
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["unit"] == "spans/s" and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_zero_steps_are_refused():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=300)
    assert res.returncode != 0 and "--steps" in res.stderr and res.stdout == ""


def test_reference_arm_other_ranks_stay_silent():
    assert _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}) == ""


def test_reference_arm_dumps_the_same_outputs_on_every_run(tmp_path):
    runs = []
    for name in ("a", "b"):
        out = _run(args=REFERENCE_ARGS + ["--dump-outputs", str(tmp_path / name)], one_cpu=True)
        assert len(out.splitlines()) == 1
        runs.append(_dumped(tmp_path / name))
    a, b = runs
    assert {"assign", "mis_rank", "counters", "topk_score", "topk_idx"} <= set(a) and set(a) == set(b)
    for k in a:
        assert a[k].dtype == np.float64 and np.all(np.isfinite(a[k])) and np.array_equal(a[k], b[k]), k
    assert a["assign"].min() >= -1 and np.array_equal(a["assign"], np.round(a["assign"]))
    # 24 services: written whole.  The empty slots of the top-K lists (past topk_cnt) are 0
    empty = np.arange(a["topk_score"].shape[1])[None, :] >= a["topk_cnt"][:, None]
    assert empty.any() and np.all(a["topk_score"][empty] == 0.0)
    assert a["topk_idx"].shape == (len(a["assign"]), 5)                  # one top-K row per tuple


def test_dump_outputs_keeps_a_fixed_sample_of_rows_under_64_mb(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    arrays = {"assign": np.arange(30_000_000, dtype=np.int32),
              "topk_score": np.arange(10_000_000, dtype=np.float64).reshape(-1, 5),
              "topk_cnt": np.full(2_000_000, 5, np.uint8),
              "counters": np.arange(4096 * 4, dtype=np.int32).reshape(-1, 4)}
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64 * 10 ** 6
    a, b = _dumped(tmp_path / "a"), _dumped(tmp_path / "b")
    assert all(np.array_equal(a[k], b[k]) for k in arrays)
    assert np.array_equal(a["counters"], arrays["counters"])                # small outputs are written whole
    s = a["assign"]
    assert 0 < len(s) < len(arrays["assign"]) and np.all(np.diff(s) > 0)    # rows of the output, in order
    t = a["topk_score"]
    assert t.shape[1] == 5 and np.all(t[:, 0] % 5 == 0) and np.all(t[:, 1:] - t[:, :-1] == 1)   # whole rows
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "c"), {"mix": np.array([1.0, np.inf])})


def test_topk_rows_regroup_the_flat_layout_per_tuple():
    """topk_idx[K * (tuple_off[p] + i*E) + r*E + e] (include/traceweaver_b200.h) -> row (tuple_off[p] + i*E + e, r),
    on two services with different callee counts."""
    sys.path.insert(0, ROOT)
    import bench
    from types import SimpleNamespace
    K = 5
    hb = SimpleNamespace(prob_ep_off=np.array([0, 2, 5]), prob_tuple_off=np.array([0, 2 * 3, 2 * 3 + 3 * 2]))
    flat = np.full(K * 12, -7, np.int32)
    want = np.zeros((12, K), np.int32)
    for p, (E, n) in enumerate(((2, 3), (3, 2))):
        for i in range(n):
            for e in range(E):
                t = int(hb.prob_tuple_off[p]) + i * E + e
                for r in range(K):
                    flat[K * (int(hb.prob_tuple_off[p]) + i * E) + r * E + e] = want[t, r] = 100 * t + r
    assert np.array_equal(bench.topk_rows(flat, hb), want)


@pytest.mark.gpu
def test_engine_arm_steps_and_dumped_outputs(tmp_path):
    """--steps sets the timed steps (the launch count of the timed window scales with it); the dump holds
    the engine's last-step arrays and repeats exactly on a second run with the same arguments."""
    base = ["--gpus", "1", "--warmup", "1", "--services", "48", "--n-in", "120", "--cpu-sample", "12", "--no-extra"]
    lines, dumps = [], []
    for k, name in ((1, "a"), (3, "b")):
        out = _run(args=base + ["--steps", str(k), "--dump-outputs", str(tmp_path / name)])
        assert len(out.splitlines()) == 1
        lines.append(json.loads(out))
        dumps.append(_dumped(tmp_path / name))
    one, three = lines
    assert one["steps"] == 1 and three["steps"] == 3
    assert one["gpu_launches"] > 0 and three["gpu_launches"] == 3 * one["gpu_launches"]
    a, b = dumps
    assert {"assign", "assign_pass0", "mis_rank", "n_cand", "counters", "topk_score", "topk_idx", "topk_cnt", "cut",
            "params_pass1"} <= set(a) and set(a) == set(b)
    for k in a:
        assert a[k].dtype == np.float64 and np.all(np.isfinite(a[k])) and np.array_equal(a[k], b[k]), k
    n_in = 48 * 120                                   # small enough to be written whole
    assert len(a["mis_rank"]) == n_in and len(a["assign"]) == three["config"]["spans_total"] - n_in
    assert len(a["counters"]) == 48 and a["assign"].min() >= -1
    empty = np.arange(a["topk_score"].shape[1])[None, :] >= a["topk_cnt"][:, None]
    assert np.all(a["topk_score"][empty] == 0.0)
    assert a["topk_idx"].shape == (len(a["assign"]), 5)
