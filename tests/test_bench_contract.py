"""bench.py's reference arm runs on the host cores (no GPU): its JSON line must carry the driver's contract --
same metric / unit / config keys as the GPU arm, `impl`, `cpu_baseline`, and an `e2e` with zero copy bytes.  Under
torchrun only rank 0 prints; the other ranks exit 0 without work.  `--dump-outputs` writes what the GPU arm's last timed
step computed, the same files from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--offers", "1500"], capture_output=True, text=True, timeout=240, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_reference_arm_line():
    lines = run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "offer-scores/sec (PxG)" and d["unit"] == "offer-scores/s"
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "pods x 1500 offers" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_stay_silent():
    assert run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []


def test_dump_outputs_sample_is_fixed_and_exact(tmp_path):
    """Short arrays are written whole; a long one as the same seeded row sample every time, its row numbers beside it."""
    from bench import DUMP_MAX_ROWS, dump_outputs

    long = np.arange(DUMP_MAX_ROWS + 12345, dtype=np.uint32) * 3
    short = np.array([-1, 0, 99_999], np.int32)
    for d in ("a", "b"):
        dump_outputs(str(tmp_path / d), {"long": long, "short": short})
    assert sorted(os.listdir(tmp_path / "a")) == ["long.npy", "long_rows.npy", "short.npy"]
    for f in os.listdir(tmp_path / "a"):
        x, y = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert x.dtype == np.float64 and np.array_equal(x, y), f
    rows = np.load(tmp_path / "a" / "long_rows.npy").astype(np.int64)
    assert len(rows) == DUMP_MAX_ROWS and (np.diff(rows) > 0).all()
    assert np.array_equal(np.load(tmp_path / "a" / "long.npy"), long[rows])
    assert np.array_equal(np.load(tmp_path / "a" / "short.npy"), short)


@pytest.mark.gpu
def test_dump_outputs_same_in_both_launch_modes(tmp_path):
    """--dump-outputs on a small workload: graph replay and eager launches write the same files, `steps` is what was
    asked for, and the dumped assignment vector and changed list are the oracle's."""
    import oracle
    import rpk

    P, G, NS = 30_000, 4_000, 20_000
    dumps = {}
    for launch in ("graph", "eager"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "4", "--warmup", "3", "--pods", str(P),
                              "--offers", str(G), "--slots", str(NS), "--no-cpu-baseline", "--no-e2e", "--no-k2-sweep",
                              "--stream-seconds", "0", "--launch", launch, "--dump-outputs", str(tmp_path / launch)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-3000:]
        line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 4 and line["parity"]["ok"]
        dumps[launch] = {f: np.load(tmp_path / launch / f) for f in os.listdir(tmp_path / launch)}
    assert sorted(dumps["graph"]) == ["best.npy", "status_changed.npy", "status_codes.npy"]
    for f, x in dumps["graph"].items():
        assert np.array_equal(x, dumps["eager"][f]), f
    want, _ = oracle.select(rpk.synth.make_offers(G), rpk.synth.make_pods(P), want_top5=False, n_threads=8)
    assert np.array_equal(dumps["graph"]["best.npy"], want)
    tabs = [rpk.synth.make_status_records(NS, 0), rpk.synth.make_status_records(NS, 1, 0.01)]
    t = oracle.StatusTable(NS)
    t.diff(tabs[0])
    changed = t.diff(tabs[1])   # the steps alternate between the two tables: either direction changes the same slots
    assert len(changed) > 0 and np.array_equal(dumps["graph"]["status_changed.npy"], changed)
    codes = dumps["graph"]["status_codes.npy"]
    assert any(np.array_equal(codes, oracle.record_codes(tab)[changed]) for tab in tabs)
