"""CPU: the bench.py JSON-line contract on the arm that runs without a GPU (`--impl reference`, tiny config), and that the
product arm refuses to run without a GPU instead of falling back.  GPU: the outputs --dump-outputs writes."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=300,
                          cwd=ROOT)


def test_reference_arm_json_line():
    r = _run("--impl", "reference", "--model", "tiny", "--batch", "2", "--ctx", "16", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-400:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1  # exactly ONE JSON line
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "tokens/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_nonzero_rank_is_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--model", "tiny", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_reference_arm_times_the_steps_it_prints_and_loads_no_product_code():
    """VERDICT r1: the reference arm printed `steps: 20` while timing <= 4 and imported the product package (which maps
    libb200spark.so into the reference process).  Now: `steps` timed steps are really run (steps x ms_per_step ~ the wall
    time of the timed region) and no b200spark module / native library is loaded."""
    code = ("import sys, json, io, contextlib, time; sys.argv = ['bench.py', '--impl', 'reference', '--model', 'tiny', '--batch', '2', "
            "'--ctx', '16', '--steps', '7', '--warmup', '2']; import bench; buf = io.StringIO(); t0 = time.perf_counter()\n"
            "with contextlib.redirect_stdout(buf): bench.main()\n"
            "wall = time.perf_counter() - t0; d = json.loads(buf.getvalue().strip().splitlines()[-1])\n"
            "maps = open('/proc/self/maps').read()\n"
            "print(json.dumps({'steps': d['steps'], 'warmup': d['warmup'], 'timed_s': d['steps'] * d['ms_per_step'] * 1e-3, 'wall': wall,\n"
            "  'b2_modules': [m for m in sys.modules if m.startswith('b200spark')], 'so': 'libb200spark' in maps or 'liballspark_b200' in maps}))")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-600:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["steps"] == 7 and d["warmup"] == 2
    assert d["b2_modules"] == [] and d["so"] is False
    assert d["timed_s"] <= d["wall"]  # the claimed timed region fits inside the run


def test_reference_arm_sets_threads_under_torchrun():
    env = dict(os.environ, RANK="0", WORLD_SIZE="2", LOCAL_RANK="0", OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--model", "tiny", "--batch", "2", "--ctx",
                        "16", "--steps", "1", "--warmup", "1", "--gpus", "2"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-400:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    sys.path.insert(0, ROOT)
    import bench
    assert d["cpu_baseline"]["cores"] == bench.physical_cores()


def test_steps_below_one_are_refused():
    r = _run("--impl", "reference", "--model", "tiny", "--steps", "0")
    assert r.returncode == 2 and "--steps" in r.stderr


def test_dump_outputs_keeps_to_64_mb(tmp_path):
    """Logits larger than the budget are cut to a seeded sample of vocabulary columns, the same from run to run."""
    import numpy as np
    import torch
    from types import SimpleNamespace
    sys.path.insert(0, ROOT)
    import bench
    logits = torch.randn(128, 152064, generator=torch.Generator().manual_seed(0)).to(torch.bfloat16)
    st = SimpleNamespace(next_ids=logits.float().argmax(1), logits=logits)
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(st, str(d))
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["logits.npy", "logits_columns.npy", "next_ids.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64_000_000
    out = {f: np.load(tmp_path / "a" / f) for f in files}
    cols = out["logits_columns.npy"]
    assert cols.dtype == np.float64 and np.all(np.diff(cols) > 0) and cols[-1] < 152064
    assert out["logits.npy"].dtype == np.float32
    assert np.array_equal(out["logits.npy"], logits.float().numpy()[:, cols.astype(np.int64)])
    assert np.array_equal(out["next_ids.npy"], st.next_ids.numpy())
    for f in files:
        assert np.array_equal(out[f], np.load(tmp_path / "b" / f))


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """--dump-outputs writes the next_ids / logits of the last timed step; the same arguments give the same arrays."""
    import numpy as np
    dumps = []
    for run in ("a", "b"):
        d = tmp_path / run
        r = _run("--model", "tiny", "--batch", "4", "--ctx", "64", "--steps", "3", "--warmup", "1", "--sub-batches", "",
                 "--no-cpu", "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr[-400:]
        dumps.append({n: np.load(d / (n + ".npy")) for n in ("next_ids", "logits")})
    ids, logits = dumps[0]["next_ids"], dumps[0]["logits"]
    assert ids.dtype == np.float64 and logits.dtype == np.float32 and logits.shape == (4, 1024)
    assert np.array_equal(ids, logits.argmax(1))
    for n in ("next_ids", "logits"):
        assert np.array_equal(dumps[0][n], dumps[1][n]), n
