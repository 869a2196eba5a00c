"""bench.py's contract on a box without a GPU: the reference arm (the CPU restatement) prints one JSON
line with the keys its readers expect, and the product arm refuses to run rather than fall back.  On
the GPU: --steps sets the number of timed runs, --dump-outputs writes what the last one computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), cwd=ROOT, env=e,
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)


def test_reference_arm_line():
    r = _run("--impl", "reference", "--shape", "small", "--ref-lattices", "24", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [x for x in r.stdout.splitlines() if x.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "arcs/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("lattice arcs/sec") and d["steps"] == 2 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "arcs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None and d["config"]["tool"] == "frame_post"


def test_reference_arm_other_ranks_stay_silent():
    r = _run("--impl", "reference", "--shape", "small", "--ref-lattices", "8", "--steps", "1", "--warmup", "0",
             env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = _run("--shape", "tiny", "--lattices", "4", "--steps", "1", "--no-tools", "--no-cpu-baseline", "--e2e-steps", "0",
             env={"CUDA_VISIBLE_DEVICES": ""})
    assert r.returncode != 0  # klu_create fails: no CPU fallback
    assert not [x for x in r.stdout.splitlines() if x.startswith("{")]


def test_steps_below_one_is_an_error():
    r = _run("--impl", "reference", "--shape", "tiny", "--ref-lattices", "4", "--steps", "0")
    assert r.returncode == 2 and "--steps" in r.stderr and not r.stdout.strip()


@pytest.mark.gpu
def test_dump_outputs_and_steps(klu, engine, tmp_path):
    """The dump holds the rows the timed tool's last step returns for a fixed sample of lattices, in
    float32 / float64 only, identical in two runs; twice the steps launch twice the kernels."""
    args = ["--shape", "tiny", "--lattices", "100", "--warmup", "1", "--no-tools", "--no-cpu-baseline",
            "--e2e-steps", "0"]
    lines, dumps = [], []
    for steps in (2, 4):
        d = tmp_path / ("steps%d" % steps)
        r = _run(*args, "--steps", str(steps), "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr[-2000:]
        lines.append(json.loads([x for x in r.stdout.splitlines() if x.startswith("{")][0]))
        dumps.append({f[:-4]: np.load(str(d / f)) for f in os.listdir(str(d))})
    assert [x["steps"] for x in lines] == [2, 4]
    assert lines[1]["gpu_launches"] == 2 * lines[0]["gpu_launches"] > 0
    a, b = dumps
    assert set(a) == set(b) == {"rows", "num_frames", "sample", "frame_row_off", "word", "logp"}
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and np.array_equal(a[k], b[k]), k
    engine.load(klu.synth_batch("tiny", 100, seed=0x5EED))
    engine.run(klu.FRAME_POST, acoustic_scale=0.1)
    off, nf, fo, w, lp = engine.fetch_frame_post_csr()
    sample = a["sample"].astype(np.int64)
    assert len(sample) == 64 and (np.diff(sample) > 0).all()
    assert np.array_equal(a["rows"], np.diff(off)) and np.array_equal(a["num_frames"], nf)
    slots = np.concatenate([[0], np.cumsum(nf.astype(np.int64) + 1)])
    for name, x, o in (("word", w, off), ("logp", lp, off), ("frame_row_off", fo, slots)):
        assert np.array_equal(a[name], np.concatenate([x[o[l]:o[l + 1]] for l in sample])), name
