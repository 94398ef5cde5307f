"""bench.py's output contract: our arm must run (here: the CPU dry run on gloo with a tiny model), print ONE JSON line with
the agreed keys, and spell the benchmark configuration exactly as the reference arm does.  The reference is not part of
this repository, so its side of the comparison is the lines its arm printed on the same arguments, stored under
tests/golden/."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "bench_reference_arm.json")
COMMON = ["--device", "cpu", "--model", "bloom-tiny", "--seq-len", "32", "--batch-per-gpu", "2", "--steps", "2", "--warmup", "3"]


def _run(extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + COMMON + extra, capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:] + out.stderr[-2000:]
    return json.loads(lines[0])


def _reference_line(extra):
    """The line ``bench.py --impl reference`` printed for COMMON + ``extra`` with the unmodified reference installed."""
    with open(GOLDEN) as f:
        return json.load(f)["lines"][" ".join(extra)]


def test_layout_and_config_helpers():
    sys.path.insert(0, ROOT)
    import argparse

    import bench

    def args(**kw):
        base = dict(gpus=8, tp=0, pp=1, model="bloom-560m", batch_per_gpu=8, seq_len=1024, microbatches=8, experts=0)
        base.update(kw)
        return argparse.Namespace(**base)

    assert bench.layout_of(args(gpus=1)) == (1, 1, 1)
    assert bench.layout_of(args(gpus=2)) == (2, 1, 1)
    assert bench.layout_of(args(gpus=8)) == (2, 1, 4)                      # BASELINE.json's headline: TP2 x DP4
    assert bench.layout_of(args(gpus=8, tp=8)) == (8, 1, 1)                # config #3 / #4
    assert bench.layout_of(args(gpus=8, tp=2, pp=2)) == (2, 2, 2)          # config #5
    cfg = bench.config_of(args(gpus=8), 2, 1, 4)
    assert cfg["parallelism"] == "tp2dp4+zero1" and cfg["global_batch"] == 64 and cfg["model"] == "bloom-560m"
    assert bench.config_of(args(gpus=8, tp=8, experts=8), 8, 1, 1)["parallelism"] == "tp8dp1+moe8e"


@pytest.mark.parametrize("extra", [["--gpus", "1"], ["--gpus", "2"], ["--gpus", "2", "--hf"]])
def test_both_arms_print_one_json_line_with_the_same_config(extra):
    ours = _run(extra)
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype",
                "data", "config", "e2e", "gpu_launches", "clocks"):
        assert key in ours, key
    assert ours["e2e"]["h2d_bytes_per_step"] > 0 and ours["e2e"]["d2h_bytes_per_step"] == 4
    if "--hf" in extra:
        return
    ref = _reference_line(extra)
    assert ref["impl"] == "reference"
    assert ref["config"] == ours["config"] and ref["metric"] == ours["metric"]
    if extra[-1] != "1":
        assert ours["numerics_ok"] is True      # the self-check ran (on CPU both engines are the library path)


def test_dump_outputs_are_reproducible_and_follow_steps(tmp_path):
    """``--dump-outputs``: the same arguments give the same outputs; one more timed step gives other weights."""
    import numpy as np

    dumps = {}
    for name, steps in (("a", "2"), ("b", "2"), ("c", "3")):
        line = _run(["--gpus", "1", "--dump-outputs", str(tmp_path / name), "--steps", steps])   # the later --steps wins
        assert line["steps"] == int(steps)
        dumps[name] = {f: np.load(tmp_path / name / f) for f in ("loss.npy", "weights_sample.npy")}
        assert float(dumps[name]["loss.npy"]) == line["final_loss"]
    a, b, c = dumps["a"], dumps["b"], dumps["c"]
    assert a["loss.npy"].dtype == np.float64 and a["loss.npy"].shape == ()
    assert a["weights_sample.npy"].dtype == np.float32 and 0 < a["weights_sample.npy"].nbytes <= 64 << 20
    for f in a:
        assert np.array_equal(a[f], b[f]), f
    assert not np.array_equal(a["weights_sample.npy"], c["weights_sample.npy"])


def test_moe_config_both_arms_and_the_reference_arm_in_bf16():
    """BASELINE.json config #4 shape (Switch-MoE, experts sharded over the tensor group).  The reference arm's line was
    recorded with the model cast to bf16 as on the GPU: its router stays fp32 (it casts its own input)."""
    extra = ["--gpus", "2", "--tp", "2", "--experts", "2"]
    ours = _run(extra + ["--no-self-check"])
    ref = _reference_line(extra)
    assert ref["impl"] == "reference" and ref["config"] == ours["config"]
    assert ours["config"]["parallelism"] == "tp2dp1+moe2e"
    for line in (ours, ref):
        assert line["final_loss"] == line["final_loss"] and 0 < line["final_loss"] < 20   # finite, of the order of ln(vocab)
