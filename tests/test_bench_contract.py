"""CPU: the parts of bench.py's contract that need no GPU -- the reference arm is rank 0's job alone (other ranks of
a torchrun launch exit 0 without work or output), and the product arm refuses to run without a CUDA device
instead of falling back to anything."""
import os
import subprocess
import sys

from conftest import ROOT

BENCH = os.path.join(ROOT, "bench.py")


def _run(args, **env):
    e = dict(os.environ, **{k: str(v) for k, v in env.items()})
    return subprocess.run([sys.executable, BENCH] + args, env=e, capture_output=True, text=True, timeout=300)


def test_reference_arm_other_ranks_exit_quietly():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"], RANK=1, WORLD_SIZE=2, LOCAL_RANK=1)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        return                                    # on a GPU box the arm runs; covered by the driver
    r = _run(["--steps", "1", "--warmup", "1", "--skip-cpu-baseline"], CUDA_VISIBLE_DEVICES="")
    assert r.returncode != 0
    assert "CUDA" in r.stderr
    assert '"metric"' not in r.stdout             # no bench line is printed without the kernels


def test_cli_flags():
    r = _run(["--help"])
    assert r.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--scaling", "--shard-degree", "--exchange",
                 "--dump-outputs"):
        assert flag in r.stdout


def test_zero_steps_is_refused():
    r = _run(["--steps", "0"])
    assert r.returncode == 2 and "--steps" in r.stderr


def test_dump_outputs_dtypes_and_values(tmp_path):
    import numpy as np
    import torch
    import bench                                  # the repository root is on sys.path (conftest)
    out = {"ids": torch.tensor([[3, 1 << 30]], dtype=torch.int32), "scores": torch.tensor([[0.5, -1.25]]),
           "u": torch.tensor([[1.5]], dtype=torch.bfloat16), "metric_sums": torch.ones(4, 3, dtype=torch.float64),
           "note": "not an array"}
    bench.dump_outputs(out, str(tmp_path / "d"))
    got = {p.stem: np.load(p) for p in (tmp_path / "d").iterdir()}
    assert set(got) == {"ids", "scores", "u", "metric_sums"}
    assert got["ids"].dtype == np.float64 and got["ids"].tolist() == [[3.0, float(1 << 30)]]
    assert got["scores"].dtype == np.float32 and got["scores"].tolist() == [[0.5, -1.25]]
    assert got["u"].dtype == np.float32 and got["metric_sums"].dtype == np.float64
