import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_reports_unavailable():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1",
                        "--steps", "5", "--warmup", "3"], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and "unavailable" in d and "TensorFlow" in d["unavailable"]


@pytest.mark.gpu
def test_bench_steps_and_dump_outputs(tmp_path):
    """`--steps` is the number of timed steps, and `--dump-outputs` writes what the last of them returned plus the
    variables they left on the ps, as float32 arrays."""
    import numpy as np
    from dist_mnist_b200.models import mlp

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "37", "--warmup", "5",
                        "--skip_e2e", "--skip_parity", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 37 and d["config"]["global_step_after_run"] == 5 + 37   # warm-up steps, then the timed ones
    spec = mlp.get_model("book", 100)
    expected = {"loss": (1,), "correct": (1,)}
    expected.update({"var_" + k.replace("/", "__"): tuple(v.shape) for k, v in mlp.init_params(spec, seed=0).items()})
    got = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert {k: v.shape for k, v in got.items()} == expected
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in got.values())
    assert 0 < got["loss"][0] < 10 and 0 <= got["correct"][0] <= 32
    init = mlp.init_params(spec, seed=0)   # the variables the run started from: training moved them
    assert any(not np.array_equal(got["var_" + k.replace("/", "__")], v.numpy()) for k, v in init.items())


def test_graft_entry_build():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    g.build()


def test_bench_defaults_and_config_are_consistent():
    sys.path.insert(0, ROOT)
    import bench
    from dist_mnist_b200.models import mlp
    from dist_mnist_b200.parallel.config import OptimizerConfig
    a = bench.parse_args([])
    assert a.gpus == 1 and a.steps >= 100 and a.warmup >= 3 and a.optimizer == "adam" and a.batch_size == 32
    assert a.dump_outputs is None and bench.parse_args(["--dump-outputs", "out"]).dump_outputs == "out"
    # the configuration bench.py derives from its defaults must validate and select the fused engine for the
    # reference's live model (784-100-10, batch 32)
    cfg = bench.engine_config(a)
    cfg.validate(OptimizerConfig("adam", 1e-4))
    assert cfg.nslots >= cfg.lanes
    assert cfg.resolve_engine(mlp.get_model(a.model, a.hidden_units), a.batch_size) == "fused"
