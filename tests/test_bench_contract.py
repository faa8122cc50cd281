"""Benchmark and build checks: the reference arm answers with a JSON line, the extension builds/imports, --dump-outputs writes
what the timed steps computed (all but the last test need no GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_reports_unavailable():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and "unavailable" in d and len(d["unavailable"]) > 10


def test_extension_is_built_and_importable():
    so = [f for f in os.listdir(os.path.join(ROOT, "lstm_tensorspark_b200")) if f.startswith("_C") and f.endswith(".so")]
    if not so:                                   # fresh checkout: build it (nvcc cross-compiles without a GPU)
        sys.path.insert(0, ROOT)
        import __graft_entry__ as g
        g.build()
    from lstm_tensorspark_b200.ops.cuda_ext import ext
    E = ext()
    assert E.ar_flag_words() == E.ar_max_blocks() * 16 * E.ar_slots()
    for name in ("gemm2", "gemm_generic", "lstm_seq_fwd", "lstm_seq_bwd", "fused_allreduce", "head_fwd", "head_bwd", "flat_adam", "lstm_pointwise_fwd"):
        assert hasattr(E._m, name)


def test_cuda_op_on_cpu_tensor_is_rejected_when_forced():
    import pytest
    import torch
    from lstm_tensorspark_b200.ops import functional as F
    F.set_backend("cuda_ext")
    try:
        with pytest.raises(RuntimeError):
            F.lstm_cell_step(torch.zeros(2, 3), torch.zeros(2, 4), torch.zeros(2, 4), torch.zeros(16, 3), torch.zeros(16, 4), torch.zeros(16))
    finally:
        F.set_backend("auto")


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_clock_sampler_degrades_without_a_gpu():
    cs = _bench_module().ClockSampler(0)
    cs.start()
    cs.mark()
    out = cs.stop()
    assert set(out) >= {"sm_mhz", "sm_max_mhz", "reasons"}


def test_dump_outputs_budget_and_fixed_sample(tmp_path):
    """Arrays above their share of the budget become the same seeded sample of their elements on every call; the others are
    written whole; float64 stays float64, every other dtype becomes float32."""
    import numpy as np
    mod = _bench_module()
    rng = np.random.default_rng(1)
    w = rng.standard_normal((300, 200))
    b = rng.standard_normal(7).astype(np.float16)
    budget = 3 * (4096 + 256)
    for d in ("a", "b"):
        mod.dump_outputs(str(tmp_path / d), {"loss": np.float32(2.5), "L/w": w, "L/b": b}, budget=budget)
    assert sorted(os.listdir(tmp_path / "a")) == ["L.b.npy", "L.w.npy", "loss.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= budget
    sw = np.load(tmp_path / "a" / "L.w.npy")
    assert sw.dtype == np.float64 and sw.shape == (4096 // 8,) and np.isin(sw, w).all()
    assert np.array_equal(sw, np.load(tmp_path / "b" / "L.w.npy"))
    sb = np.load(tmp_path / "a" / "L.b.npy")
    assert sb.dtype == np.float32 and np.array_equal(sb, b.astype(np.float32))
    assert float(np.load(tmp_path / "a" / "loss.npy")) == 2.5


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_steps(tmp_path):
    """--dump-outputs writes the loss of the last timed step and the variables it leaves.  The same arguments give the same
    inputs, so two runs agree up to summation order, while a run with more timed steps ends elsewhere."""
    import numpy as np
    small = ["--hidden_units", "256,256", "--in_features", "128", "--seq_len", "8", "--batch_size", "256", "--warmup", "2",
             "--no_baseline", "--no_e2e"]

    def run(steps, d):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                            "--dump-outputs", str(tmp_path / d)] + small, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        return {f[:-4]: np.load(tmp_path / d / f) for f in os.listdir(tmp_path / d)}

    a, b, c = run(3, "a"), run(3, "b"), run(6, "c")
    assert {"loss", "LSTMLayer0.weights_forget_x", "LSTMLayer1.bias_output", "Dense1.weights"} <= set(a) and set(a) == set(b) == set(c)
    assert all(v.dtype == np.float32 for v in a.values()) and sum(v.nbytes for v in a.values()) <= 64_000_000
    assert abs(float(a["loss"]) - float(b["loss"])) <= 1e-2 * abs(float(b["loss"]))
    cat = lambda o: np.concatenate([o[k].ravel() for k in sorted(o) if k != "loss"])
    assert np.abs(cat(a) - cat(b)).mean() < 0.1 * np.abs(cat(a) - cat(c)).mean()
