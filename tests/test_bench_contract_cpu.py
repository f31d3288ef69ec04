"""CPU check of the bench.py contract pieces that do not need a GPU: the reference arm prints one
JSON line with the agreed keys (it times the CPU oracle), and the B200 arm refuses to run without
CUDA instead of falling back."""
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]


def test_reference_arm_line():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1", "--batch", "256"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "lightpath_infer_graphs_per_sec"
    assert line["unit"] == "graphs/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["e2e"]["value"] == line["value"]


def test_reference_arm_dumps_its_last_step(tmp_path):
    """--dump-outputs writes what the last timed step returned: with --steps 3 that is the oracle on batch 2 of
    the arm's four seeded batches."""
    import numpy as np
    import torch
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "3",
                          "--warmup", "1", "--batch", "256", "--dump-outputs", str(tmp_path / "d")],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    got = np.load(tmp_path / "d" / "out.npy")
    lb = np.load(tmp_path / "d" / "lut_batch.npy")
    assert got.dtype == np.float32 and lb.dtype == np.float64
    from gnn_qot_estimation_b200 import synthetic
    from oracle import LightpathGNNOracle
    hb = synthetic.lightpath_store(4 * 256, seed=1, device="cpu").host_batch(512, 768)
    m = LightpathGNNOracle(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    m.load_state_dict(torch.load(ROOT / "tests" / "golden" / "ckpt_lightpath_model_1.pt",
                                 weights_only=False)["model_state_dict"], strict=True)
    with torch.no_grad():
        ref, ref_lb = m.eval()(hb)
    assert np.array_equal(lb, ref_lb.double().numpy())
    np.testing.assert_allclose(got, ref.numpy(), rtol=1e-5, atol=2e-6)


def test_dump_outputs_samples_rows_past_the_cap(tmp_path):
    import numpy as np
    import torch
    import bench
    out = torch.rand(1000, 3)
    idx = torch.arange(1000)
    bench.dump_outputs(str(tmp_path), {"out": out, "lut_batch": idx}, cap=8000)
    rows = np.load(tmp_path / "rows.npy")
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= 8000 + 3 * 128      # data + one .npy header each
    assert np.array_equal(np.load(tmp_path / "lut_batch.npy"), rows)
    assert np.array_equal(np.load(tmp_path / "out.npy"), out.numpy()[rows.astype(np.int64)])


def test_b200_arm_needs_cuda():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode != 0 and "CUDA" in out.stderr
