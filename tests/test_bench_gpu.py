"""GPU: bench.py's headline arm times exactly --steps steps, and --dump-outputs writes what the last of them
returned, equal to the module path on the same seeded batch."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]


def test_steps_and_dump_outputs(tmp_path, cuda):
    # 5 batches; warm-up steps 0..2, timed steps 3..9 = batches 3, 4 | 0, 1, 2, 3, 4 (two launches), last = batch 4
    G, B, K, W = 5 * 4096, 4096, 7, 3
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--graphs", str(G), "--batch", str(B),
                          "--steps", str(K), "--warmup", str(W), "--no-e2e", "--no-cpu-baseline", "--no-secondary",
                          "--dump-outputs", str(tmp_path / "d")], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == K and line["timed_steps"] == K and line["gpu_launches"] == 2
    got = np.load(tmp_path / "d" / "out.npy")
    lb = np.load(tmp_path / "d" / "lut_batch.npy")
    assert got.dtype == np.float32 and lb.dtype == np.float64

    from gnn_qot_estimation_b200 import LightpathGNN, synthetic
    m = LightpathGNN(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    m.load_state_dict(torch.load(ROOT / "tests" / "golden" / "ckpt_lightpath_model_1.pt",
                                 weights_only=False)["model_state_dict"], strict=True)
    m.to(cuda).eval()
    store = synthetic.lightpath_store(G, seed=1, device=cuda)
    assert store.verify_layout()
    with torch.no_grad():
        ref, ref_lb = m(store.collate(range(4 * B, 5 * B)))
    assert got.shape == (B, 3)
    assert np.array_equal(lb, ref_lb.double().cpu().numpy())
    np.testing.assert_allclose(got, ref.cpu().numpy(), rtol=1e-5, atol=2e-6)
