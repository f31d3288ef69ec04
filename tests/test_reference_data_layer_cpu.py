"""Check against the upstream project's own source, which this repository does not contain (runs only when
QOT_REFERENCE names a checkout of it): the REFERENCE's own data layer -- topological_training/dataset.py and
lightpath_training/dataset.py, imported unchanged from that checkout -- runs on top of the torch_geometric stand-in
(gnn_qot_estimation_b200.pyg_compat), and the batches it yields are what the models consume."""
import os
import pickle
import sys
from pathlib import Path

import networkx as nx
import numpy as np
import pytest
import torch

REF = Path(os.environ["QOT_REFERENCE"]) if os.environ.get("QOT_REFERENCE") else None   # santiagolmedo/gnn_qot_estimation
pytestmark = pytest.mark.skipif(REF is None or not (REF / "topological_training" / "dataset.py").exists(),
                                reason="QOT_REFERENCE does not name a checkout of the upstream project")


@pytest.fixture()
def reference_imports():
    from gnn_qot_estimation_b200 import pyg_compat
    pyg_compat.install()
    sys.path.insert(0, str(REF))
    yield
    sys.path.remove(str(REF))
    for k in [k for k in sys.modules if k.split(".")[0] in ("torch_geometric", "topological_training",
                                                              "lightpath_training", "constants")]:
        del sys.modules[k]


def _topo_graph(rng):
    """Shape of to_graph.create_topological_graph's output (to_graph.py:131-184): 75 nodes, one edge per
    lightpath with the four features, graph-level labels."""
    g = nx.Graph()
    g.add_nodes_from(range(1, 76))
    for _ in range(40):
        u, v = rng.choice(np.arange(1, 76), 2, replace=False)
        g.add_edge(int(u), int(v), mod_order=float(rng.choice([4, 16, 64])), path_len=float(rng.uniform(3e4, 7e6)),
                   num_spans=float(rng.integers(1, 100)), freq=float(rng.uniform(192.3, 195.7)))
    g.graph["labels"] = {"osnr": float(rng.uniform(13, 33)), "snr": float(rng.uniform(9, 29)), "ber": float(rng.uniform(1e-11, 1e-2))}
    return g


def test_reference_topological_dataset_over_the_stand_in(tmp_path, reference_imports):
    rng = np.random.default_rng(0)
    for i in range(10):
        with open(tmp_path / f"graph_{i:03d}.gpickle", "wb") as f:
            pickle.dump(_topo_graph(rng), f)
    from topological_training.dataset import TopologicalDataset          # the reference's file, unchanged
    from torch_geometric.loader import DataLoader                        # the stand-in
    ds = TopologicalDataset(directory=str(tmp_path))
    assert ds.FEATURES == ["freq", "mod_order", "num_spans", "path_len"] and ds.edge_dim == 4
    batches = list(DataLoader(ds, batch_size=4, shuffle=False))
    assert [b.num_graphs for b in batches] == [4, 4, 2]
    b = batches[0]
    assert b.x is None and b.node_ids.tolist() == list(range(75)) * 4
    assert b.edge_attr.shape == (b.edge_index.shape[1], 4) and b.y.view(-1, 3).shape == (4, 3)
    assert float(b.edge_attr.min()) >= 0.0 and float(b.edge_attr.max()) <= 1.0   # min-max scaled (constants.py)
    assert torch.equal(b.batch, torch.repeat_interleave(torch.arange(4), 75))
    # the oracle (and therefore the B200 module, parity-tested against it) accepts the batch as is
    from oracle import TopologicalGNNOracle
    ck = torch.load(Path(__file__).parent / "golden" / "ckpt_topological_model_0.pt", weights_only=False)
    m = TopologicalGNNOracle(75, 16, 3, 4, dropout_p=0.0)
    m.load_state_dict(ck["model_state_dict"], strict=True)
    out = m.eval()(b)
    assert out.shape == (4, 3) and bool(torch.isfinite(out).all())


def test_reference_lightpath_dataset_over_the_stand_in(tmp_path, reference_imports):
    rng = np.random.default_rng(1)
    for i in range(6):
        g = nx.Graph()
        n = int(rng.integers(8, 20))
        for v in range(n):
            g.add_node(v, mod_order=float(rng.choice([4, 16, 64])), path_len=float(rng.uniform(3e4, 7e6)),
                       num_spans=float(rng.integers(1, 100)), freq=float(rng.uniform(192.3, 195.7)),
                       is_lut=1.0 if v == 0 else 0.0)
        for _ in range(2 * n):
            u, v = rng.choice(n, 2, replace=False)
            g.add_edge(int(u), int(v))
        g.graph["labels"] = {"osnr": 20.0, "snr": 18.0, "ber": 1e-4}
        with open(tmp_path / f"graph_{i:03d}.gpickle", "wb") as f:
            pickle.dump(g, f)
    from lightpath_training.dataset import LightpathDataset
    from torch_geometric.loader import DataLoader
    ds = LightpathDataset(directory=str(tmp_path))
    b = next(iter(DataLoader(ds, batch_size=6, shuffle=False)))
    assert b.x.shape[1] == 5 and b.y.shape == (6, 3)
    lut_col = ds.NODE_FEATURES.index("is_lut") if hasattr(ds, "NODE_FEATURES") else 1
    assert int((b.x[:, lut_col] == 1.0).sum()) == 6
    from oracle import LightpathGNNOracle
    out, lut_batch = LightpathGNNOracle(5, 32, 3, lut_col, dropout_p=0.0).eval()(b)
    assert out.shape == (6, 3) and lut_batch.tolist() == list(range(6))


def test_reference_model_files_import_unchanged_over_the_stand_in(reference_imports):
    """The reference's OWN topological_training/models.py and lightpath_training/models.py (imported from the
    read-only checkout, not copied) build on the stand-in's layer classes -- i.e. on the B200 kernels -- with the
    constructor calls of train.py:54-60 / lightpath train.py:55-61, expose exactly the state_dict of the shipped
    checkpoints (strict load), and refuse a CPU batch loudly (there is no CPU fallback; the forward itself is
    exercised on the GPU by tests/test_layers_gpu.py through the same layer classes)."""
    from topological_training.models import TopologicalGNN as RefTopo      # the reference's files, unchanged
    from lightpath_training.models import LightpathGNN as RefLight
    import gnn_qot_estimation_b200.nn as qnn
    gold = Path(__file__).parent / "golden"
    t = RefTopo(num_nodes=75, hidden_channels=16, out_channels=3, edge_dim=4, dropout_p=0.0)
    assert isinstance(t.conv1, qnn.TransformerConv) and isinstance(t.conv2, qnn.NNConv)
    ck = torch.load(gold / "ckpt_topological_model_0.pt", weights_only=False)
    t.load_state_dict(ck["model_state_dict"], strict=True)
    l = RefLight(in_channels=5, hidden_channels=32, output_dim=3, is_lut_index=1, dropout_p=0.0)
    assert isinstance(l.conv1, qnn.GATConv) and isinstance(l.norm1, qnn.BatchNorm)
    for name in ("ckpt_lightpath_model_0.pt", "ckpt_lightpath_model_1.pt"):
        l.load_state_dict(torch.load(gold / name, weights_only=False)["model_state_dict"], strict=True)
    from gnn_qot_estimation_b200 import synthetic
    hb = synthetic.nsfnet_store(2).host_batch(0, 2)
    hb.node_ids = hb.node_ids.clamp(max=74)
    with pytest.raises(RuntimeError, match="CUDA|no CPU"):
        t(hb)
    lb = synthetic.lightpath_store(2).host_batch(0, 2)
    with pytest.raises(RuntimeError, match="CUDA|no CPU"):
        l.eval()(lb)
