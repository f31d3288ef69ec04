"""SURVEY 8(f)4 -- graph construction (to_graph.py::create_lightpath_graph + LightpathDataset tensorisation).
CPU side: the numpy restatement under oracle/ against golden vectors produced by the REFERENCE's own code
(tests/golden/make_to_graph_golden.py); when QOT_REFERENCE names a checkout of the upstream project, which this
repository does not contain, also against the reference itself on fresh seeds and corner cases."""
import os
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from conftest import load_golden

REF = Path(os.environ["QOT_REFERENCE"]) if os.environ.get("QOT_REFERENCE") else None   # santiagolmedo/gnn_qot_estimation
needs_reference = pytest.mark.skipif(REF is None or not (REF / "to_graph.py").exists(),
                                     reason="QOT_REFERENCE does not name a checkout of the upstream project")


def _oracle_all(samples):
    from oracle import lightpath_data_ref
    return [lightpath_data_ref(samples["data"][i], samples["target"][i], samples["freqs"], samples["lp_feat"], samples["metric"])
            for i in range(samples["data"].shape[0])]


def test_oracle_matches_reference_golden_vectors():
    from gnn_qot_estimation_b200 import synthetic
    gold = load_golden("to_graph_lightpath.pt")
    total_edges = loops = 0
    for (S, L, Q, seed, spacing), res in zip(gold["cases"], gold["results"]):
        samples = synthetic.network_status_samples(S, L, Q, seed=seed, spacing=spacing)
        assert float(np.abs(samples["data"]).sum(dtype=np.float64)) == res["input_checksum"]   # same inputs as the generator saw
        for (conn, x, y, ei), g in zip(_oracle_all(samples), res["graphs"]):
            assert np.array_equal(conn, g["conn_ids"].numpy())                 # node order
            assert np.array_equal(x, g["x"].numpy())                           # bit-exact features
            assert np.array_equal(y, g["y"].numpy())
            assert np.array_equal(ei, g["edge_index_sorted"].numpy())          # edge set
            assert int((x[:, 1] == 1.0).sum()) == 1                            # one LUT lightpath
            total_edges += ei.shape[1]
            loops += int((ei[0] == ei[1]).sum())
    assert total_edges > 200 and loops > 10                                     # the fixtures do exercise the join


@needs_reference
@pytest.mark.parametrize("seed,spacing", [(11, 0.0375), (12, 0.05), (13, 0.025)])
def test_oracle_matches_reference_code_on_fresh_seeds(seed, spacing):
    sys.path.insert(0, str(Path(__file__).parent / "golden"))
    try:
        import make_to_graph_golden as mk
    finally:
        sys.path.pop(0)
    from gnn_qot_estimation_b200 import synthetic
    samples = synthetic.network_status_samples(3, 9, 40, seed=seed, spacing=spacing)
    graphs = mk.reference_graphs(samples)
    datas, _ = mk.reference_data_objects(graphs)
    for (conn, x, y, ei), g, d in zip(_oracle_all(samples), graphs, datas):
        c = mk.canonical(g, d)
        assert np.array_equal(conn, c["conn_ids"].numpy()) and np.array_equal(x, c["x"].numpy())
        assert np.array_equal(y, c["y"].numpy()) and np.array_equal(ei, c["edge_index_sorted"].numpy())
    for k in [k for k in sys.modules if k.split(".")[0] == "torch_geometric"]:
        del sys.modules[k]


def test_topological_oracle_matches_reference_golden_vectors():
    """create_topological_graph + TopologicalDataset: edge ORDER, attributes (last lightpath of a node pair
    wins) and labels, bit for bit."""
    from gnn_qot_estimation_b200 import synthetic
    from oracle import topological_data_ref
    gold = load_golden("to_graph_topological.pt")
    dup = 0
    for (S, L, Q, seed, spacing, nn), res in zip(gold["cases"], gold["results"]):
        samples = synthetic.network_status_samples(S, L, Q, seed=seed, spacing=spacing, num_nodes=nn)
        for i, g in enumerate(res["graphs"]):
            ei, ea, y = topological_data_ref(samples["data"][i], samples["target"][i], samples["lp_feat"], samples["metric"])
            assert g["num_nodes"] == 75
            assert np.array_equal(ei, g["edge_index"].numpy())
            assert np.array_equal(ea, g["edge_attr"].numpy()) and np.array_equal(y, g["y"].numpy())
            n_lp = len(np.unique(samples["data"][i][0][np.any(samples["data"][i] != 0, axis=0)]))
            dup += int(ei.shape[1] < 2 * n_lp)
    assert dup >= 4                                                     # node pairs shared by several lightpaths occur


@needs_reference
def test_oracle_matches_reference_code_on_corner_cases():
    """Hand-built samples through the reference's own code and through the restatement: a single lightpath, two
    lightpaths that never share a link, two that share a link at distance exactly / just under / just over the
    threshold, a link carrying one lightpath on two adjacent channels only (skipped by to_graph.py:285), float
    conn ids (int() truncation), an empty sample."""
    sys.path.insert(0, str(Path(__file__).parent / "golden"))
    try:
        import make_to_graph_golden as mk
    finally:
        sys.path.pop(0)
    from oracle import lightpath_data_ref, topological_data_ref
    from tg_cases import corner_case_samples
    samples = corner_case_samples()
    freqs = samples["freqs"]
    graphs = mk.reference_graphs(samples)
    keep = [i for i, g in enumerate(graphs) if len(g) > 0]                 # the reference's dataset class cannot tensorise an empty graph
    datas, _ = mk.reference_data_objects([graphs[i] for i in keep])
    for i, d in zip(keep, datas):
        cn, x, y, ei = lightpath_data_ref(samples["data"][i], samples["target"][i], freqs, samples["lp_feat"], samples["metric"])
        ref = mk.canonical(graphs[i], d)
        assert np.array_equal(cn, ref["conn_ids"].numpy()) and np.array_equal(x, ref["x"].numpy()), i
        assert np.array_equal(y, ref["y"].numpy()) and np.array_equal(ei, ref["edge_index_sorted"].numpy()), i
    cn, x, y, ei = lightpath_data_ref(samples["data"][-1], samples["target"][-1], freqs, samples["lp_feat"], samples["metric"])
    assert cn.shape == (0,) and x.shape == (0, 5) and ei.shape == (2, 0)
    assert [len(g) for g in graphs] == [1, 2, 2, 2, 2, 2, 3, 0]
    assert [g.number_of_edges() for g in graphs] == [0, 0, 1, 0, 0, 0, 3, 0]
    tg = mk.reference_graphs(samples, representation="topological")
    tdatas, _ = mk.reference_topological_data_objects(tg)
    for i, d in enumerate(tdatas):
        ei, ea, yy = topological_data_ref(samples["data"][i], samples["target"][i], samples["lp_feat"], samples["metric"])
        assert np.array_equal(ei, d.edge_index.numpy()) and np.array_equal(ea, d.edge_attr.numpy().reshape(-1, 4)), i
        assert np.array_equal(yy, d.y.numpy())
    for k in [k for k in sys.modules if k.split(".")[0] == "torch_geometric"]:
        del sys.modules[k]
