"""CPU tests of the host-side logic around the kernels: the synthetic generators emit graphs in
the exact layout the reference datasets do (from_networkx edge order, feature order, y shapes;
topological_training/dataset.py:75-123, lightpath_training/dataset.py:86-123), and
PackedGraphStore.host_batch == PyG's Batch.from_data_list as restated by oracle.collate_ref."""
import networkx as nx
import numpy as np
import pytest
import torch

from gnn_qot_estimation_b200 import Batch, PackedGraphStore, synthetic
from oracle import collate_ref


def _from_networkx_edges(G):
    """Edge order of torch_geometric.utils.from_networkx (SURVEY.md A.6): G.to_directed().edges()."""
    return list(G.to_directed().edges())


def test_nsfnet_matches_networkx_order():
    G = nx.Graph()
    G.add_nodes_from(range(14))
    G.add_edges_from(synthetic.NSFNET_LINKS)
    exp = _from_networkx_edges(G)
    src, dst, lid = synthetic.directed_from_undirected(14, synthetic.NSFNET_LINKS)
    assert list(zip(src, dst)) == exp
    assert len(src) == 42 and len(set(lid)) == 21
    for (u, v), li in zip(zip(src, dst), lid):                    # each directed edge mirrors its link
        assert set(synthetic.NSFNET_LINKS[li]) == {u, v}


def test_directed_from_undirected_self_loop_once():
    G = nx.Graph()
    G.add_nodes_from(range(3))
    links = [(0, 1), (1, 1), (1, 2)]
    G.add_edges_from(links)
    src, dst, _ = synthetic.directed_from_undirected(3, links)
    assert list(zip(src, dst)) == _from_networkx_edges(G)


def test_nsfnet_store_layout():
    st = synthetic.nsfnet_store(5, seed=0)
    assert st.num_graphs == 5 and st.node_feat is None and st.edge_feat.shape == (5 * 42, 4)
    assert st.y.shape == (5, 3)
    b = st.host_batch(1, 4)
    assert b.x is None and b.num_graphs == 3
    assert b.node_ids.tolist() == list(range(14)) * 3             # dataset.py:78: arange(n) per graph
    assert b.edge_index.dtype == torch.int64 and b.edge_index.shape == (2, 126)
    # the two directions of a link carry the same attributes (undirected nx.Graph edge data)
    ei, ea = b.edge_index[:, :42], b.edge_attr[:42]
    look = {(int(u), int(v)): ea[k] for k, (u, v) in enumerate(ei.t())}
    for (u, v), a in look.items():
        assert torch.equal(a, look[(v, u)])
    assert float(b.edge_attr.min()) >= 0.0 and float(b.edge_attr.max()) < 1.0


@pytest.mark.parametrize("luts", [1, 2])
def test_lightpath_store_layout(luts):
    st = synthetic.lightpath_store(200, seed=1, lut_per_graph=luts)
    n = (st.node_ptr[1:] - st.node_ptr[:-1])
    assert int(n.min()) >= 8 and int(n.max()) <= 56
    assert st.node_feat.shape[1] == 5 and st.edge_feat is None
    lut = st.node_feat[:, 1]
    assert set(lut.unique().tolist()) <= {0.0, 1.0}
    per_graph = torch.zeros(200).index_add_(0, torch.repeat_interleave(torch.arange(200), n), lut)
    assert int(per_graph.min()) >= 1 and int(per_graph.max()) <= luts
    for g in (0, 17, 199):                                        # undirected, no self loops, no duplicates,
        e0, e1 = int(st.edge_ptr[g]), int(st.edge_ptr[g + 1])     # grouped by source ascending
        s, d = st.edge_src[e0:e1].tolist(), st.edge_dst[e0:e1].tolist()
        pairs = set(zip(s, d))
        assert len(pairs) == len(s) and all((v, u) in pairs for u, v in pairs) and all(u != v for u, v in pairs)
        assert s == sorted(s) and max(s + d) < int(n[g])
    deg = (st.edge_ptr[-1] / st.node_ptr[-1]).item()
    assert 3.0 < deg < 4.5                                        # BASELINE cfg 2: mean directed degree ~4


def test_random_topology_store_cfg5_shape():
    st = synthetic.random_topology_store(1000, 4000, seed=2)
    assert st.num_graphs == 1 and int(st.node_ptr[-1]) == 1000 and int(st.edge_ptr[-1]) == 8000
    b = st.host_batch(0, 1)
    assert b.edge_attr.shape == (8000, 4) and b.node_ids.tolist() == list(range(1000))
    assert torch.all(b.edge_index[0][1:] >= b.edge_index[0][:-1])  # grouped by source


@pytest.mark.parametrize("kind", ["nsfnet", "lightpath"])
def test_host_batch_equals_pyg_collate(kind):
    st = synthetic.nsfnet_store(12, seed=3) if kind == "nsfnet" else synthetic.lightpath_store(12, seed=3)
    graphs = []
    for g in range(2, 11):
        n0, n1 = int(st.node_ptr[g]), int(st.node_ptr[g + 1])
        e0, e1 = int(st.edge_ptr[g]), int(st.edge_ptr[g + 1])
        d = {"num_nodes": n1 - n0, "y": st.y[g:g + 1],
             "edge_index": torch.stack([st.edge_src[e0:e1], st.edge_dst[e0:e1]]).long()}
        if st.node_feat is not None:
            d["x"] = st.node_feat[n0:n1]
        else:
            d["node_ids"] = torch.arange(n1 - n0)
        if st.edge_feat is not None:
            d["edge_attr"] = st.edge_feat[e0:e1]
        graphs.append(d)
    ref = collate_ref(graphs)
    got = st.host_batch(2, 11)
    for k in ("x", "edge_index", "edge_attr", "batch", "node_ids", "y"):
        a, b = getattr(got, k), getattr(ref, k)
        assert (a is None) == (b is None), k
        if a is not None:
            assert a.dtype == b.dtype and torch.equal(a, b), k
    assert torch.equal(got.ptr, ref.ptr) and torch.equal(got.edge_ptr, ref.edge_ptr)
    assert got.num_graphs == ref.num_graphs == 9


def test_batch_container_contract():
    b = Batch(x=torch.zeros(3, 5), edge_index=torch.zeros(2, 4, dtype=torch.int64),
              batch=torch.tensor([0, 0, 1]), num_graphs=2)
    assert b.num_nodes == 3 and b.num_edges == 4
    assert b.edge_attr is None and b.node_ids is None            # attributes the modules probe exist
    c = b.to("cpu")
    assert c is not b and torch.equal(c.x, b.x) and c.num_graphs == 2
    assert b.nbytes() == 3 * 5 * 4 + 2 * 4 * 8 + 3 * 8
    assert "num_graphs=2" in repr(b)


def test_store_refuses_cpu_collate():
    st = synthetic.nsfnet_store(2, seed=0)
    with pytest.raises(RuntimeError, match="GPU"):
        st.collate(range(0, 2))


def test_numa_binding_is_best_effort():
    """bind_to_gpu_numa_node never raises: without NVML / a GPU it reports why and leaves the affinity alone."""
    import os
    from gnn_qot_estimation_b200.distributed import bind_to_gpu_numa_node
    before = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    msg = bind_to_gpu_numa_node(0)
    assert isinstance(msg, str) and msg
    os.environ["QOT_NO_NUMA_BIND"] = "1"
    try:
        assert bind_to_gpu_numa_node(0) == "numa binding off"
    finally:
        del os.environ["QOT_NO_NUMA_BIND"]
    if before is not None and "bound to" not in msg:
        assert os.sched_getaffinity(0) == before


def test_fused_topological_path_admission():
    """The block-per-graph kernels take a batch only if its largest graph fits one block's shared memory
    (and <= 512 edges: four edges per thread in the CSR build); everything else goes layer by layer."""
    from gnn_qot_estimation_b200 import ops
    assert ops.topo_fused_fits(14, 42, 14)            # NSFNET (cfg 1 / cfg 3)
    assert ops.topo_fused_fits(75, 400, 75)           # the real 75-node topology
    assert not ops.topo_fused_fits(75, 513, 75)       # too many edges for the in-block CSR build
    assert not ops.topo_fused_fits(400, 100, 75)      # node arrays beyond 227 KB
    assert not ops.topo_fused_fits(10000, 80000, 10000)   # cfg 5 stays on the layer-by-layer / tensor-core path


def test_sources_follow_from_the_destination_histogram_on_from_networkx_layouts():
    """DESIGN.md section 10.5: for the layout from_networkx emits (both directions of every link, grouped by
    source ascending; a self loop once) the source row is redundant -- src[p] is the node u with
    outptr[u] <= p < outptr[u+1], and outdeg == indeg == a histogram of the destination row."""
    import networkx as nx
    from gnn_qot_estimation_b200 import pyg_compat, synthetic
    rng = np.random.default_rng(3)
    for trial in range(20):
        n = int(rng.integers(2, 40))
        g = nx.Graph()
        g.add_nodes_from(range(n))
        for _ in range(int(rng.integers(0, 3 * n))):
            u, v = rng.integers(0, n, 2)
            g.add_edge(int(u), int(v))                      # includes self loops and repeated pairs
        ei = pyg_compat.utils.from_networkx(g).edge_index.numpy()
        src, dst = ei[0], ei[1]
        indeg = np.bincount(dst, minlength=n)
        outptr = np.concatenate([[0], np.cumsum(indeg)])
        inferred = np.searchsorted(outptr, np.arange(src.shape[0]), side="right") - 1
        assert np.array_equal(inferred, src), trial
    # the synthetic lightpath shards of the benchmark have the same layout
    st = synthetic.lightpath_store(200, seed=5)
    for gi in range(200):
        e0, e1 = int(st.edge_ptr[gi]), int(st.edge_ptr[gi + 1])
        n = int(st.node_ptr[gi + 1] - st.node_ptr[gi])
        src, dst = st.edge_src[e0:e1].numpy(), st.edge_dst[e0:e1].numpy()
        outptr = np.concatenate([[0], np.cumsum(np.bincount(dst, minlength=n))])
        assert np.array_equal(np.searchsorted(outptr, np.arange(e1 - e0), side="right") - 1, src)


def test_verify_layout_accepts_from_networkx_order_and_rejects_violations():
    """PackedGraphStore.verify_layout: the synthetic generators emit the from_networkx layout (grouped by
    source ascending, symmetric, simple); a swapped pair, a dropped direction or a duplicate must fail."""
    import torch
    from gnn_qot_estimation_b200 import synthetic
    from gnn_qot_estimation_b200.batch import PackedGraphStore
    st = synthetic.lightpath_store(50, seed=3)
    assert st.verify_layout() and st.sym_by_src
    assert st.host_batch(0, 10).sym_by_src
    assert synthetic.nsfnet_store(4).verify_layout()

    def clone(**kw):
        f = dict(node_ptr=st.node_ptr, edge_ptr=st.edge_ptr, edge_src=st.edge_src.clone(), edge_dst=st.edge_dst.clone(),
                 node_feat=st.node_feat, y=st.y, lut_col=1)
        f.update(kw)
        return PackedGraphStore(f["node_ptr"], f["edge_ptr"], f["edge_src"], f["edge_dst"], f["node_feat"], None, f["y"], f["lut_col"])
    e0, e1 = int(st.edge_ptr[0]), int(st.edge_ptr[1])
    # not grouped by source: reverse the edge order of graph 0
    s, d = st.edge_src.clone(), st.edge_dst.clone()
    s[e0:e1], d[e0:e1] = st.edge_src[e0:e1].flip(0), st.edge_dst[e0:e1].flip(0)
    assert not clone(edge_src=s, edge_dst=d).verify_layout()
    # one direction rewired: no longer symmetric
    d = st.edge_dst.clone()
    d[e0] = (d[e0] + 1) % int(st.node_ptr[1])
    assert not clone(edge_dst=d).verify_layout()
    # endpoint outside the graph
    d = st.edge_dst.clone()
    d[e0] = 1000
    assert not clone(edge_dst=d).verify_layout()


def test_derived_weight_cache_follows_parameter_updates():
    """ops._derived: re-laid-out weights are cached only while autograd is not recording, and an in-place update of a
    source (optimizer step, load_state_dict) or a new tensor at a recycled address invalidates the entry."""
    from gnn_qot_estimation_b200 import ops
    a, b = torch.nn.Parameter(torch.ones(2, 3)), torch.nn.Parameter(torch.zeros(2, 3))
    calls = []

    def make():
        calls.append(1)
        return torch.cat([a, b], dim=0)

    with torch.no_grad():
        c1 = ops._derived("t", (a, b), make)
        c2 = ops._derived("t", (a, b), make)
    assert c1 is c2 and len(calls) == 1 and not c1.requires_grad
    c3 = ops._derived("t", (a, b), make)                      # autograd recording: rebuilt, differentiable
    assert len(calls) == 2 and c3.requires_grad
    with torch.no_grad():
        a.add_(1.0)                                           # what optimizer.step() does
        c4 = ops._derived("t", (a, b), make)
    assert len(calls) == 3 and float(c4[0, 0]) == 2.0
    a.requires_grad_(False); b.requires_grad_(False)
    c5 = ops._derived("t", (a, b), make)                      # frozen weights: cached even with grad mode on
    c6 = ops._derived("t", (a, b), make)
    assert c5 is c6


def test_check_status_reads_multi_word_status_tensors(monkeypatch):
    """A tracked status tensor may hold one word per batch (the multi-batch lightpath stream): check_status() ORs its
    words, raises only when one is set, and still reads single-word tensors tracked beside it."""
    from gnn_qot_estimation_b200 import ops
    monkeypatch.setattr(ops, "_status_words", {})
    multi, single = torch.zeros(3, dtype=torch.int32), torch.zeros(1, dtype=torch.int32)
    ops._track_status("multi", multi)
    ops._track_status("single", single)
    ops.check_status(clear=False)
    multi[2] = 2
    multi[0] = 1
    with pytest.raises(RuntimeError, match=r"multi \(status 3\)") as e:
        ops.check_status(clear=False)
    assert "single" not in str(e.value)
    multi.zero_()
    single[0] = 4
    with pytest.raises(RuntimeError, match=r"single \(status 4\)"):
        ops.check_status()
    ops.check_status()                               # cleared
