"""GPU parity of LightpathGNN's every-node mode (csrc/lightpath_every_node.cu, qot_lightpath_infer_every_node through
stream_plan(..., every_node=True) / forward_stream / forward_every_node) against the fp64 oracle's literal definition
(tests/every_node_ref.py: one one-hot copy of a graph per node), against the existing one-LUT readout, on hand-built
corner cases, from raw samples, and its error paths."""
from types import SimpleNamespace

import pytest
import torch

from conftest import ABS_FLOOR, load_golden, rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-5
ATOL = ABS_FLOOR


def _model(dev, name="ckpt_lightpath_model_1.pt"):
    from gnn_qot_estimation_b200 import LightpathGNN
    sd = load_golden(name)["model_state_dict"]
    m = LightpathGNN(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    m.load_state_dict(sd, strict=True)
    return m.to(dev).eval(), sd


def _oracle64(sd, dev):
    from oracle import LightpathGNNOracle
    m = LightpathGNNOracle(5, 32, 3, is_lut_index=1, dropout_p=0.0).double()
    m.load_state_dict(sd, strict=True)
    return m.to(dev).eval()


def _ref(oracle, b, dev):
    """fp64 oracle (on the GPU: the one-hot copies of a 4096-graph batch are ~4 M nodes)."""
    from every_node_ref import lightpath_every_node_ref
    with torch.no_grad():
        return lightpath_every_node_ref(oracle, SimpleNamespace(x=b.x.to(dev).double(), edge_index=b.edge_index.to(dev),
                                                                batch=b.batch.to(dev)))


def _close(got, ref):
    assert got.shape == ref.shape
    assert torch.isfinite(got).all()
    assert rel_err(got, ref) <= RTOL
    torch.testing.assert_close(got.double().cpu(), ref.cpu(), rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("sizes", [[1], [16], [17, 1, 300], [4096, 4096, 333]])
def test_every_node_vs_oracle_both_layouts(cuda, sizes):
    from gnn_qot_estimation_b200 import synthetic
    m, sd = _model(cuda)
    o = _oracle64(sd, cuda)
    store = synthetic.lightpath_store(sum(sizes), seed=11 + len(sizes), device="cpu").to(cuda)
    assert store.verify_layout()
    dbs, g0 = [], 0
    for s in sizes:
        dbs.append(store.collate(range(g0, g0 + s)))
        g0 += s
    plan = m.stream_plan(dbs, every_node=True)
    assert plan.flags == 1
    m.forward_stream(plan)
    torch.cuda.synchronize()
    assert int(plan.status.max()) == 0
    for i, b in enumerate(dbs):
        _close(plan.result(i).out, _ref(o, b, cuda))
        assert torch.equal(plan.result(i).lut_batch, b.batch)
    for b in dbs:                                  # unverified: the launch reads the source row
        b.sym_by_src = False
    plan2 = m.stream_plan(dbs, every_node=True)
    assert plan2.flags == 0
    m.forward_stream(plan2)
    torch.cuda.synchronize()
    assert torch.equal(plan.out, plan2.out)        # same bits on both layouts


def test_every_node_agrees_with_one_lut_readout(cuda):
    """In graphs with exactly one flagged node, that node's row equals model(data) and the stream plan's row."""
    from gnn_qot_estimation_b200 import synthetic
    m, _ = _model(cuda, "ckpt_lightpath_model_0.pt")
    store = synthetic.lightpath_store(2000, seed=4, device=cuda)
    db = store.collate(range(0, 2000))
    every = m.forward_every_node(db)
    with torch.no_grad():
        mo, ml = m(db)
    lut = (db.x[:, 1] == 1.0).nonzero().flatten()
    assert torch.equal(db.batch[lut], ml)
    torch.testing.assert_close(every[lut], mo, rtol=RTOL, atol=ATOL)
    plan = m.stream_plan([db])
    m.forward_stream(plan)
    r = plan.result(0)
    n = int(r.n_lut.item())
    torch.testing.assert_close(every[r.lut_node[:n].long()], r.out[:n], rtol=RTOL, atol=ATOL)


def _hand_built(g, dev):
    from gnn_qot_estimation_b200 import Batch
    # n = 70 / 200 / 256 (70: fast path; 200, 256: generic path), zero-edge graphs, self loops and duplicates,
    # a hub row with 64 in-edges, graphs with zero or two flagged nodes, random flag values
    sizes = [1, 3, 70, 40, 2, 30, 25, 9, 200, 256, 5] + [12] * 20
    xs, eis, bts, ptr, eptr = [], [], [], [0], [0]
    off = 0
    for gi, n in enumerate(sizes):
        x = torch.rand(n, 5, generator=g)
        x[:, 1] = 0.0
        if gi not in (5, 10):
            x[n // 2, 1] = 1.0                  # graphs 5, 10: no flagged node
        if gi == 2:
            x[5, 1] = 1.0                       # two flagged nodes
        E = 0 if gi in (0, 4, 10) else 6 * n
        src = torch.randint(0, n, (E,), generator=g)
        dst = torch.randint(0, n, (E,), generator=g)   # includes self loops and duplicates
        if gi == 6:
            dst[:64] = n // 2                   # hub: 64 in-edges
        if gi == 9:
            dst[:80] = 7                        # hub in a generic-path graph
        eis.append(torch.stack([src, dst]) + off)
        xs.append(x)
        bts.append(torch.full((n,), gi, dtype=torch.int64))
        off += n
        ptr.append(off)
        eptr.append(eptr[-1] + E)
    return Batch(x=torch.cat(xs), edge_index=torch.cat(eis, 1), batch=torch.cat(bts), num_graphs=len(sizes),
                 ptr=torch.tensor(ptr), edge_ptr=torch.tensor(eptr), lut_col=1).to(dev)


def test_every_node_edge_cases(cuda):
    from gnn_qot_estimation_b200 import Batch
    m, sd = _model(cuda, "ckpt_lightpath_model_0.pt")
    o = _oracle64(sd, cuda)
    g = torch.Generator().manual_seed(0)
    db = _hand_built(g, cuda)
    empty = Batch(x=torch.zeros(0, 5, device=cuda), edge_index=torch.zeros(2, 0, dtype=torch.int64, device=cuda),
                  batch=torch.zeros(0, dtype=torch.int64, device=cuda), num_graphs=0,
                  ptr=torch.zeros(1, dtype=torch.int64, device=cuda), edge_ptr=torch.zeros(1, dtype=torch.int64,
                                                                                             device=cuda))
    plan = m.stream_plan([db, empty], every_node=True)
    m.forward_stream(plan)
    torch.cuda.synchronize()
    assert int(plan.status.max()) == 0
    assert plan.result(1).out.shape == (0, 3)
    first = plan.result(0).out.clone()
    _close(first, _ref(o, db, cuda))
    # the stored flag column has no effect: random values, then all zeros -- identical bits
    db.x[:, 1] = torch.rand(db.x.shape[0], generator=g).to(cuda)
    m.forward_stream(plan)
    torch.cuda.synchronize()
    assert torch.equal(plan.result(0).out, first)
    db.x[:, 1] = 0.0
    m.forward_stream(plan)
    torch.cuda.synchronize()
    assert torch.equal(plan.result(0).out, first)


def test_every_node_determinism_capture_and_subrange(cuda):
    from gnn_qot_estimation_b200 import synthetic
    m, _ = _model(cuda)
    store = synthetic.lightpath_store(900, seed=9, device=cuda)
    dbs = [store.collate(range(0, 300)), store.collate(range(300, 600)), store.collate(range(600, 900))]
    plan = m.stream_plan(dbs, every_node=True)
    m.forward_stream(plan)
    torch.cuda.synchronize()
    first = plan.out.clone()
    m.forward_stream(plan)
    torch.cuda.synchronize()
    assert torch.equal(plan.out, first)
    gr = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        m.forward_stream(plan)
        torch.cuda.synchronize()
        with torch.cuda.graph(gr, stream=s):
            m.forward_stream(plan)
        plan.out.zero_()
        gr.replay()
    torch.cuda.synchronize()
    assert torch.equal(plan.out, first)
    plan.out[plan.off[1]:plan.off[2]].fill_(float("nan"))
    plan.out[plan.off[0]:plan.off[1]].fill_(7.0)
    m.forward_stream(plan, 1, 1)                    # rewrites batch 1 only
    torch.cuda.synchronize()
    assert torch.equal(plan.out[plan.off[1]:], first[plan.off[1]:])
    assert bool((plan.out[plan.off[0]:plan.off[1]] == 7.0).all())


def test_every_node_from_raw_samples(cuda):
    """network-status samples -> create_lightpath_graphs(return_conn_ids=True) -> collate -> forward_every_node:
    row i is lightpath conn_ids[i] of sample batch[i]; each sample's LUT row equals forward()."""
    from gnn_qot_estimation_b200 import synthetic
    from gnn_qot_estimation_b200.to_graph import create_lightpath_graphs
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(24, seed=3)
    store, conn = create_lightpath_graphs(torch.from_numpy(smp["data"]).to(cuda), torch.from_numpy(smp["target"]),
                                          torch.from_numpy(smp["freqs"]), smp["lp_feat"], smp["metric"],
                                          return_conn_ids=True)
    db = store.collate(range(store.num_graphs))
    every = m.forward_every_node(db)
    assert every.shape == (db.x.shape[0], 3) and conn.shape[0] == db.x.shape[0]
    with torch.no_grad():
        mo, ml = m(db)
    lut = (db.x[:, 1] == 1.0).nonzero().flatten()
    assert torch.equal(db.batch[lut], ml)
    torch.testing.assert_close(every[lut], mo, rtol=RTOL, atol=ATOL)
    # rows line up with conn_ids: the same lightpath of a sample keeps its prediction when the batch is re-collated
    # with the samples in reverse order
    rev = store.collate(list(range(store.num_graphs - 1, -1, -1)))
    every_rev = m.forward_every_node(rev)
    np_ = store.node_ptr.cpu()
    for s in range(store.num_graphs):
        a, b = int(np_[s]), int(np_[s + 1])
        r0 = int(rev.ptr[store.num_graphs - 1 - s])
        assert torch.equal(every[a:b], every_rev[r0:r0 + (b - a)])
        assert len(set(conn[a:b].tolist())) == b - a              # one row per lightpath of the sample


def test_every_node_errors_and_foreign_batches(cuda):
    from gnn_qot_estimation_b200 import LightpathGNN, synthetic
    m, _ = _model(cuda)
    store = synthetic.lightpath_store(40, seed=2, device=cuda)
    db = store.collate(range(40))
    ref = m.forward_every_node(db)
    # foreign batches with grouped edges: ptr / edge_ptr derived
    foreign = SimpleNamespace(x=db.x, edge_index=db.edge_index, batch=db.batch, num_graphs=40)
    assert torch.equal(m.forward_every_node(foreign), ref)
    from gnn_qot_estimation_b200.pyg_compat import Batch as PygBatch, Data
    pyg = PygBatch.from_data_list([Data(x=store.node_feat[int(store.node_ptr[i]):int(store.node_ptr[i + 1])].cpu(),
                                        edge_index=torch.stack([store.edge_src[int(store.edge_ptr[i]):int(store.edge_ptr[i + 1])],
                                                                store.edge_dst[int(store.edge_ptr[i]):int(store.edge_ptr[i + 1])]]).long().cpu())
                                   for i in range(40)]).to(cuda)
    assert torch.equal(m.forward_every_node(pyg), ref)
    # edges not grouped by graph
    perm = torch.randperm(db.edge_index.shape[1], generator=torch.Generator().manual_seed(0)).to(cuda)
    bad = SimpleNamespace(x=db.x, edge_index=db.edge_index[:, perm], batch=db.batch, num_graphs=40)
    with pytest.raises(RuntimeError, match="not grouped by graph"):
        m.forward_every_node(bad)
    with pytest.raises(RuntimeError, match="CUDA"):
        m.forward_every_node(SimpleNamespace(x=db.x.cpu(), edge_index=db.edge_index.cpu(), batch=db.batch.cpu(),
                                             num_graphs=40))
    m.train()
    with pytest.raises(RuntimeError, match="eval"):
        m.forward_every_node(db)
    m.eval()
    odd = LightpathGNN(5, 16, 3, is_lut_index=1).to(cuda).eval()
    with pytest.raises(RuntimeError, match="reference LightpathGNN shape"):
        odd.forward_every_node(db)
