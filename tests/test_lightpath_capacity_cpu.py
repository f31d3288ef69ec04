"""CPU checks at the capacity of the lightpath network-state kernels: the dense sample builders of tests/dense_samples.py
place exactly what they claim (256 lightpaths, a hub of in-degree 255, clique density, the 6144-channel bound, the
every-node boundary stores); the chunked references equal the unchunked ones; and the oracle identities the earlier
CPU tests check on small samples still hold on a 256-lightpath sample."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import dense_samples as ds
from conftest import load_golden

TOL = dict(rtol=1e-12, atol=1e-12)
METRIC = ["osnr", "snr", "ber"]


def _oracle64():
    from oracle import LightpathGNNOracle
    m = LightpathGNNOracle(5, 32, 3, is_lut_index=1, dropout_p=0.0).double()
    m.load_state_dict(load_golden("ckpt_lightpath_model_1.pt")["model_state_dict"], strict=True)
    return m.eval()


def _graph(smp, s, thr):
    from oracle.to_graph_oracle import lightpath_data_ref
    conns, x, _, ei = lightpath_data_ref(smp["data"][s], np.zeros(3), smp["freqs"], smp["lp_feat"], METRIC, thr)
    return conns, x, ei


def _in_degree(conns, ei):
    nl = ei[0] != ei[1]
    return np.bincount(ei[1][nl], minlength=len(conns))


def _every(m, x, ei, chunk=None):
    from every_node_ref import lightpath_every_node_ref
    with torch.no_grad():
        return lightpath_every_node_ref(m, SimpleNamespace(x=torch.from_numpy(x).double(), edge_index=torch.from_numpy(ei),
                                                           batch=torch.zeros(x.shape[0], dtype=torch.int64)), chunk)


def test_hub_sample():
    smp = ds.hub()
    conns, x, ei = _graph(smp, 0, ds.HUB_THRESHOLD)
    deg = _in_degree(conns, ei)
    assert len(conns) == ds.MAX_NODES and ei.shape[1] == 510
    assert deg[1] == 255 and int(np.delete(deg, 1).max()) == 1          # node 1 is the hub, every single sees it only
    occ = np.any(smp["data"][0] != 0, axis=0)
    assert int(occ.sum()) == 128 + 255 and not occ[127, 11]
    print(f"hub: n {len(conns)}, E {ei.shape[1]}, hub in-degree {deg[1]}")


def test_clique_and_full_sparse_samples():
    smp = ds.clique()
    conns, _, ei = _graph(smp, 0, ds.CLIQUE_THRESHOLD)
    deg = _in_degree(conns, ei)
    assert len(conns) == 256 and ei.shape[1] > 20000
    assert deg.max() > 128 and deg.mean() > 64 and (deg > 64).sum() > 128
    print(f"clique: E {ei.shape[1]}, max in-degree {deg.max()}, mean {deg.mean():.1f}")
    sp = ds.full_sparse()
    assert sp["data"].shape[:1] == (4,)
    for s, cnt in enumerate((256, 255, 1, 48)):
        conns, _, _ = _graph(sp, s, ds.HUB_THRESHOLD)
        assert len(conns) == cnt


def test_occupancy_bound():
    grid = ds.full_grid()
    assert int(np.any(grid["data"][0] != 0, axis=0).sum()) == ds.MAX_CHANNELS
    conns, _, ei = _graph(grid, 0, ds.HUB_THRESHOLD)
    assert len(conns) == 256 and int((ei[0] == ei[1]).sum()) == 256   # every lightpath spans 3 slots: a self loop
    over = ds.full_grid(extra=1)
    assert int(np.any(over["data"][0] != 0, axis=0).sum()) == ds.MAX_CHANNELS + 1
    assert len(_graph(over, 0, ds.HUB_THRESHOLD)[0]) == 256
    # the builder refuses to hand out an over-capacity sample it was not asked for, or a wrong lightpath count
    b = ds.SampleBuilder(64, 97, np.random.default_rng(0))
    for k in range(256):
        b.place(list(range(8 * (k // 32), 8 * (k // 32) + 8)), 3 * (k % 32), 3)
    b.place([0], 96)
    with pytest.raises(AssertionError):
        b.place([0], 96)
    with pytest.raises(AssertionError):
        b.finish(257)
    with pytest.raises(AssertionError):
        ds.SampleBuilder(4, 4, np.random.default_rng(0)).finish(1)
    assert len(_graph(ds.count_sample(257), 0, ds.HUB_THRESHOLD)[0]) == 257


def test_boundary_stores():
    st = ds.boundary_store()
    assert st.verify_layout()
    nptr, eptr = st.node_ptr.tolist(), st.edge_ptr.tolist()
    assert [(nptr[i + 1] - nptr[i], eptr[i + 1] - eptr[i]) for i in range(4)] == ds.BOUNDARY_SHAPES
    for i in range(4):
        src, dst = st.edge_src[eptr[i]:eptr[i + 1]].long(), st.edge_dst[eptr[i]:eptr[i + 1]].long()
        deg = torch.bincount(dst[src != dst], minlength=nptr[i + 1] - nptr[i])
        assert int(deg[0]) >= 100                                          # a row of more than 64 in-neighbours
    fast = [(n, E) for n, E in ds.BOUNDARY_SHAPES if n <= ds.EN_MAX_N and E <= ds.EN_MAX_E]
    assert fast == [(128, 512), (120, 500)]


def test_chunked_references_equal_unchunked():
    from candidates_ref import candidates_ref
    from change_set_ref import change_set_ref
    from gnn_qot_estimation_b200 import synthetic
    from reconfig_ref import _rows, reconfig_ref
    m = _oracle64()
    # small: the every-node reference over a multi-graph batch, candidates and changes of a generated sample
    store = synthetic.lightpath_store(12, seed=3)
    b = store.host_batch(0, 12)
    x = b.x.double()
    with torch.no_grad():
        from every_node_ref import lightpath_every_node_ref
        full = lightpath_every_node_ref(m, SimpleNamespace(x=x, edge_index=b.edge_index, batch=b.batch))
        for chunk in (1, 7, 1000):
            part = lightpath_every_node_ref(m, SimpleNamespace(x=x, edge_index=b.edge_index, batch=b.batch), chunk)
            torch.testing.assert_close(part, full, **TOL)
    smp = synthetic.network_status_samples(2, num_links=8, num_freqs=24, seed=4, max_lightpaths=20)
    freqs, lp_feat = smp["freqs"], smp["lp_feat"]
    f = [np.float32(freqs[5]), 16, 10, 100000]
    c0, r0 = candidates_ref(m, smp["data"][0], freqs, lp_feat, [1, 2], 5, 1, f)
    c1, r1 = candidates_ref(m, smp["data"][0], freqs, lp_feat, [1, 2], 5, 1, f, chunk=1)
    torch.testing.assert_close(c1, c0, **TOL)
    assert r1.keys() == r0.keys() and all(torch.allclose(r1[k], r0[k], **TOL) for k in r0)
    conns, x, ei = _graph(smp, 0, 0.05)
    rows = list(range(len(conns)))
    torch.testing.assert_close(_rows(m, x, ei, rows, chunk=3), _rows(m, x, ei, rows), **TOL)
    # dense: the hub moved to slot 12 (255 impact rows), as a reconfiguration and as a set of one change
    hub = ds.hub()
    d, freqs = hub["data"][0], hub["freqs"]
    hub_conn = int(_graph(hub, 0, ds.HUB_THRESHOLD)[0][1])
    mv = (list(range(128)), 12, 1, [np.float32(freqs[12]), 16, 10, 100000])
    a_row, a = reconfig_ref(m, d, freqs, hub["lp_feat"], hub_conn, *mv)
    b_row, b2 = reconfig_ref(m, d, freqs, hub["lp_feat"], hub_conn, *mv, chunk=64)
    torch.testing.assert_close(b_row, a_row, **TOL)
    assert len(a) == 255 and b2.keys() == a.keys()
    assert all(b2[k][0] == a[k][0] and torch.allclose(b2[k][1], a[k][1], **TOL) for k in a)
    rows_s, s_imp = change_set_ref(m, d, freqs, hub["lp_feat"], [(hub_conn, *mv)], chunk=100)
    torch.testing.assert_close(rows_s[0], a_row, **TOL)
    assert s_imp.keys() == a.keys()
    assert all(s_imp[k][0] == a[k][0] and torch.allclose(s_imp[k][1], a[k][1], **TOL) for k in a)
    conns, x, ei = _graph(hub, 0, ds.HUB_THRESHOLD)
    torch.testing.assert_close(_every(m, x, ei, chunk=64), _every(m, x, ei), **TOL)


def test_hub_teardown_equals_every_node_of_the_sample_without_it():
    """Tearing down the hub (in-degree 255): 255 rows of kind 1, each the every-node row of the rebuilt sample."""
    from reconfig_ref import reconfig_ref
    m = _oracle64()
    hub = ds.hub()
    d, freqs, lp_feat = hub["data"][0], hub["freqs"], hub["lp_feat"]
    conns, _, _ = _graph(hub, 0, ds.HUB_THRESHOLD)
    c = int(conns[1])
    row, impact = reconfig_ref(m, d, freqs, lp_feat, c, [], 0, 1, [0.0, 0.0, 0.0, 0.0], chunk=128)
    assert row is None and len(impact) == 255 and {k for k, _ in impact.values()} == {1}
    fi = {k: i for i, k in enumerate(lp_feat)}
    rest = d.copy()
    rest[:, np.trunc(d[fi["conn_id"]]) == c] = 0.0
    conns2, x2, ei2 = _graph({**hub, "data": rest[None]}, 0, ds.HUB_THRESHOLD)
    assert ei2.shape[1] == 0
    every = _every(m, x2, ei2)
    for i, cc in enumerate(conns2):
        torch.testing.assert_close(impact[int(cc)][1], every[i], **TOL)


def test_one_change_set_equals_reconfiguration_at_capacity():
    """A set of one change on the clique sample equals the reconfiguration reference: a lightpath moved onto a free
    slot of three links, with well over 64 old and new neighbours."""
    from change_set_ref import change_set_ref
    from reconfig_ref import reconfig_ref
    m = _oracle64()
    cl = ds.clique()
    d, freqs, lp_feat = cl["data"][0], cl["freqs"], cl["lp_feat"]
    conns, _, ei = _graph(cl, 0, ds.CLIQUE_THRESHOLD)
    c = int(conns[_in_degree(conns, ei).argmax()])
    fi = {k: i for i, k in enumerate(lp_feat)}
    mine = np.trunc(d[fi["conn_id"]]) == c
    free = ~np.any(d != 0, axis=0) | mine
    links = [0, 3, 5]
    q = next(q for q in range(256) if free[links, q].all() and not mine[:, q].any())
    ch = (links, q, 1, [np.float32(freqs[q]), 16, 10, 100000])
    row, impact = reconfig_ref(m, d, freqs, lp_feat, c, *ch, freq_threshold=ds.CLIQUE_THRESHOLD, chunk=32)
    rows, s_imp = change_set_ref(m, d, freqs, lp_feat, [(c, *ch)], freq_threshold=ds.CLIQUE_THRESHOLD, chunk=32)
    assert len(impact) > 128 and {k for k, _ in impact.values()} >= {1, 2, 3}
    torch.testing.assert_close(rows[0], row, **TOL)
    assert s_imp.keys() == impact.keys()
    for k, (kind, r) in impact.items():
        assert s_imp[k][0] == kind
        torch.testing.assert_close(s_imp[k][1], r, **TOL)
    print(f"clique move: {len(impact)} impact rows")
