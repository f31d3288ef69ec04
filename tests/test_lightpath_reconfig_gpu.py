"""GPU parity of LightpathGNN's reconfiguration QoT (qot_lightpath_reconfigure through
LightpathGNN.forward_reconfigurations) against the fp64 oracle's literal definition (tests/reconfig_ref.py), against
forward_candidates for insertions (bit for bit) and against forward_every_node for no-op moves and teardowns, on every
status bit, and its determinism, CUDA-graph capture and error paths."""
import numpy as np
import pytest
import torch

from conftest import ABS_FLOOR, load_golden, rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-5
ATOL = ABS_FLOOR


def _model(dev):
    from gnn_qot_estimation_b200 import LightpathGNN
    sd = load_golden("ckpt_lightpath_model_1.pt")["model_state_dict"]
    m = LightpathGNN(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    m.load_state_dict(sd, strict=True)
    return m.to(dev).eval(), sd


def _oracle64(sd):
    from oracle import LightpathGNNOracle
    m = LightpathGNNOracle(5, 32, 3, is_lut_index=1, dropout_p=0.0).double()
    m.load_state_dict(sd, strict=True)
    return m.eval()


def _state(smp, dev, thr=0.05):
    from gnn_qot_estimation_b200.to_graph import lightpath_network_state
    return lightpath_network_state(torch.from_numpy(smp["data"]).to(dev), torch.from_numpy(smp["freqs"]),
                                   smp["lp_feat"], thr)


def _changes(rows, dev):
    """[(node, sample, links, q0, width, feat)] -> LightpathChanges on dev."""
    from gnn_qot_estimation_b200.to_graph import LightpathChanges
    lp = np.cumsum([0] + [len(r[2]) for r in rows])
    links = [l for r in rows for l in r[2]]
    return LightpathChanges(torch.tensor([r[0] for r in rows], dtype=torch.int64),
                            torch.tensor([r[1] for r in rows], dtype=torch.int64),
                            torch.tensor(lp, dtype=torch.int64), torch.tensor(links, dtype=torch.int32),
                            torch.tensor([r[3] for r in rows], dtype=torch.int32),
                            torch.tensor([r[4] for r in rows], dtype=torch.int32),
                            torch.tensor(np.array([r[5] for r in rows], dtype=np.float32).reshape(-1, 4))).to(dev)


def _rows_of(c):
    out = []
    for k in range(c.sample.shape[0]):
        a, b = int(c.link_ptr[k]), int(c.link_ptr[k + 1])
        out.append((int(c.node[k]), int(c.sample[k]), c.links[a:b].tolist(), int(c.q0[k]), int(c.width[k]),
                    c.feat[k].tolist()))
    return out


def _lightpaths(smp, state):
    """[(sample, node, conn_id, own links, q0, width, feat of the first channel)] of every lightpath of the state."""
    data, fi = smp["data"], {k: i for i, k in enumerate(smp["lp_feat"])}
    conn_ids, ptr = state.conn_ids.cpu(), state.batch.ptr.cpu()
    occ = np.any(data != 0, axis=1)
    out = []
    for s in range(data.shape[0]):
        conn = np.trunc(data[s, fi["conn_id"]])
        for v in range(int(ptr[s]), int(ptr[s + 1])):
            c = int(conn_ids[v])
            ls, qs = np.nonzero(occ[s] & (conn == c))
            feat = [data[s, fi[k], ls[0], qs[0]] for k in ("freq", "mod_order", "num_spans", "path_len")]
            out.append((s, v, c, sorted(set(ls.tolist())), int(qs.min()), int(qs.max() - qs.min() + 1), feat))
    return out


def _check_vs_ref(m, o, smp, state, rows, dev, max_impact=64):
    from reconfig_ref import reconfig_ref
    r = m.forward_reconfigurations(state, _changes(rows, dev), max_impact)
    torch.cuda.synchronize()
    conn = state.conn_ids.cpu()
    assert int(r.status.max()) == 0, r.status
    got_rows, ref_rows, kinds = [], [], []
    for k, (node, s, links, q0, w, feat) in enumerate(rows):
        row, impact = reconfig_ref(o, smp["data"][s], smp["freqs"], smp["lp_feat"],
                                   None if node < 0 else int(conn[node]), links, q0, w, feat)
        n = int(r.n_impact[k])
        assert n == len(impact)
        nodes = r.impact_node[k, :n].cpu()
        assert bool((nodes[1:] > nodes[:-1]).all())                      # ascending node order
        assert bool((r.impact_node[k, n:] == -1).all()) and bool(torch.isnan(r.impact_out[k, n:]).all())
        assert bool((r.impact_kind[k, n:] == 0).all())
        assert {int(conn[v]) for v in nodes} == set(impact)
        if row is None:
            assert bool(torch.isnan(r.out[k]).all())
        else:
            got_rows.append(r.out[k])
            ref_rows.append(row)
        for i, v in enumerate(nodes.tolist()):
            kind, ref = impact[int(conn[v])]
            assert int(r.impact_kind[k, i]) == kind
            kinds.append(kind)
            got_rows.append(r.impact_out[k, i])
            ref_rows.append(ref)
    got, ref = torch.stack(got_rows).double().cpu(), torch.stack(ref_rows)
    assert torch.isfinite(got).all()
    assert rel_err(got, ref) <= RTOL
    torch.testing.assert_close(got, ref, rtol=RTOL, atol=ATOL)
    return r, kinds


def test_reconfig_vs_oracle_fresh_seeds(cuda):
    """Generated retunes, reroutes, teardowns and insertions, plus: retunes by one slot that overlap a super-channel's
    own slots, reroutes that keep the lightpath's links and add one (kind 3 rows), moves to width 3, and moves next to
    a lightpath met on several links."""
    from gnn_qot_estimation_b200 import synthetic
    m, sd = _model(cuda)
    o = _oracle64(sd)
    smp = synthetic.network_status_samples(6, num_links=16, num_freqs=32, seed=31, super_channel_p=0.3)
    state = _state(smp, cuda)
    rows = _rows_of(synthetic.lightpath_changes(smp, state, 12, seed=32))
    occ = np.any(smp["data"] != 0, axis=1)
    freqs = smp["freqs"]
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    lps = _lightpaths(smp, state)
    extra = dict(overlap=0, keep=0, wide=0, multi=0)
    for s, v, c, links, q0, w, feat in lps:
        free = ~occ[s] | (occ[s] & (np.trunc(smp["data"][s, fi["conn_id"]]) == c))
        f = lambda q: [np.float32(freqs[q]), feat[1], feat[2], feat[3]]
        ok = lambda ls, q, ww: 0 <= q and q + ww <= 32 and free[np.ix_(ls, range(q, q + ww))].all()
        if w == 2 and extra["overlap"] < 6:
            for q in (q0 + 1, q0 - 1):
                if ok(links, q, 2):
                    rows.append((v, s, links, q, 2, f(q)))
                    extra["overlap"] += 1
                    break
        if extra["keep"] < 8:
            more = [l for l in range(16) if l not in links and ok([l], q0, w)]
            if more:
                rows.append((v, s, links + more[:1], q0, w, f(q0)))
                extra["keep"] += 1
        if extra["wide"] < 4:
            for q in range(max(q0 - 2, 0), q0 + 1):
                if ok(links, q, 3):
                    rows.append((v, s, links, q, 3, f(q)))
                    extra["wide"] += 1
                    break
        if len(links) >= 2 and extra["multi"] < 6:               # another lightpath moves next to j on j's links
            movers = [u for s2, u, *_ in lps if s2 == s and u != v]
            for q in (q0 + w, q0 - 1):
                if movers and 0 <= q < 32 and not occ[s][links, q].any():
                    rows.append((movers[0], s, links, q, 1, f(q)))
                    extra["multi"] += 1
                    break
    assert min(extra.values()) >= 2, extra
    r, kinds = _check_vs_ref(m, o, smp, state, rows, cuda)
    assert {1, 2, 3} <= set(kinds)
    nd = torch.tensor([row[0] for row in rows])
    assert bool((nd < 0).any()) and bool((nd >= 0).any())
    assert int(r.n_impact.max()) >= 3


def test_reconfig_threshold_boundary_and_empty_sample(cuda):
    """Spacing 0.05 on a 0.05 threshold (adjacency decided by fp64 rounding, as numpy decides it) for moves of every
    lightpath to every free slot of its links; insertions into an empty sample."""
    from gnn_qot_estimation_b200 import synthetic
    m, sd = _model(cuda)
    o = _oracle64(sd)
    smp = synthetic.network_status_samples(3, num_links=6, num_freqs=24, seed=5, spacing=0.05, max_lightpaths=14)
    smp["data"][2] = 0.0
    state = _state(smp, cuda)
    occ = np.any(smp["data"] != 0, axis=1)
    rows = []
    for s, v, c, links, q0, w, feat in _lightpaths(smp, state):
        for q in range(24 - w + 1):
            if q != q0 and not occ[s][np.ix_(links, range(q, q + w))].any():
                rows.append((v, s, links, q, w, [np.float32(smp["freqs"][q]), feat[1], feat[2], feat[3]]))
    rows = rows[::3]
    rows += [(-1, 2, [0, 3], 4, 2, [np.float32(smp["freqs"][4]), 8, 2, 90000]),
             (-1, 2, [5], 7, 1, [192.55, 4, 9, 80000])]
    r, kinds = _check_vs_ref(m, o, smp, state, rows, cuda)
    assert int(r.n_impact[-1]) == 0 and int(r.n_impact[-2]) == 0
    assert int((r.n_impact > 0).sum()) > 20 and {1, 2} <= set(kinds)      # kind 3: test_reconfig_vs_oracle_fresh_seeds


def test_insertions_are_bit_identical_to_candidates(cuda):
    from gnn_qot_estimation_b200 import synthetic
    from gnn_qot_estimation_b200.to_graph import LightpathChanges
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(16, seed=41, super_channel_p=0.2)
    state = _state(smp, cuda)
    c = synthetic.lightpath_candidates(smp, 64, seed=42).to(cuda)
    ch = LightpathChanges(torch.full_like(c.sample, -1), *c)
    for mi in (64, 1):
        a = m.forward_candidates(state, c, mi)
        b = m.forward_reconfigurations(state, ch, mi)
        torch.cuda.synchronize()
        for name in ("out", "status", "n_impact", "impact_node", "impact_out"):
            x, y = getattr(a, name), getattr(b, name)
            assert torch.equal(x.nan_to_num(7.0) if x.is_floating_point() else x,
                               y.nan_to_num(7.0) if y.is_floating_point() else y), name
        rows = torch.arange(mi, device=cuda)[None, :] < torch.clamp(b.n_impact.long(), max=mi)[:, None]
        assert bool((b.impact_kind[rows] == 2).all()) and bool((b.impact_kind[~rows] == 0).all())
    assert int(a.n_impact.max()) > 1


def test_noop_moves_and_teardowns_vs_every_node(cuda):
    """Every lightpath of 24 samples re-placed where it is: its row and its neighbours' rows are forward_every_node's
    rows of the state (kind 3).  Every lightpath torn down: the rows are forward_every_node's rows of the state without
    it (kind 1), matched by conn_id; n_impact is its degree, self loop excluded."""
    from gnn_qot_estimation_b200 import synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(24, seed=13, super_channel_p=0.2)
    data, fi = smp["data"], {k: i for i, k in enumerate(smp["lp_feat"])}
    state = _state(smp, cuda)
    every = m.forward_every_node(state.batch)
    lps = _lightpaths(smp, state)
    noop = [(v, s, links, q0, w, feat) for s, v, c, links, q0, w, feat in lps]
    r = m.forward_reconfigurations(state, _changes(noop, cuda), 64)
    torch.cuda.synchronize()
    assert int(r.status.max()) == 0
    sel = torch.arange(64, device=cuda)[None, :] < r.n_impact.long()[:, None]
    assert bool((r.impact_kind[sel] == 3).all())
    torch.testing.assert_close(r.out, every, rtol=RTOL, atol=ATOL)
    torch.testing.assert_close(r.impact_out[sel], every[r.impact_node[sel]], rtol=RTOL, atol=ATOL)
    assert int(sel.sum()) > 100
    ei = state.batch.edge_index
    deg = torch.bincount(ei[0][ei[0] != ei[1]], minlength=state.batch.x.shape[0])
    nodes = torch.tensor([v for _, v, *_ in lps], device=cuda)
    assert torch.equal(r.n_impact.long(), deg[nodes])
    # teardowns against the reduced states
    tear = [(v, s, [], 0, 1, feat) for s, v, c, links, q0, w, feat in lps]
    t = m.forward_reconfigurations(state, _changes(tear, cuda), 64)
    torch.cuda.synchronize()
    assert int(t.status.max()) == 0 and bool(torch.isnan(t.out).all())
    assert torch.equal(t.n_impact.long(), deg[nodes])
    reduced = []
    occ = np.any(data != 0, axis=1)
    for s, v, c, *_ in lps:
        rest = data[s].copy()
        rest[:, occ[s] & (np.trunc(data[s, fi["conn_id"]]) == c)] = 0.0
        reduced.append(rest)
    st2 = _state(dict(smp, data=np.stack(reduced)), cuda)
    after = m.forward_every_node(st2.batch)
    conn0, conn2, ptr2 = state.conn_ids, st2.conn_ids.cpu(), st2.batch.ptr.cpu()
    got, ref = [], []
    for k in range(len(lps)):
        n = int(t.n_impact[k])
        assert bool((t.impact_kind[k, :n] == 1).all())
        row_of = {int(conn2[u]): u for u in range(int(ptr2[k]), int(ptr2[k + 1]))}
        for i in range(n):
            got.append(t.impact_out[k, i])
            ref.append(after[row_of[int(conn0[t.impact_node[k, i]])]])
    torch.testing.assert_close(torch.stack(got), torch.stack(ref), rtol=RTOL, atol=ATOL)
    assert len(got) > 100


def test_reconfig_status_bits(cuda):
    from gnn_qot_estimation_b200 import ops, synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(3, num_links=8, num_freqs=20, seed=7, max_lightpaths=20,
                                           super_channel_p=0.4)
    smp["data"][2] = 0.0
    state = _state(smp, cuda)
    lps = _lightpaths(smp, state)
    occ = np.any(smp["data"] != 0, axis=1)
    s, v, c, links, q0, w, feat = next(lp for lp in lps if lp[0] == 0)
    ptr = state.batch.ptr.cpu()
    busy_l, busy_q = next((l, q) for l in range(8) for q in range(20)
                          if occ[0, l, q] and not (l in links and q0 <= q < q0 + w))
    f = [np.float32(smp["freqs"][3]), 16, 10, 100000]
    N = int(state.batch.x.shape[0])
    rows = [
        (int(ptr[1]), 0, [1], 3, 1, f),                   # 0: a node of sample 1 named in sample 0
        (N + 5, 0, [1], 3, 1, f),                         # 1: a node out of range
        (-7, 0, [1], 3, 1, f),                            # 2: a negative node other than -1
        (-1, 0, [], 3, 1, f),                             # 3: a teardown of nothing
        (v, 0, [busy_l], busy_q, 1, f),                   # 4: another lightpath's channel
        (v, 0, links, q0, w, feat),                       # 5: its own channels: fine
        (v, 3, [1], 3, 1, f),                             # 6: sample out of range
        (v, 0, [], 99, -4, f),                            # 7: a teardown ignores q0 and width
        (v, 0, [9], 3, 1, f),                             # 8: link out of range
    ]
    r = m.forward_reconfigurations(state, _changes(rows, cuda), 64)
    torch.cuda.synchronize()
    st = r.status.cpu().tolist()
    assert st[0:3] == [ops.CAND_BAD_NODE] * 3
    assert st[3] == ops.CAND_BAD_PATH
    assert st[4] == ops.CAND_OCCUPIED
    assert st[5] == 0 and bool(torch.isfinite(r.out[5]).all())
    assert st[6] == ops.CAND_BAD_SAMPLE
    assert st[7] == 0 and bool(torch.isnan(r.out[7]).all())
    assert st[8] == ops.CAND_BAD_PATH
    for k in (0, 1, 2, 3, 4, 6, 8):
        assert bool(torch.isnan(r.out[k]).all()) and int(r.n_impact[k]) == 0
        assert bool((r.impact_node[k] == -1).all()) and bool((r.impact_kind[k] == 0).all())
        assert bool(torch.isnan(r.impact_out[k]).all())
    # max_impact overflow: the first rows and kinds are kept, the true count reported
    gen = _rows_of(synthetic.lightpath_changes(smp, state, 20, seed=3))
    full = m.forward_reconfigurations(state, _changes(gen, cuda), 64)
    n = full.n_impact.cpu()
    k = int(torch.argmax(n))
    assert int(n[k]) >= 2
    cut = int(n[k]) - 1
    over = m.forward_reconfigurations(state, _changes(gen, cuda), cut)
    torch.cuda.synchronize()
    assert int(over.status[k]) == ops.CAND_IMPACT_OVERFLOW and int(over.n_impact[k]) == int(n[k])
    assert torch.equal(over.out[k].nan_to_num(7.0), full.out[k].nan_to_num(7.0))
    assert torch.equal(over.impact_node[k], full.impact_node[k, :cut])
    assert torch.equal(over.impact_kind[k], full.impact_kind[k, :cut])
    assert torch.equal(over.impact_out[k], full.impact_out[k, :cut])
    zero = m.forward_reconfigurations(state, _changes(gen, cuda), 0)
    assert zero.impact_out.shape == (len(gen), 0, 3) and zero.impact_kind.shape == (len(gen), 0)
    assert torch.equal(zero.out.nan_to_num(7.0), full.out.nan_to_num(7.0))
    assert torch.equal(zero.status.cpu() == ops.CAND_IMPACT_OVERFLOW, n > 0)


def test_reconfig_determinism_capture_errors_and_nodes(cuda):
    from gnn_qot_estimation_b200 import LightpathGNN, synthetic
    from gnn_qot_estimation_b200.to_graph import LightpathChanges, lightpath_nodes
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(16, seed=17)
    state = _state(smp, cuda)
    c = synthetic.lightpath_changes(smp, state, 64, seed=18).to(cuda)
    a = m.forward_reconfigurations(state, c)
    b = m.forward_reconfigurations(state, c)
    torch.cuda.synchronize()
    same = lambda x, y: torch.equal(x.nan_to_num(7.0) if x.is_floating_point() else x,
                                    y.nan_to_num(7.0) if y.is_floating_point() else y)
    assert all(same(x, y) for x, y in zip(a, b))
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    holder = {}
    with torch.cuda.stream(s):
        m.forward_reconfigurations(state, c)
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            holder["r"] = m.forward_reconfigurations(state, c)
        g.replay()
    torch.cuda.synchronize()
    assert all(same(x, y) for x, y in zip(holder["r"], a))
    # errors
    m.train()
    with pytest.raises(RuntimeError, match="eval"):
        m.forward_reconfigurations(state, c)
    m.eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        m.forward_reconfigurations(state, c.to("cpu"))
    with pytest.raises(TypeError, match="node"):
        m.forward_reconfigurations(state, c._replace(node=c.node.int()))
    with pytest.raises(TypeError, match="links"):
        m.forward_reconfigurations(state, c._replace(links=c.links.long()))
    with pytest.raises(ValueError, match="node"):
        m.forward_reconfigurations(state, c._replace(node=c.node[:-1]))
    with pytest.raises(ValueError, match="link_ptr"):
        m.forward_reconfigurations(state, c._replace(link_ptr=c.link_ptr[:-1]))
    with pytest.raises(ValueError, match="max_impact"):
        m.forward_reconfigurations(state, c, -1)
    odd = LightpathGNN(5, 16, 3, is_lut_index=1).to(cuda).eval()
    with pytest.raises(RuntimeError, match="reference LightpathGNN shape"):
        odd.forward_reconfigurations(state, c)
    empty = LightpathChanges(*(t[:0] for t in c))._replace(link_ptr=c.link_ptr[:1])
    r = m.forward_reconfigurations(state, empty)
    assert r.out.shape == (0, 3) and r.impact_out.shape == (0, 64, 3) and r.impact_kind.shape == (0, 64)
    # lightpath_nodes: conn_ids -> nodes of state.batch, -1 where the sample has no such lightpath
    nodes = torch.arange(state.conn_ids.shape[0], device=cuda)
    got = lightpath_nodes(state, state.batch.batch, state.conn_ids)
    assert torch.equal(got, nodes)
    smp_of = state.batch.batch
    absent = state.conn_ids.max() + 1
    miss = lightpath_nodes(state, torch.cat([smp_of[:5], torch.tensor([-1, 16, 1], device=cuda)]),
                           torch.cat([state.conn_ids[:5] + 10 ** 6, state.conn_ids[:2], absent[None]]))
    assert bool((miss == -1).all())
    perm = torch.randperm(nodes.numel(), generator=torch.Generator().manual_seed(0)).to(cuda)
    assert torch.equal(lightpath_nodes(state, smp_of[perm], state.conn_ids[perm].cpu()), perm)
