"""GPU parity of LightpathGNN's candidate QoT (csrc/lightpath_candidates.cu through to_graph.lightpath_network_state
and LightpathGNN.forward_candidates) against the fp64 oracle's literal definition (tests/candidates_ref.py), against
every-node mode by leave-one-out, on every status bit, and its determinism, CUDA-graph capture and error paths."""
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


def _cands(rows, dev):
    """[(sample, links, q0, width, feat)] -> LightpathCandidates on dev."""
    from gnn_qot_estimation_b200.to_graph import LightpathCandidates
    lp = np.cumsum([0] + [len(r[1]) for r in rows])
    links = [l for r in rows for l in r[1]]
    return LightpathCandidates(torch.tensor([r[0] for r in rows], dtype=torch.int64),
                               torch.tensor(lp, dtype=torch.int64), torch.tensor(links, dtype=torch.int32),
                               torch.tensor([r[2] for r in rows], dtype=torch.int32),
                               torch.tensor([r[3] for r in rows], dtype=torch.int32),
                               torch.tensor(np.array([r[4] for r in rows], dtype=np.float32).reshape(-1, 4))).to(dev)


def _rows_of(c):
    out = []
    for k in range(c.sample.shape[0]):
        a, b = int(c.link_ptr[k]), int(c.link_ptr[k + 1])
        out.append((int(c.sample[k]), c.links[a:b].tolist(), int(c.q0[k]), int(c.width[k]), c.feat[k].tolist()))
    return out


def _state(smp, dev, thr=0.05):
    from gnn_qot_estimation_b200.to_graph import lightpath_network_state
    return lightpath_network_state(torch.from_numpy(smp["data"]).to(dev), torch.from_numpy(smp["freqs"]),
                                   smp["lp_feat"], thr)


def _check_vs_ref(m, o, smp, state, rows, dev, max_impact=64):
    from candidates_ref import candidates_ref
    r = m.forward_candidates(state, _cands(rows, dev), max_impact)
    torch.cuda.synchronize()
    conn = state.conn_ids.cpu()
    assert int(r.status.max()) == 0
    got_rows, ref_rows = [], []
    for k, (s, links, q0, w, feat) in enumerate(rows):
        row, impact = candidates_ref(o, smp["data"][s], smp["freqs"], smp["lp_feat"], links, q0, w, feat)
        n = int(r.n_impact[k])
        assert n == len(impact)
        nodes = r.impact_node[k, :n].cpu()
        assert bool((nodes[1:] > nodes[:-1]).all())                      # ascending node order
        assert bool((r.impact_node[k, n:] == -1).all()) and bool(torch.isnan(r.impact_out[k, n:]).all())
        assert {int(conn[v]) for v in nodes} == set(impact)
        got_rows.append(r.out[k])
        ref_rows.append(row)
        for i, v in enumerate(nodes.tolist()):
            got_rows.append(r.impact_out[k, i])
            ref_rows.append(impact[int(conn[v])])
    got, ref = torch.stack(got_rows).double().cpu(), torch.stack(ref_rows)
    assert torch.isfinite(got).all()
    assert rel_err(got, ref) <= RTOL
    torch.testing.assert_close(got, ref, rtol=RTOL, atol=ATOL)
    return r


def test_candidates_vs_oracle_fresh_seeds(cuda):
    from gnn_qot_estimation_b200 import synthetic
    m, sd = _model(cuda)
    o = _oracle64(sd)
    smp = synthetic.network_status_samples(6, num_links=16, num_freqs=32, seed=21, super_channel_p=0.3)
    state = _state(smp, cuda)
    rows = _rows_of(synthetic.lightpath_candidates(smp, 10, seed=22))
    # wide super-channel candidates and a lightpath met on several links: next to a multi-link lightpath on all of
    # its links, on a free slot
    data = smp["data"]
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    occ = np.any(data != 0, axis=1)
    multi = 0
    for s in range(6):
        conn = np.trunc(data[s, fi["conn_id"]])
        for c in np.unique(conn[occ[s]]):
            ls, qs = np.nonzero(occ[s] & (conn == c))
            links = sorted(set(ls.tolist()))
            if len(links) < 2:
                continue
            for q in (int(qs.max()) + 1, int(qs.min()) - 1, int(qs.max()) + 2):
                if 0 <= q < 32 and not occ[s][links, q].any():
                    rows.append((s, links, q, 1, [np.float32(smp["freqs"][q]), 32, 20, 500000]))
                    multi += 1
                    break
        free = np.flatnonzero(~occ[s][[0, 1]].any(axis=0))
        runs = [q for q in free if q + 2 < 32 and all(q + u in free for u in range(3))]
        if runs:
            rows.append((s, [1, 0, 1], int(runs[0]), 3, [np.float32(smp["freqs"][runs[0]]), 64, 3, 30000]))
    assert multi >= 3
    r = _check_vs_ref(m, o, smp, state, rows, cuda)
    assert int(r.n_impact.max()) >= 3


def test_candidates_threshold_boundary_and_no_neighbours(cuda):
    """Spacing 0.05 on a 0.05 threshold (adjacency decided by fp64 rounding, as numpy decides it); an empty sample
    and an empty link (no neighbours)."""
    from gnn_qot_estimation_b200 import synthetic
    m, sd = _model(cuda)
    o = _oracle64(sd)
    smp = synthetic.network_status_samples(3, num_links=6, num_freqs=24, seed=5, spacing=0.05, max_lightpaths=16)
    smp["data"][2] = 0.0                                                  # an empty sample
    smp["data"][1][:, 5, :] = 0.0                                         # an empty link
    state = _state(smp, cuda)
    occ = np.any(smp["data"] != 0, axis=1)
    rows = []
    for s in range(2):
        for l in range(6):
            for q in np.flatnonzero(~occ[s, l]):
                rows.append((s, [l], int(q), 1, [np.float32(smp["freqs"][q]), 16, 40, 2000000]))
    rows += [(2, [0, 3], 4, 2, [np.float32(smp["freqs"][4]), 8, 2, 90000]), (1, [5], 7, 1, [192.55, 4, 9, 80000])]
    r = _check_vs_ref(m, o, smp, state, rows, cuda)
    assert int(r.n_impact[-1]) == 0 and int(r.n_impact[-2]) == 0
    assert int((r.n_impact > 0).sum()) > 20


def test_leave_one_out_vs_every_node(cuda):
    """Every lightpath of 24 samples, removed from its sample and offered back as a candidate: the candidate row is
    forward_every_node's row for it in the original state, the impact rows are the original rows of its neighbours
    (matched by conn_id)."""
    from gnn_qot_estimation_b200 import synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(24, seed=13, super_channel_p=0.2)
    data, fi = smp["data"], {k: i for i, k in enumerate(smp["lp_feat"])}
    state = _state(smp, cuda)
    every = m.forward_every_node(state.batch).cpu()
    conn0, ptr0 = state.conn_ids.cpu(), state.batch.ptr.cpu()
    before = {(s, int(conn0[v])): every[v] for s in range(24) for v in range(int(ptr0[s]), int(ptr0[s + 1]))}
    occ = np.any(data != 0, axis=1)
    reduced, rows, who = [], [], []
    for s in range(24):
        conn = np.trunc(data[s, fi["conn_id"]])
        for c in np.unique(conn[occ[s]]):
            mine = occ[s] & (conn == c)
            ls, qs = np.nonzero(mine)
            links = sorted(set(ls.tolist()))
            q0, w = int(qs.min()), int(qs.max() - qs.min() + 1)
            feat = [data[s, fi[k], ls[0], qs[0]] for k in ("freq", "mod_order", "num_spans", "path_len")]
            rest = data[s].copy()
            rest[:, mine] = 0.0
            rows.append((len(reduced), links, q0, w, feat))
            reduced.append(rest)
            who.append((s, int(c)))
    red = dict(smp, data=np.stack(reduced))
    st2 = _state(red, cuda)
    r = m.forward_candidates(st2, _cands(rows, cuda), 64)
    torch.cuda.synchronize()
    assert int(r.status.max()) == 0
    conn2 = st2.conn_ids.cpu()
    got, ref = [r.out.cpu()], [torch.stack([before[w_] for w_ in who])]
    for k, (s, c) in enumerate(who):
        n = int(r.n_impact[k])
        nodes = r.impact_node[k, :n].cpu()
        got.append(r.impact_out[k, :n].cpu())
        ref.append(torch.stack([before[(s, int(conn2[v]))] for v in nodes]) if n else torch.zeros(0, 3))
    got, ref = torch.cat(got), torch.cat(ref)
    assert got.shape[0] > len(who) + 100
    torch.testing.assert_close(got, ref, rtol=RTOL, atol=ATOL)
    # n_impact is the lightpath's degree in the original graph (self loops aside)
    ei = state.batch.edge_index.cpu()
    deg = torch.bincount(ei[0][ei[0] != ei[1]], minlength=conn0.shape[0])
    node_of = {(s, int(conn0[v])): v for s in range(24) for v in range(int(ptr0[s]), int(ptr0[s + 1]))}
    assert torch.equal(r.n_impact.cpu().long(), torch.stack([deg[node_of[w_]] for w_ in who]))


def test_candidate_status_bits(cuda):
    from gnn_qot_estimation_b200 import ops, synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(3, num_links=8, num_freqs=20, seed=7, max_lightpaths=20)
    smp["data"][2] = 0.0
    state = _state(smp, cuda)
    occ = np.any(smp["data"] != 0, axis=1)
    l_busy, q_busy = [int(v[0]) for v in np.nonzero(occ[0])]
    f = [np.float32(smp["freqs"][3]), 16, 10, 100000]
    good = synthetic.lightpath_candidates(smp, 2, seed=1)
    gl = _rows_of(good)
    rows = [
        (0, [l_busy], q_busy, 1, f),                      # 0: occupied
        (0, [0, 8], 3, 1, f),                             # 1: link out of range
        (0, [], 3, 1, f),                                 # 2: empty path
        (0, [1], 19, 2, f),                               # 3: slot range past Q
        (0, [1], -1, 1, f),                               # 4: slot range before 0
        (0, [1], 3, 0, f),                                # 5: width 0
        (3, [1], 3, 1, f),                                # 6: sample out of range
        (-1, [1], 3, 1, f),                               # 7: negative sample
        (2, [1, 2], 3, 1, f),                             # 8: empty sample: fine, no neighbours
    ] + gl
    dup = [(s, ls + ls[::-1] + ls, q0, w, ft) for s, ls, q0, w, ft in gl]   # duplicate links
    rows += dup
    r = m.forward_candidates(state, _cands(rows, cuda), 64)
    torch.cuda.synchronize()
    st = r.status.cpu().tolist()
    assert st[0] == ops.CAND_OCCUPIED
    assert st[1:6] == [ops.CAND_BAD_PATH] * 5
    assert st[6:8] == [ops.CAND_BAD_SAMPLE] * 2
    assert st[8] == 0 and int(r.n_impact[8]) == 0 and bool(torch.isfinite(r.out[8]).all())
    for k in range(8):
        assert bool(torch.isnan(r.out[k]).all()) and int(r.n_impact[k]) == 0
        assert bool((r.impact_node[k] == -1).all()) and bool(torch.isnan(r.impact_out[k]).all())
    ng = len(gl)
    base = 9
    for k in range(ng):                                    # duplicates change nothing
        a, b = base + k, base + ng + k
        assert st[a] == st[b] == 0
        assert torch.equal(r.out[a], r.out[b]) and torch.equal(r.n_impact[a], r.n_impact[b])
        assert torch.equal(r.impact_node[a], r.impact_node[b])
        torch.testing.assert_close(r.impact_out[a], r.impact_out[b], rtol=0, atol=0, equal_nan=True)
    # max_impact overflow: the first rows are written, the true count reported
    full = m.forward_candidates(state, _cands(gl, cuda), 64)
    n = full.n_impact.cpu()
    k = int(torch.argmax(n))
    assert int(n[k]) >= 2
    cut = int(n[k]) - 1
    over = m.forward_candidates(state, _cands(gl, cuda), cut)
    torch.cuda.synchronize()
    assert int(over.status[k]) == ops.CAND_IMPACT_OVERFLOW and int(over.n_impact[k]) == int(n[k])
    assert torch.equal(over.out[k], full.out[k])
    assert torch.equal(over.impact_node[k], full.impact_node[k, :cut])
    assert torch.equal(over.impact_out[k], full.impact_out[k, :cut])
    zero = m.forward_candidates(state, _cands(gl, cuda), 0)
    assert zero.impact_out.shape == (len(gl), 0, 3)
    assert torch.equal(zero.out, full.out)
    assert torch.equal(zero.status.cpu() == ops.CAND_IMPACT_OVERFLOW, n > 0)


def test_candidates_determinism_capture_and_errors(cuda):
    from gnn_qot_estimation_b200 import LightpathGNN, synthetic
    from gnn_qot_estimation_b200.to_graph import LightpathCandidates
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(16, seed=17)
    state = _state(smp, cuda)
    c = synthetic.lightpath_candidates(smp, 64, seed=18).to(cuda)
    a = m.forward_candidates(state, c)
    b = m.forward_candidates(state, c)
    torch.cuda.synchronize()
    for x, y in zip(a, b):
        assert torch.equal(x.nan_to_num(7.0) if x.is_floating_point() else x,
                           y.nan_to_num(7.0) if y.is_floating_point() else y)
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    holder = {}
    with torch.cuda.stream(s):
        m.forward_candidates(state, c)
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            holder["r"] = m.forward_candidates(state, c)
        g.replay()
    torch.cuda.synchronize()
    for x, y in zip(holder["r"], a):
        assert torch.equal(x.nan_to_num(7.0) if x.is_floating_point() else x,
                           y.nan_to_num(7.0) if y.is_floating_point() else y)
    # the state's batch serves forward_every_node directly
    assert m.forward_every_node(state.batch).shape == (state.batch.x.shape[0], 3)
    # errors
    m.train()
    with pytest.raises(RuntimeError, match="eval"):
        m.forward_candidates(state, c)
    m.eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        m.forward_candidates(state, c.to("cpu"))
    with pytest.raises(TypeError, match="links"):
        m.forward_candidates(state, c._replace(links=c.links.long()))
    with pytest.raises(TypeError, match="feat"):
        m.forward_candidates(state, c._replace(feat=c.feat.double()))
    with pytest.raises(ValueError, match="link_ptr"):
        m.forward_candidates(state, c._replace(link_ptr=c.link_ptr[:-1]))
    with pytest.raises(ValueError, match="feat"):
        m.forward_candidates(state, c._replace(feat=c.feat[:, :3]))
    with pytest.raises(ValueError, match="max_impact"):
        m.forward_candidates(state, c, -1)
    odd = LightpathGNN(5, 16, 3, is_lut_index=1).to(cuda).eval()
    with pytest.raises(RuntimeError, match="reference LightpathGNN shape"):
        odd.forward_candidates(state, c)
    empty = LightpathCandidates(*(t[:0] for t in c))._replace(link_ptr=c.link_ptr[:1])
    r = m.forward_candidates(state, empty)
    assert r.out.shape == (0, 3) and r.impact_out.shape == (0, 64, 3)
    with pytest.raises(RuntimeError, match="CUDA"):
        from gnn_qot_estimation_b200.to_graph import lightpath_network_state
        lightpath_network_state(torch.from_numpy(smp["data"]), torch.from_numpy(smp["freqs"]), smp["lp_feat"])
