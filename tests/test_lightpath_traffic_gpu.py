"""GPU checks of LightpathGNN's dynamic traffic (qot_lightpath_traffic through LightpathGNN.forward_traffic and
to_graph.commit_traffic): bit-identity with the round loop of forward_reconfigurations teardowns, forward_placements and
rebuilds (tests/traffic_ref.py), the reduction to forward_provision without releases, hand-built release sequences,
capacity samples, parity with the fp64 literal reference, the commit, every status bit, determinism, CUDA-graph replay
and the error paths."""
import ctypes as C

import numpy as np
import pytest
import torch

from test_lightpath_provision_gpu import (ATOL, RTOL, _builder, _demands, _model, _node_bound, _oracle64, _pack,
                                          _same, _state)

pytestmark = pytest.mark.gpu
FIELDS = ("option", "q0", "out", "margin", "n_free", "n_feasible", "status", "n_impact", "impact_conn", "impact_out",
          "conn_id", "release_status", "release_conn_id", "release_n_impact", "release_impact_conn",
          "release_impact_out", "release_margin")


def _assert_same(r, ref, fields=FIELDS):
    for f in fields:
        assert _same(getattr(r, f), getattr(ref, f)), f


def _rel(rows, dev):
    """[(sample, before, demand, conn_id)] -> LightpathReleases on dev."""
    from gnn_qot_estimation_b200.to_graph import LightpathReleases
    cols = list(zip(*rows)) if rows else [[], [], [], []]
    return LightpathReleases(*(torch.tensor(list(c), dtype=torch.int64, device=dev) for c in cols))


def _round_loop(m, smp, dev, d, rel, policy, metric=0, maximize=True, bound=None, max_impact=64, thr=0.05):
    from traffic_ref import round_loop
    data = torch.from_numpy(smp["data"]).to(dev).contiguous()
    return round_loop(m, data, torch.from_numpy(smp["freqs"]).to(dev), smp["lp_feat"], d, rel, policy, metric,
                      maximize, bound, max_impact, thr)


def _mixed(seed=41):
    """5 samples, demands interleaved, releases by demand and by conn_id, ties in before, before = 0 and = D, and a
    sample (4) with releases only."""
    from gnn_qot_estimation_b200 import synthetic
    smp = synthetic.network_status_samples(5, num_links=12, num_freqs=40, seed=seed, super_channel_p=0.3)
    d, r = synthetic.lightpath_traffic(smp, 10, 4.0, seed=seed + 1, bound_range=(0.0, 0.5), release_existing=0.3)
    keep = d.sample != 4
    # sample 4 keeps its releases by conn_id only; its demands go to sample 0
    d = d._replace(sample=torch.where(keep, d.sample, torch.zeros_like(d.sample)))
    byd = r.demand >= 0
    r = r._replace(sample=torch.where(byd, d.sample[r.demand.clamp(min=0)], r.sample))
    D = int(d.sample.shape[0])
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    x = smp["data"][4]
    c4 = sorted(set(np.trunc(x[fi["conn_id"]][np.any(x != 0, axis=0)]).astype(int).tolist()))
    extra = [(4, 0, -1, c4[0]), (4, D, -1, c4[1]), (1, 0, -1, -5), (2, D, -1, 999999)]
    from gnn_qot_estimation_b200.to_graph import LightpathReleases
    r = LightpathReleases(*(torch.cat([a, torch.tensor([e[i] for e in extra])]) for i, a in enumerate(r)))
    return smp, d, r


# ------------------------------------------------------------------------------------------------ round loop
def test_round_loop_bit_identity(cuda):
    """Every policy, both senses, each metric column, with and without a bound: every demand and release output equal
    bit for bit to the round loop."""
    m, _ = _model(cuda)
    smp, d, r = _mixed()
    state = _state(smp, cuda)
    d, r = d.to(cuda), r.to(cuda)
    assert int(((r.before == int(d.sample.shape[0])) & (r.demand >= 0)).sum()) > 0
    assert int(torch.unique(r.before, return_counts=True)[1].max()) > 1
    released = accepted = 0
    for metric, mx in ((0, True), (1, True), (2, False), (0, False)):
        for bound in (None, _node_bound(m, state, metric, mx, 43 + metric, spread=0.05)):
            for policy in (0, 1, 2):
                t = m.forward_traffic(state, d, r, policy, metric, mx, bound)
                ref, _ = _round_loop(m, smp, cuda, d, r, policy, metric, mx, bound)
                torch.cuda.synchronize()
                _assert_same(t, ref)
                accepted += int((t.conn_id >= 0).sum())
                released += int((t.release_conn_id >= 0).sum())
    assert accepted > 100 and released > 100


def test_without_releases_equals_provision(cuda):
    from gnn_qot_estimation_b200 import synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(6, num_links=16, num_freqs=40, seed=51, super_channel_p=0.3)
    state = _state(smp, cuda)
    d = synthetic.lightpath_demands(smp, 8, seed=52, bound_range=(0.0, 0.5)).to(cuda)
    none = _rel([], cuda)
    for policy in (0, 1, 2):
        for b in (None, _node_bound(m, state, 0, True, 53)):
            t = m.forward_traffic(state, d, none, policy, 0, True, b)
            p = m.forward_provision(state, d, policy, 0, True, b)
            _assert_same(t, p, FIELDS[:11])
            assert t.release_status.numel() == 0


# ------------------------------------------------------------------------------------------------ hand-built
def test_hand_built_releases(cuda):
    """First fit takes the slots a release just freed; releasing the top lightpath then accepting gives top + 1 of the
    call, not a reused id; double release, release of a later demand and an unknown conn give TRAF_BAD_REF; release of
    a blocked demand gives TRAF_NOT_ACCEPTED; the lowest, a middle and the highest stable id released, each followed
    by arrivals; all against the round loop."""
    from gnn_qot_estimation_b200 import ops
    m, _ = _model(cuda)
    b = _builder(4, 24, 3)
    b.place([0], 0, 2)
    b.place([1, 2], 5)
    b.place([1], 6)
    b.place([2], 20)                                      # an interfering pair never released: the round loop's
    b.place([2], 21)                                      # rebuilds need a state with at least one edge
    b.place([3], 10)
    smp = _pack([b])
    state = _state(smp, cuda)
    cn = state.conn_ids.tolist()                          # node order (first channel): stable ids 0..5
    top = max(cn)
    f = (16, 10, 300000)
    ninf = -np.inf
    rows = [(0, [([0], 2, f, ninf)]),                     # 0: q0 2
            (0, [([0], 2, f, ninf)]),                     # 1: q0 0 after conn on slots 0-1 left; first fit
            (0, [([1], 1, f, np.inf)]),                   # 2: blocked
            (0, [([3], 1, f, ninf)]),                     # 3
            (0, [([0], 1, f, ninf)])]                     # 4
    d = _demands(rows, cuda)
    rel = [(0, 1, -1, cn[0]),                             # before 1: the lowest stable id (the slot-0 lightpath)
           (0, 3, 2, -1),                                 # release of the blocked demand 2: NOT_ACCEPTED
           (0, 3, 0, -1),                                 # demand 0 (top + 1)
           (0, 3, 1, -1),                                 # demand 1 (top + 2): the sample's largest id leaves
           (0, 3, 0, -1),                                 # demand 0 again: BAD_REF
           (0, 3, 4, -1),                                 # a later demand: BAD_REF
           (0, 3, -1, 424242),                            # unknown conn: BAD_REF
           (0, 4, -1, cn[1]),                             # a middle stable id
           (0, 5, 3, -1),                                 # the highest stable id (the last accepted)
           (0, 5, -1, cn[5])]
    r = _rel(rel, cuda)
    t = m.forward_traffic(state, d, r, ops.PLACE_FIRST_FIT)
    torch.cuda.synchronize()
    assert int(t.q0[0]) == 2 and int(t.q0[1]) == 0                # the freed slots 0-1 taken again
    assert t.conn_id.tolist()[:2] == [top + 1, top + 2] and int(t.conn_id[2]) == -1
    assert t.conn_id.tolist()[3:] == [top + 3, top + 4]           # top + 1, top + 2 released: never reused
    st = t.release_status.tolist()
    assert st[1] == ops.TRAF_NOT_ACCEPTED and st[4] == st[5] == st[6] == ops.TRAF_BAD_REF
    assert [st[k] & ~ops.CAND_IMPACT_OVERFLOW for k in (0, 2, 3, 7, 8, 9)] == [0] * 6
    assert t.release_conn_id.tolist() == [cn[0], -1, top + 1, top + 2, -1, -1, -1, cn[1], top + 3, cn[5]]
    ref, _ = _round_loop(m, smp, cuda, d, r, ops.PLACE_FIRST_FIT)
    _assert_same(t, ref)
    for policy in (1, 2):
        for bound in (None, _node_bound(m, state, 0, True, 5, spread=0.2)):
            t = m.forward_traffic(state, d, r, policy, 0, True, bound)
            ref, _ = _round_loop(m, smp, cuda, d, r, policy, 0, True, bound)
            _assert_same(t, ref)


def test_release_below_bound(cuda):
    """A release that takes a bounded neighbour below its bound gives a negative release_margin (reported, not
    refused), and the remaining bounds still bind later demands."""
    from gnn_qot_estimation_b200 import ops
    m, _ = _model(cuda)
    b = _builder(3, 24, 4)
    b.place([0], 4)
    b.place([0], 5)
    b.place([0], 6)
    b.place([1], 10)                                      # the round loop's rebuilds need at least one edge left
    b.place([1], 11)
    smp = _pack([b])
    state = _state(smp, cuda)
    every = m.forward_every_node(state.batch)[:, 0]
    conns = state.conn_ids.tolist()
    f = (16, 10, 300000)
    for k in range(len(conns)):
        # bound every lightpath exactly at its present value: any change of a neighbour row moves one side of it
        bound = every.clone().contiguous()
        r = _rel([(0, 0, -1, conns[k])], cuda)
        d = _demands([(0, [([0], 1, f, -np.inf), ([1], 1, f, -np.inf)])], cuda)
        t = m.forward_traffic(state, d, r, ops.PLACE_MAX_MARGIN, 0, True, bound)
        ref, _ = _round_loop(m, smp, cuda, d, r, ops.PLACE_MAX_MARGIN, 0, True, bound)
        torch.cuda.synchronize()
        _assert_same(t, ref)
        n = int(t.release_n_impact[0])
        assert n > 0
        mins = (t.release_impact_out[0, :n, 0] - bound[[conns.index(c) for c in t.release_impact_conn[0, :n].tolist()]])
        assert float(t.release_margin[0]) == float(mins.min())
    neg = []
    for k in range(len(conns)):
        t = m.forward_traffic(state, d, _rel([(0, 0, -1, conns[k])], cuda), ops.PLACE_MAX_MARGIN, 0, True,
                              every.contiguous())
        neg.append(float(t.release_margin[0]))
    assert min(neg) < 0


# ------------------------------------------------------------------------------------------------ capacity
def test_capacity(cuda):
    """A 256-lightpath sample reports PROV_FULL, then accepts after one release; the channel limit with a route past
    the 768-entry fallback; the hub and clique samples (more than 64 neighbour rows on a release: IMPACT_OVERFLOW)."""
    import dense_samples as ds
    from gnn_qot_estimation_b200 import ops
    m, _ = _model(cuda)
    f = (16, 10, 300000)
    smp = ds.full_sparse(3, counts=(256,))
    state = _state(smp, cuda, ds.HUB_THRESHOLD)
    c0 = int(state.conn_ids[0])
    d = _demands([(0, [([0], 1, f, -np.inf)])] * 2, cuda)
    r = _rel([(0, 1, -1, c0)], cuda)
    t = m.forward_traffic(state, d, r, ops.PLACE_FIRST_FIT)
    torch.cuda.synchronize()
    assert int(t.status[0]) & ops.PROV_FULL and int(t.conn_id[0]) == -1
    assert (int(t.status[1]) & ~ops.CAND_IMPACT_OVERFLOW) == 0 and int(t.conn_id[1]) >= 0
    ref, _ = _round_loop(m, smp, cuda, d, r, ops.PLACE_FIRST_FIT, thr=ds.HUB_THRESHOLD)
    _assert_same(t, ref)
    # channels: 254 lightpaths of 8 links x 3 slots on L = 64, Q = 97; a 9-link route on slot column 96 holds 864
    # channels of known lightpaths (the entry-list fallback); a 6-wide 8-link route is over the channel limit until
    # one lightpath leaves
    b = _builder(64, 97, 11)
    for k in range(254):
        b.place(list(range(8 * (k // 32), 8 * (k // 32) + 8)), 3 * (k % 32), 3)
    g = _pack([b])
    gs = _state(g, cuda, ds.HUB_THRESHOLD)
    rows = [(0, [(list(range(9)), 1, f, -np.inf)]), (0, [(list(range(56, 64)), 6, f, -np.inf)]),
            (0, [(list(range(56, 64)), 6, f, -np.inf)])]
    d = _demands(rows, cuda)
    victim = int(gs.conn_ids[gs.chan_node[0, 0, 0] - 0])
    r = _rel([(0, 2, -1, victim), (0, 2, -1, int(gs.conn_ids[gs.chan_node[0, 56, 3]]))], cuda)
    for policy, bound in ((0, None), (2, _node_bound(m, gs, 0, True, 12, spread=0.2))):
        t = m.forward_traffic(gs, d, r, policy, 0, True, bound, 256)
        ref, _ = _round_loop(m, g, cuda, d, r, policy, 0, True, bound, 256, ds.HUB_THRESHOLD)
        torch.cuda.synchronize()
        _assert_same(t, ref)
        if policy == 0:
            assert int(t.conn_id[0]) >= 0 and int(t.status[1]) & ops.PROV_FULL and int(t.conn_id[2]) >= 0
    over = 0
    for smp, thr in ((ds.hub(7), ds.HUB_THRESHOLD), (ds.clique(8, n=200), ds.CLIQUE_THRESHOLD)):
        st = _state(smp, cuda, thr)
        L = smp["data"].shape[2]
        rng = np.random.default_rng(9)
        rows = [(0, [(sorted(rng.choice(L, 2, replace=False).tolist()), 1, f, -np.inf), ([0], 1, f, 0.2)])
                for _ in range(6)]
        d = _demands(rows, cuda)
        cs = st.conn_ids.tolist()
        r = _rel([(0, 0, -1, cs[0]), (0, 2, -1, cs[len(cs) // 2]), (0, 3, 1, -1), (0, 6, -1, cs[-1])], cuda)
        bound = _node_bound(m, st, 0, True, 10, spread=0.2)
        for policy, bb in ((0, None), (2, bound)):
            t = m.forward_traffic(st, d, r, policy, 0, True, bb, 32)
            ref, _ = _round_loop(m, smp, cuda, d, r, policy, 0, True, bb, 32, thr)
            _assert_same(t, ref)
            over += int(((t.release_status & ops.CAND_IMPACT_OVERFLOW) != 0).sum())
    assert over > 0


# ------------------------------------------------------------------------------------------------ fp64
def test_vs_fp64_reference(cuda):
    """traffic_ref on the fp64 oracle, following the kernel's choices: every demand's own and impact rows and every
    release's neighbour rows at 1e-5, and the releases' conn_ids."""
    from gnn_qot_estimation_b200 import synthetic
    from traffic_ref import traffic_ref
    m, sd = _model(cuda)
    o = _oracle64(sd, cuda)
    smp = synthetic.network_status_samples(1, num_links=5, num_freqs=20, seed=61, spacing=0.05, max_lightpaths=8,
                                           super_channel_p=0.3)
    state = _state(smp, cuda)
    f1, f2 = (16, 40, 2000000), (64, 9, 80000)
    opts = [[([0], 1, f1, -np.inf), ([1, 2], 2, f2, -np.inf)], [([0], 1, f1, -np.inf)], [([0, 3], 1, f2, -np.inf)],
            [([2], 1, f2, -np.inf)]]
    c0 = sorted(state.conn_ids.tolist())
    rel = [(0, 1, -1, c0[0]), (0, 2, 0, -1), (0, 4, -1, c0[-1]), (0, 4, 1, -1)]
    d = _demands([(0, o_) for o_ in opts], cuda)
    t = m.forward_traffic(state, d, _rel(rel, cuda), 0, 0, True, None, 256)
    torch.cuda.synchronize()
    seq = [("d", opts[0]), ("r", c0[0]), ("d", opts[1]), ("rd", 0), ("d", opts[2]), ("d", opts[3]), ("r", c0[-1]),
           ("rd", 2)]
    dix = {0: 0, 2: 1, 4: 2, 5: 3}
    follow = [(int(t.option[k]), int(t.q0[k])) if int(t.conn_id[k]) >= 0 else None for k in range(4)]
    steps, _ = traffic_ref(o, smp["data"][0], smp["freqs"], smp["lp_feat"], seq, 0, follow=follow, device=cuda)
    rix = {1: 0, 3: 1, 6: 2, 7: 3}
    for e, st in enumerate(steps):
        if e in dix:
            k = dix[e]
            if follow[k] is None:
                continue
            row, imp, _ = st["table"][follow[k]]
            torch.testing.assert_close(t.out[k].double().cpu(), row, rtol=RTOL, atol=ATOL)
            n = int(t.n_impact[k])
            assert n == len(imp) and set(t.impact_conn[k, :n].tolist()) == set(imp)
        else:
            k = rix[e]
            assert int(t.release_conn_id[k]) == (st["conn"] if st["conn"] is not None else -1)
            n = int(t.release_n_impact[k])
            assert n == len(st["rows"])
            for i in range(n):
                torch.testing.assert_close(t.release_impact_out[k, i].double().cpu(),
                                           st["rows"][int(t.release_impact_conn[k, i])], rtol=RTOL, atol=ATOL)


# ------------------------------------------------------------------------------------------------ commit
def test_commit_traffic(cuda):
    """commit_traffic equals the round loop's final state (x, edges, conn_ids, chan_node) and the samples it wrote."""
    from gnn_qot_estimation_b200.to_graph import commit_traffic
    m, _ = _model(cuda)
    smp, d, r = _mixed(71)
    state = _state(smp, cuda)
    d, r = d.to(cuda), r.to(cuda)
    t = m.forward_traffic(state, d, r, 2)
    data = torch.from_numpy(smp["data"]).to(cuda).contiguous()
    new = commit_traffic(data, state, d, r, t)
    _, fin = _round_loop(m, smp, cuda, d, r, 2)
    for f in ("x", "edge_index", "ptr", "batch"):
        assert torch.equal(getattr(new.batch, f), getattr(fin.batch, f)), f
    for f in ("rowptr", "conn_ids", "chan_node"):
        assert torch.equal(getattr(new, f), getattr(fin, f)), f
    assert int((t.release_conn_id >= 0).sum()) > 10 and int((t.conn_id >= 0).sum()) > 10


# ------------------------------------------------------------------------------------------------ status, errors
def _c_call(m, state, d, r, order, sp, rel_order, rel_ptr, max_impact=4):
    from gnn_qot_estimation_b200 import _lib, ops
    from gnn_qot_estimation_b200.ops import _demands_desc, _state_desc, ptr, stream
    D, P, R, dev = int(d.sample.shape[0]), int(d.width.shape[0]), int(r.sample.shape[0]), state.batch.x.device
    i32 = lambda n: torch.full((n,), 99, dtype=torch.int32, device=dev)
    i64 = lambda *s: torch.full(s, 99, dtype=torch.int64, device=dev)
    res = ops.TrafficQoT(i32(D), i32(D), torch.zeros(D, 3, device=dev), torch.zeros(D, device=dev), i32(D), i32(D),
                         i32(D), i32(D), i64(D, max_impact), torch.zeros(D, max_impact, 3, device=dev), i64(D),
                         i32(R), i64(R), i32(R), i64(R, max_impact), torch.zeros(R, max_impact, 3, device=dev),
                         torch.zeros(R, device=dev))
    keep = []
    cw = torch.empty_like(state.chan_node)
    rel = _lib.QotLpReleases(R, ptr(r.sample), ptr(r.before), ptr(r.demand), ptr(r.conn_id))
    rc = _lib.lib().qot_lightpath_traffic(
        C.byref(_state_desc(state, keep)), C.byref(_demands_desc(d, D, P, keep)), ptr(order), ptr(sp), None, 0, 1, 0,
        ptr(m.prepared()), 1, max_impact, ptr(cw), None, *(ptr(x) for x in res[:8]), ptr(res.conn_id),
        ptr(res.impact_conn), ptr(res.impact_out), C.byref(rel), ptr(rel_order),
        ptr(rel_ptr), *(ptr(x) for x in res[11:]), stream())
    torch.cuda.synchronize()
    return rc, res


def test_status_bits_and_c_groupings(cuda):
    """CAND_BAD_SAMPLE and CAND_BAD_STATE on releases, before outside [0, D], a demand of another sample, and every
    malformed release grouping through the C entry point: every demand and release output PROV_BAD_GROUPING alone."""
    from gnn_qot_estimation_b200 import ops, synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(3, num_links=8, num_freqs=32, seed=81)
    state = _state(smp, cuda)
    f = (16, 10, 300000)
    d = _demands([(0, [([0], 1, f, -np.inf)]), (1, [([1], 1, f, -np.inf)]), (0, [([2], 1, f, -np.inf)])], cuda)
    c1 = int(state.conn_ids[int(state.batch.ptr[1])])
    r = _rel([(5, 0, -1, 1), (-1, 0, -1, 1), (0, -1, -1, c1), (0, 4, -1, c1), (0, 2, 1, -1), (1, 3, -1, c1)], cuda)
    t = m.forward_traffic(state, d, r, 0, max_impact=0)
    torch.cuda.synchronize()
    assert t.release_status.tolist()[:5] == [ops.CAND_BAD_SAMPLE] * 2 + [ops.TRAF_BAD_REF] * 3
    assert (int(t.release_status[5]) & ~ops.CAND_IMPACT_OVERFLOW) == 0 and int(t.release_conn_id[5]) == c1
    assert t.release_conn_id.tolist()[:5] == [-1] * 5 and bool(torch.isnan(t.release_margin).all())
    # a sample whose graph is inconsistent: node n0's out-run of sample 1 ends before it starts
    bad = state._replace(rowptr=state.rowptr.clone())
    n0 = int(state.batch.ptr[1])
    bad.rowptr[n0 + 1] = bad.rowptr[n0] - 1
    tb = m.forward_traffic(bad, d, _rel([(1, 3, -1, c1), (0, 0, -1, int(state.conn_ids[0]))], cuda), 0)
    torch.cuda.synchronize()
    assert int(tb.release_status[0]) == ops.CAND_BAD_STATE and int(tb.release_conn_id[1]) >= 0
    # D = 0 with releases: a sample with releases only
    e = d._replace(sample=d.sample[:0], opt_ptr=d.opt_ptr[:1], link_ptr=d.link_ptr[:1], links=d.links[:0],
                   width=d.width[:0], feat=d.feat[:0], own_bound=d.own_bound[:0])
    te = m.forward_traffic(state, e, _rel([(1, 0, -1, c1), (1, 0, -1, c1)], cuda), 0)
    torch.cuda.synchronize()
    assert te.release_conn_id.tolist() == [c1, -1] and int(te.release_status[1]) == ops.TRAF_BAD_REF
    # malformed release groupings through the C ABI
    g = _rel([(0, 1, -1, 100001), (1, 0, -1, 100002), (0, 0, -1, 100003)], cuda)
    i64 = lambda v: torch.tensor(v, dtype=torch.int64, device=cuda)
    order, sp = i64([0, 2, 1]), i64([0, 2, 3, 3])
    rc, ok = _c_call(m, state, d, g, order, sp, i64([2, 0, 1]), i64([0, 2, 3, 3]))
    assert rc == 0 and int(ok.status.max()) == 0 and ok.release_status.tolist() == [ops.TRAF_BAD_REF] * 3
    for ro, rp in (([0, 2, 1], [0, 2, 3, 3]),       # not by before within sample 0
                   ([2, 1, 0], [0, 2, 3, 3]),       # release 1 is not sample 0's
                   ([2, 0, 1], [1, 2, 3, 3]),       # rel_ptr[0] != 0
                   ([2, 0, 1], [0, 2, 1, 3]),       # decreasing
                   ([2, 0, 1], [0, 2, 2, 2]),       # a release left out
                   ([2, 0, 7], [0, 2, 3, 3]),       # rel_order outside [0, R)
                   ([2, 2, 1], [0, 2, 3, 3])):      # a release twice
        rc, res = _c_call(m, state, d, g, order, sp, i64(ro), i64(rp))
        assert rc == 0
        assert res.status.tolist() == [ops.PROV_BAD_GROUPING] * 3, (ro, rp)
        assert res.release_status.tolist() == [ops.PROV_BAD_GROUPING] * 3, (ro, rp)
        assert res.conn_id.tolist() == [-1] * 3 and res.release_conn_id.tolist() == [-1] * 3
        assert res.release_n_impact.tolist() == [0] * 3 and bool(torch.isnan(res.release_impact_out).all())
        assert bool((res.release_impact_conn == -1).all()) and bool(torch.isnan(res.release_margin).all())


def test_determinism_capture_and_errors(cuda):
    m, _ = _model(cuda)
    smp, d, r = _mixed(91)
    state = _state(smp, cuda)
    d, r = d.to(cuda), r.to(cuda)
    bound = _node_bound(m, state, 0, True, 93)
    cn = state.chan_node.clone()
    a = m.forward_traffic(state, d, r, 2, 0, True, bound)
    b = m.forward_traffic(state, d, r, 2, 0, True, bound)
    torch.cuda.synchronize()
    _assert_same(a, b)
    assert torch.equal(state.chan_node, cn)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        m.forward_traffic(state, d, r, 2, 0, True, bound)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c = m.forward_traffic(state, d, r, 2, 0, True, bound)
    g.replay()
    torch.cuda.synchronize()
    _assert_same(a, c)
    with pytest.raises(ValueError):
        m.forward_traffic(state, d, r, 7)
    with pytest.raises(ValueError):
        m.forward_traffic(state, d, r._replace(before=r.before[:-1]), 0)
    with pytest.raises(TypeError):
        m.forward_traffic(state, d, r._replace(demand=r.demand.int()), 0)
    with pytest.raises(RuntimeError):
        m.forward_traffic(state, d, r.to("cpu"), 0)
    with pytest.raises(ValueError):
        m.forward_traffic(state, d, r, 0, bound=bound[:-1])
    m.train()
    with pytest.raises(RuntimeError):
        m.forward_traffic(state, d, r, 0)
    m.eval()
