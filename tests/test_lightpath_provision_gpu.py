"""GPU checks of LightpathGNN's sequential provisioning (qot_lightpath_provision through
LightpathGNN.forward_provision and to_graph.commit_provision): bit-identity with the round loop of forward_placements
and rebuilds (tests/provision_ref.py), the reduction to forward_placements, sequential effects on hand-built samples,
parity with the fp64 literal reference, the commit, capacity samples, every status bit, determinism, CUDA-graph
replay and the error paths."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import ABS_FLOOR, load_golden

pytestmark = pytest.mark.gpu
RTOL = 1e-5
ATOL = ABS_FLOOR
FIELDS = ("option", "q0", "out", "margin", "n_free", "n_feasible", "status", "n_impact", "impact_conn", "impact_out",
          "conn_id")


def _model(dev):
    from gnn_qot_estimation_b200 import LightpathGNN
    sd = load_golden("ckpt_lightpath_model_1.pt")["model_state_dict"]
    m = LightpathGNN(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    m.load_state_dict(sd, strict=True)
    return m.to(dev).eval(), sd


def _oracle64(sd, dev):
    from oracle import LightpathGNNOracle
    m = LightpathGNNOracle(5, 32, 3, is_lut_index=1, dropout_p=0.0).double()
    m.load_state_dict(sd, strict=True)
    return m.to(dev).eval()


def _state(smp, dev, thr=0.05):
    from gnn_qot_estimation_b200.to_graph import lightpath_network_state
    return lightpath_network_state(torch.from_numpy(smp["data"]).to(dev), torch.from_numpy(smp["freqs"]),
                                   smp["lp_feat"], thr)


def _demands(rows, dev):
    """[(sample, [(links, width, (mod_order, num_spans, path_len), own_bound)])] -> LightpathDemands on dev."""
    from gnn_qot_estimation_b200.to_graph import LightpathDemands
    opts = [o for _, os_ in rows for o in os_]
    optr = np.cumsum([0] + [len(os_) for _, os_ in rows])
    lptr = np.cumsum([0] + [len(o[0]) for o in opts])
    return LightpathDemands(torch.tensor([r[0] for r in rows], dtype=torch.int64),
                            torch.tensor(optr, dtype=torch.int64), torch.tensor(lptr, dtype=torch.int64),
                            torch.tensor([l for o in opts for l in o[0]], dtype=torch.int32),
                            torch.tensor([o[1] for o in opts], dtype=torch.int32),
                            torch.tensor(np.array([o[2] for o in opts], dtype=np.float32).reshape(-1, 3)),
                            torch.tensor(np.array([o[3] for o in opts], dtype=np.float32))).to(dev)


def _same(a, b):
    a, b = a.cpu(), b.cpu()
    if a.is_floating_point():
        return torch.equal(a.nan_to_num(7.0), b.nan_to_num(7.0)) and torch.equal(torch.isnan(a), torch.isnan(b))
    return torch.equal(a, b)


def _assert_same(r, ref, fields=FIELDS):
    for f in fields:
        assert _same(getattr(r, f), getattr(ref, f)), f


def _node_bound(m, state, metric, maximize, seed, spread=0.02):
    every = m.forward_every_node(state.batch)[:, metric]
    g = torch.Generator(device="cpu").manual_seed(seed)
    delta = (torch.rand(every.shape[0], generator=g) * 2 - 1).to(every.device) * spread
    return (every - delta if maximize else every + delta).contiguous()


def _round_loop(m, smp, dev, d, policy, metric, maximize, bound, max_impact=64, thr=0.05):
    from provision_ref import round_loop
    data = torch.from_numpy(smp["data"]).to(dev).contiguous()
    return round_loop(m, data, torch.from_numpy(smp["freqs"]).to(dev), smp["lp_feat"], d, policy, metric, maximize,
                      bound, max_impact, thr)


def _builder(L, Q, seed, spacing=0.0375):
    from dense_samples import SampleBuilder
    return SampleBuilder(L, Q, np.random.default_rng(seed), spacing)


def _pack(builders):
    data = np.stack([b.finish(b.count) for b in builders])
    b = builders[0]
    return {"data": data, "freqs": b.freqs, "lp_feat": b.lp_feat, "metric": b.metric}


# ------------------------------------------------------------------------------------------------ round loop
def test_round_loop_bit_identity(cuda):
    """Every policy, both senses, each metric column, with and without a bound: 10 demands per sample on average,
    interleaved across 5 samples (one of them empty), every output equal bit for bit to the round loop."""
    from gnn_qot_estimation_b200 import synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(5, num_links=12, num_freqs=40, seed=41, super_channel_p=0.3)
    smp["data"][4] = 0.0
    state = _state(smp, cuda)
    d = synthetic.lightpath_demands(smp, 10, seed=42, bound_range=(0.0, 0.5)).to(cuda)
    assert int(torch.bincount(d.sample.cpu(), minlength=5).min()) >= 4
    accepted = 0
    for metric, mx in ((0, True), (1, True), (2, False), (0, False)):
        for bound in (None, _node_bound(m, state, metric, mx, 43 + metric, spread=0.05)):
            for policy in (0, 1, 2):
                r = m.forward_provision(state, d, policy, metric, mx, bound)
                ref, _ = _round_loop(m, smp, cuda, d, policy, metric, mx, bound)
                torch.cuda.synchronize()
                _assert_same(r, ref)
                accepted += int((r.conn_id >= 0).sum())
    assert accepted > 100


def test_reduces_to_placements(cuda):
    """One demand per sample: forward_provision equals forward_placements bit for bit (impact nodes as conn_ids)."""
    from gnn_qot_estimation_b200 import synthetic
    from provision_ref import rounds
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(6, num_links=16, num_freqs=40, seed=51, super_channel_p=0.3)
    state = _state(smp, cuda)
    d = synthetic.lightpath_demands(smp, 3, seed=52).to(cuda)
    _, one = rounds(d, state.S)[0]
    bound = _node_bound(m, state, 0, True, 53)
    for policy in (0, 1, 2):
        for b in (None, bound):
            r = m.forward_provision(state, one, policy, 0, True, b, max_impact=4)
            p = m.forward_placements(state, one, policy, 0, True, b, max_impact=4)
            _assert_same(r, p, FIELDS[:8] + ("impact_out",))
            ic = torch.where(p.impact_node >= 0, state.conn_ids[p.impact_node.clamp(min=0)], p.impact_node)
            assert _same(r.impact_conn, ic)
            assert bool(((r.conn_id >= 0) == ((p.option >= 0) & ((p.status & ~8) == 0))).all())


# ------------------------------------------------------------------------------------------------ sequential effects
def test_sequential_effects(cuda):
    """Hand-built: two identical first-fit demands (the second takes the next free range), adjacent-slot demands that
    interfere with each other, a demand whose best slot would break an accepted demand's own_bound, a blocked demand
    followed by one that fits.  Each against the round loop as well."""
    from gnn_qot_estimation_b200 import ops
    m, _ = _model(cuda)
    b = _builder(4, 24, 3)
    b.place([0], 0, 2)
    b.place([1, 2], 5)
    b.place([1], 6)                          # next to the one at slot 5: the state has an edge
    smp = _pack([b])
    state = _state(smp, cuda)
    f = (16, 10, 300000)
    ninf = -np.inf
    rows = [(0, [([0], 2, f, ninf)]), (0, [([0], 2, f, ninf)]),            # first fit: q0 = 2, then 4
            (0, [([3], 1, f, ninf)]), (0, [([3], 1, f, ninf)]),            # adjacent on link 3: 0, then 1
            (0, [([1], 1, f, np.inf)]),                                    # blocked: nothing is feasible
            (0, [([1], 1, f, ninf)])]                                      # fits after the blocked one
    d = _demands(rows, cuda)
    r = m.forward_provision(state, d, ops.PLACE_FIRST_FIT)
    torch.cuda.synchronize()
    assert r.q0.tolist() == [2, 4, 0, 1, -1, 0]
    top = int(state.conn_ids.max())
    assert r.conn_id.tolist() == [top + 1, top + 2, top + 3, top + 4, -1, top + 5]
    # the two demands on link 3 interfere: the first is the second's impact row
    assert int(r.n_impact[3]) == 1 and int(r.impact_conn[3, 0]) == top + 3
    ref, _ = _round_loop(m, smp, cuda, d, ops.PLACE_FIRST_FIT, 0, True, None)
    _assert_same(r, ref)
    # an accepted demand's own_bound binds later placements: the first demand is accepted with margin 0, so a later
    # placement is feasible only where the first's row stays at or above its own value
    e = _demands([(0, [([3], 1, f, ninf)])], cuda)
    bnd = torch.full_like(state.batch.x[:, 0], -1e9)
    own = float(m.forward_provision(state, e, ops.PLACE_FIRST_FIT, 0, True, bnd).out[0, 0])
    rows2 = [(0, [([3], 1, f, own)])] + [(0, [([3], 1, f, ninf), ([2, 3], 1, f, ninf)])] * 3
    d2 = _demands(rows2, cuda)
    for policy in (0, 1, 2):
        r2 = m.forward_provision(state, d2, policy, 0, True, bnd)
        ref2, _ = _round_loop(m, smp, cuda, d2, policy, 0, True, bnd)
        torch.cuda.synchronize()
        _assert_same(r2, ref2)
        assert int(r2.q0[0]) == 0 and int(r2.conn_id[0]) == top + 1 and float(r2.margin[0]) == 0.0
        for k in range(1, 4):
            n = int(r2.n_impact[k])
            hit = (r2.impact_conn[k, :n] == top + 1).nonzero().flatten().tolist()
            if int(r2.option[k]) >= 0 and hit:
                assert float(r2.impact_out[k, hit[0], 0]) >= own
    # without the bound the first free slot (next to it) is taken by first fit; with it, only if that keeps the bound
    r3 = m.forward_provision(state, d2, ops.PLACE_FIRST_FIT, 0, True, None)
    r4 = m.forward_provision(state, d2, ops.PLACE_FIRST_FIT, 0, True, bnd)
    torch.cuda.synchronize()
    assert int(r3.q0[1]) == 1
    assert int(r4.n_feasible[1]) <= int(r3.n_feasible[1])


# ------------------------------------------------------------------------------------------------ fp64
def test_vs_fp64_reference(cuda):
    """provision_ref on the fp64 oracle, following the kernel's choices: every step's chosen own row and impact rows
    at 1e-5, n_free, and the choice feasible and policy-optimal within the tolerance band."""
    from gnn_qot_estimation_b200 import synthetic
    from provision_ref import provision_ref
    m, sd = _model(cuda)
    o = _oracle64(sd, cuda)
    smp = synthetic.network_status_samples(2, num_links=5, num_freqs=20, seed=61, spacing=0.05, max_lightpaths=8,
                                           super_channel_p=0.3)
    state = _state(smp, cuda)
    f1, f2 = (16, 40, 2000000), (64, 9, 80000)
    per = {0: [[([0], 1, f1, 0.1), ([1, 2], 2, f2, 0.2)], [([0], 1, f1, 0.1)], [([0, 3], 1, f2, -np.inf)],
               [([0], 2, f1, 0.15), ([4], 1, f2, 0.1)]],
           1: [[([2], 1, f2, 0.1)], [([2, 3], 1, f1, -np.inf)], [([2], 1, f2, 0.3)]]}
    rows = [(s, per[s][i]) for i in range(4) for s in (0, 1) if i < len(per[s])]     # interleaved
    d = _demands(rows, cuda)
    for policy in (0, 2):
        r = m.forward_provision(state, d, policy, 0, True, None, 256)
        torch.cuda.synchronize()
        for s in (0, 1):
            ks = [k for k, (ss, _) in enumerate(rows) if ss == s]
            follow = [(int(r.option[k]), int(r.q0[k])) if int(r.conn_id[k]) >= 0 else None for k in ks]
            steps, _ = provision_ref(o, smp["data"][s], smp["freqs"], smp["lp_feat"], per[s], policy, follow=follow,
                                     device=cuda)
            for k, st in zip(ks, steps):
                table = st["table"]
                assert int(r.n_free[k]) == st["n_free"]
                if follow[ks.index(k)] is None:
                    assert st["choice"] is None or table[st["choice"]][2] < 1e-5
                    continue
                kb = follow[ks.index(k)]
                row, imp, mg = table[kb]
                assert mg >= -1e-5
                torch.testing.assert_close(r.out[k].double().cpu(), row, rtol=RTOL, atol=ATOL)
                best = st["choice"]
                if policy == 0:
                    assert all(table[x][2] < 1e-5 for x in table if x < kb)
                else:
                    assert best is None or mg >= table[best][2] - 1e-5
                n = int(r.n_impact[k])
                assert n == len(imp) and set(r.impact_conn[k, :n].tolist()) == set(imp)
                if n:
                    torch.testing.assert_close(r.impact_out[k, :n].double().cpu(),
                                               torch.stack([imp[int(c)] for c in r.impact_conn[k, :n].tolist()]),
                                               rtol=RTOL, atol=ATOL)


# ------------------------------------------------------------------------------------------------ commit
def test_commit(cuda):
    """commit_provision equals lightpath_network_state of the samples written in numpy, field by field and bit for
    bit; forward_every_node on it gives each accepted demand its provisioned own row (1e-5)."""
    from gnn_qot_estimation_b200 import synthetic
    from gnn_qot_estimation_b200.to_graph import commit_provision
    from candidates_ref import insert_candidate
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(4, num_links=12, num_freqs=40, seed=71, super_channel_p=0.3)
    state = _state(smp, cuda)
    d = synthetic.lightpath_demands(smp, 6, seed=72, bound_range=(-1.0, 0.2)).to(cuda)
    r = m.forward_provision(state, d, 2)
    data = torch.from_numpy(smp["data"]).to(cuda).contiguous()
    new = commit_provision(data, state, d, r)
    ref = np.array(smp["data"], copy=True)
    optr, lptr, lk = d.opt_ptr.tolist(), d.link_ptr.tolist(), d.links.tolist()
    n_acc = 0
    for k in range(d.sample.shape[0]):
        if int(r.conn_id[k]) < 0:
            continue
        s, p, q0 = int(d.sample[k]), optr[k] + int(r.option[k]), int(r.q0[k])
        ref[s], conn = insert_candidate(ref[s], smp["lp_feat"], lk[lptr[p]:lptr[p + 1]], q0, int(d.width[p]),
                                        [np.float32(smp["freqs"][q0])] + d.feat[p].tolist())
        assert conn == int(r.conn_id[k])
        n_acc += 1
    assert n_acc > 5
    assert torch.equal(data.cpu(), torch.from_numpy(ref))
    want = _state(dict(smp, data=ref), cuda)
    for f in ("x", "edge_index", "ptr", "batch"):
        assert torch.equal(getattr(new.batch, f), getattr(want.batch, f)), f
    for f in ("rowptr", "conn_ids", "chan_node"):
        assert torch.equal(getattr(new, f), getattr(want, f)), f
    every = m.forward_every_node(new.batch)
    acc = r.conn_id >= 0
    from gnn_qot_estimation_b200.to_graph import lightpath_nodes
    nodes = lightpath_nodes(new, d.sample[acc], r.conn_id[acc])
    assert bool((nodes >= 0).all())
    # the own row of a demand is its row in the state it was placed against; later demands may change it, so only the
    # last accepted demand of each sample is compared
    last = {}
    for k in torch.nonzero(acc).flatten().tolist():
        last[int(d.sample[k])] = k
    ks = torch.tensor(sorted(last.values()), device=cuda)
    nl = lightpath_nodes(new, d.sample[ks], r.conn_id[ks])
    torch.testing.assert_close(every[nl], r.out[ks], rtol=RTOL, atol=ATOL)


# ------------------------------------------------------------------------------------------------ capacity
def test_capacity(cuda):
    """A sample at 255 lightpaths accepts one demand and then reports PROV_FULL; the channel limit (the full grid, whose
    routes also take the entry-list fallback); the hub and clique samples against the round loop."""
    import dense_samples as ds
    from gnn_qot_estimation_b200 import ops
    m, _ = _model(cuda)
    f = (16, 10, 300000)
    smp = ds.full_sparse(3, counts=(255,))
    state = _state(smp, cuda, ds.HUB_THRESHOLD)
    free = np.flatnonzero(~np.any(smp["data"][0] != 0, axis=0)[0])
    assert free.size >= 3
    d = _demands([(0, [([0], 1, f, -np.inf)])] * 3, cuda)
    r = m.forward_provision(state, d, ops.PLACE_FIRST_FIT)
    torch.cuda.synchronize()
    assert (int(r.status[0]) & ~ops.CAND_IMPACT_OVERFLOW) == 0 and int(r.conn_id[0]) >= 0
    assert int(r.status[1]) & ops.PROV_FULL and int(r.conn_id[1]) == -1 and int(r.option[1]) == 0
    assert int(r.q0[1]) == int(r.q0[2])                                  # nothing was committed
    ref, _ = _round_loop(m, smp, cuda, d, ops.PLACE_FIRST_FIT, 0, True, None, thr=ds.HUB_THRESHOLD)
    _assert_same(r, ref)
    # channels: 254 lightpaths of 8 links x 3 slots (6096 channels) on L = 64, Q = 97; slot column 96 is free.  A
    # 9-link route on that column holds 864 channels of known lightpaths: the entry-list fallback.
    b = _builder(64, 97, 11)
    for k in range(254):
        b.place(list(range(8 * (k // 32), 8 * (k // 32) + 8)), 3 * (k % 32), 3)
    g = _pack([b])
    gstate = _state(g, cuda, ds.HUB_THRESHOLD)
    rows = [(0, [(list(range(9)), 1, f, -np.inf)]),                      # 6105 channels, 255 lightpaths: accepted
            (0, [(list(range(56, 64)), 6, f, -np.inf)]),                 # 6153 channels: PROV_FULL
            (0, [([9], 1, f, -np.inf)]),                                 # 6106 channels, 256 lightpaths: accepted
            (0, [([10], 1, f, -np.inf)])]                                # 257 lightpaths: PROV_FULL
    d = _demands(rows, cuda)
    for policy, bound in ((0, None), (2, _node_bound(m, gstate, 0, True, 12, spread=0.2))):
        r = m.forward_provision(gstate, d, policy, 0, True, bound, 256)
        ref, _ = _round_loop(m, g, cuda, d, policy, 0, True, bound, 256, ds.HUB_THRESHOLD)
        torch.cuda.synchronize()
        _assert_same(r, ref)
        if policy == 0:
            assert [int(v) & ops.PROV_FULL for v in r.status.tolist()] == [0, ops.PROV_FULL, 0, ops.PROV_FULL]
            assert (r.conn_id >= 0).tolist() == [True, False, True, False]
            assert int(r.n_impact[0]) > 0
    for smp, thr in ((ds.hub(7), ds.HUB_THRESHOLD), (ds.clique(8, n=200), ds.CLIQUE_THRESHOLD)):
        st = _state(smp, cuda, thr)
        L = smp["data"].shape[2]
        rng = np.random.default_rng(9)
        rows = [(0, [(sorted(rng.choice(L, 2, replace=False).tolist()), 1, f, -np.inf), ([0], 1, f, 0.2)])
                for _ in range(8)]
        d = _demands(rows, cuda)
        bound = _node_bound(m, st, 0, True, 10, spread=0.2)
        for policy, b in ((0, None), (2, bound)):
            r = m.forward_provision(st, d, policy, 0, True, b, 32)
            ref, _ = _round_loop(m, smp, cuda, d, policy, 0, True, b, 32, thr)
            _assert_same(r, ref)


# ------------------------------------------------------------------------------------------------ status, errors
def _c_call(m, state, d, order, sample_ptr, bound=None, max_impact=4):
    """qot_lightpath_provision through the C entry point with a caller-made grouping."""
    from gnn_qot_estimation_b200 import _lib, ops
    from gnn_qot_estimation_b200.ops import _demands_desc, _state_desc, ptr, stream
    D, P, dev = int(d.sample.shape[0]), int(d.width.shape[0]), state.batch.x.device
    res = ops.ProvisionQoT(*(torch.full((D,), 99, dtype=torch.int32, device=dev) for _ in range(2)),
                           torch.zeros(D, 3, device=dev), torch.zeros(D, device=dev),
                           *(torch.full((D,), 99, dtype=torch.int32, device=dev) for _ in range(4)),
                           torch.full((D, max_impact), 99, dtype=torch.int64, device=dev),
                           torch.zeros(D, max_impact, 3, device=dev), torch.full((D,), 99, dtype=torch.int64,
                                                                                 device=dev))
    keep = []
    cw = torch.empty_like(state.chan_node)
    rc = _lib.lib().qot_lightpath_provision(
        C.byref(_state_desc(state, keep)), C.byref(_demands_desc(d, D, P, keep)), ptr(order),
        ptr(sample_ptr), None, 0, 1, 0, ptr(m.prepared()), 1, max_impact, ptr(cw), None, ptr(res.option),
        ptr(res.q0), ptr(res.out), ptr(res.margin), ptr(res.n_free), ptr(res.n_feasible), ptr(res.status),
        ptr(res.n_impact), ptr(res.conn_id), ptr(res.impact_conn), ptr(res.impact_out), stream())
    torch.cuda.synchronize()
    return rc, res


def test_status_bits_and_c_groupings_through_structs(cuda):
    """BAD_SAMPLE, BAD_PATH (each kind), BAD_STATE, IMPACT_OVERFLOW (accepted), PROV_FULL (above), BAD_GROUPING through
    the C entry point (each malformation), an empty sample and D = 0."""
    from gnn_qot_estimation_b200 import ops, synthetic
    from gnn_qot_estimation_b200.to_graph import LightpathDemands
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(3, num_links=8, num_freqs=32, seed=81)
    smp["data"][2] = 0.0
    state = _state(smp, cuda)
    f = (16, 10, 300000)
    ninf = -np.inf
    rows = [(5, [([0], 1, f, ninf)]), (-1, [([0], 1, f, ninf)]),
            (0, [([], 1, f, ninf)]), (0, [([9], 1, f, ninf)]), (0, [([0], 0, f, ninf)]), (0, [([0], 33, f, ninf)]),
            (0, [([0], 1, f, ninf)] * 33),
            (1, [(list(range(8)), 1, f, ninf)]),
            (2, [([0], 1, f, ninf)]), (2, [([0], 1, f, ninf)])]
    d = _demands(rows, cuda)
    r = m.forward_provision(state, d, 0, max_impact=0)
    torch.cuda.synchronize()
    st = r.status.tolist()
    assert st[:2] == [ops.CAND_BAD_SAMPLE] * 2
    assert st[2:7] == [ops.CAND_BAD_PATH] * 5
    for k in range(7):
        assert int(r.option[k]) == -1 and int(r.conn_id[k]) == -1 and int(r.n_free[k]) == 0
        assert bool(torch.isnan(r.out[k]).all()) and bool(torch.isnan(r.margin[k]))
    assert st[7] == (ops.CAND_IMPACT_OVERFLOW if int(r.n_impact[7]) else 0)      # an overflow is still accepted
    assert (int(r.conn_id[7]) >= 0) == (int(r.option[7]) >= 0)
    assert r.q0.tolist()[8:] == [0, 1] and r.conn_id.tolist()[8:] == [1, 2]      # the empty sample: ids from 1
    # BAD_STATE: a state whose chan_node names a node of another sample
    bad = state._replace(chan_node=state.chan_node.clone())
    bad.chan_node[1, 0, :] = 0
    rb = m.forward_provision(bad, _demands([(1, [([0], 1, f, ninf)]), (0, [([0], 1, f, ninf)])], cuda), 0)
    torch.cuda.synchronize()
    assert int(rb.status[0]) == ops.CAND_BAD_STATE and int(rb.status[1]) == 0
    # D = 0; S = 0
    e = LightpathDemands(d.sample[:0], d.opt_ptr[:1], d.link_ptr[:1], d.links[:0], d.width[:0], d.feat[:0],
                         d.own_bound[:0])
    assert m.forward_provision(state, e, 0).status.numel() == 0
    # malformed groupings through the C ABI: every demand says BAD_GROUPING alone
    g = _demands([(0, [([0], 1, f, ninf)]), (1, [([1], 1, f, ninf)]), (0, [([2], 1, f, ninf)])], cuda)
    i64 = lambda v: torch.tensor(v, dtype=torch.int64, device=cuda)
    rc, ok = _c_call(m, state, g, i64([0, 2, 1]), i64([0, 2, 3, 3]))
    assert rc == 0 and int(ok.status.max()) == 0
    for order, sp in (([2, 0, 1], [0, 2, 3, 3]),       # not ascending within sample 0
                      ([0, 1, 2], [0, 2, 3, 3]),       # demand 1 is not sample 0's
                      ([0, 2, 1], [1, 2, 3, 3]),       # sample_ptr[0] != 0
                      ([0, 2, 1], [0, 2, 1, 3]),       # decreasing
                      ([0, 2, 1], [0, 2, 2, 2]),       # a demand left out
                      ([0, 2, 7], [0, 2, 3, 3]),       # order outside [0, D)
                      ([0, 0, 1], [0, 2, 3, 3])):      # a demand twice
        rc, res = _c_call(m, state, g, i64(order), i64(sp))
        assert rc == 0
        assert res.status.tolist() == [ops.PROV_BAD_GROUPING] * 3, (order, sp)
        assert res.option.tolist() == [-1] * 3 and res.conn_id.tolist() == [-1] * 3
        assert res.n_free.tolist() == [0] * 3 and bool(torch.isnan(res.out).all())
        assert bool((res.impact_conn == -1).all()) and bool(torch.isnan(res.impact_out).all())


def test_determinism_capture_and_errors(cuda):
    """Two calls and a CUDA-graph replay are bit-identical; the state is not modified; the host error paths."""
    from gnn_qot_estimation_b200 import ops, synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(8, num_links=16, num_freqs=48, seed=91, super_channel_p=0.3)
    state = _state(smp, cuda)
    d = synthetic.lightpath_demands(smp, 8, seed=92).to(cuda)
    bound = _node_bound(m, state, 0, True, 93)
    cn = state.chan_node.clone()
    a = m.forward_provision(state, d, 2, 0, True, bound)
    b = m.forward_provision(state, d, 2, 0, True, bound)
    torch.cuda.synchronize()
    _assert_same(a, b)
    assert torch.equal(state.chan_node, cn)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        m.forward_provision(state, d, 2, 0, True, bound)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c = m.forward_provision(state, d, 2, 0, True, bound)
    g.replay()
    torch.cuda.synchronize()
    _assert_same(a, c)
    with pytest.raises(ValueError):
        m.forward_provision(state, d, 7)
    with pytest.raises(ValueError):
        m.forward_provision(state, d, 0, metric=3)
    with pytest.raises(ValueError):
        m.forward_provision(state, d, 0, max_impact=-1)
    with pytest.raises(ValueError):
        m.forward_provision(state, d, 0, bound=bound[:-1])
    with pytest.raises(TypeError):
        m.forward_provision(state, d._replace(width=d.width.long()), 0)
    with pytest.raises(RuntimeError):
        m.forward_provision(state, d.to("cpu"), 0)
    m.train()
    with pytest.raises(RuntimeError):
        m.forward_provision(state, d, 0)
    m.eval()
