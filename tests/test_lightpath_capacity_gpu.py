"""GPU parity of the lightpath network-state kernels at sample capacity (QOT_TG_MAX_NODES = 256 lightpaths,
QOT_TG_MAX_CHANNELS = 6144 occupied channels, QOT_SET_MAX_CHANGES = 64 changes, the every-node fast-path bounds), on
the dense samples of tests/dense_samples.py, against the fp64 oracle's literal definitions (run on the GPU, chunked):
to_graph and the channel map, every-node mode on both layouts, candidates, reconfigurations and change sets with
max_impact = 256 so that every impact row is compared, and the max_impact overflow prefix.  Each test prints the
largest n_impact, in-row length, set size and sample-local neighbour index it reached."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import dense_samples as ds
from conftest import rel_err
from test_lightpath_reconfig_gpu import ATOL, RTOL, _changes, _lightpaths, _model, _oracle64, _state

pytestmark = pytest.mark.gpu
MI = 256            # every impact row of a 256-lightpath sample
CHUNK = 32          # one-hot copies per oracle call: 32 copies of the clique graph are ~1 M edges


@pytest.fixture(scope="module")
def models(cuda):
    m, sd = _model(cuda)
    return m, _oracle64(sd).to(cuda)


@pytest.fixture(scope="module")
def hub(cuda):
    smp = ds.hub()
    return smp, _state(smp, cuda, ds.HUB_THRESHOLD), ds.HUB_THRESHOLD


@pytest.fixture(scope="module")
def clique(cuda):
    smp = ds.clique()
    return smp, _state(smp, cuda, ds.CLIQUE_THRESHOLD), ds.CLIQUE_THRESHOLD


@pytest.fixture(scope="module")
def sparse(cuda):
    smp = ds.full_sparse()
    return smp, _state(smp, cuda, ds.HUB_THRESHOLD), ds.HUB_THRESHOLD


class Reach:
    """The largest n_impact, in-row length (state in-degree of an impact row, self loop included), set size and
    sample-local neighbour index a test compared."""

    def __init__(self, state):
        self.rowptr, self.ptr, self.b = state.rowptr.cpu(), state.batch.ptr.cpu(), state.batch.batch.cpu()
        self.n_impact = self.in_row = self.set_size = self.nbr_index = 0

    def add(self, nodes, set_size=1):
        self.n_impact = max(self.n_impact, len(nodes))
        self.set_size = max(self.set_size, set_size)
        for v in nodes:
            self.in_row = max(self.in_row, int(self.rowptr[v + 1] - self.rowptr[v]))
            self.nbr_index = max(self.nbr_index, int(v - self.ptr[self.b[v]]))

    def report(self, what):
        print(f"\n{what}: n_impact {self.n_impact}, in-row {self.in_row}, set size {self.set_size}, "
              f"neighbour index {self.nbr_index}")
        return self


def _impact(r, u, conn, impact, kinds, got, ref, reach, set_size=1):
    """Impact rows of unit u (a candidate, change or set) of result r (on the CPU) against ``impact`` {conn_id: (kind,
    row)}: n_impact exact, nodes ascending, kinds right, every slot past n_impact -1 / NaN (kind 0)."""
    n = int(r.n_impact[u])
    assert n == len(impact)
    nodes = r.impact_node[u, :n]
    assert bool((nodes[1:] > nodes[:-1]).all())
    assert bool((r.impact_node[u, n:] == -1).all()) and bool(torch.isnan(r.impact_out[u, n:]).all())
    assert {int(conn[v]) for v in nodes} == set(impact)
    if kinds:
        assert bool((r.impact_kind[u, n:] == 0).all())
    for i, v in enumerate(nodes.tolist()):
        kind, row = impact[int(conn[v])]
        if kinds:
            assert int(r.impact_kind[u, i]) == kind
        got.append(r.impact_out[u, i])
        ref.append(row)
    reach.add(nodes.tolist(), set_size)


def _close(got, ref):
    got, ref = torch.stack(got).double().cpu(), torch.stack(ref).double().cpu()
    assert torch.isfinite(got).all()
    assert rel_err(got, ref) <= RTOL
    torch.testing.assert_close(got, ref, rtol=RTOL, atol=ATOL)


def _cpu(r):
    return type(r)(*(t.cpu() for t in r))


def _same(a, b, names=None):
    for name in names or a._fields:
        x, y = getattr(a, name), getattr(b, name)
        assert torch.equal(x.nan_to_num(7.0) if x.is_floating_point() else x,
                           y.nan_to_num(7.0) if y.is_floating_point() else y), name


def _prefix(full, over, units, cut, kinds=True):
    """``over`` (max_impact = cut) is exactly the first ``cut`` impact rows of ``full`` (max_impact = MI)."""
    from gnn_qot_estimation_b200 import ops
    n = full.n_impact
    assert torch.equal(over.n_impact, n)
    assert torch.equal((over.status if not hasattr(over, "set_status") else over.set_status) & ops.CAND_IMPACT_OVERFLOW
                       != 0, n > cut)
    assert torch.equal(over.out.nan_to_num(7.0), full.out.nan_to_num(7.0))
    assert torch.equal(over.impact_node, full.impact_node[:, :cut])
    assert torch.equal(over.impact_out.nan_to_num(7.0), full.impact_out[:, :cut].nan_to_num(7.0))
    if kinds:
        assert torch.equal(over.impact_kind, full.impact_kind[:, :cut])
    assert int((n > cut).sum()) >= units


def _hub_node(smp, state):
    lps = _lightpaths(smp, state)
    return next(lp for lp in lps if len(lp[3]) == 128), lps


def _f(freqs, q, feat=(16, 10, 100000)):
    return [np.float32(freqs[q]), *feat]


# --------------------------------------------------------------------------------------------- a. to_graph
def test_to_graph_and_channel_map_at_capacity(cuda, hub, clique, sparse):
    """Every dense shape builds with status 0 and matches the numpy oracle's nodes, x and edges, and the channel map
    names the right node on every channel; 256 lightpaths and 6144 occupied channels build, 257 and 6145 do not."""
    from oracle.to_graph_oracle import lightpath_data_ref
    grid = ds.full_grid()
    cases = [hub, clique, sparse, (grid, _state(grid, cuda, ds.HUB_THRESHOLD), ds.HUB_THRESHOLD),
             (ds.count_sample(256), None, ds.HUB_THRESHOLD)]
    top_n = top_e = 0
    for smp, state, thr in cases:
        if state is None:
            state = _state(smp, cuda, thr)
        ptr, bt = state.batch.ptr.cpu(), state.batch.batch.cpu()
        ei = state.batch.edge_index.cpu()
        chan = state.chan_node.cpu()
        for s in range(smp["data"].shape[0]):
            ec, ex, _, eei = lightpath_data_ref(smp["data"][s], np.zeros(3), smp["freqs"], smp["lp_feat"],
                                                ["osnr", "snr", "ber"], thr)
            n0, n1 = int(ptr[s]), int(ptr[s + 1])
            assert np.array_equal(state.conn_ids[n0:n1].cpu().numpy(), ec)
            assert np.array_equal(state.batch.x[n0:n1].cpu().numpy(), ex)
            mine = bt[ei[0]] == s
            assert np.array_equal((ei[:, mine] - n0).numpy(), eei)
            fi = {k: i for i, k in enumerate(smp["lp_feat"])}
            occ = np.any(smp["data"][s] != 0, axis=0)
            node_of = {int(c): n0 + i for i, c in enumerate(ec)}
            want = np.where(occ, np.vectorize(lambda c: node_of.get(int(c), -2))(
                np.trunc(smp["data"][s, fi["conn_id"]])), -1)
            assert np.array_equal(chan[s].numpy(), want)
            top_n, top_e = max(top_n, n1 - n0), max(top_e, eei.shape[1])
    from gnn_qot_estimation_b200.to_graph import lightpath_network_state
    for over in (ds.count_sample(257), ds.full_grid(extra=1)):
        with pytest.raises(RuntimeError, match="capacity"):
            lightpath_network_state(torch.from_numpy(over["data"]).to(cuda), torch.from_numpy(over["freqs"]),
                                    over["lp_feat"])
    print(f"\nto_graph: up to {top_n} nodes, {top_e} edges, {ds.MAX_CHANNELS} occupied channels")


# --------------------------------------------------------------------------------------------- b. every-node
def _every_ref(o, b, dev):
    from every_node_ref import lightpath_every_node_ref
    with torch.no_grad():
        return lightpath_every_node_ref(o, SimpleNamespace(x=b.x.to(dev).double(), edge_index=b.edge_index.to(dev),
                                                           batch=b.batch.to(dev)), CHUNK)


def _both_layouts(m, b):
    """forward_every_node of a verified-layout batch, then of the same tensors without the layout flag: same bits."""
    assert b.sym_by_src
    sym = m.forward_every_node(b)
    plain = m.forward_every_node(SimpleNamespace(x=b.x, edge_index=b.edge_index, batch=b.batch, ptr=b.ptr,
                                                 edge_ptr=b.edge_ptr, num_graphs=b.num_graphs))
    assert torch.equal(sym, plain)
    return sym


def test_every_node_dense_shapes_both_layouts(cuda, models, hub, clique, sparse):
    m, o = models
    grid = ds.full_grid()
    deg = 0
    for smp, state, _ in (hub, clique, sparse, (grid, _state(grid, cuda, ds.HUB_THRESHOLD), None)):
        b = state.batch
        got = _both_layouts(m, b)
        _close(list(got), list(_every_ref(o, b, cuda)))
        deg = max(deg, int(torch.diff(state.rowptr).max()))
    print(f"\nevery-node dense: in-row up to {deg}")


def test_every_node_fast_path_boundary_stores(cuda, models):
    """(n, E) = (128, 512) and (120, 500) take the fast path, (129, 512) and (128, 514) the generic one; each graph
    has a row of 100+ in-neighbours."""
    m, o = models
    store = ds.boundary_store().to(cuda)
    assert store.verify_layout()
    b = store.collate(range(store.num_graphs))
    got = _both_layouts(m, b)
    _close(list(got), list(_every_ref(o, b, cuda)))
    hub_rows = [int((b.edge_index[1] == int(b.ptr[g])).sum()) for g in range(store.num_graphs)]
    print(f"\nevery-node boundary: shapes {ds.BOUNDARY_SHAPES}, hub in-rows {hub_rows}")


# --------------------------------------------------------------------------------------------- c. candidates
def _check_candidates(m, o, smp, state, thr, rows, dev, max_impact=MI):
    """rows: [(sample, links, q0, width, feat)]; returns the CPU result after checking every row."""
    from candidates_ref import candidates_ref
    from gnn_qot_estimation_b200.to_graph import LightpathCandidates
    cands = LightpathCandidates(*_changes([(-1, *c) for c in rows], dev)[1:])
    r = _cpu(m.forward_candidates(state, cands, max_impact))
    assert int(r.status.max()) == 0, r.status
    conn = state.conn_ids.cpu()
    got, ref, reach = [], [], Reach(state)
    for k, (s, links, q0, w, feat) in enumerate(rows):
        row, impact = candidates_ref(o, smp["data"][s], smp["freqs"], smp["lp_feat"], links, q0, w, feat, thr,
                                     chunk=CHUNK, device=dev)
        got.append(r.out[k])
        ref.append(row)
        _impact(r, k, conn, {c: (2, v) for c, v in impact.items()}, False, got, ref, reach)
    _close(got, ref)
    return r, cands, reach


def _hub_candidates(smp):
    fr = smp["freqs"]
    return [(0, [127], 11, 1, _f(fr, 11)),                       # next to the hub: its row has 255 + 1 + 1 messages
            (0, list(range(115, 127)), 12, 1, _f(fr, 12)),       # neighbours: the slot-11 singles, nodes 232..254
            (0, [127], 8, 1, _f(fr, 8, (4, 3, 2000000))),        # neighbour: node 255
            (0, list(range(100, 128)), 8, 1, _f(fr, 8)),         # 28 neighbours, nodes 201..255
            (0, [64, 127], 12, 1, _f(fr, 12))]


def _clique_candidates(smp):
    free = ~np.any(smp["data"][0] != 0, axis=0)
    fr = smp["freqs"]
    out = []
    for links in ([0], [1, 2], [0, 3, 5], [4, 6, 7], [2, 5, 7]):
        q = [q for q in range(256) if free[links, q].all()]
        out += [(0, links, q[0], 1, _f(fr, q[0])), (0, links, q[-1], 1, _f(fr, q[-1], (64, 100, 7000000)))]
    return out


def test_candidates_at_capacity(cuda, models, hub, clique, sparse):
    """Candidates next to the hub, with neighbours among nodes 224..255, with more than 64 impact rows in the clique:
    each sample' holds 257 lightpaths, one over to_graph's capacity and inside the kernel's.  Node -1 changes are
    bit-identical."""
    from gnn_qot_estimation_b200 import synthetic
    from gnn_qot_estimation_b200.to_graph import LightpathChanges
    m, o = models
    for (smp, state, thr), rows in ((hub, _hub_candidates(hub[0])), (clique, _clique_candidates(clique[0])),
                                    (sparse, None)):
        if rows is None:
            c = synthetic.lightpath_candidates(smp, 3, seed=7)
            rows = [(int(c.sample[k]), c.links[int(c.link_ptr[k]):int(c.link_ptr[k + 1])].tolist(), int(c.q0[k]),
                     int(c.width[k]), c.feat[k].tolist()) for k in range(c.sample.shape[0])]
        r, cands, reach = _check_candidates(m, o, smp, state, thr, rows, cuda)
        reach.report(f"candidates ({len(rows)})")
        rec = _cpu(m.forward_reconfigurations(state, LightpathChanges(torch.full_like(cands.sample, -1), *cands), MI))
        _same(r, rec, ("out", "status", "n_impact", "impact_node", "impact_out"))
        if smp is hub[0]:
            assert reach.in_row == 255 and reach.nbr_index == 255
        if smp is clique[0]:
            assert reach.n_impact > 128


# --------------------------------------------------------------------------------------------- d. reconfiguration
def _check_changes(m, o, smp, state, thr, rows, dev):
    """rows: [(node, sample, links, q0, width, feat)] -> the CPU result, every row checked against reconfig_ref."""
    from reconfig_ref import reconfig_ref
    r = _cpu(m.forward_reconfigurations(state, _changes(rows, dev), MI))
    assert int(r.status.max()) == 0, r.status
    conn = state.conn_ids.cpu()
    got, ref, reach = [], [], Reach(state)
    for k, (node, s, links, q0, w, feat) in enumerate(rows):
        row, impact = reconfig_ref(o, smp["data"][s], smp["freqs"], smp["lp_feat"],
                                   None if node < 0 else int(conn[node]), links, q0, w, feat, thr, chunk=CHUNK,
                                   device=dev)
        if row is None:
            assert bool(torch.isnan(r.out[k]).all())
        else:
            got.append(r.out[k])
            ref.append(row)
        _impact(r, k, conn, impact, True, got, ref, reach)
    _close(got, ref)
    return r, reach


def _clique_moves(smp, state):
    lps = _lightpaths(smp, state)
    deg = torch.diff(state.rowptr).cpu()
    occ = np.any(smp["data"][0] != 0, axis=0)
    fr = smp["freqs"]
    rows = []
    for s, v, c, links, q0, w, feat in sorted(lps, key=lambda lp: -int(deg[lp[1]]))[:3]:
        new = [0, 3, 5]
        q = next(q for q in range(256) if not occ[new, q].any())
        rows += [(v, 0, new, q, 1, [np.float32(fr[q]), *feat[1:]]), (v, 0, [], 0, 1, feat)]
    return rows


def test_reconfigurations_at_capacity(cuda, models, hub, clique):
    """The hub moved to slot 12 (its 255 old neighbours and 127 new ones), torn down (255 rows of kind 1) and moved
    where it is (every-node rows of the state); the clique's busiest lightpaths moved and torn down."""
    m, o = models
    smp, state, thr = hub
    (_, v, c, links, q0, w, feat), _ = _hub_node(smp, state)
    fr = smp["freqs"]
    rows = [(v, 0, links, 12, 1, [np.float32(fr[12]), *feat[1:]]), (v, 0, [], 0, 1, feat),
            (v, 0, links, q0, w, feat)]
    r, reach = _check_changes(m, o, smp, state, thr, rows, cuda)
    reach.report("hub reconfigurations")
    assert r.n_impact.tolist() == [255, 255, 255]
    assert set(r.impact_kind[0, :255].tolist()) == {1, 3} and bool((r.impact_kind[1, :255] == 1).all())
    assert bool((r.impact_kind[2, :255] == 3).all())
    every = m.forward_every_node(state.batch).cpu()
    torch.testing.assert_close(r.out[2], every[v], rtol=RTOL, atol=ATOL)
    torch.testing.assert_close(r.impact_out[2, :255], every[r.impact_node[2, :255]], rtol=RTOL, atol=ATOL)
    smp, state, thr = clique
    r, reach = _check_changes(m, o, smp, state, thr, _clique_moves(smp, state), cuda)
    reach.report("clique reconfigurations")
    assert reach.n_impact > 128 and {1, 2, 3} <= set(r.impact_kind[r.impact_kind > 0].tolist())


# --------------------------------------------------------------------------------------------- e. change sets
def _set_ptr(sizes, dev):
    return torch.tensor(np.cumsum([0] + list(sizes)), dtype=torch.int64, device=dev)


def _check_sets(m, o, smp, state, thr, sets, dev):
    """sets: [[(node, sample, links, q0, width, feat)]] -> the CPU result, every row checked against change_set_ref."""
    from change_set_ref import change_set_ref
    rows = [c for st in sets for c in st]
    r = _cpu(m.forward_change_sets(state, _changes(rows, dev), _set_ptr([len(st) for st in sets], dev), MI))
    assert int(r.set_status.max()) == 0 and int(r.status.max()) == 0, r.set_status
    conn = state.conn_ids.cpu()
    got, ref, reach, k = [], [], Reach(state), 0
    for g, st in enumerate(sets):
        own, impact = change_set_ref(o, smp["data"][st[0][1]], smp["freqs"], smp["lp_feat"],
                                     [(None if c[0] < 0 else int(conn[c[0]]), *c[2:]) for c in st], thr,
                                     chunk=CHUNK, device=dev)
        for row in own:
            if row is None:
                assert bool(torch.isnan(r.out[k]).all())
            else:
                got.append(r.out[k])
                ref.append(row)
            k += 1
        _impact(r, g, conn, impact, True, got, ref, reach, len(st))
    _close(got, ref)
    return r, reach


def _hub_set(smp, state):
    """64 changes: the slot-9 singles of links 0..15 torn down, those of links 16..31 moved to slot 20, then 32
    insertions into the freed slot 9 of links 0..31 -- every insertion is adjacent to the hub and sits at set index
    >= 32."""
    (_, hv, *_), lps = _hub_node(smp, state)
    fr = smp["freqs"]
    single = {(lp[3][0], lp[4]): lp for lp in lps if len(lp[3]) == 1}
    out = []
    for l in range(32):
        s, v, c, links, q0, w, feat = single[(l, 9)]
        out.append((v, 0, [], 0, 1, feat) if l < 16 else (v, 0, [l], 20, 1, [np.float32(fr[20]), *feat[1:]]))
    out += [(-1, 0, [l], 9, 1, _f(fr, 9, (8, 20 + l, 50000 + 1000 * l))) for l in range(32)]
    return out, hv


def _clique_set(smp, state, moves=20, inserts=24):
    """Changes that all use link 0 (so all are adjacent to each other and to every lightpath left on link 0): the first
    ``moves`` single-slot lightpaths of link 0 moved to free slots of link 0 alone, then ``inserts`` insertions."""
    lps = _lightpaths(smp, state)
    occ = np.any(smp["data"][0] != 0, axis=0)
    fr = smp["freqs"]
    free = [q for q in range(256) if not occ[0, q]]
    on0 = [lp for lp in lps if 0 in lp[3] and lp[5] == 1][:moves]
    out = [(v, 0, [0], free[i], 1, [np.float32(fr[free[i]]), *feat[1:]]) for i, (_, v, _, _, _, _, feat) in
           enumerate(on0)]
    out += [(-1, 0, [0], q, 1, _f(fr, q)) for q in free[moves:moves + inserts]]
    assert len(out) == moves + inserts
    return out


def test_change_sets_at_capacity(cuda, models, hub, clique):
    """The 64-change hub set: the hub's row is its in-row without the 32 removed singles, the 32 adjacent insertions
    and its self loop.  A 44-change clique set on one link: adjacency bits >= 32 and a second ballot pass over the
    changes.  A permuted set changes no row; single-change sets are bit-identical to forward_reconfigurations."""
    m, o = models
    smp, state, thr = hub
    hset, hv = _hub_set(smp, state)
    r, reach = _check_sets(m, o, smp, state, thr, [hset], cuda)
    reach.report("hub set")
    assert r.impact_node[0, :int(r.n_impact[0])].tolist() == [hv] and int(r.impact_kind[0, 0]) == 3
    smp, state, thr = clique
    cset = _clique_set(smp, state)
    perm = np.random.default_rng(0).permutation(len(cset))
    r, reach = _check_sets(m, o, smp, state, thr, [cset, [cset[i] for i in perm]], cuda)
    reach.report("clique sets")
    assert reach.set_size == 44 and reach.n_impact > 64
    n = int(r.n_impact[0])
    assert int(r.n_impact[1]) == n and torch.equal(r.impact_node[1], r.impact_node[0])
    assert torch.equal(r.impact_kind[1], r.impact_kind[0])
    torch.testing.assert_close(r.impact_out[1, :n], r.impact_out[0, :n], rtol=RTOL, atol=ATOL)
    torch.testing.assert_close(r.out[44 + np.argsort(perm)], r.out[:44], rtol=RTOL, atol=ATOL)
    # one change per set, at capacity: the hub and clique changes of the reconfiguration test and both sets' changes
    for (smp, state, _), rows in ((hub, hset), (clique, cset + _clique_moves(smp, state))):
        ch = _changes(rows, cuda)
        a = _cpu(m.forward_reconfigurations(state, ch, MI))
        b = _cpu(m.forward_change_sets(state, ch, torch.arange(len(rows) + 1, device=cuda), MI))
        _same(a, b, ("out", "status", "n_impact", "impact_node", "impact_kind", "impact_out"))
        assert torch.equal(b.set_status, b.status)


# --------------------------------------------------------------------------------------------- f. overflow
def test_overflow_prefix_at_scale(cuda, models, hub, clique):
    """max_impact = 64: exactly the first 64 rows of the max_impact = 256 output, for every entry point."""
    from gnn_qot_estimation_b200.to_graph import LightpathCandidates
    m, _ = models
    cut = 64
    for smp, state, _ in (hub, clique):
        cands = _clique_candidates(smp) if smp is clique[0] else _hub_candidates(smp)
        cc = LightpathCandidates(*_changes([(-1, *c) for c in cands], cuda)[1:])
        full, over = (_cpu(m.forward_candidates(state, cc, mi)) for mi in (MI, cut))
        _prefix(full, over, 0 if smp is hub[0] else 5, cut, kinds=False)
        if smp is hub[0]:
            (_, v, c, links, q0, w, feat), _ = _hub_node(smp, state)
            rows = [(v, 0, links, 12, 1, [np.float32(smp["freqs"][12]), *feat[1:]]), (v, 0, [], 0, 1, feat)]
            sets = [_hub_set(smp, state)[0]]
        else:
            rows = _clique_moves(smp, state)
            sets = [_clique_set(smp, state), _clique_set(smp, state, 2, 3)]
        ch = _changes(rows, cuda)
        full, over = (_cpu(m.forward_reconfigurations(state, ch, mi)) for mi in (MI, cut))
        _prefix(full, over, 2, cut)
        flat = _changes([c for st in sets for c in st], cuda)
        sp = _set_ptr([len(st) for st in sets], cuda)
        full, over = (_cpu(m.forward_change_sets(state, flat, sp, mi)) for mi in (MI, cut))
        _prefix(full, over, len(sets) if smp is clique[0] else 0, cut)
        assert torch.equal(over.status & ~8, full.status)
