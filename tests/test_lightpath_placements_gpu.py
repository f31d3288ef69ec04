"""GPU checks of LightpathGNN's placement search (qot_lightpath_placements through LightpathGNN.forward_placements):
bit-identity with forward_candidates on the expanded placement list and a torch selection over it, parity with the
fp64 literal reference (tests/placement_ref.py), the slot-grid edges, capacity samples, every status bit, determinism,
CUDA-graph replay and the error paths."""
import numpy as np
import pytest
import torch

from conftest import ABS_FLOOR, load_golden

pytestmark = pytest.mark.gpu
RTOL = 1e-5
ATOL = ABS_FLOOR


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


def _rows_of(d):
    out = []
    lp, lk = d.link_ptr.tolist(), d.links.tolist()
    for k in range(d.sample.shape[0]):
        opts = []
        for p in range(int(d.opt_ptr[k]), int(d.opt_ptr[k + 1])):
            opts.append((lk[lp[p]:lp[p + 1]], int(d.width[p]), d.feat[p].tolist(), float(d.own_bound[p])))
        out.append((int(d.sample[k]), opts))
    return out


def _expand(state, d):
    """Every free placement of every demand, from chan_node on the host: ([(demand, option p, q0)], candidates)."""
    from gnn_qot_estimation_b200.to_graph import LightpathCandidates
    cn = state.chan_node.cpu().numpy()
    freqs = state.freqs.cpu().numpy()
    lp, lk = d.link_ptr.cpu().tolist(), d.links.cpu().tolist()
    width, feat = d.width.cpu().tolist(), d.feat.cpu().numpy()
    who, smp, lptr, links, q0s, ws, feats = [], [], [0], [], [], [], []
    for k in range(d.sample.shape[0]):
        s = int(d.sample[k])
        for p in range(int(d.opt_ptr[k]), int(d.opt_ptr[k + 1])):
            route, w = lk[lp[p]:lp[p + 1]], width[p]
            occ = (cn[s, route] != -1).any(axis=0)
            for q0 in range(cn.shape[2] - w + 1):
                if occ[q0:q0 + w].any():
                    continue
                who.append((k, p, q0))
                smp.append(s)
                links.extend(route)
                lptr.append(len(links))
                q0s.append(q0)
                ws.append(w)
                feats.append([np.float32(freqs[q0])] + feat[p].tolist())
    dev = state.batch.x.device
    c = LightpathCandidates(torch.tensor(smp, dtype=torch.int64), torch.tensor(lptr, dtype=torch.int64),
                            torch.tensor(links, dtype=torch.int32), torch.tensor(q0s, dtype=torch.int32),
                            torch.tensor(ws, dtype=torch.int32),
                            torch.tensor(np.array(feats, dtype=np.float32).reshape(-1, 4))).to(dev)
    return who, c


def _select(who, cand, d, policy, metric, maximize, bound):
    """Torch selection over the expansion (fp32 margins): per demand (option, q0, margin, n_free, n_feasible)."""
    from gnn_qot_estimation_b200 import ops
    ob = d.own_bound.cpu()
    v = cand.out[:, metric].cpu()
    pidx = torch.tensor([p for _, p, _ in who], dtype=torch.int64)
    mg = (v - ob[pidx]) if maximize else (ob[pidx] - v)
    if bound is not None:
        n = cand.n_impact.cpu().long()
        assert n.numel() == 0 or int(n.max()) <= cand.impact_out.shape[1]
        iv = cand.impact_out[:, :, metric].cpu()
        nd = cand.impact_node.cpu().clamp(min=0)
        b = bound.cpu()[nd]
        im = (iv - b) if maximize else (b - iv)
        im = torch.where(torch.arange(im.shape[1])[None, :] < n[:, None], im, torch.full_like(im, float("inf")))
        mg = torch.minimum(mg, im.min(dim=1).values) if im.shape[1] else mg
    D = d.sample.shape[0]
    res = []
    opt_ptr = d.opt_ptr.cpu().tolist()
    by = {}
    for i, (k, p, q0) in enumerate(who):
        by.setdefault(k, []).append(i)
    for k in range(D):
        idx = by.get(k, [])
        feas = [i for i in idx if bool(mg[i] >= 0)]
        best = None
        if feas:
            if policy == ops.PLACE_FIRST_FIT:
                best = feas[0]
            else:
                score = (v if maximize else -v) if policy == ops.PLACE_BEST_QOT else mg
                top = max(float(score[i]) for i in feas)
                best = next(i for i in feas if float(score[i]) == top)
        if best is None:
            res.append((-1, -1, float("nan"), len(idx), 0, None))
        else:
            _, p, q0 = who[best]
            res.append((p - opt_ptr[k], q0, float(mg[best]), len(idx), len(feas), best))
    return res, mg


def _same(a, b):
    return torch.equal(a.nan_to_num(7.0), b.nan_to_num(7.0)) and torch.equal(torch.isnan(a), torch.isnan(b))


def _check_vs_expansion(m, state, d, policies=(0, 1, 2), metrics=(0, 1, 2), senses=(True, False), bounds=(None,),
                        max_impact=64):
    """forward_placements(return_all=True) against forward_candidates over every free placement and a torch selection
    over it.  Returns the number of demands with a feasible choice."""
    from gnn_qot_estimation_b200 import ops
    who, c = _expand(state, d)
    cand = m.forward_candidates(state, c, 256)
    torch.cuda.synchronize()
    assert c.sample.numel() == 0 or int(cand.status.max()) == 0
    P, Q = d.width.shape[0], state.Q
    chosen = 0
    for bound in bounds:
        for policy in policies:
            for metric in metrics:
                for mx in senses:
                    r = m.forward_placements(state, d, policy, metric, mx, bound, max_impact, return_all=True)
                    torch.cuda.synchronize()
                    # every free placement's own row is forward_candidates' row, bit for bit; NaN elsewhere
                    flat = r.all_out.view(P * Q, 3).cpu()
                    at = torch.tensor([p * Q + q0 for _, p, q0 in who], dtype=torch.int64)
                    assert torch.equal(flat[at], cand.out.cpu())
                    free = torch.zeros(P * Q, dtype=torch.bool)
                    free[at] = True
                    assert bool(torch.isnan(flat[~free]).all())
                    assert bool(torch.isnan(r.all_margin.view(-1).cpu()[~free]).all())
                    ref, mg = _select(who, cand, d, policy, metric, mx, bound)
                    assert _same(r.all_margin.view(-1).cpu()[at], mg)
                    assert r.option.cpu().tolist() == [x[0] for x in ref]
                    assert r.q0.cpu().tolist() == [x[1] for x in ref]
                    assert r.n_free.cpu().tolist() == [x[3] for x in ref]
                    assert r.n_feasible.cpu().tolist() == [x[4] for x in ref]
                    assert _same(r.margin.cpu(), torch.tensor([x[2] for x in ref], dtype=torch.float32))
                    for k, x in enumerate(ref):
                        if x[5] is None:
                            assert int(r.status[k]) == 0 and int(r.n_impact[k]) == 0
                            assert bool(torch.isnan(r.out[k]).all()) and bool((r.impact_node[k] == -1).all())
                            continue
                        chosen += 1
                        i = x[5]
                        n = int(cand.n_impact[i])
                        rows = min(n, max_impact)
                        assert torch.equal(r.out[k].cpu(), cand.out[i].cpu())
                        assert int(r.n_impact[k]) == n
                        assert int(r.status[k]) == (ops.CAND_IMPACT_OVERFLOW if n > max_impact else 0)
                        assert torch.equal(r.impact_node[k, :rows], cand.impact_node[i, :rows])
                        assert torch.equal(r.impact_out[k, :rows], cand.impact_out[i, :rows])
                        assert bool((r.impact_node[k, rows:] == -1).all())
                        assert bool(torch.isnan(r.impact_out[k, rows:]).all())
    return chosen


def _node_bound(m, state, metric, maximize, seed, spread=0.02):
    """[N] bound around each lightpath's every-node value: some impact rows pass it, some fail."""
    every = m.forward_every_node(state.batch)[:, metric]
    g = torch.Generator(device="cpu").manual_seed(seed)
    delta = (torch.rand(every.shape[0], generator=g) * 2 - 1).to(every.device) * spread
    return (every - delta if maximize else every + delta).contiguous()


def test_placements_bit_identical_to_candidates_fresh_seeds(cuda):
    from gnn_qot_estimation_b200 import synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(6, num_links=16, num_freqs=40, seed=31, super_channel_p=0.3)
    state = _state(smp, cuda)
    d = synthetic.lightpath_demands(smp, 3, seed=32).to(cuda)
    n = _check_vs_expansion(m, state, d, bounds=(None, _node_bound(m, state, 0, True, 33)))
    assert n > 0
    # a bound on the metric and sense actually selected, tight enough that it excludes placements
    for metric, mx in ((0, True), (2, False)):
        b = _node_bound(m, state, metric, mx, 34 + metric, spread=0.005)
        d2 = d._replace(own_bound=torch.full_like(d.own_bound, -float("inf") if mx else float("inf")))
        _check_vs_expansion(m, state, d2, metrics=(metric,), senses=(mx,), bounds=(b,), max_impact=4)
        r0 = m.forward_placements(state, d2, 0, metric, mx)
        r1 = m.forward_placements(state, d2, 0, metric, mx, b)
        assert int(r1.n_feasible.sum()) < int(r0.n_feasible.sum()) == int(r0.n_free.sum())


def _parity_case(cuda, smp, rows, policies=(0, 1, 2), thr=0.05, bound_of=None):
    """forward_placements vs placement_ref (fp64 oracle): every free placement's own row at 1e-5, the chosen
    placement's impact rows, and the choice (or, where it differs, a reference score within tolerance of the best)."""
    from placement_ref import choose, placement_table
    m, sd = _model(cuda)
    o = _oracle64(sd, cuda)
    state = _state(smp, cuda, thr)
    d = _demands(rows, cuda)
    conn = state.conn_ids.cpu()
    bound = None
    if bound_of is not None:
        bound = torch.tensor([bound_of(int(c)) for c in conn.tolist()], dtype=torch.float32, device=cuda)
    tables = []
    for s, opts in rows:
        bmap = None if bound is None else {int(conn[v]): float(bound[v]) for v in
                                           range(int(state.batch.ptr[s]), int(state.batch.ptr[s + 1]))}
        tables.append(placement_table(o, smp["data"][s], smp["freqs"], smp["lp_feat"], opts, 0, True, bmap, thr,
                                      device=cuda))
    for policy in policies:
        r = m.forward_placements(state, d, policy, 0, True, bound, 256, return_all=True)
        torch.cuda.synchronize()
        assert int(r.status.max()) == 0
        opt_ptr = d.opt_ptr.tolist()
        for k, (s, opts) in enumerate(rows):
            table = tables[k]
            best, n_free, n_feas = choose(table, policy)
            assert int(r.n_free[k]) == n_free
            got = torch.stack([r.all_out[opt_ptr[k] + p, q0] for (p, q0) in table]).double().cpu() \
                if table else torch.zeros(0, 3, dtype=torch.float64)
            ref = torch.stack([t[0] for t in table.values()]) if table else torch.zeros(0, 3, dtype=torch.float64)
            torch.testing.assert_close(got, ref, rtol=RTOL, atol=ATOL)
            if best is None:
                assert int(r.option[k]) == -1 or table[(int(r.option[k]), int(r.q0[k]))][2] > -1e-5
                continue
            kb = (int(r.option[k]), int(r.q0[k]))
            assert kb in table
            if kb != best:                          # a near tie decided by fp32 rounding
                if policy == 0:
                    assert table[kb][2] >= -1e-5 and all(table[x][2] < 1e-5 for x in table if x < kb)
                elif policy == 1:
                    assert float(table[kb][0][0]) >= float(table[best][0][0]) - 1e-5
                else:
                    assert table[kb][2] >= table[best][2] - 1e-5
            _, imp, _ = table[kb]
            n = int(r.n_impact[k])
            assert n == len(imp)
            nodes = r.impact_node[k, :n].cpu()
            assert {int(conn[v]) for v in nodes} == set(imp)
            if n:
                torch.testing.assert_close(r.impact_out[k, :n].double().cpu(),
                                           torch.stack([imp[int(conn[v])] for v in nodes]), rtol=RTOL, atol=ATOL)


def test_placements_vs_fp64_reference(cuda):
    """Spacing 0.05 at the 0.05 threshold, widths 1..3, a route meeting a multi-link lightpath on several links, a
    route with duplicate links, an empty sample; with and without a per-lightpath bound."""
    from gnn_qot_estimation_b200 import synthetic
    smp = synthetic.network_status_samples(3, num_links=6, num_freqs=24, seed=5, spacing=0.05, max_lightpaths=14,
                                           super_channel_p=0.3)
    smp["data"][2] = 0.0
    data, fi = smp["data"], {k: i for i, k in enumerate(smp["lp_feat"])}
    occ = np.any(data != 0, axis=1)
    multi = None
    for s in range(2):
        conn = np.trunc(data[s, fi["conn_id"]])
        for c in np.unique(conn[occ[s]]):
            ls = sorted(set(np.nonzero(occ[s] & (conn == c))[0].tolist()))
            if len(ls) >= 2:
                multi = (s, ls)
                break
        if multi:
            break
    assert multi is not None
    rows = [
        (0, [([0], 1, (16, 40, 2000000), 0.2), ([1, 2], 2, (8, 3, 90000), 0.3), ([3], 3, (64, 9, 80000), 0.1)]),
        (1, [([4, 5, 4], 1, (32, 20, 500000), 0.25), ([4, 5], 2, (4, 60, 4000000), -np.inf)]),
        (multi[0], [(multi[1], 1, (16, 10, 300000), 0.3), (multi[1], 2, (64, 10, 300000), 0.2)]),
        (2, [([0, 3], 2, (8, 2, 90000), 0.2)]),
    ]
    _parity_case(cuda, smp, rows)
    rng = np.random.default_rng(6)
    cache = {}
    _parity_case(cuda, smp, rows[:3], policies=(2,), bound_of=lambda c: cache.setdefault(c, rng.uniform(0.0, 0.4)))


def _builder(L, Q, seed, spacing=0.0375):
    from dense_samples import SampleBuilder
    return SampleBuilder(L, Q, np.random.default_rng(seed), spacing)


def _pack(builders):
    data = np.stack([b.finish(b.count) for b in builders])
    b = builders[0]
    return {"data": data, "freqs": b.freqs, "lp_feat": b.lp_feat, "metric": b.metric}


def test_word_carry_q_not_multiple_of_32_and_ties(cuda):
    """Q = 40: a link whose only free run is slots 31..32 (crossing the first 32-slot word); two identical options
    (the lower wins).  Q = 41 on a grid mirrored about slot 20 with a mirrored sample: starts q and 40 - q give
    bit-identical rows, so every choice is a tie that the lower q0 wins."""
    m, _ = _model(cuda)
    b = _builder(3, 40, 1)
    for q in list(range(0, 30, 2)) + [33, 35, 37]:
        b.place([0], q, 2)
    b.place([0], 30)
    b.place([0], 39)
    b.place([1], 20)
    assert np.flatnonzero(b.free()[0]).tolist() == [31, 32]
    mir = _builder(3, 41, 2)
    mir.freqs = 192.2 + 0.0375 * np.abs(np.arange(41) - 20)     # freqs[q] == freqs[40 - q]
    vec = mir.vector()
    for q in (19, 21):                                          # one lightpath vector on both sides of slot 20
        mir.put(vec, 2, q)
    mir.count += 1
    mir.place([2], 20)
    state = _state(_pack([b]), cuda)
    mstate = _state(_pack([mir]), cuda)
    f = (16, 10, 300000)
    rows = [(0, [([0], 2, f, -np.inf)]),                          # one free start: q0 = 31
            (0, [([0, 1], 1, f, -np.inf)]),                       # 31, 32
            (0, [([1], 2, f, -np.inf), ([1], 2, f, -np.inf)])]    # identical options
    d = _demands(rows, cuda)
    md = _demands([(0, [([0, 1, 2], 1, f, -1.0)])], cuda)
    _check_vs_expansion(m, state, d)
    _check_vs_expansion(m, mstate, md)
    for policy in (0, 1, 2):
        r = m.forward_placements(state, d, policy, return_all=True)
        torch.cuda.synchronize()
        assert (int(r.option[0]), int(r.q0[0]), int(r.n_free[0])) == (0, 31, 1)
        assert int(r.n_free[1]) == 2 and int(r.option[2]) == 0
        assert _same(r.all_out[2], r.all_out[3])                                # options 2 and 3 are the same
        r = m.forward_placements(mstate, md, policy, return_all=True)
        torch.cuda.synchronize()
        row, q0 = r.all_out[0].cpu(), int(r.q0[0])
        assert int(r.n_free[0]) == 38 and 0 <= q0 < 20
        assert _same(row[:20], row.flip(0)[:20])                               # start q is start 40 - q
        assert torch.equal(r.out[0].cpu(), row[40 - q0])                       # the twin ties, the lower wins
    assert int(r.n_free[0]) == 38 and not torch.equal(row[18], row[17])


def test_q1024_and_bounds(cuda):
    """Q = 1024 (the largest grid), own_bound -inf / +inf, and a bound that excludes exactly the placements adjacent
    to one lightpath."""
    from gnn_qot_estimation_b200 import ops, synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(2, num_links=6, num_freqs=1024, seed=9, spacing=0.005, max_lightpaths=24)
    state = _state(smp, cuda)
    d = synthetic.lightpath_demands(smp, 2, seed=10, options=(1, 2)).to(cuda)
    _check_vs_expansion(m, state, d, metrics=(0,), senses=(True,))
    lo = d._replace(own_bound=torch.full_like(d.own_bound, -float("inf")))
    hi = d._replace(own_bound=torch.full_like(d.own_bound, float("inf")))
    r = m.forward_placements(state, lo, ops.PLACE_FIRST_FIT)
    assert torch.equal(r.n_feasible, r.n_free) and int(r.n_free.min()) > 0
    r = m.forward_placements(state, hi, ops.PLACE_MAX_MARGIN)
    torch.cuda.synchronize()
    assert int(r.n_feasible.max()) == 0 and bool((r.option == -1).all()) and bool((r.q0 == -1).all())
    assert bool(torch.isnan(r.out).all()) and bool(torch.isnan(r.margin).all()) and int(r.n_impact.max()) == 0
    assert int(r.status.max()) == 0 and bool((r.impact_node == -1).all())
    # the bound excludes exactly the placements adjacent to lightpath v
    smp2 = synthetic.network_status_samples(3, num_links=10, num_freqs=40, seed=11)
    st2 = _state(smp2, cuda)
    d2 = synthetic.lightpath_demands(smp2, 4, seed=12)
    d2 = d2._replace(own_bound=torch.full_like(d2.own_bound, -float("inf"))).to(cuda)
    who, c = _expand(st2, d2)
    cand = m.forward_candidates(st2, c, 256)
    nodes = cand.impact_node[cand.impact_node >= 0]
    v = int(torch.mode(nodes.cpu()).values)
    bound = torch.full((st2.batch.x.shape[0],), -float("inf"), device=cuda)
    bound[v] = float("inf")
    r = m.forward_placements(st2, d2, ops.PLACE_FIRST_FIT, bound=bound, max_impact=0, return_all=True)
    torch.cuda.synchronize()
    adj = (cand.impact_node == v).any(dim=1).cpu()
    at = torch.tensor([p * st2.Q + q0 for _, p, q0 in who])
    mg = r.all_margin.view(-1).cpu()[at]
    assert int(adj.sum()) > 0
    assert bool((mg[adj] == -float("inf")).all()) and bool((mg[~adj] == float("inf")).all())
    assert torch.equal(r.n_free - r.n_feasible,
                       torch.bincount(torch.tensor([k for k, _, _ in who])[adj], minlength=d2.sample.shape[0])
                       .to(r.n_free))


def test_max_impact_zero_and_overflow(cuda):
    from gnn_qot_estimation_b200 import ops, synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(4, num_links=12, num_freqs=32, seed=13, max_lightpaths=30)
    state = _state(smp, cuda)
    d = synthetic.lightpath_demands(smp, 4, seed=14)
    d = d._replace(own_bound=torch.full_like(d.own_bound, -float("inf"))).to(cuda)
    _check_vs_expansion(m, state, d, policies=(1,), metrics=(0,), senses=(True,), max_impact=1)
    full = m.forward_placements(state, d, ops.PLACE_BEST_QOT)
    zero = m.forward_placements(state, d, ops.PLACE_BEST_QOT, max_impact=0)
    torch.cuda.synchronize()
    assert zero.impact_out.shape == (d.sample.shape[0], 0, 3)
    for f in ("option", "q0", "out", "margin", "n_free", "n_feasible", "n_impact"):
        assert _same(getattr(zero, f).float(), getattr(full, f).float())
    assert torch.equal(zero.status == ops.CAND_IMPACT_OVERFLOW, full.n_impact > 0)
    assert int((full.n_impact > 1).sum()) > 0


def _against_expansion_at_capacity(cuda, smp, thr, rows, bounds=(None,)):
    m, _ = _model(cuda)
    state = _state(smp, cuda, thr)
    d = _demands(rows, cuda)
    return m, state, d, _check_vs_expansion(m, state, d, policies=(0, 2), metrics=(0,), senses=(True,),
                                            bounds=bounds)


def test_capacity_full_grid_clique_hub(cuda):
    """full_grid (no free placement), clique (255-row impact sets, each counted towards feasibility; the collected
    channels overflow the per-warp list and the chan_node rows are scanned again) and hub."""
    import dense_samples as ds
    from gnn_qot_estimation_b200 import ops
    m, _ = _model(cuda)
    f = (16, 10, 300000)
    # full grid: every channel occupied
    g = ds.full_grid(seed=1)
    st = _state(g, cuda, ds.HUB_THRESHOLD)
    d = _demands([(0, [(list(range(8 * k, 8 * k + 8)), w, f, -np.inf) for k in range(8) for w in (1, 3)])], cuda)
    r = m.forward_placements(st, d, ops.PLACE_FIRST_FIT, return_all=True)
    torch.cuda.synchronize()
    assert int(r.status[0]) == 0 and int(r.n_free[0]) == 0 and int(r.option[0]) == -1
    assert bool(torch.isnan(r.all_out).all())
    # clique: the grid is wide, every lightpath on a shared link is a neighbour
    c = ds.clique(seed=2)
    free = ~np.any(c["data"][0] != 0, axis=0)
    routes = [[0, 1, 2, 3], list(range(8)), list(range(8)) * 2, [5]]     # 16 links: over the collected channels
    rows = [(0, [(rt, w, f, -np.inf) for rt in routes for w in (1, 2)])]
    m, state, d, n = _against_expansion_at_capacity(cuda, c, ds.CLIQUE_THRESHOLD, rows)
    assert n > 0 and bool(free.any())
    who, cand = _expand(state, d)
    cand = m.forward_candidates(state, cand, 256)
    torch.cuda.synchronize()
    assert int(cand.n_impact.max()) >= 150
    hits = torch.bincount(cand.impact_node[cand.impact_node >= 0].cpu(), minlength=state.batch.x.shape[0])
    X = cand.out.shape[0]
    v = int(torch.argmin((hits - X // 2).abs() + X * (hits == 0) + X * (hits == X)))
    assert 0 < int(hits[v]) < X
    bound = torch.full((state.batch.x.shape[0],), -float("inf"), device=cuda)
    bound[v] = float("inf")                                     # a lightpath some placements meet and some do not
    _check_vs_expansion(m, state, d, policies=(2,), metrics=(0,), senses=(True,), bounds=(bound,), max_impact=8)
    r = m.forward_placements(state, d, ops.PLACE_MAX_MARGIN, bound=bound, max_impact=8)
    torch.cuda.synchronize()
    assert 0 < int(r.n_feasible[0]) < int(r.n_free[0])
    # hub: the hub's own in-row holds 255 messages
    hb = ds.hub(seed=3)
    rows = [(0, [([127], 1, f, -np.inf), ([126, 127], 1, f, -np.inf), (list(range(128)), 1, f, -np.inf)])]
    m, state, d, n = _against_expansion_at_capacity(cuda, hb, ds.HUB_THRESHOLD, rows,
                                                    bounds=(None, _node_bound(m, _state(hb, cuda), 0, True, 4)))
    assert n > 0


def test_status_bits(cuda):
    from gnn_qot_estimation_b200 import ops, synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(3, num_links=8, num_freqs=20, seed=7, max_lightpaths=20)
    state = _state(smp, cuda)
    f = (16, 10, 100000)
    rows = [
        (0, [([1], 1, f, -np.inf)]),                      # 0: fine
        (3, [([1], 1, f, -np.inf)]),                      # 1: sample out of range
        (-1, [([1], 1, f, -np.inf)]),                     # 2: negative sample
        (0, [([1], 1, f, -np.inf), ([0, 8], 1, f, 0.0)]), # 3: a link out of range
        (0, [([], 1, f, -np.inf)]),                       # 4: an empty route
        (0, [([2], 0, f, -np.inf)]),                      # 5: width 0
        (0, [([2], 21, f, -np.inf)]),                     # 6: width over Q
        (0, [([2], 20, f, -np.inf)]),                     # 7: width Q: fine
    ]
    d = _demands(rows, cuda)
    r = m.forward_placements(state, d, ops.PLACE_FIRST_FIT, return_all=True)
    torch.cuda.synchronize()
    st = r.status.cpu().tolist()
    assert st == [0, 1, 1, 2, 2, 2, 2, 0]

    def nan_demand(r, k, opts=()):
        assert int(r.option[k]) == -1 and int(r.q0[k]) == -1
        assert bool(torch.isnan(r.out[k]).all()) and bool(torch.isnan(r.margin[k]))
        assert int(r.n_free[k]) == int(r.n_feasible[k]) == int(r.n_impact[k]) == 0
        assert bool((r.impact_node[k] == -1).all()) and bool(torch.isnan(r.impact_out[k]).all())
        for p in opts:
            assert bool(torch.isnan(r.all_out[p]).all()) and bool(torch.isnan(r.all_margin[p]).all())

    for k in range(1, 7):
        nan_demand(r, k, range(int(d.opt_ptr[k]), int(d.opt_ptr[k + 1])))
    assert int(r.option[0]) == 0 and int(r.n_free[0]) > 0
    # zero options, more than 32, a malformed opt_ptr / link_ptr
    many = _demands([(0, [([1], 1, f, -np.inf)] * 33), (0, [([1], 1, f, -np.inf)] * 32)], cuda)
    r = m.forward_placements(state, many, ops.PLACE_FIRST_FIT)
    assert r.status.cpu().tolist() == [ops.CAND_BAD_PATH, 0]
    four = _demands([(0, [([1], 1, f, -np.inf)])] * 4, cuda)
    for optr, want in (([0, 1, 1, 0, 4], [0, 2, 2, 0]),                 # zero options, a decreasing range
                       ([0, 1, 2, 3, 5], [0, 0, 0, 2]),                 # a range past P
                       ([-1, 1, 2, 3, 4], [2, 0, 0, 0])):               # a range before 0
        r = m.forward_placements(state, four._replace(opt_ptr=torch.tensor(optr, device=cuda)), 0)
        torch.cuda.synchronize()
        assert r.status.cpu().tolist() == want
    for lptr, want in (([0, 3, 2, 3, 4], [0, 2, 0, 0]),                 # option 1's range decreasing
                       ([0, 1, 2, 3, 5], [0, 0, 0, 2])):                # a range past the links
        r = m.forward_placements(state, four._replace(link_ptr=torch.tensor(lptr, device=cuda)), 0)
        torch.cuda.synchronize()
        assert r.status.cpu().tolist() == want
    # BAD_STATE: a channel of option 0's route holding a node outside the sample
    cn = state.chan_node.clone()
    cn[0, 1, 0] = int(state.batch.ptr[2])
    r = m.forward_placements(state._replace(chan_node=cn), d, ops.PLACE_FIRST_FIT, return_all=True)
    torch.cuda.synchronize()
    assert int(r.status[0]) == ops.CAND_BAD_STATE
    nan_demand(r, 0, [0])
    assert int(r.status[7]) == 0
    # IMPACT_OVERFLOW on the chosen placement only
    g = synthetic.lightpath_demands(smp, 6, seed=8)
    g = g._replace(own_bound=torch.full_like(g.own_bound, -float("inf"))).to(cuda)
    full = m.forward_placements(state, g, ops.PLACE_BEST_QOT)
    over = m.forward_placements(state, g, ops.PLACE_BEST_QOT, max_impact=1)
    torch.cuda.synchronize()
    assert torch.equal(over.status == ops.CAND_IMPACT_OVERFLOW, full.n_impact > 1)
    assert torch.equal(over.option, full.option) and _same(over.out, full.out)


def test_determinism_capture_and_errors(cuda):
    from gnn_qot_estimation_b200 import LightpathGNN, ops, synthetic
    from gnn_qot_estimation_b200.to_graph import LightpathDemands
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(16, seed=17)
    state = _state(smp, cuda)
    d = synthetic.lightpath_demands(smp, 16, seed=18).to(cuda)
    bound = _node_bound(m, state, 0, True, 19)
    a = m.forward_placements(state, d, ops.PLACE_MAX_MARGIN, bound=bound, return_all=True)
    b = m.forward_placements(state, d, ops.PLACE_MAX_MARGIN, bound=bound, return_all=True)
    torch.cuda.synchronize()
    for x, y in zip(a, b):
        assert _same(x, y) if x.is_floating_point() else torch.equal(x, y)
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    holder = {}
    with torch.cuda.stream(s):
        m.forward_placements(state, d, ops.PLACE_MAX_MARGIN, bound=bound, return_all=True)
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            holder["r"] = m.forward_placements(state, d, ops.PLACE_MAX_MARGIN, bound=bound, return_all=True)
        g.replay()
    torch.cuda.synchronize()
    for x, y in zip(holder["r"], a):
        assert _same(x, y) if x.is_floating_point() else torch.equal(x, y)
    assert int((a.option >= 0).sum()) > 0
    # errors
    m.train()
    with pytest.raises(RuntimeError, match="eval"):
        m.forward_placements(state, d, 0)
    m.eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        m.forward_placements(state, d.to("cpu"), 0)
    with pytest.raises(RuntimeError, match="CUDA"):
        m.forward_placements(state, d, 0, bound=bound.cpu())
    with pytest.raises(TypeError, match="links"):
        m.forward_placements(state, d._replace(links=d.links.long()), 0)
    with pytest.raises(TypeError, match="own_bound"):
        m.forward_placements(state, d._replace(own_bound=d.own_bound.double()), 0)
    with pytest.raises(TypeError, match="bound"):
        m.forward_placements(state, d, 0, bound=bound.double())
    with pytest.raises(ValueError, match="opt_ptr"):
        m.forward_placements(state, d._replace(opt_ptr=d.opt_ptr[:-1]), 0)
    with pytest.raises(ValueError, match="feat"):
        m.forward_placements(state, d._replace(feat=torch.zeros(d.feat.shape[0], 4, device=cuda)), 0)
    with pytest.raises(ValueError, match="bound"):
        m.forward_placements(state, d, 0, bound=bound[:-1])
    with pytest.raises(ValueError, match="policy"):
        m.forward_placements(state, d, 3)
    with pytest.raises(ValueError, match="metric"):
        m.forward_placements(state, d, 0, metric=3)
    with pytest.raises(ValueError, match="max_impact"):
        m.forward_placements(state, d, 0, max_impact=-1)
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError, match="cuda"):
            m.forward_placements(state, d._replace(width=d.width.to("cuda:1")), 0)
    odd = LightpathGNN(5, 16, 3, is_lut_index=1).to(cuda).eval()
    with pytest.raises(RuntimeError, match="reference LightpathGNN shape"):
        odd.forward_placements(state, d, 0)
    big = synthetic.network_status_samples(1, num_links=2, num_freqs=1025, seed=1)
    with pytest.raises(ValueError, match="1024"):
        m.forward_placements(_state(big, cuda), d, 0)
    empty = LightpathDemands(*(t[:0] for t in d))._replace(opt_ptr=d.opt_ptr[:1], link_ptr=d.link_ptr[:1])
    r = m.forward_placements(state, empty, 0)
    assert r.out.shape == (0, 3) and r.impact_out.shape == (0, 64, 3)
