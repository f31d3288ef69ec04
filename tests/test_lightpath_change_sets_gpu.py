"""GPU parity of LightpathGNN's change-set QoT (qot_lightpath_change_sets through LightpathGNN.forward_change_sets)
against the fp64 oracle's literal definition (tests/change_set_ref.py), against forward_reconfigurations for sets of
one change (bit for bit), against forward_every_node of rebuilt states for link teardowns, on every status bit, and its
determinism, CUDA-graph capture and error paths."""
import numpy as np
import pytest
import torch

from conftest import rel_err
from test_lightpath_reconfig_gpu import ATOL, RTOL, _changes, _lightpaths, _model, _oracle64, _rows_of, _state

pytestmark = pytest.mark.gpu


def _set_ptr(sizes, dev):
    return torch.tensor(np.cumsum([0] + list(sizes)), dtype=torch.int64, device=dev)


def _check_vs_ref(m, o, smp, state, sets, dev, max_impact=64):
    """sets: [[(node, sample, links, q0, width, feat)]] -> the result, after checking every row against the reference."""
    from change_set_ref import change_set_ref
    rows = [c for st in sets for c in st]
    r = m.forward_change_sets(state, _changes(rows, dev), _set_ptr([len(st) for st in sets], dev), max_impact)
    torch.cuda.synchronize()
    conn = state.conn_ids.cpu()
    assert int(r.set_status.max()) == 0 and int(r.status.max()) == 0, r.set_status
    got, ref, kinds, k = [], [], [], 0
    for g, st in enumerate(sets):
        s = st[0][1]
        own, impact = change_set_ref(o, smp["data"][s], smp["freqs"], smp["lp_feat"],
                                     [(None if c[0] < 0 else int(conn[c[0]]), *c[2:]) for c in st])
        for row in own:
            if row is None:
                assert bool(torch.isnan(r.out[k]).all())
            else:
                got.append(r.out[k])
                ref.append(row)
            k += 1
        n = int(r.n_impact[g])
        assert n == len(impact)
        nodes = r.impact_node[g, :n].cpu()
        assert bool((nodes[1:] > nodes[:-1]).all())
        assert bool((r.impact_node[g, n:] == -1).all()) and bool(torch.isnan(r.impact_out[g, n:]).all())
        assert {int(conn[v]) for v in nodes} == set(impact)
        for i, v in enumerate(nodes.tolist()):
            kind, row = impact[int(conn[v])]
            assert int(r.impact_kind[g, i]) == kind
            kinds.append(kind)
            got.append(r.impact_out[g, i])
            ref.append(row)
    got, ref = torch.stack(got).double().cpu(), torch.stack(ref)
    assert torch.isfinite(got).all()
    assert rel_err(got, ref) <= RTOL
    torch.testing.assert_close(got, ref, rtol=RTOL, atol=ATOL)
    return r, kinds


def _gen_sets(smp, state, per, seed):
    from gnn_qot_estimation_b200 import synthetic
    c, sp = synthetic.lightpath_change_sets(smp, state, per, seed=seed)
    rows = _rows_of(c)
    return [rows[int(sp[g]):int(sp[g + 1])] for g in range(sp.numel() - 1)]


def test_change_sets_vs_oracle_fresh_seeds_width3_and_empty_sample(cuda):
    """Every generated set kind on fresh seeds, super-channels widened to 3 slots, insertions into an empty sample."""
    from gnn_qot_estimation_b200 import synthetic
    m, sd = _model(cuda)
    o = _oracle64(sd)
    smp = synthetic.network_status_samples(6, num_links=16, num_freqs=32, seed=51, super_channel_p=0.3)
    smp["data"][5] = 0.0
    state = _state(smp, cuda)
    sets = _gen_sets(smp, state, 12, 52)
    occ = np.any(smp["data"] != 0, axis=1)
    freqs = smp["freqs"]
    wide = []                                            # two lightpaths of a sample retuned together, one to width 3
    lps = _lightpaths(smp, state)
    for s in range(5):
        mine = [lp for lp in lps if lp[0] == s]
        for (_, v, c, links, q0, w, feat), (_, v2, c2, l2, q2, w2, f2) in zip(mine[::2], mine[1::2]):
            fi = {k: i for i, k in enumerate(smp["lp_feat"])}
            conn = np.trunc(smp["data"][s, fi["conn_id"]])
            free = ~occ[s] | (conn == c) | (conn == c2)
            q = next((q for q in range(30) if free[np.ix_(links, range(q, q + 3))].all() and
                      free[np.ix_(l2, range(q2, q2 + w2))].all() and
                      not (set(links) & set(l2) and q < q2 + w2 and q2 < q + 3)), None)
            if q is not None:
                wide.append([(v, s, links, q, 3, [np.float32(freqs[q]), *feat[1:]]), (v2, s, l2, q2, w2, f2)])
                break
    assert len(wide) >= 3
    r, kinds = _check_vs_ref(m, o, smp, state, sets + wide + [[(-1, 5, [0, 3], 4, 2, [np.float32(freqs[4]), 8, 2,
                                                                                       90000]),
                                                                (-1, 5, [3], 7, 1, [192.55, 4, 9, 80000])]], cuda)
    assert {1, 2, 3} <= set(kinds)
    assert int(r.n_impact[-1]) == 0 and bool(torch.isfinite(r.out[-2:]).all())
    assert max(len(st) for st in sets) >= 4


def test_change_sets_threshold_boundary(cuda):
    """Spacing 0.05 on a 0.05 threshold: adjacency between changes and to the state decided by fp64 rounding."""
    from gnn_qot_estimation_b200 import synthetic
    m, sd = _model(cuda)
    o = _oracle64(sd)
    smp = synthetic.network_status_samples(4, num_links=6, num_freqs=24, seed=5, spacing=0.05, max_lightpaths=14)
    state = _state(smp, cuda)
    _, kinds = _check_vs_ref(m, o, smp, state, _gen_sets(smp, state, 10, 6), cuda)
    assert {1, 2} <= set(kinds)


def test_single_change_sets_are_bit_identical_to_reconfigurations(cuda):
    from gnn_qot_estimation_b200 import synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(16, seed=41, super_channel_p=0.2)
    state = _state(smp, cuda)
    c = synthetic.lightpath_changes(smp, state, 64, seed=42).to(cuda)
    sp = torch.arange(c.sample.shape[0] + 1, device=cuda)
    for mi in (64, 1):
        a = m.forward_reconfigurations(state, c, mi)
        b = m.forward_change_sets(state, c, sp, mi)
        torch.cuda.synchronize()
        for name in ("out", "status", "n_impact", "impact_node", "impact_kind", "impact_out"):
            x, y = getattr(a, name), getattr(b, name)
            assert torch.equal(x.nan_to_num(7.0) if x.is_floating_point() else x,
                               y.nan_to_num(7.0) if y.is_floating_point() else y), name
        assert torch.equal(b.set_status, b.status)
    assert int(a.n_impact.max()) > 1


def _free(smp, s):
    return ~np.any(smp["data"][s] != 0, axis=0)


def test_joint_insertion_sees_the_interaction_and_a_swap_is_legal(cuda):
    """Two new lightpaths on adjacent slots of a shared link: each row matches the reference and differs from its
    forward_candidates row, which leaves the other out.  Two lightpaths of equal width swapping slots: no OCCUPIED."""
    from gnn_qot_estimation_b200 import ops, synthetic
    from gnn_qot_estimation_b200.to_graph import LightpathCandidates
    m, sd = _model(cuda)
    o = _oracle64(sd)
    smp = synthetic.network_status_samples(4, num_links=6, num_freqs=32, seed=9, max_lightpaths=12)
    state = _state(smp, cuda)
    freqs = smp["freqs"]
    free = _free(smp, 0)
    l, q = next((l, q) for l in range(6) for q in range(31) if free[l, q] and free[l, q + 1])
    f = lambda q: [np.float32(freqs[q]), 16, 10, 100000]
    pair = [(-1, 0, [l], q, 1, f(q)), (-1, 0, [l], q + 1, 1, f(q + 1))]
    r, _ = _check_vs_ref(m, o, smp, state, [pair], cuda)
    cands = LightpathCandidates(*_changes(pair, cuda)[1:])
    alone = m.forward_candidates(state, cands, 64)
    assert not torch.allclose(alone.out, r.out, rtol=1e-4, atol=1e-4)
    # a swap: every pair of equal-width lightpaths whose exchanged placements are free once both are cleared
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    swaps = []
    for s in range(4):
        lps = [lp for lp in _lightpaths(smp, state) if lp[0] == s]
        occ = ~_free(smp, s)
        conn = np.trunc(smp["data"][s, fi["conn_id"]])
        for a in lps:
            for b in lps:
                if a[1] >= b[1] or a[5] != b[5] or a[4] == b[4]:
                    continue
                others = occ & (conn != a[2]) & (conn != b[2])
                w = a[5]
                if others[np.ix_(a[3], range(b[4], b[4] + w))].any() or \
                        others[np.ix_(b[3], range(a[4], a[4] + w))].any():
                    continue
                if not set(a[3]) & set(b[3]) or abs(a[4] - b[4]) < w:
                    continue                               # share a link, so that each half alone is blocked
                swaps.append([(a[1], s, a[3], b[4], w, [np.float32(freqs[b[4]]), *a[6][1:]]),
                              (b[1], s, b[3], a[4], w, [np.float32(freqs[a[4]]), *b[6][1:]])])
    assert swaps
    r, _ = _check_vs_ref(m, o, smp, state, swaps[:8], cuda)
    rec = m.forward_reconfigurations(state, _changes([c for st in swaps[:8] for c in st], cuda), 64)
    torch.cuda.synchronize()
    assert bool((r.status & ops.CAND_OCCUPIED == 0).all())
    assert bool((rec.status & ops.CAND_OCCUPIED != 0).any())       # each half alone is blocked by the other


def test_link_teardowns_vs_every_node_of_rebuilt_states(cuda):
    """For every link of 24 samples, the set tearing down every lightpath on it: the listed rows (kind 1) and every
    unlisted row equal forward_every_node of the state rebuilt from the cleared data."""
    from gnn_qot_estimation_b200 import synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(24, seed=13, super_channel_p=0.2)
    data, fi = smp["data"], {k: i for i, k in enumerate(smp["lp_feat"])}
    state = _state(smp, cuda)
    every = m.forward_every_node(state.batch).cpu()
    conn_ids, ptr = state.conn_ids.cpu(), state.batch.ptr.cpu()
    occ = np.any(data != 0, axis=1)
    L = data.shape[2]
    sets, cleared = [], []
    for s in range(24):
        conn = np.trunc(data[s, fi["conn_id"]])
        node_of = {int(conn_ids[v]): v for v in range(int(ptr[s]), int(ptr[s + 1]))}
        for l in range(L):
            gone = sorted({int(c) for c in conn[l][occ[s, l]]})
            if not gone or len(gone) > 64:
                continue
            sets.append([(node_of[c], s, [], 0, 1, [0.0, 0.0, 0.0, 0.0]) for c in gone])
            rest = data[s].copy()
            rest[:, occ[s] & np.isin(conn, gone)] = 0.0
            cleared.append((s, set(gone), rest))
    rows = [c for st in sets for c in st]
    r = m.forward_change_sets(state, _changes(rows, cuda), _set_ptr([len(st) for st in sets], cuda), 64)
    torch.cuda.synchronize()
    assert int(r.set_status.max()) == 0 and bool(torch.isnan(r.out).all())
    st2 = _state(dict(smp, data=np.stack([c[2] for c in cleared])), cuda)
    after = m.forward_every_node(st2.batch).cpu()
    conn2, ptr2 = st2.conn_ids.cpu(), st2.batch.ptr.cpu()
    got, ref, n_unlisted = [], [], 0
    for g, (s, gone, _) in enumerate(cleared):
        n = int(r.n_impact[g])
        assert bool((r.impact_kind[g, :n] == 1).all())
        listed = {int(v): i for i, v in enumerate(r.impact_node[g, :n].tolist())}
        for u in range(int(ptr2[g]), int(ptr2[g + 1])):
            v = next(v for v in range(int(ptr[s]), int(ptr[s + 1])) if int(conn_ids[v]) == int(conn2[u]))
            got.append(r.impact_out[g, listed[v]].cpu() if v in listed else every[v])
            ref.append(after[u])
            n_unlisted += v not in listed
        assert len(listed) + len(gone) <= int(ptr[s + 1] - ptr[s])
    torch.testing.assert_close(torch.stack(got), torch.stack(ref), rtol=RTOL, atol=ATOL)
    assert len(got) - n_unlisted > 100 and n_unlisted > 100


def test_change_set_status_bits(cuda):
    from gnn_qot_estimation_b200 import ops, synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(3, num_links=8, num_freqs=20, seed=7, max_lightpaths=20,
                                           super_channel_p=0.4)
    state = _state(smp, cuda)
    lps = _lightpaths(smp, state)
    s, v, c, links, q0, w, feat = next(lp for lp in lps if lp[0] == 0)
    v2 = next(lp[1] for lp in lps if lp[0] == 0 and lp[1] != v)
    ptr = state.batch.ptr.cpu()
    free = _free(smp, 0)
    fl, fq = next((l, q) for l in range(8) for q in range(19) if free[l, q] and free[l, q + 1])
    f = [np.float32(smp["freqs"][3]), 16, 10, 100000]
    good = (-1, 0, [fl], fq, 1, f)
    sets = [
        [good, (-1, 1, [1], 3, 1, f)],                                   # 0: two samples
        [(v, 0, links, q0, w, feat), (v, 0, [], 0, 1, f)],               # 1: v moved and torn down
        [good, (-1, 0, [fl], fq, 1, f)],                                 # 2: the same channel twice
        [good, (int(ptr[1]), 0, [1], 3, 1, f)],                          # 3: a node of another sample
        [(v, 0, links, q0, w, feat), (v2, 0, [], 0, 1, f)],              # 4: fine
        [good] * 65,                                                     # 5: over the limit
        [],                                                              # 6: empty
        [good, (-1, 0, [9], 3, 1, f)],                                   # 7: a bad link
    ]
    rows = [x for st in sets for x in st]
    ch = _changes(rows, cuda)
    r = m.forward_change_sets(state, ch, _set_ptr([len(st) for st in sets], cuda), 64)
    torch.cuda.synchronize()
    ss, st = r.set_status.cpu().tolist(), r.status.cpu().tolist()
    assert ss[0] == ops.SET_BAD_SET and st[0:2] == [0, ops.SET_BAD_SET]
    assert ss[1] == ops.SET_DUPLICATE and st[2:4] == [ops.SET_DUPLICATE] * 2
    assert ss[2] == ops.SET_CONFLICT and st[4:6] == [ops.SET_CONFLICT] * 2
    assert ss[3] == ops.CAND_BAD_NODE
    assert ss[4] == 0 and bool(torch.isfinite(r.out[8]).all()) and bool(torch.isnan(r.out[9]).all())
    assert ss[5] == ops.SET_BAD_SET and set(st[10:75]) == {ops.SET_BAD_SET}
    assert ss[6] == 0 and int(r.n_impact[6]) == 0
    assert ss[7] == ops.CAND_BAD_PATH
    for g in (0, 1, 2, 3, 5, 7):
        assert int(r.n_impact[g]) == 0 and bool((r.impact_node[g] == -1).all())
        assert bool((r.impact_kind[g] == 0).all()) and bool(torch.isnan(r.impact_out[g]).all())
    bad_k = [0, 1, 2, 3, 4, 5, 6, 7] + list(range(10, 77))
    assert bool(torch.isnan(r.out[bad_k]).all())
    # a malformed set_ptr: nothing is evaluated, every change and set says BAD_SET
    for sp in ([0, 3, 2, len(rows)], [1, len(rows)], [0, len(rows) - 1], [0, len(rows) + 1]):
        b = m.forward_change_sets(state, ch, torch.tensor(sp, device=cuda), 64)
        torch.cuda.synchronize()
        assert bool((b.status == ops.SET_BAD_SET).all()) and bool((b.set_status == ops.SET_BAD_SET).all())
        assert bool(torch.isnan(b.out).all()) and bool((b.n_impact == 0).all())
        assert bool(torch.isnan(b.impact_out).all()) and bool((b.impact_node == -1).all())
    # max_impact overflow: the first rows kept, the true count reported, every change flagged
    sets = _gen_sets(smp, state, 20, 3)
    rows = [x for st in sets for x in st]
    sp = _set_ptr([len(st) for st in sets], cuda)
    full = m.forward_change_sets(state, _changes(rows, cuda), sp, 64)
    n = full.n_impact.cpu()
    g = int(torch.argmax(n))
    assert int(n[g]) >= 2
    cut = int(n[g]) - 1
    over = m.forward_change_sets(state, _changes(rows, cuda), sp, cut)
    torch.cuda.synchronize()
    k0, k1 = int(sp[g]), int(sp[g + 1])
    assert int(over.set_status[g]) == ops.CAND_IMPACT_OVERFLOW and int(over.n_impact[g]) == int(n[g])
    assert bool((over.status[k0:k1] == ops.CAND_IMPACT_OVERFLOW).all())
    assert torch.equal(over.out[k0:k1].nan_to_num(7.0), full.out[k0:k1].nan_to_num(7.0))
    assert torch.equal(over.impact_node[g], full.impact_node[g, :cut])
    assert torch.equal(over.impact_kind[g], full.impact_kind[g, :cut])
    assert torch.equal(over.impact_out[g], full.impact_out[g, :cut])


def test_change_sets_determinism_capture_and_errors(cuda):
    from gnn_qot_estimation_b200 import LightpathGNN, synthetic
    from gnn_qot_estimation_b200.to_graph import LightpathChanges
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(16, seed=17)
    state = _state(smp, cuda)
    c, sp = synthetic.lightpath_change_sets(smp, state, 32, seed=18)
    c, sp = c.to(cuda), sp.to(cuda)
    a = m.forward_change_sets(state, c, sp)
    b = m.forward_change_sets(state, c, sp)
    torch.cuda.synchronize()
    same = lambda x, y: torch.equal(x.nan_to_num(7.0) if x.is_floating_point() else x,
                                    y.nan_to_num(7.0) if y.is_floating_point() else y)
    assert all(same(x, y) for x, y in zip(a, b))
    assert int(a.set_status.max()) == 0
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    holder = {}
    with torch.cuda.stream(s):
        m.forward_change_sets(state, c, sp)
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            holder["r"] = m.forward_change_sets(state, c, sp)
        g.replay()
    torch.cuda.synchronize()
    assert all(same(x, y) for x, y in zip(holder["r"], a))
    m.train()
    with pytest.raises(RuntimeError, match="eval"):
        m.forward_change_sets(state, c, sp)
    m.eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        m.forward_change_sets(state, c.to("cpu"), sp)
    with pytest.raises(RuntimeError, match="set_ptr"):
        m.forward_change_sets(state, c, sp.cpu())
    with pytest.raises(TypeError, match="set_ptr"):
        m.forward_change_sets(state, c, sp.int())
    with pytest.raises(ValueError, match="set_ptr"):
        m.forward_change_sets(state, c, sp[None])
    with pytest.raises(TypeError, match="node"):
        m.forward_change_sets(state, c._replace(node=c.node.int()), sp)
    with pytest.raises(ValueError, match="max_impact"):
        m.forward_change_sets(state, c, sp, -1)
    odd = LightpathGNN(5, 16, 3, is_lut_index=1).to(cuda).eval()
    with pytest.raises(RuntimeError, match="reference LightpathGNN shape"):
        odd.forward_change_sets(state, c, sp)
    empty = LightpathChanges(*(t[:0] for t in c))._replace(link_ptr=c.link_ptr[:1])
    r = m.forward_change_sets(state, empty, sp[:1])
    assert r.out.shape == (0, 3) and r.impact_out.shape == (0, 64, 3) and r.set_status.shape == (0,)
    r = m.forward_change_sets(state, empty, torch.zeros(3, dtype=torch.int64, device=cuda))
    torch.cuda.synchronize()
    assert r.set_status.tolist() == [0, 0] and r.n_impact.tolist() == [0, 0]


def _pair_setup(cuda, seed=21):
    """A small state, and per sample with two or more lightpaths: lightpaths A and B (as _lightpaths gives them), B's
    first channel (bl, bq), and a free channel (fl, fq) whose next slot is free too."""
    from gnn_qot_estimation_b200 import synthetic
    smp = synthetic.network_status_samples(3, num_links=8, num_freqs=24, seed=seed, max_lightpaths=16,
                                           super_channel_p=0.3)
    state = _state(smp, cuda)
    lps = _lightpaths(smp, state)
    out = {}
    for s in range(3):
        mine = [lp for lp in lps if lp[0] == s]
        free = _free(smp, s)
        fc = next(((l, q) for l in range(8) for q in range(23) if free[l, q] and free[l, q + 1]), None)
        if len(mine) >= 2 and fc:
            out[s] = (mine[0], mine[1], (mine[1][3][0], mine[1][4]), fc)
    return smp, state, out


def _assert_fatal(r, sp, g, status, set_status):
    """Set g failed with exactly these per-change status words and this set status: its out rows are NaN, n_impact is
    0 and its impact slots hold -1 / 0 / NaN."""
    k0, k1 = int(sp[g]), int(sp[g + 1])
    assert r.status[k0:k1].cpu().tolist() == status
    assert int(r.set_status[g]) == set_status
    assert bool(torch.isnan(r.out[k0:k1]).all()) and int(r.n_impact[g]) == 0
    assert bool((r.impact_node[g] == -1).all()) and bool((r.impact_kind[g] == 0).all())
    assert bool(torch.isnan(r.impact_out[g]).all())


def test_change_set_occupied_and_bad_sample(cuda):
    """OCCUPIED means a channel held by a lightpath the set leaves in place: (a) an insertion on it, (b) a move onto it
    are OCCUPIED, (c) the same move with the holder moved away is clean.  (d) A sample outside the state is BAD_SAMPLE.
    A fatal change makes its whole set NaN; the other sets are untouched."""
    from gnn_qot_estimation_b200 import ops
    m, _ = _model(cuda)
    smp, state, pick = _pair_setup(cuda)
    (_, va, _, _, _, _, fa), (_, vb, _, _, _, _, fb), (bl, bq), (fl, fq) = pick[0]
    freqs = smp["freqs"]
    f = lambda q: [np.float32(freqs[q]), 16, 10, 100000]
    good = (-1, 0, [fl], fq, 1, f(fq))
    a_on_b = (va, 0, [bl], bq, 1, [np.float32(freqs[bq]), *fa[1:]])
    sets = [
        [good, (-1, 0, [bl], bq, 1, f(bq))],                             # 0 (a): insertion on B's channel
        [a_on_b],                                                        # 1 (b): A onto B's channel, B stays
        [a_on_b, (vb, 0, [fl], fq, 1, [np.float32(freqs[fq]), *fb[1:]])],  # 2 (c): B moves away: clean
        [(-1, 3, [1], 3, 1, f(3))],                                      # 3 (d): sample 3 of 3
        [(-1, 3, [1], 3, 1, f(3)), (-1, 3, [2], 5, 1, f(5))],            # 4 (d): twice
        [good],                                                          # 5: fine
    ]
    rows = [x for st in sets for x in st]
    sp = _set_ptr([len(st) for st in sets], cuda)
    r = m.forward_change_sets(state, _changes(rows, cuda), sp, 64)
    torch.cuda.synchronize()
    _assert_fatal(r, sp, 0, [0, ops.CAND_OCCUPIED], ops.CAND_OCCUPIED)
    _assert_fatal(r, sp, 1, [ops.CAND_OCCUPIED], ops.CAND_OCCUPIED)
    assert r.status[3:5].tolist() == [0, 0] and int(r.set_status[2]) == 0
    assert bool(torch.isfinite(r.out[3:5]).all())
    _assert_fatal(r, sp, 3, [ops.CAND_BAD_SAMPLE], ops.CAND_BAD_SAMPLE)
    _assert_fatal(r, sp, 4, [ops.CAND_BAD_SAMPLE] * 2, ops.CAND_BAD_SAMPLE)
    assert int(r.set_status[5]) == 0 and bool(torch.isfinite(r.out[8]).all())
    # (b) against forward_reconfigurations, which applies the same occupancy rule to one change
    rec = m.forward_reconfigurations(state, _changes([a_on_b], cuda), 64)
    assert int(rec.status[0]) == ops.CAND_OCCUPIED


def test_mixed_sets_vs_oracle(cuda):
    """Insertions mixed with moves and teardowns: a teardown and an insertion into the freed slot (restoration), a move
    and an insertion right next to it, and a move onto a channel the set frees by moving its holder away."""
    m, sd = _model(cuda)
    o = _oracle64(sd)
    smp, state, pick = _pair_setup(cuda)
    freqs = smp["freqs"]
    f = lambda q: [np.float32(freqs[q]), 16, 10, 100000]
    sets = []
    for s, ((_, va, _, _, _, _, fa), (_, vb, _, _, _, _, fb), (bl, bq), (fl, fq)) in pick.items():
        mv = lambda v, ft, l, q: (v, s, [l], q, 1, [np.float32(freqs[q]), *ft[1:]])
        sets += [[(vb, s, [], 0, 1, fb), (-1, s, [bl], bq, 1, f(bq))],
                 [mv(va, fa, fl, fq), (-1, s, [fl], fq + 1, 1, f(fq + 1))],
                 [mv(va, fa, bl, bq), mv(vb, fb, fl, fq)]]
    assert len(sets) >= 6
    r, kinds = _check_vs_ref(m, o, smp, state, sets, cuda)
    assert len(kinds) >= 4                   # rows that lose a lightpath and gain its replacement are kind 3
    # the insertion next to the moved lightpath is one of its neighbours: the joint row differs from the move alone
    alone = m.forward_reconfigurations(state, _changes([sets[1][0]], cuda), 64)
    assert not torch.allclose(alone.out[0], r.out[2], rtol=1e-4, atol=1e-4)


def test_bad_in_row_makes_the_whole_set_nan(cuda):
    """A state whose edge list sends an impact row's in-row outside its sample: the pre-check reports BAD_STATE on the
    set's first change before any row is written, so the whole set is NaN; a set of another sample is unaffected."""
    from types import SimpleNamespace
    from gnn_qot_estimation_b200 import ops
    m, _ = _model(cuda)
    smp, state, pick = _pair_setup(cuda)
    lps = _lightpaths(smp, state)
    ei, rp = state.batch.edge_index, state.rowptr
    src, dst = ei[0].cpu(), ei[1].cpu()
    j = next(lp for lp in lps if lp[0] == 0 and bool(((src == lp[1]) & (dst != lp[1])).any()))
    i = int(dst[(src == j[1]) & (dst != j[1])][0])                     # a neighbour of j: an impact row of j's move
    other = next(lp for lp in lps if lp[0] == 1)
    fl, fq = pick[0][3]
    sets = [[(-1, 0, [fl], fq, 1, [np.float32(smp["freqs"][fq]), 16, 10, 100000]), (j[1], 0, *j[3:])],
            [(other[1], 1, *other[3:])]]
    rows = [x for st in sets for x in st]
    sp = _set_ptr([len(st) for st in sets], cuda)
    ch = _changes(rows, cuda)
    ok = m.forward_change_sets(state, ch, sp, 64)
    bad_ei = ei.clone()
    bad_ei[1, int(rp[i])] = state.batch.x.shape[0] + 5
    bad = state._replace(batch=SimpleNamespace(x=state.batch.x, edge_index=bad_ei, ptr=state.batch.ptr))
    r = m.forward_change_sets(bad, ch, sp, 64)
    torch.cuda.synchronize()
    assert int(ok.set_status.max()) == 0 and i in ok.impact_node[0].tolist()
    _assert_fatal(r, sp, 0, [ops.CAND_BAD_STATE, 0], ops.CAND_BAD_STATE)
    same = lambda x, y: torch.equal(x.nan_to_num(7.0), y.nan_to_num(7.0))
    assert int(r.set_status[1]) == 0 and same(r.out[2], ok.out[2]) and same(r.impact_out[1], ok.impact_out[1])
