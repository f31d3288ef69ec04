"""GPU checks of LightpathGNN's 1+1 protected provisioning (qot_lightpath_protect through
LightpathGNN.forward_protection and to_graph.commit_protection): bit-identity with the round loop of
forward_placements and rebuilds (tests/protection_ref.py), the reduction to forward_provision, hand-built rollbacks,
partner-less demands, slots and ties, capacity samples, parity with the fp64 literal reference, the commit, every status
bit, determinism, CUDA-graph replay and the error paths."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from test_lightpath_provision_gpu import (ATOL, FIELDS, RTOL, _builder, _demands, _model, _node_bound, _oracle64,
                                          _pack, _same, _state)

pytestmark = pytest.mark.gpu
BFIELDS = FIELDS + tuple("backup_" + f for f in FIELDS)


def _assert_same(r, ref, fields=BFIELDS):
    for f in fields:
        assert _same(getattr(r, f), getattr(ref, f)), f


def _round_loop(m, smp, dev, d, protect, policy, metric, maximize, bound, max_impact=64, thr=0.05):
    from protection_ref import round_loop
    data = torch.from_numpy(smp["data"]).to(dev).contiguous()
    res, state = round_loop(m, data, torch.from_numpy(smp["freqs"]).to(dev), smp["lp_feat"], d, protect, policy,
                            metric, maximize, bound, max_impact, thr)
    return res, state, data


def _protect(D, dev, seed, share=0.5):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.rand(D, generator=g) < share).to(dev)


def _flags(v, dev):
    return torch.tensor(v, dtype=torch.bool, device=dev)


# ------------------------------------------------------------------------------------------------ round loop
def test_round_loop_bit_identity(cuda):
    """Every policy, both senses, each metric column, with and without a bound: 10 interleaved demands per sample on
    average over 5 samples (one of them empty), about half protected, every output equal bit for bit to the round
    loop; accepted and partner-less demands occur."""
    from gnn_qot_estimation_b200 import ops, synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(5, num_links=12, num_freqs=40, seed=41, super_channel_p=0.3)
    smp["data"][4] = 0.0
    state = _state(smp, cuda)
    d = synthetic.lightpath_demands(smp, 10, options=(2, 4), seed=42, bound_range=(0.0, 0.5)).to(cuda)
    prot = _protect(d.sample.shape[0], cuda, 44)
    seen = {"acc": 0, "partner": 0}
    for metric, mx in ((0, True), (1, True), (2, False), (0, False)):
        for bound in (None, _node_bound(m, state, metric, mx, 43 + metric, spread=0.05)):
            for policy in (0, 1, 2):
                r = m.forward_protection(state, d, prot, policy, metric, mx, bound)
                ref, _, _ = _round_loop(m, smp, cuda, d, prot, policy, metric, mx, bound)
                torch.cuda.synchronize()
                _assert_same(r, ref)
                seen["acc"] += int((r.backup_conn_id >= 0).sum())
                seen["partner"] += int((r.status & ops.PROT_NO_PARTNER != 0).sum())
    assert seen["acc"] > 50 and seen["partner"] > 0, seen


def _c_call(m, state, d, order, sample_ptr, protect, max_impact=4):
    """qot_lightpath_protect through the C entry point with a caller-made grouping (protect may be None: NULL)."""
    from gnn_qot_estimation_b200 import _lib, ops
    from gnn_qot_estimation_b200.ops import _demands_desc, _state_desc, ptr, stream
    D, P, dev = int(d.sample.shape[0]), int(d.width.shape[0]), state.batch.x.device

    def outs():
        return [torch.full((D,), 99, dtype=torch.int32, device=dev) for _ in range(2)] + \
               [torch.zeros(D, 3, device=dev), torch.zeros(D, device=dev)] + \
               [torch.full((D,), 99, dtype=torch.int32, device=dev) for _ in range(4)] + \
               [torch.full((D, max_impact), 99, dtype=torch.int64, device=dev), torch.zeros(D, max_impact, 3, device=dev),
                torch.full((D,), 99, dtype=torch.int64, device=dev)]
    res = ops.ProtectionQoT(*outs(), *outs())
    keep = []
    cw = torch.empty_like(state.chan_node)
    co = ops._C_ORDER
    rc = _lib.lib().qot_lightpath_protect(
        C.byref(_state_desc(state, keep)), C.byref(_demands_desc(d, D, P, keep)), ptr(order), ptr(sample_ptr), None,
        0, 1, 0, ptr(m.prepared()), 1, max_impact, ptr(cw), None, *(ptr(res[k]) for k in co),
        None if protect is None else ptr(protect), *(ptr(res[11 + k]) for k in co), stream())
    torch.cuda.synchronize()
    return rc, res


def _empty_backup(r):
    assert bool((r.backup_option == -1).all()) and bool((r.backup_q0 == -1).all())
    assert bool(torch.isnan(r.backup_out).all()) and bool(torch.isnan(r.backup_margin).all())
    assert int(r.backup_n_free.abs().sum()) == 0 and int(r.backup_n_feasible.abs().sum()) == 0
    assert int(r.backup_status.abs().sum()) == 0 and int(r.backup_n_impact.abs().sum()) == 0
    assert bool((r.backup_impact_conn == -1).all()) and bool(torch.isnan(r.backup_impact_out).all())
    assert bool((r.backup_conn_id == -1).all())


def test_reduces_to_provision(cuda):
    """protect all False, and a NULL protect through the C entry point: forward_provision's outputs bit for bit, the
    backup fields empty."""
    from gnn_qot_estimation_b200 import ops, synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(6, num_links=16, num_freqs=40, seed=51, super_channel_p=0.3)
    state = _state(smp, cuda)
    d = synthetic.lightpath_demands(smp, 6, options=(2, 4), seed=52).to(cuda)
    D = int(d.sample.shape[0])
    bound = _node_bound(m, state, 0, True, 53)
    for policy in (0, 1, 2):
        for b in (None, bound):
            r = m.forward_protection(state, d, torch.zeros(D, dtype=torch.bool, device=cuda), policy, 0, True, b, 4)
            p = m.forward_provision(state, d, policy, 0, True, b, 4)
            torch.cuda.synchronize()
            _assert_same(r, p, FIELDS)
            _empty_backup(r)
    order, sp = ops.provision_grouping(d.sample, state.S)
    rc, r = _c_call(m, state, d, order, sp, None)
    p = m.forward_provision(state, d, 0, 0, True, None, 4)
    torch.cuda.synchronize()
    assert rc == 0
    _assert_same(r, p, FIELDS)
    _empty_backup(r)


# ------------------------------------------------------------------------------------------------ hand-built
def test_rollback_is_invisible(cuda):
    """The working path's only partner is full: NO_BACKUP, conn_ids -1, the working placement reported; every later
    demand's outputs, conn_ids included, equal those of the same call without that demand."""
    from gnn_qot_estimation_b200 import ops
    m, _ = _model(cuda)
    b = _builder(4, 8, 3)
    for q in range(8):
        b.place([2], q)                              # link 2 full
    b.place([0], 4)
    smp = _pack([b])
    state = _state(smp, cuda)
    f = (16, 10, 300000)
    ninf = -np.inf
    blocked = (0, [([0], 1, f, ninf), ([2], 1, f, ninf)])
    later = [(0, [([0], 1, f, ninf)]), (0, [([0], 1, f, ninf), ([1], 1, f, ninf)]), (0, [([1, 3], 1, f, ninf)])]
    d = _demands([blocked] + later, cuda)
    d2 = _demands(later, cuda)
    for policy in (0, 2):
        r = m.forward_protection(state, d, _flags([True, False, True, True], cuda), policy)
        r2 = m.forward_protection(state, d2, _flags([False, True, True], cuda), policy)
        ref, _, _ = _round_loop(m, smp, cuda, d, _flags([True, False, True, True], cuda), policy, 0, True, None)
        torch.cuda.synchronize()
        _assert_same(r, ref)
        assert int(r.status[0]) & ops.PROT_NO_BACKUP and int(r.conn_id[0]) == -1 and int(r.backup_conn_id[0]) == -1
        assert int(r.option[0]) == 0 and int(r.q0[0]) >= 0 and int(r.backup_n_free[0]) == 0
        for f_ in BFIELDS:
            assert _same(getattr(r, f_)[1:], getattr(r2, f_)), f_
        top = int(state.conn_ids.max())
        assert int(r.conn_id[1]) == top + 1                               # nothing consumed by the rollback


def test_no_partner(cuda):
    """One option, or every route sharing a link: NO_PARTNER with nothing placed and n_free = 0; unprotected, the same
    demands are placed."""
    from gnn_qot_estimation_b200 import ops
    m, _ = _model(cuda)
    b = _builder(4, 16, 5)
    b.place([0], 3)
    b.place([2], 8)
    b.place([2], 9)                                  # an interfering pair: the state has an edge
    smp = _pack([b])
    state = _state(smp, cuda)
    f = (16, 10, 300000)
    ninf = -np.inf
    rows = [(0, [([1], 1, f, ninf)]), (0, [([1], 1, f, ninf), ([1, 3], 1, f, ninf), ([3, 1, 1], 2, f, ninf)])]
    d = _demands(rows, cuda)
    r = m.forward_protection(state, d, _flags([True, True], cuda), 0)
    torch.cuda.synchronize()
    assert r.status.tolist() == [ops.PROT_NO_PARTNER] * 2
    assert r.option.tolist() == [-1, -1] and r.n_free.tolist() == [0, 0] and r.conn_id.tolist() == [-1, -1]
    assert bool(torch.isnan(r.out).all())
    _empty_backup(r)
    u = m.forward_protection(state, d, _flags([False, False], cuda), 0)
    torch.cuda.synchronize()
    assert (u.conn_id >= 0).all()


def test_slots_and_mirrored_ties(cuda):
    """Later demands cannot take either path's slots; on an empty sample a tie between mirrored options goes to the
    lower option for the working path, the other route being the backup."""
    m, _ = _model(cuda)
    b = _builder(4, 16, 7)
    b.place([3], 10)
    b.place([3], 11)
    smp = _pack([b])
    state = _state(smp, cuda)
    f = (16, 10, 300000)
    ninf = -np.inf
    rows = [(0, [([0], 1, f, ninf), ([1, 2], 1, f, ninf)]), (0, [([0], 1, f, ninf)]), (0, [([1], 1, f, ninf)]),
            (0, [([2], 1, f, ninf)])]
    d = _demands(rows, cuda)
    prot = _flags([True, False, False, False], cuda)
    r = m.forward_protection(state, d, prot, 0)
    torch.cuda.synchronize()
    assert (int(r.option[0]), int(r.q0[0]), int(r.backup_option[0]), int(r.backup_q0[0])) == (0, 0, 1, 0)
    assert r.q0.tolist()[1:] == [1, 1, 1]                             # slot 0 taken on links 0, 1 and 2
    ref, _, _ = _round_loop(m, smp, cuda, d, prot, 0, 0, True, None)
    _assert_same(r, ref)
    far = _builder(4, 16, 8)
    far.place([3], 8)                                                  # interferes with neither option
    far.place([3], 9)
    far = _pack([far])
    est = _state(far, cuda)
    for rows2 in ([(0, [([0], 1, f, ninf), ([1], 1, f, ninf)])], [(0, [([1], 1, f, ninf), ([0], 1, f, ninf)])]):
        d2 = _demands(rows2, cuda)
        for policy in (0, 1, 2):
            r2 = m.forward_protection(est, d2, _flags([True], cuda), policy)
            ref2, _, _ = _round_loop(m, far, cuda, d2, _flags([True], cuda), policy, 0, True, None)
            torch.cuda.synchronize()
            _assert_same(r2, ref2)
            assert int(r2.option[0]) == 0 and int(r2.backup_option[0]) == 1


def test_backup_bound_refuses_a_neighbour_break(cuda):
    """With a bound above every lightpath's current value, each backup slot next to one of them (slots 1, 3, .., 15
    on link 2) would take it below its bound and is infeasible; the others stay feasible.  Every output equals the
    round loop's."""
    m, _ = _model(cuda)
    b = _builder(4, 24, 9)
    for q in (2, 6, 10, 14):
        b.place([2], q)
    b.place([3], 20)
    b.place([3], 21)                                 # an interfering pair away from the demand's routes
    smp = _pack([b])
    state = _state(smp, cuda)
    f = (16, 10, 300000)
    ninf = -np.inf
    d = _demands([(0, [([0], 1, f, ninf), ([2], 1, f, ninf)])], cuda)
    bound = (m.forward_every_node(state.batch)[:, 0] + 1.0).contiguous()
    prot = _flags([True], cuda)
    r0 = m.forward_protection(state, d, prot, 0, 0, True, None)
    r1 = m.forward_protection(state, d, prot, 0, 0, True, bound)
    ref, _, _ = _round_loop(m, smp, cuda, d, prot, 0, 0, True, bound)
    torch.cuda.synchronize()
    _assert_same(r1, ref)
    assert int(r1.backup_n_free[0]) == int(r0.backup_n_free[0]) == 20
    assert int(r0.backup_n_feasible[0]) == 20 and int(r1.backup_n_feasible[0]) == 12
    assert int(r1.backup_conn_id[0]) >= 0 and int(r1.backup_q0[0]) not in range(1, 16, 2)
    assert int(r1.backup_n_impact[0]) == 0


# ------------------------------------------------------------------------------------------------ capacity
def _count_sample(n, seed):
    """n single-slot lightpaths on links 2..7 of L = 8, Q = 64; links 0 and 1 free."""
    b = _builder(8, 64, seed)
    for k in range(n):
        b.place([2 + k // 64], k % 64)
    return _pack([b])


def test_capacity(cuda):
    """254 lightpaths: one protected demand is accepted (256), the next gets PROV_FULL.  255: the working path fits,
    the backup gets PROV_FULL and the demand rolls back, a following unprotected demand is accepted.  A backup route
    past the 768-entry fallback.  Hub and clique samples with IMPACT_OVERFLOW on the backup.  Each against the round
    loop."""
    import dense_samples as ds
    from gnn_qot_estimation_b200 import ops
    m, _ = _model(cuda)
    f = (16, 10, 300000)
    ninf = -np.inf
    pair = (0, [([0], 1, f, ninf), ([1], 1, f, ninf)])
    for n, prot in ((254, [True, False]), (255, [True, False])):
        smp = _count_sample(n, 21)
        state = _state(smp, cuda)
        d = _demands([pair, (0, [([0], 1, f, ninf)])], cuda)
        r = m.forward_protection(state, d, _flags(prot, cuda), 0)
        ref, _, _ = _round_loop(m, smp, cuda, d, _flags(prot, cuda), 0, 0, True, None)
        torch.cuda.synchronize()
        _assert_same(r, ref)
        st = r.status.tolist()
        if n == 254:
            assert int(r.conn_id[0]) >= 0 and int(r.backup_conn_id[0]) >= 0
            assert st[1] & ops.PROV_FULL and int(r.conn_id[1]) == -1
        else:
            assert int(r.backup_status[0]) & ops.PROV_FULL and st[0] & ops.PROT_NO_BACKUP
            assert int(r.conn_id[0]) == -1 and int(r.conn_id[1]) >= 0 and (st[1] & ~ops.CAND_IMPACT_OVERFLOW) == 0
    # 254 lightpaths of 8 links x 3 slots on L = 64, Q = 97 (slot column 96 free): the backup on a 9-link route of 864
    # known channels takes the entry-list fallback
    b = _builder(64, 97, 11)
    for k in range(254):
        b.place(list(range(8 * (k // 32), 8 * (k // 32) + 8)), 3 * (k % 32), 3)
    g = _pack([b])
    gstate = _state(g, cuda, ds.HUB_THRESHOLD)
    d = _demands([(0, [([60], 1, f, ninf), (list(range(9)), 1, f, ninf)])], cuda)
    for policy, bound in ((0, None), (2, _node_bound(m, gstate, 0, True, 12, spread=0.2))):
        r = m.forward_protection(gstate, d, _flags([True], cuda), policy, 0, True, bound, 256)
        ref, _, _ = _round_loop(m, g, cuda, d, _flags([True], cuda), policy, 0, True, bound, 256, ds.HUB_THRESHOLD)
        torch.cuda.synchronize()
        _assert_same(r, ref)
        if policy == 0:
            assert int(r.backup_option[0]) == 1 and int(r.backup_q0[0]) == 96 and int(r.backup_n_impact[0]) > 0
    overflow = 0
    for smp, thr in ((ds.hub(7), ds.HUB_THRESHOLD), (ds.clique(8, n=200), ds.CLIQUE_THRESHOLD)):
        st = _state(smp, cuda, thr)
        L = smp["data"].shape[2]
        rng = np.random.default_rng(9)
        rows = [(0, [([0], 1, f, 0.2)] + [(sorted(rng.choice(np.arange(1, L), 2, replace=False).tolist()), 1, f, ninf)
                                          for _ in range(2)]) for _ in range(8)]
        d = _demands(rows, cuda)
        prot = _protect(8, cuda, 10, share=0.75)
        bound = _node_bound(m, st, 0, True, 10, spread=0.2)
        for policy, bnd in ((0, None), (2, bound)):
            r = m.forward_protection(st, d, prot, policy, 0, True, bnd, 4)
            ref, _, _ = _round_loop(m, smp, cuda, d, prot, policy, 0, True, bnd, 4, thr)
            torch.cuda.synchronize()
            _assert_same(r, ref)
            overflow += int((r.backup_status & ops.CAND_IMPACT_OVERFLOW != 0).sum())
    assert overflow > 0


# ------------------------------------------------------------------------------------------------ fp64
def test_vs_fp64_reference(cuda):
    """protection_ref on the fp64 oracle, following the kernel's choices: both searches' chosen own rows and impact
    rows at 1e-5, n_free of both, rollbacks and partner-less demands where the kernel has them."""
    from gnn_qot_estimation_b200 import ops, synthetic
    from protection_ref import PROT_NO_BACKUP, PROT_NO_PARTNER, protection_ref
    m, sd = _model(cuda)
    o = _oracle64(sd, cuda)
    smp = synthetic.network_status_samples(2, num_links=5, num_freqs=20, seed=61, spacing=0.05, max_lightpaths=8,
                                           super_channel_p=0.3)
    state = _state(smp, cuda)
    f1, f2 = (16, 40, 2000000), (64, 9, 80000)
    per = {0: [[([0], 1, f1, 0.1), ([1, 2], 2, f2, 0.2)], [([0], 1, f1, 0.1)], [([0, 3], 1, f2, -np.inf),
                                                                                ([4], 1, f1, -np.inf)],
               [([0], 2, f1, 0.15), ([4], 1, f2, 0.1), ([0, 4], 1, f1, -np.inf)]],
           1: [[([2], 1, f2, 0.1), ([3], 1, f2, -np.inf)], [([2, 3], 1, f1, -np.inf)], [([2], 1, f2, 0.3),
                                                                                          ([1, 4], 1, f1, 0.0)]]}
    pr = {0: [True, True, True, False], 1: [True, False, True]}
    rows = [(s, per[s][i]) for i in range(4) for s in (0, 1) if i < len(per[s])]
    prot = [pr[s][i] for i in range(4) for s in (0, 1) if i < len(per[s])]
    d = _demands(rows, cuda)
    for policy in (0, 2):
        r = m.forward_protection(state, d, _flags(prot, cuda), policy, 0, True, None, 256)
        torch.cuda.synchronize()
        for s in (0, 1):
            ks = [k for k, (ss, _) in enumerate(rows) if ss == s]
            follow = []
            for k in ks:
                placed = int(r.conn_id[k]) >= 0 or int(r.status[k]) & ops.PROT_NO_BACKUP
                work = (int(r.option[k]), int(r.q0[k])) if placed else None
                back = (int(r.backup_option[k]), int(r.backup_q0[k])) if int(r.backup_conn_id[k]) >= 0 else None
                follow.append((work, back))
            steps, _ = protection_ref(o, smp["data"][s], smp["freqs"], smp["lp_feat"], per[s], pr[s], policy,
                                      follow=follow, device=cuda)
            for k, st, (work, back) in zip(ks, steps, follow):
                assert int(r.n_free[k]) == st["n_free"]
                assert (int(r.status[k]) & PROT_NO_PARTNER) == st["status"] & PROT_NO_PARTNER
                assert (int(r.status[k]) & PROT_NO_BACKUP) == st["status"] & PROT_NO_BACKUP
                for w, tab, out, n_imp, ic, io in ((work, st["table"], r.out, r.n_impact, r.impact_conn,
                                                    r.impact_out),
                                                   (back, st["b_table"], r.backup_out, r.backup_n_impact,
                                                    r.backup_impact_conn, r.backup_impact_out)):
                    if w is None:
                        continue
                    row, imp, mg = tab[w]
                    assert mg >= -1e-5
                    torch.testing.assert_close(out[k].double().cpu(), row, rtol=RTOL, atol=ATOL)
                    n = int(n_imp[k])
                    assert n == len(imp) and set(ic[k, :n].tolist()) == set(imp)
                    if n:
                        torch.testing.assert_close(io[k, :n].double().cpu(),
                                                   torch.stack([imp[int(c)] for c in ic[k, :n].tolist()]),
                                                   rtol=RTOL, atol=ATOL)
                if work is not None and int(r.status[k]) & ops.PROT_NO_BACKUP == 0 and pr[s][ks.index(k)]:
                    assert int(r.backup_n_free[k]) == st["b_n_free"]


# ------------------------------------------------------------------------------------------------ commit
def test_commit(cuda):
    """commit_protection equals the round loop's final samples and state, field by field and bit for bit."""
    from gnn_qot_estimation_b200 import synthetic
    from gnn_qot_estimation_b200.to_graph import commit_protection
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(4, num_links=12, num_freqs=40, seed=71, super_channel_p=0.3)
    state = _state(smp, cuda)
    d = synthetic.lightpath_demands(smp, 6, options=(2, 4), seed=72, bound_range=(-1.0, 0.2)).to(cuda)
    prot = _protect(d.sample.shape[0], cuda, 73)
    r = m.forward_protection(state, d, prot, 2)
    data = torch.from_numpy(smp["data"]).to(cuda).contiguous()
    new = commit_protection(data, state, d, r)
    ref, rstate, rdata = _round_loop(m, smp, cuda, d, prot, 2, 0, True, None)
    torch.cuda.synchronize()
    _assert_same(r, ref)
    assert int((r.backup_conn_id >= 0).sum()) > 2
    assert torch.equal(data, rdata)
    for f in ("x", "edge_index", "ptr", "batch"):
        assert torch.equal(getattr(new.batch, f), getattr(rstate.batch, f)), f
    for f in ("rowptr", "conn_ids", "chan_node"):
        assert torch.equal(getattr(new, f), getattr(rstate, f)), f


# ------------------------------------------------------------------------------------------------ status, errors
def test_status_bits_and_c_groupings(cuda):
    """BAD_SAMPLE, BAD_PATH, BAD_STATE with empty backups; BAD_GROUPING through the C entry point for each
    malformation, the backup outputs empty; D = 0."""
    from gnn_qot_estimation_b200 import ops, synthetic
    from gnn_qot_estimation_b200.to_graph import LightpathDemands
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(3, num_links=8, num_freqs=32, seed=81)
    state = _state(smp, cuda)
    f = (16, 10, 300000)
    ninf = -np.inf
    two = [([0], 1, f, ninf), ([1], 1, f, ninf)]
    rows = [(5, two), (-1, two), (0, [([], 1, f, ninf)] + two), (0, [([9], 1, f, ninf)] + two),
            (0, [([0], 0, f, ninf)] + two), (0, two * 17), (1, two)]
    d = _demands(rows, cuda)
    r = m.forward_protection(state, d, torch.ones(len(rows), dtype=torch.bool, device=cuda), 0, max_impact=0)
    torch.cuda.synchronize()
    st = r.status.tolist()
    assert st[:2] == [ops.CAND_BAD_SAMPLE] * 2 and st[2:6] == [ops.CAND_BAD_PATH] * 4
    assert r.option.tolist()[:6] == [-1] * 6 and r.conn_id.tolist()[:6] == [-1] * 6
    assert int(r.backup_conn_id[6]) >= 0
    _empty_backup(SimpleNamespace(**{k: getattr(r, k)[:6] for k in r._fields}))
    bad = state._replace(chan_node=state.chan_node.clone())
    bad.chan_node[1, 0, :] = 0
    rb = m.forward_protection(bad, _demands([(1, two), (0, two)], cuda), _flags([True, True], cuda), 0)
    torch.cuda.synchronize()
    assert int(rb.status[0]) == ops.CAND_BAD_STATE and int(rb.status[1]) == 0 and int(rb.backup_conn_id[1]) >= 0
    e = LightpathDemands(d.sample[:0], d.opt_ptr[:1], d.link_ptr[:1], d.links[:0], d.width[:0], d.feat[:0],
                         d.own_bound[:0])
    assert m.forward_protection(state, e, _flags([], cuda), 0).status.numel() == 0
    g = _demands([(0, two), (1, two), (0, two)], cuda)
    i64 = lambda v: torch.tensor(v, dtype=torch.int64, device=cuda)
    pg = _flags([True, True, True], cuda)
    rc, ok = _c_call(m, state, g, i64([0, 2, 1]), i64([0, 2, 3, 3]), pg)
    assert rc == 0 and int(ok.status.max()) == 0
    for order, sp in (([2, 0, 1], [0, 2, 3, 3]), ([0, 1, 2], [0, 2, 3, 3]), ([0, 2, 1], [1, 2, 3, 3]),
                      ([0, 2, 1], [0, 2, 1, 3]), ([0, 2, 1], [0, 2, 2, 2]), ([0, 2, 7], [0, 2, 3, 3]),
                      ([0, 0, 1], [0, 2, 3, 3])):
        rc, res = _c_call(m, state, g, i64(order), i64(sp), pg)
        assert rc == 0
        assert res.status.tolist() == [ops.PROV_BAD_GROUPING] * 3, (order, sp)
        assert res.option.tolist() == [-1] * 3 and res.conn_id.tolist() == [-1] * 3
        _empty_backup(res)


def test_determinism_capture_and_errors(cuda):
    """Two calls and a CUDA-graph replay are bit-identical; the state is not modified; the host error paths, protect's
    dtype, shape and device among them."""
    from gnn_qot_estimation_b200 import synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(8, num_links=16, num_freqs=48, seed=91, super_channel_p=0.3)
    state = _state(smp, cuda)
    d = synthetic.lightpath_demands(smp, 8, options=(2, 4), seed=92).to(cuda)
    D = int(d.sample.shape[0])
    prot = _protect(D, cuda, 94)
    bound = _node_bound(m, state, 0, True, 93)
    cn = state.chan_node.clone()
    a = m.forward_protection(state, d, prot, 2, 0, True, bound)
    b = m.forward_protection(state, d, prot, 2, 0, True, bound)
    torch.cuda.synchronize()
    _assert_same(a, b)
    assert torch.equal(state.chan_node, cn)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        m.forward_protection(state, d, prot, 2, 0, True, bound)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c = m.forward_protection(state, d, prot, 2, 0, True, bound)
    g.replay()
    torch.cuda.synchronize()
    _assert_same(a, c)
    with pytest.raises(TypeError):
        m.forward_protection(state, d, prot.to(torch.uint8), 0)
    with pytest.raises(ValueError):
        m.forward_protection(state, d, prot[:-1], 0)
    with pytest.raises(RuntimeError):
        m.forward_protection(state, d, prot.cpu(), 0)
    with pytest.raises(ValueError):
        m.forward_protection(state, d, prot, 7)
    with pytest.raises(ValueError):
        m.forward_protection(state, d, prot, 0, bound=bound[:-1])
    m.train()
    with pytest.raises(RuntimeError):
        m.forward_protection(state, d, prot, 0)
    m.eval()

