"""GPU checks of LightpathGNN's failure restoration (qot_lightpath_restore through LightpathGNN.forward_restoration):
bit-identity of every cut lightpath's outputs with the expansion through forward_traffic on replicated samples
(tests/restoration_ref.py), the end rows against forward_every_node on the committed end state, end_margin / n_below
against the kernel's own end rows, hand-built edge cases, capacity samples, parity with the fp64 literal reference,
every status bit, the state left unchanged, determinism, CUDA-graph replay and the error paths."""
import ctypes as C

import numpy as np
import pytest
import torch

from test_lightpath_candidates_gpu import ATOL, RTOL
from test_lightpath_provision_gpu import _builder, _model, _node_bound, _oracle64, _pack, _same, _state

pytestmark = pytest.mark.gpu
CUT_FIELDS = ("cut_node", "option", "q0", "out", "margin", "n_free", "n_feasible", "cut_status", "status", "n_cut",
              "n_restored")


def _fail(rows, dev):
    """[(sample, [links])] -> LightpathFailures on dev."""
    from gnn_qot_estimation_b200.to_graph import LightpathFailures
    lptr = np.cumsum([0] + [len(l) for _, l in rows])
    return LightpathFailures(torch.tensor([s for s, _ in rows], dtype=torch.int64, device=dev),
                             torch.tensor(lptr, dtype=torch.int64, device=dev),
                             torch.tensor([x for _, l in rows for x in l], dtype=torch.int32, device=dev))


def _cat(a, b):
    from gnn_qot_estimation_b200.to_graph import LightpathFailures
    n = int(a.link_ptr[-1])
    return LightpathFailures(torch.cat([a.sample, b.sample]), torch.cat([a.link_ptr, b.link_ptr[1:] + n]),
                             torch.cat([a.links, b.links]))


def _end_consistent(r, state, options, fails, bound, metric, maximize):
    """end_margin / n_below recomputed from the kernel's own end rows: each row's margin in fp32 against bound[node]
    for a survivor and the chosen option's own_bound for a restored lightpath."""
    from types import SimpleNamespace
    ptr, conn = state.batch.ptr.tolist(), state.conn_ids.tolist()
    optr, own = options.opt_ptr.tolist(), options.own_bound.cpu()
    r = SimpleNamespace(**{k: getattr(r, k).cpu() for k in r._fields})
    bound = None if bound is None else bound.cpu()
    for f in range(r.status.shape[0]):
        if int(r.status[f]) & ~(1 << 15):
            assert int(r.n_cut[f]) == 0 and int(r.n_below[f]) == 0 and bool(torch.isnan(r.end_margin[f]))
            continue
        nt = int((r.end_conn[f] >= 0).sum())
        if bound is None or nt == 0:
            assert bool(torch.isnan(r.end_margin[f])) and (bound is not None or int(r.n_below[f]) == 0)
            continue
        s = int(fails.sample[f])
        rest = {}                                       # conn -> own_bound of the restored lightpaths
        for i in range(min(int(r.n_cut[f]), r.cut_node.shape[1])):
            v, o = int(r.cut_node[f, i]), int(r.option[f, i])
            if o >= 0 and not int(r.cut_status[f, i]) & 512:
                rest[conn[v]] = float(own[optr[v] + o])
        b = []
        for c in r.end_conn[f, :nt].tolist():
            if c in rest:
                b.append(rest[c])
            else:
                v = next(u for u in range(ptr[s], ptr[s + 1]) if conn[u] == c)
                b.append(float(bound[v]))
        b = torch.tensor(b, dtype=torch.float32)
        v = r.end_out[f, :nt, metric]
        m = v - b if maximize else b - v
        below = int((~(m >= 0)).sum())
        assert int(r.n_below[f]) == below
        want = float("nan") if bool(torch.isnan(m).any()) else float(m.min())
        got = float(r.end_margin[f])
        assert (np.isnan(want) and np.isnan(got)) or got == want


def _check(m, smp, state, options, fails, policy, metric=0, maximize=True, bound=None, max_cut=64):
    """forward_restoration against expand(): every per-cut and count output bit for bit, end_conn exactly, end_out at
    the candidate tolerance; returns (result, how many end rows were bit-identical, end rows)."""
    from restoration_ref import expand
    r = m.forward_restoration(state, options, fails, policy, metric, maximize, bound, max_cut, return_end=True)
    ref = expand(m, smp, state, options, fails, policy, metric, maximize, bound, max_cut)
    torch.cuda.synchronize()
    for f in CUT_FIELDS:
        assert _same(getattr(r, f), getattr(ref, f)), f
    assert _same(r.end_conn, ref.end_conn)
    torch.testing.assert_close(r.end_out, ref.end_out, rtol=RTOL, atol=ATOL, equal_nan=True)
    live = r.end_conn >= 0
    same = int((r.end_out[live] == ref.end_out[live]).all(1).sum())
    _end_consistent(r, state, options, fails, bound, metric, maximize)
    return r, same, int(live.sum())


# ------------------------------------------------------------------------------------------------ expansion
def test_bit_identity_with_expand(cuda):
    """Every policy, both senses, each metric column, with and without a bound, on every single-link failure of 5
    samples (consecutive scenarios of one sample run on different blocks at once) and on shared-risk groups."""
    from gnn_qot_estimation_b200 import synthetic
    from gnn_qot_estimation_b200.to_graph import single_link_failures
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(5, num_links=12, num_freqs=40, seed=41, super_channel_p=0.3)
    state = _state(smp, cuda)
    options = synthetic.lightpath_restoration_options(smp, state, (1, 4), seed=42, bound_range=(0.0, 0.5)).to(cuda)
    fails = _cat(single_link_failures(state), _fail([(0, [0, 1]), (1, [2, 5, 7]), (3, [11, 0]), (4, [3, 4, 5, 6])],
                                                    cuda))
    assert int(fails.sample.shape[0]) > 40
    restored = cut = same = rows = 0
    for metric, mx in ((0, True), (1, True), (2, False), (0, False)):
        for bound in (None, _node_bound(m, state, metric, mx, 43 + metric, spread=0.05)):
            for policy in (0, 1, 2):
                r, sm, n = _check(m, smp, state, options, fails, policy, metric, mx, bound)
                restored += int(r.n_restored.sum())
                cut += int(r.n_cut.sum())
                same += sm
                rows += n
                assert int((r.cut_status & 8192 != 0).sum()) > 0
    assert restored > 200 and cut > restored
    print(f"end rows bit-identical to forward_every_node: {same} of {rows}")


# ------------------------------------------------------------------------------------------------ hand-built
def test_edge_cases(cuda):
    """A link with no lightpath (nothing cut; the end rows are the state's every-node rows), a failure of every link
    (every lightpath cut), REST_NO_OPTION, REST_CUT_OVERFLOW with max_cut = 2 (all still restored and counted)."""
    from gnn_qot_estimation_b200 import ops, synthetic
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(2, num_links=10, num_freqs=40, seed=5, max_lightpaths=12)
    state = _state(smp, cuda)
    L = state.L
    smp["data"][0][:, L - 1] = 0.0                      # sample 0 leaves its last link unused
    state = _state(smp, cuda)
    empty = L - 1
    options = synthetic.lightpath_restoration_options(smp, state, (2, 4), seed=6).to(cuda)
    fails = _fail([(0, [empty]), (0, list(range(L))), (1, list(range(L))), (1, [0])], cuda)
    every = m.forward_every_node(state.batch)
    for policy in (0, 2):
        bound = _node_bound(m, state, 0, True, 7, spread=0.1) if policy == 2 else None
        r, _, _ = _check(m, smp, state, options, fails, policy, 0, True, bound)
        n0, n1 = int(state.batch.ptr[0]), int(state.batch.ptr[1])
        assert int(r.n_cut[0]) == 0 and int(r.n_restored[0]) == 0 and int(r.status[0]) == 0
        assert r.end_conn[0, :n1 - n0].tolist() == state.conn_ids[n0:n1].tolist()
        torch.testing.assert_close(r.end_out[0, :n1 - n0], every[n0:n1], rtol=RTOL, atol=ATOL)
        assert int(r.n_cut[1]) == n1 - n0 and int(r.n_restored[1]) == 0                # every link failed
        assert bool((r.cut_status[1, :n1 - n0] == ops.REST_NO_OPTION).all())
        assert bool((r.end_conn[1] == -1).all()) and bool(torch.isnan(r.end_out[1]).all())
    # max_cut = 2: the first two reported, every one restored and counted
    r2, _, _ = _check(m, smp, state, options, fails, 0, max_cut=2)
    full = m.forward_restoration(state, options, fails, 0, max_cut=64)
    assert int(r2.status[1]) & ops.REST_CUT_OVERFLOW
    assert r2.n_restored.tolist() == full.n_restored.tolist() and r2.n_cut.tolist() == full.n_cut.tolist()
    for f in ("option", "q0", "cut_status", "cut_node"):
        assert _same(getattr(r2, f), getattr(full, f)[:, :2]), f


def test_capacity(cuda):
    """PROV_FULL: 254 lightpaths of 8 links x 3 slots (6 096 channels); failing link 0 cuts 32 of them, whose only
    surviving option is a 16-link, 3-wide route (48 channels against the 24 freed each): the 18th does not fit.  That
    route holds 9 x 96 channels of known lightpaths, past the 768-entry list.  Then the 256-lightpath, hub and clique
    samples on every single-link failure."""
    import dense_samples as ds
    from gnn_qot_estimation_b200 import ops, synthetic
    from gnn_qot_estimation_b200.to_graph import LightpathDemands, single_link_failures
    m, _ = _model(cuda)
    b = _builder(64, 200, 11)
    for k in range(254):
        b.place(list(range(8 * (k // 32), 8 * (k // 32) + 8)), 3 * (k % 32), 3)
    g = _pack([b])
    gs = _state(g, cuda, ds.HUB_THRESHOLD)
    N = int(gs.batch.x.shape[0])
    f = [16.0, 10.0, 300000.0]
    own = [sorted(set(torch.nonzero((gs.chan_node[0] == v).any(1)).flatten().tolist())) for v in range(N)]
    routes = [[own[v], list(range(1, 17))] for v in range(N)]
    lptr = np.cumsum([0] + [len(x) for r_ in routes for x in r_])
    options = LightpathDemands(torch.zeros(N, dtype=torch.int64), torch.arange(0, 2 * N + 1, 2),
                               torch.tensor(lptr), torch.tensor([l for r_ in routes for x in r_ for l in x],
                                                                dtype=torch.int32),
                               torch.tensor([3, 3] * N, dtype=torch.int32), torch.tensor([f] * (2 * N)),
                               torch.full((2 * N,), -np.inf)).to(cuda)
    fails = _fail([(0, [0])], cuda)
    for policy, bound in ((0, None), (2, _node_bound(m, gs, 0, True, 12, spread=0.2))):
        r, _, _ = _check(m, g, gs, options, fails, policy, 0, True, bound)
        assert int(r.n_cut[0]) == 32
        if policy == 0:
            assert int(r.n_restored[0]) == 17 and bool((r.option[0, :32] == 1).all())
            assert int(((r.cut_status[0, :32] & ops.PROV_FULL) != 0).sum()) == 15
    # the capacity samples, every single-link failure (a subset of links for the dense ones)
    for smp, thr in ((ds.full_sparse(3, counts=(256,)), ds.HUB_THRESHOLD), (ds.hub(7), ds.HUB_THRESHOLD),
                     (ds.clique(8, n=200), ds.CLIQUE_THRESHOLD)):
        st = _state(smp, cuda, thr)
        opts = synthetic.lightpath_restoration_options(smp, st, (1, 4), seed=9).to(cuda)
        fl = single_link_failures(st)
        keep = torch.arange(0, int(fl.sample.shape[0]), max(1, int(fl.sample.shape[0]) // 12), device=cuda)
        fl = _fail([(int(fl.sample[k]), [int(fl.links[k])]) for k in keep.tolist()], cuda)
        for policy, bb in ((0, None), (2, _node_bound(m, st, 0, True, 10, spread=0.2))):
            r, _, _ = _check(m, smp, st, opts, fl, policy, 0, True, bb)
            assert int(r.n_cut.sum()) > 0


# ------------------------------------------------------------------------------------------------ fp64
def test_vs_fp64_reference(cuda):
    """restoration_ref on the fp64 oracle, following the kernel's choices: every restored lightpath's own row and
    every end row at 1e-5, the cut set and the end conn_ids."""
    from gnn_qot_estimation_b200 import synthetic
    from restoration_ref import _all_opts, restoration_ref
    m, sd = _model(cuda)
    o = _oracle64(sd, cuda)
    smp = synthetic.network_status_samples(1, num_links=5, num_freqs=20, seed=61, spacing=0.05, max_lightpaths=8,
                                           super_channel_p=0.3)
    state = _state(smp, cuda)
    options = synthetic.lightpath_restoration_options(smp, state, (2, 4), seed=62, bound_range=(-1.0, -0.5)).to(cuda)
    conn = state.conn_ids.tolist()
    every = _all_opts(options)
    checked = 0
    for failed in ([0], [1], [2, 3]):
        r = m.forward_restoration(state, options, _fail([(0, failed)], cuda), 0, return_end=True)
        torch.cuda.synchronize()
        nc = int(r.n_cut[0])
        cut_k = r.cut_node[0, :nc].tolist()
        follow = []
        for i, v in enumerate(cut_k):
            keep = [j for j, (links, *_) in enumerate(every[v]) if not set(links) & set(failed)]
            if not keep:
                continue
            oi = int(r.option[0, i])
            follow.append((keep.index(oi), int(r.q0[0, i])) if oi >= 0 and int(r.cut_status[0, i]) == 0 else None)
        cut, steps, keep, final, (st, rows) = restoration_ref(o, smp["data"][0], smp["freqs"], smp["lp_feat"], conn,
                                                              every, failed, 0, follow=follow, device=cuda)
        assert cut == cut_k
        d = 0
        for i, v in enumerate(cut_k):
            if int(r.cut_status[0, i]) & 8192:
                continue
            if follow[d] is not None:
                row, _, _ = steps[d]["table"][follow[d]]
                torch.testing.assert_close(r.out[0, i].double().cpu(), row, rtol=RTOL, atol=ATOL)
                checked += 1
            d += 1
        n = int(st.batch.ptr[1])
        torch.testing.assert_close(r.end_out[0, :n].double(), rows, rtol=RTOL, atol=ATOL)
        assert int((r.end_conn[0] >= 0).sum()) == n
    assert checked > 0


# ------------------------------------------------------------------------------------------------ status, errors
def _c_call(m, state, options, fails_struct, max_cut=4):
    from gnn_qot_estimation_b200 import _lib, ops
    from gnn_qot_estimation_b200.ops import _demands_desc, _state_desc, ptr, stream
    dev = state.batch.x.device
    F = fails_struct.F
    i32 = lambda *s: torch.full(s, 99, dtype=torch.int32, device=dev)
    res = ops.RestorationQoT(torch.full((F, max_cut), 99, dtype=torch.int64, device=dev), i32(F, max_cut),
                             i32(F, max_cut), torch.zeros(F, max_cut, 3, device=dev), torch.zeros(F, max_cut, device=dev),
                             i32(F, max_cut), i32(F, max_cut), i32(F, max_cut), i32(F), i32(F), i32(F),
                             torch.zeros(F, device=dev), i32(F), torch.full((F, 256), 99, dtype=torch.int64, device=dev),
                             torch.zeros(F, 256, 3, device=dev))
    keep = []
    D, P = int(options.sample.shape[0]), int(options.width.shape[0])
    cw = torch.empty(3, state.L, state.Q, dtype=torch.int32, device=dev)
    rc = _lib.lib().qot_lightpath_restore(
        C.byref(_state_desc(state, keep)), C.byref(_demands_desc(options, D, P, keep)), C.byref(fails_struct), 0, 0, 1,
        None, ptr(m.prepared()), 1, max_cut, ptr(cw), None, 3, *(ptr(x) for x in res), stream())
    torch.cuda.synchronize()
    return rc, res


def test_status_bits(cuda):
    """Scenario bits: a sample outside [0, S), an empty link set, a link outside [0, L), a malformed link_ptr through
    the C entry point, an inconsistent state; per cut lightpath: options of another sample, a bad option route, width
    or count.  Nothing is done with a scenario-level bit."""
    from gnn_qot_estimation_b200 import _lib, ops, synthetic
    from gnn_qot_estimation_b200.to_graph import LightpathDemands
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(3, num_links=8, num_freqs=32, seed=81)
    state = _state(smp, cuda)
    options = synthetic.lightpath_restoration_options(smp, state, (1, 3), seed=82).to(cuda)
    fails = _fail([(5, [0]), (-1, [0]), (0, []), (0, [8]), (0, [-1]), (0, [0]), (1, [1, 1])], cuda)
    r = m.forward_restoration(state, options, fails, 0, return_end=True)
    torch.cuda.synchronize()
    assert r.status.tolist()[:5] == [ops.CAND_BAD_SAMPLE] * 2 + [ops.REST_BAD_FAILURE] * 3
    assert r.status.tolist()[5:] == [0, 0] and int(r.n_cut[5]) > 0
    for f in range(5):
        assert int(r.n_cut[f]) == 0 and int(r.n_restored[f]) == 0 and bool((r.cut_node[f] == -1).all())
        assert bool(torch.isnan(r.out[f]).all()) and bool((r.end_conn[f] == -1).all())
        assert bool(torch.isnan(r.end_out[f]).all())
    # a duplicated link in a group changes nothing
    one = m.forward_restoration(state, options, _fail([(1, [1])], cuda), 0, return_end=True)
    for f in CUT_FIELDS[:-3] + ("end_conn", "end_out"):
        assert _same(getattr(r, f)[6], getattr(one, f)[0]), f
    # malformed link_ptr through the C ABI: decreasing, past n_links, negative
    i64 = lambda v: torch.tensor(v, dtype=torch.int64, device=cuda)
    smp_t, links = i64([0, 0, 0]), torch.tensor([0, 1], dtype=torch.int32, device=cuda)
    for lp in ([0, 2, 1, 2], [0, 1, 2, 3], [-1, 1, 1, 2]):
        lpt = i64(lp)
        fs = _lib.QotLpFailures(3, 2, smp_t.data_ptr(), lpt.data_ptr(), links.data_ptr())
        rc, res = _c_call(m, state, options, fs)
        assert rc == 0
        bad = [k for k in range(3) if not (0 <= lp[k] < lp[k + 1] <= 2)]
        assert bad and all(int(res.status[k]) == ops.REST_BAD_FAILURE for k in bad), lp
        assert all(int(res.n_cut[k]) == 0 and bool((res.end_conn[k] == -1).all()) for k in bad)
    # an inconsistent state: node n0's out-run of sample 1 ends before it starts
    bad = state._replace(rowptr=state.rowptr.clone())
    n0 = int(state.batch.ptr[1])
    bad.rowptr[n0 + 1] = bad.rowptr[n0] - 1
    rb = m.forward_restoration(bad, options, _fail([(1, [0]), (0, [0])], cuda), 0)
    torch.cuda.synchronize()
    assert int(rb.status[0]) == ops.CAND_BAD_STATE and int(rb.n_cut[0]) == 0 and int(rb.status[1]) == 0
    # per cut lightpath: options of another sample, a link outside [0, L), a zero width, 33 options
    N = int(state.batch.x.shape[0])
    cut0 = torch.nonzero((state.chan_node[0, 0] >= 0)).flatten()
    vs = sorted(set(state.chan_node[0, 0, cut0].tolist()))
    assert len(vs) >= 1
    v = vs[0]
    rows = [None if u == v else [([2], 1)] for u in range(N)]

    def with_opts(u_opts, u_sample=None):
        opts = [o_ if o_ is not None else u_opts for o_ in rows]
        flat = [x for o_ in opts for x in o_]
        smp_ = state.batch.batch.to(torch.int64).clone()
        if u_sample is not None:
            smp_[v] = u_sample
        return LightpathDemands(smp_, torch.tensor(np.cumsum([0] + [len(o_) for o_ in opts])),
                                torch.tensor(np.cumsum([0] + [len(x[0]) for x in flat])),
                                torch.tensor([l for x in flat for l in x[0]], dtype=torch.int32),
                                torch.tensor([x[1] for x in flat], dtype=torch.int32),
                                torch.tensor([[16.0, 10.0, 3e5]] * len(flat)), torch.full((len(flat),), -np.inf)).to(cuda)
    cases = [(with_opts([([3], 1)], u_sample=1), ops.CAND_BAD_SAMPLE),
             (with_opts([([3], 1), ([8], 1)]), ops.CAND_BAD_PATH),           # a link outside [0, L)
             (with_opts([([3], 0)]), ops.CAND_BAD_PATH),                     # width 0
             (with_opts([([3], 1)] * 33), ops.CAND_BAD_PATH),                # 33 options
             (with_opts([([0, 3], 1)]), ops.REST_NO_OPTION),                 # crosses the failure
             (with_opts([]), ops.REST_NO_OPTION)]                            # no option
    for o_, bit in cases:
        r = m.forward_restoration(state, o_, _fail([(0, [0])], cuda), 0)
        torch.cuda.synchronize()
        i = r.cut_node[0].tolist().index(v)
        assert int(r.cut_status[0, i]) == bit and int(r.option[0, i]) == -1 and int(r.n_free[0, i]) == 0
        assert int(r.status[0]) == 0


def test_state_unchanged_determinism_capture_and_errors(cuda):
    from gnn_qot_estimation_b200 import synthetic
    from gnn_qot_estimation_b200.to_graph import single_link_failures
    m, _ = _model(cuda)
    smp = synthetic.network_status_samples(4, num_links=12, num_freqs=40, seed=91, super_channel_p=0.3)
    state = _state(smp, cuda)
    options = synthetic.lightpath_restoration_options(smp, state, seed=92).to(cuda)
    fails = single_link_failures(state)
    bound = _node_bound(m, state, 0, True, 93)
    cn = state.chan_node.clone()
    a = m.forward_restoration(state, options, fails, 2, 0, True, bound, return_end=True)
    b = m.forward_restoration(state, options, fails, 2, 0, True, bound, return_end=True)
    torch.cuda.synchronize()
    assert torch.equal(state.chan_node, cn)
    for f in a._fields:
        assert _same(getattr(a, f), getattr(b, f)), f
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        m.forward_restoration(state, options, fails, 2, 0, True, bound, return_end=True)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c = m.forward_restoration(state, options, fails, 2, 0, True, bound, return_end=True)
    g.replay()
    torch.cuda.synchronize()
    for f in a._fields:
        assert _same(getattr(a, f), getattr(c, f)), f
    with pytest.raises(ValueError):
        m.forward_restoration(state, options, fails, 7)
    with pytest.raises(ValueError):
        m.forward_restoration(state, options, fails._replace(link_ptr=fails.link_ptr[:-1]), 0)
    with pytest.raises(TypeError):
        m.forward_restoration(state, options, fails._replace(links=fails.links.long()), 0)
    with pytest.raises(RuntimeError):
        m.forward_restoration(state, options, fails.to("cpu"), 0)
    with pytest.raises(ValueError):
        m.forward_restoration(state, options._replace(sample=options.sample[:-1], opt_ptr=options.opt_ptr[:-1]),
                              fails, 0)
    with pytest.raises(ValueError):
        m.forward_restoration(state, options, fails, 0, max_cut=-1)
    with pytest.raises(ValueError):
        m.forward_restoration(state, options, fails, 0, bound=bound[:-1])
    m.train()
    with pytest.raises(RuntimeError):
        m.forward_restoration(state, options, fails, 0)
    m.eval()
    e = m.forward_restoration(state, options, fails._replace(sample=fails.sample[:0], link_ptr=fails.link_ptr[:1]), 0)
    assert e.status.numel() == 0
