"""CPU checks of failure restoration's host side: the C ABI declares and binds qot_lightpath_restore, the literal
reference (tests/restoration_ref.py) is traffic_ref on the releases and filtered demands, single_link_failures lists
what numpy finds, and synthetic.lightpath_restoration_options draws what it documents."""
import ctypes as C
import re
from types import SimpleNamespace

import numpy as np
import torch

from test_lightpath_provision_cpu import _oracle, _sample
from test_lightpath_reconfig_cpu import HEADER, _header_arity


def test_header_declares_and_ctypes_binds_restore():
    from gnn_qot_estimation_b200 import _lib, ops
    name = "qot_lightpath_restore"
    args = _lib.SIGNATURES[name][1]
    assert len(args) == _header_arity(name) == 29
    # the state, the options as demands, the failures
    assert args[:3] == [C.POINTER(_lib.QotLpState), C.POINTER(_lib.QotLpDemands), C.POINTER(_lib.QotLpFailures)]
    assert args[3:6] == [C.c_int32] * 3 and args[12] == C.c_int32          # policy, metric, maximize; n_blocks
    assert C.sizeof(_lib.QotLpFailures) == 40
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    body = re.search(r"typedef struct \{([^}]*)\}\s*qot_lp_failures_t\s*;", text).group(1)
    names = [d.strip().split()[-1].lstrip("*") for d in body.split(";") if d.strip()]
    assert names == [f for f, _ in _lib.QotLpFailures._fields_]
    for bit, v in (("QOT_REST_NO_OPTION", ops.REST_NO_OPTION), ("QOT_REST_BAD_FAILURE", ops.REST_BAD_FAILURE),
                   ("QOT_REST_CUT_OVERFLOW", ops.REST_CUT_OVERFLOW)):
        assert int(re.search(r"#define " + bit + r"\s+(\d+)", HEADER.read_text()).group(1)) == v
    assert (ops.REST_NO_OPTION, ops.REST_BAD_FAILURE, ops.REST_CUT_OVERFLOW) == (8192, 16384, 32768)
    assert ops.RestorationQoT._fields[:8] == ("cut_node", "option", "q0", "out", "margin", "n_free", "n_feasible",
                                              "cut_status")


def test_restore_rejects_bad_arguments_without_a_gpu():
    """QOT_E_BADARG with a message naming the query: NULL descriptors, n_blocks < 1, options not one per node."""
    from gnn_qot_estimation_b200 import _lib
    L = _lib.lib()
    cfg = _lib.QotLpGraphCfg(F=10, L=4, Q=16, T=3, i_conn=0)
    st = _lib.QotLpState(cfg, 1, 3, 0)
    d = _lib.QotLpDemands(3, 0, 0)
    fl = _lib.QotLpFailures(1, 1)
    prep = C.create_string_buffer(64)
    aligned = (C.addressof(prep) + 15) & ~15
    call = lambda s, o, f, n_blocks=1: L.qot_lightpath_restore(s, o, f, 0, 0, 1, None, aligned, 1, 4, None, None,
                                                                n_blocks, *([None] * 15), None)
    assert call(None, C.byref(d), C.byref(fl)) != 0
    assert b"qot_lightpath_restore" in L.qot_last_error()
    assert call(C.byref(st), C.byref(d), None) != 0
    assert b"failures" in L.qot_last_error()
    assert call(C.byref(st), C.byref(d), C.byref(fl), 0) != 0
    assert call(C.byref(st), C.byref(_lib.QotLpDemands(2, 0, 0)), C.byref(fl)) != 0
    assert b"one demand per node" in L.qot_last_error()


def _opts(links_list, f=(16, 10, 300000), ob=-np.inf):
    return [(links, 1, f, ob) for links in links_list]


def test_restoration_ref_is_traffic_ref_on_the_sequence():
    """The literal reference is traffic_ref on (the cut lightpaths released, then their filtered options), and its cut
    set is every lightpath with a channel on a failed link: a single link and a two-link group, an option list that
    loses its first route, one that keeps all and one that loses all (no demand)."""
    from restoration_ref import cut_set, restoration_ref
    from traffic_ref import traffic_ref
    o = _oracle()
    smp = _sample()
    s0, freqs, lp_feat = smp["data"][0], smp["freqs"], smp["lp_feat"]
    fi = {k: i for i, k in enumerate(lp_feat)}
    cid = np.trunc(s0[fi["conn_id"]]).astype(int)
    occ = np.any(s0 != 0, axis=0)
    conns = sorted(set(cid[occ].tolist()))
    first = {c: min((l * s0.shape[2] + q) for l, q in zip(*np.nonzero(occ & (cid == c)))) for c in conns}
    conn_of = sorted(conns, key=lambda c: first[c])                  # node order: first channel
    opts_of = [_opts([[0], [1], [2, 3]]) for _ in conn_of]
    for failed in ([0], [1, 3]):
        on = {c for c in conns if np.any(occ[failed] & (cid[failed] == c))}
        assert cut_set(s0, lp_feat, failed) == on and on
        cut, steps, keep, final, end = restoration_ref(o, s0, freqs, lp_feat, conn_of, opts_of, failed, 0, end=False)
        assert end is None and cut == [i for i, c in enumerate(conn_of) if c in on]
        want = [k for k, (links, *_) in enumerate(opts_of[0]) if not set(links) & set(failed)]
        assert keep == [want] * len(cut)
        seq = [("r", conn_of[i]) for i in cut] + [("d", [opts_of[i][k] for k in want]) for i in cut]
        ref, rfinal = traffic_ref(o, s0, freqs, lp_feat, seq, 0)
        assert np.array_equal(final, rfinal)
        assert [(x["choice"], x["n_free"], x["n_feasible"]) for x in steps] == \
               [(x["choice"], x["n_free"], x["n_feasible"]) for x in ref[len(cut):]]
        assert all(x["conn"] is not None for x in ref[:len(cut)])
    # every option crosses the failure: the cut lightpaths are released and nothing is placed
    cut, steps, keep, final, _ = restoration_ref(o, s0, freqs, lp_feat, conn_of, [_opts([[0]])] * len(conn_of), [0],
                                                 0, end=False)
    assert cut and steps == [] and keep == []
    assert not np.any(np.isin(np.trunc(final[fi["conn_id"]]).astype(int)[np.any(final != 0, axis=0)],
                              [conn_of[i] for i in cut]))


def test_single_link_failures_matches_numpy():
    from gnn_qot_estimation_b200.to_graph import single_link_failures
    g = torch.Generator().manual_seed(3)
    S, L, Q = 4, 7, 9
    chan = torch.randint(-1, 5, (S, L, Q), generator=g, dtype=torch.int32)
    chan[chan == 4] = torch.iinfo(torch.int32).min                 # a lightpath the state does not know
    chan[2] = -1                                                   # an empty sample
    f = single_link_failures(SimpleNamespace(chan_node=chan, S=S, L=L, Q=Q))
    c = chan.numpy()
    want = [(s, l) for s in range(S) for l in range(L) if np.any(c[s, l] >= 0)]
    assert list(zip(f.sample.tolist(), f.links.tolist())) == want
    assert f.link_ptr.tolist() == list(range(len(want) + 1))
    assert f.sample.dtype == torch.int64 and f.links.dtype == torch.int32 and f.link_ptr.dtype == torch.int64


def test_synthetic_restoration_options():
    """One demand per node, in the node's sample; option 0 is the lightpath's current route (the links it occupies)
    and width with its own features; the count in range; deterministic under a seed."""
    from gnn_qot_estimation_b200 import synthetic
    smp = synthetic.network_status_samples(3, num_links=10, num_freqs=24, seed=5, super_channel_p=0.4)
    data = smp["data"]
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    # a host stand-in for the state: nodes by first channel, chan_node from the raw samples
    S, _, L, Q = data.shape
    chan = np.full((S, L, Q), -1, dtype=np.int32)
    ptr, conns, n0 = [0], [], 0
    for s in range(S):
        cid = np.trunc(data[s, fi["conn_id"]]).astype(int)
        occ = np.any(data[s] != 0, axis=0)
        cs = sorted(set(cid[occ].tolist()), key=lambda c: np.flatnonzero((occ & (cid == c)).ravel())[0])
        for k, c in enumerate(cs):
            chan[s][occ & (cid == c)] = n0 + k
        n0 += len(cs)
        ptr.append(n0)
        conns += cs
    state = SimpleNamespace(chan_node=torch.from_numpy(chan), S=S, batch=SimpleNamespace(ptr=torch.tensor(ptr)))
    o = synthetic.lightpath_restoration_options(smp, state, options=(2, 5), seed=7)
    assert o.sample.tolist() == [s for s in range(S) for _ in range(ptr[s], ptr[s + 1])]
    optr, lptr = o.opt_ptr.tolist(), o.link_ptr.tolist()
    for s in range(S):
        for v in range(ptr[s], ptr[s + 1]):
            assert 2 <= optr[v + 1] - optr[v] <= 5
            p = optr[v]
            ll, qq = np.nonzero(chan[s] == v)
            assert o.links[lptr[p]:lptr[p + 1]].tolist() == sorted(set(ll.tolist()))
            assert int(o.width[p]) == int((ll == ll.min()).sum())
            assert o.feat[p].tolist() == [float(data[s, fi[n], ll[0], qq[0]]) for n in ("mod_order", "num_spans",
                                                                                            "path_len")]
    o2 = synthetic.lightpath_restoration_options(smp, state, options=(2, 5), seed=7)
    assert all(torch.equal(a, b) for a, b in zip(o, o2))
    o3 = synthetic.lightpath_restoration_options(smp, state, options=(2, 5), seed=8)
    assert not torch.equal(o.width, o3.width) or not torch.equal(o.opt_ptr, o3.opt_ptr)
