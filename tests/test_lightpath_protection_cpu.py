"""CPU checks of protected provisioning's host side: the C ABI declares and binds qot_lightpath_protect, the entry
point refuses malformed arguments without a GPU, the literal reference (tests/protection_ref.py) is provision_ref when
nothing is protected, its option filters are set disjointness, and the round loop's conn_id bookkeeping survives a
rollback."""
import ctypes as C
import re

import numpy as np
import torch

from test_lightpath_provision_cpu import _oracle, _sample
from test_lightpath_reconfig_cpu import HEADER, _header_arity


def test_header_declares_and_ctypes_binds_protect():
    from gnn_qot_estimation_b200 import _lib, ops
    name = "qot_lightpath_protect"
    args = _lib.SIGNATURES[name][1]
    assert len(args) == _header_arity(name) == 37
    # qot_lightpath_provision's arguments but the stream, then protect and the eleven backup outputs
    assert args[:24] == _lib.SIGNATURES["qot_lightpath_provision"][1][:24]
    assert args[24:] == [C.c_void_p] * 13
    text = HEADER.read_text()
    for bit, v in (("QOT_PROT_NO_PARTNER", ops.PROT_NO_PARTNER), ("QOT_PROT_NO_BACKUP", ops.PROT_NO_BACKUP)):
        assert int(re.search(r"#define " + bit + r"\s+(\d+)", text).group(1)) == v
    assert (ops.PROT_NO_PARTNER, ops.PROT_NO_BACKUP) == (65536, 131072)
    # no other status bit of the header takes these values
    values = [int(v) for n, v in re.findall(r"#define (QOT_[A-Z_]+) (\d+)\s*/\*", text) if "PROT" not in n]
    assert 65536 not in values and 131072 not in values
    want = ops.ProvisionQoT._fields + tuple("backup_" + f for f in ops.ProvisionQoT._fields)
    assert ops.ProtectionQoT._fields == want


def test_protect_rejects_bad_arguments_without_a_gpu():
    """QOT_E_BADARG with a message naming the query: NULL descriptors, L over QOT_TG_MAX_LINKS, NULL backup outputs."""
    from gnn_qot_estimation_b200 import _lib
    L = _lib.lib()
    prep = C.create_string_buffer(64)
    aligned = (C.addressof(prep) + 15) & ~15
    x = C.create_string_buffer(64)
    ptr = C.addressof(x)

    def call(st, d, backup=None):
        outs = [ptr] * 11
        return L.qot_lightpath_protect(st, d, ptr, ptr, None, 0, 1, 0, aligned, 1, 0, ptr, None, *outs, None,
                                       *(backup if backup is not None else [ptr] * 11), None)
    cfg = _lib.QotLpGraphCfg(F=10, L=4, Q=16, T=3, i_conn=0)
    st = _lib.QotLpState(cfg, 1, 3, 0)
    d = _lib.QotLpDemands(2, 2, 2)
    assert call(None, C.byref(d)) != 0
    assert b"qot_lightpath_protect" in L.qot_last_error()
    wide = _lib.QotLpState(_lib.QotLpGraphCfg(F=10, L=1025, Q=16, T=3, i_conn=0), 1, 3, 0)
    assert call(C.byref(wide), C.byref(d)) != 0
    assert b"QOT_TG_MAX_LINKS" in L.qot_last_error()
    assert call(C.byref(st), C.byref(d), [None] * 11) != 0
    assert b"backup" in L.qot_last_error()


def test_protection_ref_is_provision_ref_when_nothing_is_protected():
    from protection_ref import protection_ref
    from provision_ref import provision_ref
    o = _oracle()
    smp = _sample()
    s0, freqs, lp_feat = smp["data"][0], smp["freqs"], smp["lp_feat"]
    f = (16, 10, 300000)
    demands = [[([0], 1, f, -np.inf), ([1, 2], 1, f, -np.inf)], [([0], 1, f, -np.inf)], [([0, 3], 2, f, -np.inf)],
               [([0], 1, f, np.inf)], [([1], 1, f, -np.inf), ([2, 3], 1, f, -np.inf)]]
    for policy in (0, 2):
        steps, final = protection_ref(o, s0, freqs, lp_feat, demands, [False] * len(demands), policy)
        psteps, pfinal = provision_ref(o, s0, freqs, lp_feat, demands, policy)
        assert np.array_equal(final, pfinal)
        for a, b in zip(steps, psteps):
            for k in ("choice", "n_free", "n_feasible", "written", "conn"):
                assert a[k] == b[k], k
            assert a["status"] == 0 and a["b_written"] is None and a["b_conn"] is None


def test_protection_ref_protected_steps():
    """A protected demand: its working path is the provision choice over its eligible options, its backup link-disjoint
    and written as top + 2; a demand whose backup cannot be placed leaves the sample as it was; no partner: nothing."""
    from protection_ref import PROT_NO_BACKUP, PROT_NO_PARTNER, protection_ref
    o = _oracle()
    smp = _sample()
    s0, freqs, lp_feat = smp["data"][0], smp["freqs"], smp["lp_feat"]
    fi = {k: i for i, k in enumerate(lp_feat)}
    top = int(np.trunc(s0[fi["conn_id"]]).max(initial=0))
    f = (16, 10, 300000)
    ninf = -np.inf
    demands = [[([0], 1, f, ninf), ([0, 1], 1, f, ninf), ([2, 3], 1, f, ninf)],     # working 0 or 1, backup [2, 3]
               [([1], 1, f, ninf), ([1, 2], 1, f, ninf)],                          # every route shares link 1
               [([0], 1, f, ninf), ([3], 1, f, np.inf)],                           # the only partner is infeasible
               [([1], 1, f, ninf), ([2], 1, f, ninf)]]
    steps, final = protection_ref(o, s0, freqs, lp_feat, demands, [True] * 4, 0)
    a, b, c, d = steps
    assert a["status"] == 0 and a["written"][0] in (0, 1) and a["b_written"][0] == 2
    assert (a["conn"], a["b_conn"]) == (top + 1, top + 2)
    assert b["status"] == PROT_NO_PARTNER and b["n_free"] == 0 and b["written"] is None
    assert c["status"] == PROT_NO_BACKUP and c["written"] is not None and c["conn"] is None
    assert c["b_n_free"] > 0 and c["b_n_feasible"] == 0
    assert (d["conn"], d["b_conn"]) == (top + 3, top + 4)              # the rolled-back demand took no conn_id
    # the final sample holds exactly the four accepted paths
    ids = set(np.trunc(final[fi["conn_id"]]).astype(int)[np.any(final != 0, axis=0)].tolist())
    assert {top + 1, top + 2, top + 3, top + 4} <= ids and top + 5 not in ids


def test_option_filters_are_set_disjointness():
    from protection_ref import disjoint_from, partner_eligible
    rng = np.random.default_rng(4)
    for _ in range(300):
        n = int(rng.integers(1, 9))
        routes = [rng.integers(0, 12, int(rng.integers(1, 5))).tolist() for _ in range(n)]   # duplicates allowed
        m = np.zeros((n, 12), dtype=bool)
        for p, r in enumerate(routes):
            m[p, r] = True
        share = (m[:, None, :] & m[None, :, :]).any(2)
        assert partner_eligible(routes) == (~share).any(1).tolist()
        w = int(rng.integers(0, n))
        assert disjoint_from(routes, routes[w]) == (~share[w]).tolist()
        assert not disjoint_from(routes, routes[w])[w]


def test_round_loop_conn_ids_across_a_rollback():
    """A rolled-back demand takes no conn_id and leaves its sample's running top; the next accepted demand of that
    sample takes top + 1 as if the rolled-back one had never been offered."""
    from protection_ref import conn_ids
    top = torch.tensor([5, 0, 9])
    s = torch.tensor([0, 1, 2])
    t = lambda *v: torch.tensor(v)
    conn, bconn, top2 = conn_ids(top, s, t(True, True, True), t(False, True, False), t(True, True, False))
    assert conn.tolist() == [-1, 1, 10] and bconn.tolist() == [-1, 2, -1]
    assert top2.tolist() == [5, 2, 10]
    conn, bconn, top3 = conn_ids(top2, s[:1], t(True), t(True), t(True))
    assert conn.tolist() == [6] and bconn.tolist() == [7] and top3.tolist() == [7, 2, 10]
    conn, bconn, top4 = conn_ids(top3, s[:1], t(False), t(False), t(True))
    assert conn.tolist() == [-1] and bconn.tolist() == [-1] and torch.equal(top4, top3)
