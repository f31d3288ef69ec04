"""CPU checks of sequential provisioning's host side: the C ABI declares and binds it, the literal reference
(tests/provision_ref.py) is consistent with placement_ref and insert_candidate, and the device grouping of demands by
sample is a stable sort."""
import ctypes as C

import numpy as np
import torch

from conftest import load_golden
from test_lightpath_reconfig_cpu import _header_arity


def test_header_declares_and_ctypes_binds_provision():
    from gnn_qot_estimation_b200 import _lib
    name = "qot_lightpath_provision"
    assert len(_lib.SIGNATURES[name][1]) == _header_arity(name) == 25
    # the state, the demands, then the grouping
    assert _lib.SIGNATURES[name][1][:4] == [C.POINTER(_lib.QotLpState), C.POINTER(_lib.QotLpDemands), C.c_void_p,
                                            C.c_void_p]


def _oracle():
    from oracle import LightpathGNNOracle
    m = LightpathGNNOracle(5, 32, 3, is_lut_index=1, dropout_p=0.0).double()
    m.load_state_dict(load_golden("ckpt_lightpath_model_1.pt")["model_state_dict"], strict=True)
    return m.eval()


def _sample():
    from gnn_qot_estimation_b200 import synthetic
    return synthetic.network_status_samples(1, num_links=4, num_freqs=16, seed=3, spacing=0.05, max_lightpaths=8)


def test_provision_ref_steps():
    """The first step is placement_ref on the sample; every written placement is free in the sample it was written
    into (so accepted placements are disjoint); conn_ids go top + 1, top + 2, ...; the written vectors are
    insert_candidate's."""
    from candidates_ref import insert_candidate
    from placement_ref import free_starts, placement_ref
    from provision_ref import provision_ref
    o = _oracle()
    smp = _sample()
    s0, freqs, lp_feat = smp["data"][0], smp["freqs"], smp["lp_feat"]
    f = (16, 10, 300000)
    demands = [[([0], 1, f, -np.inf), ([1, 2], 1, f, -np.inf)], [([0], 1, f, -np.inf)], [([0, 3], 2, f, -np.inf)],
               [([0], 1, f, np.inf)]]
    steps, final = provision_ref(o, s0, freqs, lp_feat, demands, 2)
    choice, n_free, n_feas, _ = placement_ref(o, s0, freqs, lp_feat, demands[0], 2)
    assert (steps[0]["choice"], steps[0]["n_free"], steps[0]["n_feasible"]) == (choice, n_free, n_feas)
    fi = {k: i for i, k in enumerate(lp_feat)}
    top = int(np.trunc(s0[fi["conn_id"]]).max(initial=0))
    cur = np.array(s0, copy=True)
    want = top
    for opts, st in zip(demands, steps):
        if st["written"] is None:
            assert st["conn"] is None
            continue
        p, q0 = st["written"]
        links, width = opts[p][0], opts[p][1]
        assert q0 in free_starts(cur, links, width)
        cur, conn = insert_candidate(cur, lp_feat, links, q0, width, [np.float32(freqs[q0])] + list(opts[p][2]))
        want += 1
        assert conn == st["conn"] == want
    assert steps[3]["written"] is None and want >= top + 2
    assert np.array_equal(cur, final)


def test_provision_ref_follow():
    """follow= writes the given placements whatever the reference would choose, and None writes nothing."""
    from provision_ref import provision_ref
    o = _oracle()
    smp = _sample()
    f = (16, 10, 300000)
    demands = [[([0], 1, f, -np.inf)], [([0], 1, f, -np.inf)]]
    steps, final = provision_ref(o, smp["data"][0], smp["freqs"], smp["lp_feat"], demands, 0, follow=[None, (0, 15)])
    assert steps[0]["conn"] is None and steps[1]["written"] == (0, 15)
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    assert final[fi["conn_id"], 0, 15] == steps[1]["conn"]
    assert final[fi["osnr"], 0, 15] == -1.0


def test_grouping_is_stable():
    """provision_grouping: order lists each sample's demands in increasing index, samples outside [0, S) last and
    outside every range; sample_ptr[0] = 0 and sample_ptr[S] = the demands with a valid sample."""
    from gnn_qot_estimation_b200.ops import provision_grouping
    g = torch.Generator().manual_seed(0)
    sample = torch.randint(-1, 6, (500,), generator=g)
    order, sp = provision_grouping(sample, 5)
    assert int(sp[0]) == 0 and int(sp[-1]) == int(((sample >= 0) & (sample < 5)).sum())
    for s in range(5):
        got = order[int(sp[s]):int(sp[s + 1])].tolist()
        assert got == torch.nonzero(sample == s).flatten().tolist()
    assert sorted(order.tolist()) == list(range(500))
    empty, sp0 = provision_grouping(torch.zeros(0, dtype=torch.int64), 3)
    assert empty.numel() == 0 and sp0.tolist() == [0, 0, 0, 0]
