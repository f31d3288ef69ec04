"""CPU checks of dynamic traffic's host side: the C ABI declares and binds qot_lightpath_traffic, the literal reference
(tests/traffic_ref.py) without releases is provision_ref, the device grouping of releases is the stable (sample,
before, k) order, and synthetic.lightpath_traffic draws what it documents."""
import ctypes as C

import numpy as np
import torch

from test_lightpath_provision_cpu import _oracle, _sample
from test_lightpath_reconfig_cpu import _header_arity


def test_header_declares_and_ctypes_binds_traffic():
    from gnn_qot_estimation_b200 import _lib
    name = "qot_lightpath_traffic"
    args = _lib.SIGNATURES[name][1]
    assert len(args) == _header_arity(name) == 34
    # the provision arguments first, in their order, then the releases struct and its grouping, the release outputs
    assert args[:24] == _lib.SIGNATURES["qot_lightpath_provision"][1][:24]
    assert args[24] == C.POINTER(_lib.QotLpReleases) and args[25:33] == [C.c_void_p] * 8
    assert C.sizeof(_lib.QotLpReleases) == 40


def test_traffic_ref_without_releases_is_provision_ref():
    from provision_ref import provision_ref
    from traffic_ref import traffic_ref
    o = _oracle()
    smp = _sample()
    s0, freqs, lp_feat = smp["data"][0], smp["freqs"], smp["lp_feat"]
    f = (16, 10, 300000)
    demands = [[([0], 1, f, -np.inf), ([1, 2], 1, f, -np.inf)], [([0], 1, f, -np.inf)], [([0, 3], 2, f, -np.inf)],
               [([0], 1, f, np.inf)]]
    a, fa = provision_ref(o, s0, freqs, lp_feat, demands, 2)
    b, fb = traffic_ref(o, s0, freqs, lp_feat, [("d", x) for x in demands], 2)
    assert np.array_equal(fa, fb)
    for x, y in zip(a, b):
        assert (x["choice"], x["n_free"], x["n_feasible"], x["written"], x["conn"]) == \
               (y["choice"], y["n_free"], y["n_feasible"], y["written"], y["conn"])


def test_traffic_ref_release_then_arrival():
    """A release by demand frees the slots (first fit takes them again) and the next id is top + 2, not a reused one;
    releasing it twice names nothing."""
    from traffic_ref import traffic_ref
    o = _oracle()
    smp = _sample()
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    s0 = smp["data"][0]
    top = int(np.trunc(s0[fi["conn_id"]]).max())
    f = (16, 10, 300000)
    seq = [("d", [([0], 1, f, -np.inf)]), ("rd", 0), ("d", [([0], 1, f, -np.inf)]), ("rd", 0)]
    steps, final = traffic_ref(o, s0, smp["freqs"], smp["lp_feat"], seq, 0)
    assert steps[0]["conn"] == top + 1 and steps[1]["conn"] == top + 1
    assert steps[2]["written"] == steps[0]["written"] and steps[2]["conn"] == top + 2
    assert steps[3]["conn"] is None
    q0 = steps[2]["written"][1]
    assert final[fi["conn_id"], 0, q0] == top + 2


def test_traffic_grouping_is_stable():
    """traffic_grouping: each sample's releases by (before, k), samples outside [0, S) last and outside every range,
    before outside [0, D] kept in its sample's range."""
    from gnn_qot_estimation_b200.ops import traffic_grouping
    g = torch.Generator().manual_seed(0)
    sample = torch.randint(-1, 6, (400,), generator=g)
    before = torch.randint(-2, 12, (400,), generator=g)
    order, rp = traffic_grouping(sample, before, 5, 10)
    assert int(rp[0]) == 0 and int(rp[-1]) == int(((sample >= 0) & (sample < 5)).sum())
    for s in range(5):
        got = order[int(rp[s]):int(rp[s + 1])].tolist()
        want = sorted(torch.nonzero(sample == s).flatten().tolist(), key=lambda k: (int(before[k]), k))
        assert got == want
    assert sorted(order.tolist()) == list(range(400))
    e, rp0 = traffic_grouping(torch.zeros(0, dtype=torch.int64), torch.zeros(0, dtype=torch.int64), 3, 0)
    assert e.numel() == 0 and rp0.tolist() == [0, 0, 0, 0]


def test_synthetic_traffic():
    """Each release by demand names an earlier demand of its sample and its before is the number of demands that
    arrived before the departure (so before > demand); releases by conn_id name a lightpath of their sample; the draw
    is deterministic under a seed and differs across seeds."""
    from gnn_qot_estimation_b200 import synthetic
    smp = synthetic.network_status_samples(4, num_links=12, num_freqs=40, seed=5)
    d, r = synthetic.lightpath_traffic(smp, 8, 3.0, seed=6, release_existing=0.3)
    D = int(d.sample.shape[0])
    assert D == 32 and int(r.sample.shape[0]) > D
    ds = d.sample.tolist()
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    for s, b, dm, c in zip(r.sample.tolist(), r.before.tolist(), r.demand.tolist(), r.conn_id.tolist()):
        assert 0 <= b <= D
        if dm >= 0:
            assert ds[dm] == s and dm < b and c == -1
        else:
            x = smp["data"][s]
            assert c in set(np.trunc(x[fi["conn_id"]][np.any(x != 0, axis=0)]).astype(int).tolist())
    assert (r.demand >= 0).sum() == D and (r.demand == -1).sum() > 0
    assert sorted(r.demand[r.demand >= 0].tolist()) == list(range(D))
    # the departure times reproduce before: recompute from the same seed's draws
    d2, r2 = synthetic.lightpath_traffic(smp, 8, 3.0, seed=6, release_existing=0.3)
    assert all(torch.equal(a, b) for a, b in zip(d, d2)) and all(torch.equal(a, b) for a, b in zip(r, r2))
    d3, r3 = synthetic.lightpath_traffic(smp, 8, 3.0, seed=7, release_existing=0.3)
    assert not torch.equal(r.before, r3.before) or not torch.equal(d.sample, d3.sample)


def test_synthetic_traffic_before_is_searchsorted():
    """before[k] of a release by demand is the count of arrivals strictly before its departure: with load -> large,
    arrivals are dense, and every demand's departure lies after its own arrival (before > demand)."""
    from gnn_qot_estimation_b200 import synthetic
    smp = synthetic.network_status_samples(2, num_links=8, num_freqs=32, seed=8)
    for load in (0.5, 20.0):
        d, r = synthetic.lightpath_traffic(smp, 30, load, seed=9)
        byd = r.demand >= 0
        assert bool((r.before[byd] > r.demand[byd]).all())
    # a low load: holding times outlast few arrivals, so befores cluster near the demand; a high load: far after it
    _, lo = synthetic.lightpath_traffic(smp, 30, 0.5, seed=9)
    _, hi = synthetic.lightpath_traffic(smp, 30, 20.0, seed=9)
    gap = lambda x: float((x.before - x.demand).double().mean())
    assert gap(hi) > gap(lo)
