"""CPU checks of LightpathGNN's placement search: the C ABI declares and binds it, the literal reference definition
(tests/placement_ref.py) agrees with candidates_ref, with its own per-placement table and with every-node mode on the
oracle, the seeded demand generator, and the timing script's arguments and arithmetic."""
import ctypes as C
import importlib.util
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from test_lightpath_reconfig_cpu import HEADER, TOL, _every, _header_arity, _oracle64

ROOT = Path(__file__).resolve().parents[1]


def test_placements_take_state_and_demands_structs():
    from gnn_qot_estimation_b200 import _lib, ops
    name = "qot_lightpath_placements"
    assert name in _lib.SIGNATURES
    assert len(_lib.SIGNATURES[name][1]) == _header_arity(name) == 22
    # the state, then the demands
    assert _lib.SIGNATURES[name][1][:2] == [C.POINTER(_lib.QotLpState), C.POINTER(_lib.QotLpDemands)]
    text = HEADER.read_text()
    vals = {n: int(re.search(r"#define QOT_PLACE_" + n + r"\s+(\d+)", text).group(1))
            for n in ("MAX_OPTIONS", "MAX_SLOTS", "FIRST_FIT", "BEST_QOT", "MAX_MARGIN")}
    assert vals == dict(MAX_OPTIONS=ops.PLACE_MAX_OPTIONS, MAX_SLOTS=ops.PLACE_MAX_SLOTS,
                        FIRST_FIT=ops.PLACE_FIRST_FIT, BEST_QOT=ops.PLACE_BEST_QOT, MAX_MARGIN=ops.PLACE_MAX_MARGIN)
    assert vals == dict(MAX_OPTIONS=32, MAX_SLOTS=1024, FIRST_FIT=0, BEST_QOT=1, MAX_MARGIN=2)
    assert (ops.CAND_BAD_SAMPLE, ops.CAND_BAD_PATH, ops.CAND_IMPACT_OVERFLOW, ops.CAND_BAD_STATE) == (1, 2, 8, 16)
    assert set(ops.CandidateQoT._fields) < set(ops.PlacementQoT._fields)
    import placement_ref
    assert (placement_ref.FIRST_FIT, placement_ref.BEST_QOT, placement_ref.MAX_MARGIN) == (0, 1, 2)


def _samples(n=3, seed=3, Q=24):
    from gnn_qot_estimation_b200 import synthetic
    return synthetic.network_status_samples(n, num_links=8, num_freqs=Q, seed=seed, max_lightpaths=12,
                                            super_channel_p=0.3)


def test_single_free_start_equals_candidates_ref():
    """A demand with one option and exactly one free start slot is candidates_ref at that slot."""
    from candidates_ref import candidates_ref
    from placement_ref import FIRST_FIT, placement_ref
    m = _oracle64()
    smp = _samples()
    sample = smp["data"][0].copy()
    occ = np.any(sample != 0, axis=0)
    link = int(np.argmin(occ.sum(axis=1)))
    free = np.flatnonzero(~occ[link])
    keep = int(free[len(free) // 2])
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    for q in free:                                          # fill every other free slot of the link with a lightpath
        if q != keep:
            sample[fi["conn_id"], link, q] = 900 + q
            sample[fi["freq"], link, q] = smp["freqs"][q]
            sample[fi["mod_order"], link, q] = 16
    feat3 = (32, 12, 400000)
    best, n_free, n_feas, table = placement_ref(m, sample, smp["freqs"], smp["lp_feat"],
                                                [([link], 1, feat3, -np.inf)], FIRST_FIT)
    assert best == (0, keep) and n_free == n_feas == 1
    row, imp = candidates_ref(m, sample, smp["freqs"], smp["lp_feat"], [link], keep, 1,
                              [np.float32(smp["freqs"][keep])] + list(feat3))
    torch.testing.assert_close(table[best][0], row, **TOL)
    assert set(table[best][1]) == set(imp) and len(imp) > 0
    for c, r in imp.items():
        torch.testing.assert_close(table[best][1][c], r, **TOL)


def test_choice_is_brute_force_over_the_table():
    """placement_ref's choice is a brute-force argmax over its own table, for each policy, both senses and with a
    per-lightpath bound."""
    from placement_ref import BEST_QOT, FIRST_FIT, MAX_MARGIN, choose, placement_table
    m = _oracle64()
    smp = _samples(seed=4)
    s = 1
    _, conns, _ = _every(m, smp["data"][s], smp["freqs"], smp["lp_feat"])
    rng = np.random.default_rng(5)
    opts = [([0, 3], 1, (16, 20, 100000), 0.25), ([5], 2, (64, 3, 30000), 0.2), ([0, 3], 3, (4, 90, 5000000), 0.3)]
    n_pick = 0
    for bound in (None, {int(c): float(rng.uniform(0.0, 0.5)) for c in conns}):
        for mx in (True, False):
            ob = [(l, w, f, b if mx else b + 0.1) for l, w, f, b in opts]
            table = placement_table(m, smp["data"][s], smp["freqs"], smp["lp_feat"], ob, 0, mx, bound)
            assert len(table) > 10
            keys = sorted(table)
            for policy in (FIRST_FIT, BEST_QOT, MAX_MARGIN):
                best, n_free, n_feas = choose(table, policy, 0, mx)
                feas = [k for k in keys if table[k][2] >= 0]
                assert n_free == len(keys) and n_feas == len(feas)
                if not feas:
                    assert best is None
                    continue
                sign = 1.0 if mx else -1.0
                score = {FIRST_FIT: lambda k: 0.0, BEST_QOT: lambda k: sign * float(table[k][0][0]),
                         MAX_MARGIN: lambda k: table[k][2]}[policy]
                top = max(score(k) for k in feas)
                assert best == [k for k in feas if score(k) == top][0]
                n_pick += 1
            # the margins by hand
            for (p, q0), (row, imp, mg) in table.items():
                ms = [(float(row[0]) - ob[p][3]) * (1 if mx else -1)]
                if bound is not None:
                    ms += [(float(r[0]) - bound[c]) * (1 if mx else -1) for c, r in imp.items()]
                assert mg == min(ms)
    assert n_pick >= 6


def test_leave_one_out_row_is_every_node_row():
    """A lightpath written with insert_candidate (freq = float32(freqs[q0])) into a sample: offered back as a demand on
    the sample without it, the reference's row at its q0 is the every-node row of the sample with it, and its impact
    rows are the every-node rows of its neighbours there."""
    from candidates_ref import insert_candidate
    from placement_ref import FIRST_FIT, free_starts, placement_ref
    m = _oracle64()
    smp = _samples(seed=6)
    n = 0
    for s, (links, q0, w, feat3) in enumerate([([1, 4], 5, 1, (16, 30, 700000)), ([2], 9, 2, (64, 4, 60000)),
                                               ([0, 6, 7], 13, 1, (8, 50, 2000000))]):
        base = smp["data"][s]
        if q0 not in free_starts(base, links, w):
            continue
        feat = [np.float32(smp["freqs"][q0])] + list(feat3)
        with_it, conn = insert_candidate(base, smp["lp_feat"], links, q0, w, feat)
        every, _, _ = _every(m, with_it, smp["freqs"], smp["lp_feat"])
        _, _, _, table = placement_ref(m, base, smp["freqs"], smp["lp_feat"], [(links, w, feat3, -np.inf)],
                                       FIRST_FIT)
        row, imp, _ = table[(0, q0)]
        torch.testing.assert_close(row, every[conn], **TOL)
        for c, r in imp.items():
            torch.testing.assert_close(r, every[c], **TOL)
        n += 1
    assert n >= 2


def test_demand_generator_is_seeded_and_in_range():
    from gnn_qot_estimation_b200 import synthetic
    from gnn_qot_estimation_b200.to_graph import LightpathDemands
    smp = _samples(n=4, seed=7, Q=32)
    a = synthetic.lightpath_demands(smp, 8, seed=9)
    b = synthetic.lightpath_demands(smp, 8, seed=9)
    c = synthetic.lightpath_demands(smp, 8, seed=10)
    assert isinstance(a, LightpathDemands)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    assert not torch.equal(a.links, c.links) or not torch.equal(a.width, c.width)
    D, P = a.sample.shape[0], a.width.shape[0]
    assert D == 32 and a.opt_ptr.shape == (D + 1,) and a.link_ptr.shape == (P + 1,) and a.feat.shape == (P, 3)
    assert a.sample.dtype == torch.int64 and a.links.dtype == torch.int32 and a.own_bound.dtype == torch.float32
    assert bool(((a.sample >= 0) & (a.sample < 4)).all())
    n_opt = a.opt_ptr[1:] - a.opt_ptr[:-1]
    assert int(n_opt.min()) >= 1 and int(n_opt.max()) <= 4 and int(a.opt_ptr[-1]) == P
    rl = a.link_ptr[1:] - a.link_ptr[:-1]
    assert int(rl.min()) >= 1 and int(rl.max()) <= 6 and bool(((a.links >= 0) & (a.links < 8)).all())
    assert int(a.width.min()) >= 1 and int(a.width.max()) <= 3
    for p in range(P):                                        # distinct links per route
        r = a.links[a.link_ptr[p]:a.link_ptr[p + 1]].tolist()
        assert len(set(r)) == len(r)
    assert set(a.feat[:, 0].tolist()) <= {4.0, 8.0, 16.0, 32.0, 64.0}
    assert bool(((a.feat[:, 1] >= 1) & (a.feat[:, 1] <= 106)).all())
    # repeated routes with another format, and all three kinds of bound
    routes = [tuple(a.links[a.link_ptr[p]:a.link_ptr[p + 1]].tolist()) for p in range(P)]
    assert len(set(routes)) < len(routes)
    ob = a.own_bound
    assert bool(torch.isneginf(ob).any()) and bool(torch.isposinf(ob).any()) and bool(torch.isfinite(ob).any())
    one = synthetic.lightpath_demands(smp, 2, options=(1, 1), seed=1)
    assert bool((one.opt_ptr[1:] - one.opt_ptr[:-1] == 1).all())
    with pytest.raises(ValueError):
        synthetic.lightpath_demands(smp, 2, options=(0, 2))


def _script():
    spec = importlib.util.spec_from_file_location("time_placements", ROOT / "scripts" / "time_placements.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_timing_script_arguments_and_arithmetic():
    mod = _script()
    a = mod.parse_args([])
    assert (a.states, a.links, a.freqs, a.demands, a.max_impact) == (64, 60, 80, 8192, 64)
    with pytest.raises(SystemExit):
        mod.parse_args(["--freqs", "1025"])
    with pytest.raises(SystemExit):
        mod.parse_args(["--demands", "3", "--states", "4"])
    # 2 demands, 3 options, 5 route links on a 4-slot grid, 2 chosen impact rows with 3 edges, max_impact 1
    assert mod.algorithmic_bytes(2, 3, 5, 4, 2, 3, 1) == 2 * (16 + 40 + 20) + 3 * 28 + 5 * (4 + 16) + 40 * 2 + 8 * 3
    assert mod.head_mmas(16) == 240 and mod.head_mmas(40) == 600
