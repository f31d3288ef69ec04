"""CPU checks of LightpathGNN's change-set QoT: the C ABI declares and binds it, the literal reference definition
(tests/change_set_ref.py) agrees with the reconfiguration reference and with every-node mode on the oracle, the seeded
set generator, and the timing script's arguments and byte arithmetic."""
import ctypes as C
import importlib.util
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from test_lightpath_reconfig_cpu import HEADER, TOL, _every, _header_arity, _oracle64, fake_state

ROOT = Path(__file__).resolve().parents[1]


def test_change_sets_take_state_and_changes_structs():
    from gnn_qot_estimation_b200 import _lib, ops
    name = "qot_lightpath_change_sets"
    assert name in _lib.SIGNATURES
    assert len(_lib.SIGNATURES[name][1]) == _header_arity(name) == 15
    # the state, the changes, then G and set_ptr
    assert _lib.SIGNATURES[name][1][:4] == [C.POINTER(_lib.QotLpState), C.POINTER(_lib.QotLpChanges), C.c_int64,
                                            C.c_void_p]
    text = HEADER.read_text()
    bits = {n: int(re.search(r"#define QOT_SET_" + n + r"\s+(\d+)", text).group(1))
            for n in ("MAX_CHANGES", "BAD_SET", "DUPLICATE", "CONFLICT")}
    assert bits == dict(MAX_CHANGES=ops.SET_MAX_CHANGES, BAD_SET=ops.SET_BAD_SET, DUPLICATE=ops.SET_DUPLICATE,
                        CONFLICT=ops.SET_CONFLICT) == dict(MAX_CHANGES=64, BAD_SET=64, DUPLICATE=128, CONFLICT=256)
    cand = (ops.CAND_BAD_SAMPLE | ops.CAND_BAD_PATH | ops.CAND_OCCUPIED | ops.CAND_IMPACT_OVERFLOW |
            ops.CAND_BAD_STATE | ops.CAND_BAD_NODE)
    assert cand & (ops.SET_BAD_SET | ops.SET_DUPLICATE | ops.SET_CONFLICT) == 0
    assert set(ops.ChangeSetQoT._fields) == set(ops.ReconfigQoT._fields) | {"set_status"}


def _sets(c, set_ptr, conn_ids):
    """[(sample, [(conn_id or None, links, q0, width, feat)])] of generated sets."""
    out = []
    for g in range(set_ptr.numel() - 1):
        ch = []
        for k in range(int(set_ptr[g]), int(set_ptr[g + 1])):
            a, b = int(c.link_ptr[k]), int(c.link_ptr[k + 1])
            nd = int(c.node[k])
            ch.append((None if nd < 0 else int(conn_ids[nd]), c.links[a:b].tolist(), int(c.q0[k]), int(c.width[k]),
                       c.feat[k].tolist()))
        out.append((int(c.sample[int(set_ptr[g])]), ch))
    return out


def _generated(n=3, per=10, seed=8):
    from gnn_qot_estimation_b200 import synthetic
    smp = synthetic.network_status_samples(n, num_links=12, num_freqs=24, seed=seed, max_lightpaths=14,
                                           super_channel_p=0.3)
    st = fake_state(smp)
    c, sp = synthetic.lightpath_change_sets(smp, st, per, seed=seed + 1)
    return smp, st, c, sp


def test_one_change_set_is_reconfig_ref_and_unlisted_rows_are_unchanged():
    """A set of one change equals reconfig_ref (bit for bit on the oracle); for every generated set, every row the set
    does not list (and does not name) is the every-node row of the original sample, and every listed row is the
    every-node row of the rebuilt sample."""
    from change_set_ref import apply_set, change_set_ref
    from reconfig_ref import reconfig_ref
    m = _oracle64()
    smp, st, c, sp = _generated()
    freqs, lp_feat = smp["freqs"], smp["lp_feat"]
    n = dict(single=0, multi=0, unchanged=0)
    for s, ch in _sets(c, sp, st.conn_ids):
        sample = smp["data"][s]
        rows, imp = change_set_ref(m, sample, freqs, lp_feat, ch)
        if len(ch) == 1:
            row, rimp = reconfig_ref(m, sample, freqs, lp_feat, *ch[0])
            assert (row is None) == (rows[0] is None) and (row is None or torch.equal(row, rows[0]))
            assert set(rimp) == set(imp)
            for o, (kind, r) in rimp.items():
                assert imp[o][0] == kind and torch.equal(imp[o][1], r)
            n["single"] += 1
            continue
        n["multi"] += 1
        s2, conns = apply_set(sample, lp_feat, ch)
        before, _, _ = _every(m, sample, freqs, lp_feat)
        after, _, _ = _every(m, s2, freqs, lp_feat)
        named = {cc for cc, *_ in ch if cc is not None}
        for o, r in before.items():
            if o not in named and o not in imp:
                torch.testing.assert_close(after[o], r, **TOL)
                n["unchanged"] += 1
        for o, (_, r) in imp.items():
            torch.testing.assert_close(after[o], r, **TOL)
        for cc, r in zip(conns, rows):
            if r is not None:
                torch.testing.assert_close(after[cc], r, **TOL)
    assert n["single"] >= 3 and n["multi"] >= 10 and n["unchanged"] > 50, n


def test_teardown_only_restoration_is_every_node_without_them():
    """Tear down every lightpath on one link: the listed rows (all kind 1) are the every-node rows of the sample rebuilt
    without them, and nothing else changes."""
    from change_set_ref import change_set_ref
    m = _oracle64()
    smp, st, _, _ = _generated(n=2)
    freqs, lp_feat = smp["freqs"], smp["lp_feat"]
    fi = {k: i for i, k in enumerate(lp_feat)}
    checked = 0
    for s in range(2):
        sample = smp["data"][s]
        occ = np.any(sample != 0, axis=0)
        conn = np.trunc(sample[fi["conn_id"]])
        for l in range(12):
            gone = sorted({int(v) for v in conn[l][occ[l]]})
            if not gone:
                continue
            rows, imp = change_set_ref(m, sample, freqs, lp_feat, [(cc, [], 0, 1, [0, 0, 0, 0]) for cc in gone])
            assert all(r is None for r in rows) and all(k == 1 for k, _ in imp.values())
            rest = sample.copy()
            rest[:, occ & np.isin(conn, gone)] = 0.0
            without, _, _ = _every(m, rest, freqs, lp_feat)
            for o, (_, r) in imp.items():
                torch.testing.assert_close(r, without[o], **TOL)
            checked += len(imp)
    assert checked > 20


def test_permuting_a_set_changes_no_row():
    from change_set_ref import change_set_ref
    m = _oracle64()
    smp, st, c, sp = _generated(seed=11)
    rng = np.random.default_rng(0)
    n = 0
    for s, ch in _sets(c, sp, st.conn_ids):
        if len(ch) < 2:
            continue
        perm = rng.permutation(len(ch))
        rows, imp = change_set_ref(m, smp["data"][s], smp["freqs"], smp["lp_feat"], ch)
        prows, pimp = change_set_ref(m, smp["data"][s], smp["freqs"], smp["lp_feat"], [ch[i] for i in perm])
        for i, p in enumerate(perm):
            assert (rows[p] is None) == (prows[i] is None)
            if rows[p] is not None:
                torch.testing.assert_close(prows[i], rows[p], **TOL)
        assert set(imp) == set(pimp)
        for o, (k, r) in imp.items():
            assert pimp[o][0] == k
            torch.testing.assert_close(pimp[o][1], r, **TOL)
        n += 1
    assert n >= 10


def test_synthetic_change_sets_are_seeded_legal_and_mixed():
    from gnn_qot_estimation_b200 import synthetic
    smp = synthetic.network_status_samples(6, num_links=20, num_freqs=32, seed=4, super_channel_p=0.3)
    smp["data"][5] = 0.0                                            # an empty sample: batch insertions only
    st = fake_state(smp)
    c, sp = synthetic.lightpath_change_sets(smp, st, 24, seed=3)
    c2, sp2 = synthetic.lightpath_change_sets(smp, st, 24, seed=3)
    assert all(torch.equal(a, b) for a, b in zip(c, c2)) and torch.equal(sp, sp2)
    assert not torch.equal(c.q0, synthetic.lightpath_change_sets(smp, st, 24, seed=4)[0].q0)
    K, G = c.sample.shape[0], sp.shape[0] - 1
    assert sp.dtype == torch.int64 and int(sp[0]) == 0 and int(sp[-1]) == K and 130 <= G <= 144
    sizes = (sp[1:] - sp[:-1]).tolist()
    assert min(sizes) >= 1 and max(sizes) <= 64
    data, occ = smp["data"], np.any(smp["data"] != 0, axis=1)
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    kinds = dict(single=0, insert_adjacent=0, swap=0, teardown=0, restore=0)
    for s, ch in _sets(c, sp, st.conn_ids):
        conn = np.trunc(data[s, fi["conn_id"]])
        free = ~occ[s]
        for cc, *_ in ch:
            if cc is not None:
                free = free | (occ[s] & (conn == cc))
        taken = np.zeros_like(free)
        named = [cc for cc, *_ in ch if cc is not None]
        assert len(named) == len(set(named))
        for cc, links, q0, w, feat in ch:
            if not links:
                kinds["teardown"] += 1
                continue
            chans = np.zeros_like(free)
            chans[np.ix_(links, range(q0, q0 + w))] = True
            assert not (chans & ~free).any() and not (chans & taken).any()
            taken |= chans
        kinds["single"] += len(ch) == 1
        olds = {cc: (np.nonzero(occ[s] & (conn == cc))[1].min()) for cc in named}
        kinds["swap"] += any(a[0] is not None and b[0] is not None and a[0] != b[0] and a[2] == olds[b[0]] and
                             b[2] == olds[a[0]] and a[1] and b[1] for a in ch for b in ch)
        ins = [x for x in ch if x[0] is None]
        kinds["insert_adjacent"] += any(set(a[1]) & set(b[1]) and (a[2] + a[3] == b[2] or b[2] + b[3] == a[2])
                                        for i, a in enumerate(ins) for b in ins[i + 1:])
        old_links = [set(np.nonzero(occ[s] & (conn == cc))[0].tolist()) for cc in named]
        common = set.intersection(*old_links) if len(named) == len(ch) >= 2 else set()
        kinds["restore"] += any(all(l not in x[1] for x in ch) for l in common)
    assert min(kinds.values()) > 0, kinds


def _script():
    import sys
    sys.path.insert(0, str(ROOT / "scripts"))
    spec = importlib.util.spec_from_file_location("time_change_sets", ROOT / "scripts" / "time_change_sets.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_timing_script_arguments_and_bytes():
    mod = _script()
    a = mod.parse_args([])
    assert (a.states, a.links, a.freqs, a.sets_per_state, a.expand, a.max_impact) == (64, 60, 80, 256, 512, 64)
    a = mod.parse_args(["--states", "2", "--sets-per-state", "8", "--expand", "3", "--max-impact", "0"])
    assert (a.states, a.sets_per_state, a.expand, a.max_impact) == (2, 8, 3, 0)
    for bad in (["--expand", "0"], ["--sets-per-state", "0"], ["--max-impact", "-1"]):
        with pytest.raises(SystemExit):
            mod.parse_args(bad)
    tr = importlib.util.spec_from_file_location("time_reconfig", ROOT / "scripts" / "time_reconfig.py")
    trm = importlib.util.module_from_spec(tr)
    tr.loader.exec_module(trm)
    # per change: node, the change arrays, out and status (8 + 40 + 16 B); per set: set_ptr, set_status and n_impact
    # (16 B) and 21 B per impact slot; plus 16 B per pair of changes whose paths are compared
    K, G, MI = 10, 4, 7
    got = mod.algorithmic_bytes(K, G, 5, 80, 7, 30, MI, 3, 6, 11)
    assert got == K * (8 + 40 + 16) + 5 * (4 + 4 * 80) + 36 * 7 + 8 * 30 + 16 * 3 + 8 * 6 + G * (16 + 21 * MI) + 16 * 11
    # one change per set, no pairs: the reconfiguration bytes plus set_ptr and set_status (12 B per set)
    assert mod.algorithmic_bytes(K, K, 5, 80, 7, 30, MI, 3, 6, 0) == trm.algorithmic_bytes(K, 5, 80, 7, 30, MI, 3, 6) \
        + 12 * K
