"""CPU checks of LightpathGNN's reconfiguration QoT: the C ABI declares and binds it, the literal reference definition
(tests/reconfig_ref.py) agrees with every-node mode and with the candidate reference on the oracle, the seeded change
generator, and the timing script's argument parsing, byte arithmetic and expansion inputs."""
import ctypes as C
import importlib.util
import re
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from conftest import load_golden

ROOT = Path(__file__).resolve().parents[1]
HEADER = ROOT / "include" / "qot_b200.h"
TOL = dict(rtol=1e-12, atol=1e-12)


def _header_arity(name):
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", text, flags=re.S)
    assert m, name
    return m.group(1).count(",") + 1


def test_reconfigure_takes_state_and_changes_structs():
    from gnn_qot_estimation_b200 import _lib, ops
    name = "qot_lightpath_reconfigure"
    assert name in _lib.SIGNATURES
    assert len(_lib.SIGNATURES[name][1]) == _header_arity(name) == 12
    # the state, then the changes
    assert _lib.SIGNATURES[name][1][:2] == [C.POINTER(_lib.QotLpState), C.POINTER(_lib.QotLpChanges)]
    bit = int(re.search(r"#define QOT_CAND_BAD_NODE\s+(\d+)", HEADER.read_text()).group(1))
    assert bit == ops.CAND_BAD_NODE == 32
    assert (ops.KIND_LOST, ops.KIND_GAINED, ops.KIND_KEPT) == (1, 2, 3)
    assert set(ops.ReconfigQoT._fields) == set(ops.CandidateQoT._fields) | {"impact_kind"}


def _oracle64():
    from oracle import LightpathGNNOracle
    m = LightpathGNNOracle(5, 32, 3, is_lut_index=1, dropout_p=0.0).double()
    m.load_state_dict(load_golden("ckpt_lightpath_model_1.pt")["model_state_dict"], strict=True)
    return m.eval()


def _every(m, sample, freqs, lp_feat):
    """{conn_id: every-node row} of a sample, through the oracle's to_graph and the every-node reference."""
    from every_node_ref import lightpath_every_node_ref
    from oracle.to_graph_oracle import lightpath_data_ref
    conns, x, _, ei = lightpath_data_ref(sample, np.zeros(3), freqs, lp_feat, ["osnr", "snr", "ber"])
    if len(conns) == 0:
        return {}, conns, ei
    with torch.no_grad():
        every = lightpath_every_node_ref(m, SimpleNamespace(
            x=torch.from_numpy(x).double(), edge_index=torch.from_numpy(ei),
            batch=torch.zeros(x.shape[0], dtype=torch.int64)))
    return {int(c): every[i] for i, c in enumerate(conns)}, conns, ei


def _placement(sample, lp_feat, conn):
    from test_lightpath_candidates_cpu import lightpath_as_candidate
    return lightpath_as_candidate(sample, lp_feat, conn)


def _unlisted_unchanged(m, smp, s, sample2, conn, listed):
    before, _, _ = _every(m, smp["data"][s], smp["freqs"], smp["lp_feat"])
    after, _, _ = _every(m, sample2, smp["freqs"], smp["lp_feat"])
    n = 0
    for c, row in before.items():
        if c != conn and c not in listed:
            torch.testing.assert_close(after[c], row, **TOL)
            n += 1
    return after, n


def test_oracle_identities_noop_teardown_and_move():
    """On every lightpath j of a few samples: re-placing j where it is reproduces the every-node rows (all kind 3);
    a teardown's rows are the every-node rows of the sample without j (all kind 1); a real move is candidates_ref on
    the sample without j for j's row and the rows that gain j, every_node_ref of the sample without j for the rows
    that only lose it.  Every row the change does not list is the same before and after it."""
    from candidates_ref import candidates_ref
    from gnn_qot_estimation_b200 import synthetic
    from reconfig_ref import reconfig_ref, rewrite_lightpath
    m = _oracle64()
    smp = synthetic.network_status_samples(3, num_links=12, num_freqs=24, seed=8, max_lightpaths=14,
                                           super_channel_p=0.3)
    freqs, lp_feat = smp["freqs"], smp["lp_feat"]
    fi = {k: i for i, k in enumerate(lp_feat)}
    rng = np.random.default_rng(3)
    counts = dict(noop=0, tear=0, move=0, lost=0, gained=0, kept=0, unchanged=0)
    for s in range(3):
        sample = smp["data"][s]
        every, conns, ei = _every(m, sample, freqs, lp_feat)
        occ = np.any(sample != 0, axis=0)
        for j, c in enumerate(int(v) for v in conns):
            nbr = {int(conns[d]) for a, d in ei.T if a == j and d != j}
            rest, links, q0, width, feat = _placement(sample, lp_feat, c)
            # no-op move
            row, imp = reconfig_ref(m, sample, freqs, lp_feat, c, links, q0, width, feat)
            torch.testing.assert_close(row, every[c], **TOL)
            assert set(imp) == nbr and all(k == 3 for k, _ in imp.values())
            for o, (_, r) in imp.items():
                torch.testing.assert_close(r, every[o], **TOL)
            counts["noop"] += 1
            # teardown
            row, imp = reconfig_ref(m, sample, freqs, lp_feat, c, [], 0, 1, feat)
            assert row is None and set(imp) == nbr and all(k == 1 for k, _ in imp.values())
            without, _, _ = _every(m, rest, freqs, lp_feat)
            for o, (_, r) in imp.items():
                torch.testing.assert_close(r, without[o], **TOL)
            _, n = _unlisted_unchanged(m, smp, s, rest, c, imp)
            counts["tear"] += 1
            counts["unchanged"] += n
            # a real move: its own slots on other links, or another slot on its own links
            free = ~occ | (occ & (np.trunc(sample[fi["conn_id"]]) == c))
            for _try in range(32):
                path = sorted(rng.choice(12, size=int(rng.integers(1, 4)), replace=False).tolist())
                ok = [q for q in range(24 - width + 1) if free[np.ix_(path, range(q, q + width))].all()]
                if ok:
                    break
            else:
                continue
            q1 = int(rng.choice(ok))
            f1 = [np.float32(freqs[q1]), feat[1], float(rng.integers(1, 107)), float(rng.integers(24214, 7834746))]
            row, imp = reconfig_ref(m, sample, freqs, lp_feat, c, path, q1, width, f1)
            crow, cimp = candidates_ref(m, rest, freqs, lp_feat, path, q1, width, f1)
            torch.testing.assert_close(row, crow, **TOL)
            assert {o for o, (k, _) in imp.items() if k & 2} == set(cimp)
            assert {o for o, (k, _) in imp.items() if k & 1} == nbr
            for o, (k, r) in imp.items():
                if k & 2:
                    torch.testing.assert_close(r, cimp[o], **TOL)
                    counts["kept" if k == 3 else "gained"] += 1
                else:
                    torch.testing.assert_close(r, without[o], **TOL)
                    counts["lost"] += 1
            s2 = rewrite_lightpath(sample, lp_feat, c, path, q1, width, f1)
            after, n = _unlisted_unchanged(m, smp, s, s2, c, imp)
            torch.testing.assert_close(after[c], row, **TOL)
            for o, (_, r) in imp.items():
                torch.testing.assert_close(after[o], r, **TOL)
            counts["move"] += 1
            counts["unchanged"] += n
    assert counts["noop"] >= 20 and counts["move"] >= 15 and counts["unchanged"] > 100
    assert min(counts["lost"], counts["gained"], counts["kept"]) > 0, counts


def test_reconfig_ref_insertion_is_candidates_ref():
    from candidates_ref import candidates_ref
    from gnn_qot_estimation_b200 import synthetic
    from reconfig_ref import reconfig_ref
    m = _oracle64()
    smp = synthetic.network_status_samples(2, num_links=8, num_freqs=20, seed=6, max_lightpaths=16)
    c = synthetic.lightpath_candidates(smp, 6, seed=1)
    for k in range(c.sample.shape[0]):
        s, a, b = int(c.sample[k]), int(c.link_ptr[k]), int(c.link_ptr[k + 1])
        args = (smp["data"][s], smp["freqs"], smp["lp_feat"])
        rest = (c.links[a:b].tolist(), int(c.q0[k]), int(c.width[k]), c.feat[k].tolist())
        row, imp = reconfig_ref(m, *args, None, *rest)
        crow, cimp = candidates_ref(m, *args, *rest)
        assert torch.equal(row, crow) and set(imp) == set(cimp)
        for o, (kind, r) in imp.items():
            assert kind == 2 and torch.equal(r, cimp[o])


def fake_state(smp):
    """What synthetic.lightpath_changes reads of a network state (conn_ids, batch.ptr), from the oracle's to_graph:
    its node order is create_lightpath_graphs' (tests/test_to_graph_cpu.py)."""
    from oracle.to_graph_oracle import lightpath_data_ref
    conns = [lightpath_data_ref(d, np.zeros(3), smp["freqs"], smp["lp_feat"], ["osnr", "snr", "ber"])[0]
             for d in smp["data"]]
    ptr = np.cumsum([0] + [len(c) for c in conns])
    return SimpleNamespace(conn_ids=torch.from_numpy(np.concatenate(conns).astype(np.int64)),
                           batch=SimpleNamespace(ptr=torch.from_numpy(ptr.astype(np.int64))))


def test_synthetic_changes_are_seeded_legal_and_mixed():
    from gnn_qot_estimation_b200 import synthetic
    smp = synthetic.network_status_samples(6, num_links=20, num_freqs=32, seed=4, super_channel_p=0.3)
    smp["data"][5] = 0.0                                            # an empty sample: insertions only
    st = fake_state(smp)
    c = synthetic.lightpath_changes(smp, st, 60, seed=3)
    c2 = synthetic.lightpath_changes(smp, st, 60, seed=3)
    assert all(torch.equal(a, b) for a, b in zip(c, c2))
    assert not torch.equal(c.q0, synthetic.lightpath_changes(smp, st, 60, seed=4).q0)
    K = c.sample.shape[0]
    assert 330 <= K <= 360
    assert [t.dtype for t in c] == [torch.int64, torch.int64, torch.int64, torch.int32, torch.int32, torch.int32,
                                    torch.float32]
    assert c.link_ptr.shape == (K + 1,) and int(c.link_ptr[0]) == 0 and int(c.link_ptr[-1]) == c.links.numel()
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    data, freqs = smp["data"], smp["freqs"]
    occ = np.any(data != 0, axis=1)
    ptr = st.batch.ptr.numpy()
    kinds = dict(insert=0, retune=0, overlap=0, reroute=0, teardown=0)
    for k in range(K):
        s, node, q0, w = int(c.sample[k]), int(c.node[k]), int(c.q0[k]), int(c.width[k])
        links = c.links[int(c.link_ptr[k]):int(c.link_ptr[k + 1])].numpy()
        assert len(set(links.tolist())) == len(links) <= 6
        if node < 0:
            kinds["insert"] += 1
            assert len(links) >= 1 and not occ[s][np.ix_(links, range(q0, q0 + w))].any()
            continue
        assert ptr[s] <= node < ptr[s + 1] and s != 5
        conn = int(st.conn_ids[node])
        mine = occ[s] & (np.trunc(data[s, fi["conn_id"]]) == conn)
        assert mine.any()                                            # the node is that lightpath of that sample
        ls, qs = np.nonzero(mine)
        own_links, q_own, w_own = sorted(set(ls.tolist())), int(qs.min()), int(qs.max() - qs.min() + 1)
        assert w == w_own
        assert c.feat[k, 1].item() == data[s, fi["mod_order"], ls[0], qs[0]]
        if len(links) == 0:
            kinds["teardown"] += 1
            continue
        assert c.feat[k, 0].item() == np.float32(freqs[q0])
        chans = np.zeros_like(mine)
        chans[np.ix_(links, range(q0, q0 + w))] = True
        assert not (chans & occ[s] & ~mine).any()                   # free or the lightpath's own
        if sorted(links.tolist()) == own_links:
            kinds["retune"] += 1
            kinds["overlap"] += int((chans & mine).any())
        else:
            kinds["reroute"] += 1
    assert min(kinds.values()) > 0, kinds


def _script():
    import sys
    sys.path.insert(0, str(ROOT / "scripts"))
    spec = importlib.util.spec_from_file_location("time_reconfig", ROOT / "scripts" / "time_reconfig.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_timing_script_arguments_and_bytes():
    mod = _script()
    a = mod.parse_args([])
    assert (a.states, a.links, a.freqs, a.changes, a.expand, a.max_impact) == (64, 60, 80, 65536, 4096, 64)
    a = mod.parse_args(["--states", "2", "--changes", "8", "--expand", "3", "--max-impact", "0"])
    assert (a.states, a.changes, a.expand, a.max_impact) == (2, 8, 3, 0)
    for bad in (["--expand", "0"], ["--states", "4", "--changes", "3"], ["--max-impact", "-1"]):
        with pytest.raises(SystemExit):
            mod.parse_args(bad)
    # K (48 + 20 + 21 MI) + links (4 + 4 Q) + 36 impact rows + 8 row edges + 16 moved + 8 moved edges
    assert mod.algorithmic_bytes(2, 5, 80, 7, 30, 4, 1, 6) == 2 * 152 + 5 * 324 + 252 + 240 + 16 + 48
    tc = importlib.util.spec_from_file_location("time_candidates", ROOT / "scripts" / "time_candidates.py")
    tcm = importlib.util.module_from_spec(tc)
    tc.loader.exec_module(tcm)
    # with no node / kind bytes and no moved lightpath, the candidate terms
    assert mod.algorithmic_bytes(3, 5, 80, 7, 30, 0, 0, 0) - 3 * 8 == tcm.algorithmic_bytes(3, 5, 80, 7, 30, 0)


def test_timing_script_expansion_inputs():
    """Moves clear the lightpath's conn_id and write its first channel with the new feat; insertions take a new
    conn_id; teardowns write nothing."""
    from gnn_qot_estimation_b200 import synthetic
    mod = _script()
    smp = synthetic.network_status_samples(3, num_links=10, num_freqs=20, seed=1)
    st = fake_state(smp)
    c = synthetic.lightpath_changes(smp, st, 12, seed=2)
    X = 30
    smp_k, conn, vec, ck, cl, cq = mod.expansion_inputs(smp, c, st.conn_ids.numpy(), X)
    assert torch.equal(smp_k, c.sample[:X])
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    data = smp["data"]
    seen = set()
    for k in range(X):
        s, node = int(smp_k[k]), int(c.node[k])
        top = np.trunc(data[s, fi["conn_id"]]).max()
        if node < 0:
            assert int(conn[k]) == top + 1 and float(vec[k, fi["osnr"]]) == -1.0
            seen.add("insert")
        else:
            assert int(conn[k]) == int(st.conn_ids[node])
            mine = np.any(data[s] != 0, axis=0) & (np.trunc(data[s, fi["conn_id"]]) == int(conn[k]))
            ls, qs = np.nonzero(mine)
            first = data[s, :, ls[0], qs[0]]
            for name in ("conn_id", "src_id", "dst_id", "osnr", "snr", "ber"):
                assert float(vec[k, fi[name]]) == first[fi[name]]
        for i, name in enumerate(("freq", "mod_order", "num_spans", "path_len")):
            assert float(vec[k, fi[name]]) == float(c.feat[k, i])
        got = {(int(l), int(q)) for l, q in zip(cl[ck == k], cq[ck == k])}
        links = c.links[int(c.link_ptr[k]):int(c.link_ptr[k + 1])].tolist()
        want = {(l, q) for l in links for q in range(int(c.q0[k]), int(c.q0[k]) + int(c.width[k]))}
        assert got == want
        if node >= 0 and not links:
            seen.add("teardown")
    assert seen == {"insert", "teardown"}
