"""CPU checks of LightpathGNN's candidate QoT: the C ABI declares and binds it, the literal reference definition
(tests/candidates_ref.py) agrees with every-node mode by leave-one-out on the oracle, the seeded candidate generator
uses free channels only, and the timing script's argument parsing and byte arithmetic."""
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
CANDIDATES = ("qot_lightpath_channel_map", "qot_lightpath_candidates")


def _header_arity(name):
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", text, flags=re.S)
    assert m, name
    return m.group(1).count(",") + 1


def test_candidate_family_takes_state_and_changes_structs():
    from gnn_qot_estimation_b200 import _lib, ops
    for name in CANDIDATES:
        assert name in _lib.SIGNATURES, name
        assert len(_lib.SIGNATURES[name][1]) == _header_arity(name), name
    assert _header_arity("qot_lightpath_candidates") == 11
    # the state, then the candidates
    assert _lib.SIGNATURES["qot_lightpath_candidates"][1][:2] == [C.POINTER(_lib.QotLpState),
                                                                  C.POINTER(_lib.QotLpChanges)]
    text = HEADER.read_text()
    bits = {name: int(re.search(r"#define " + name + r"\s+(\d+)", text).group(1))
            for name in ("QOT_CAND_BAD_SAMPLE", "QOT_CAND_BAD_PATH", "QOT_CAND_OCCUPIED", "QOT_CAND_IMPACT_OVERFLOW",
                         "QOT_CAND_BAD_STATE")}
    assert bits == {"QOT_CAND_BAD_SAMPLE": ops.CAND_BAD_SAMPLE, "QOT_CAND_BAD_PATH": ops.CAND_BAD_PATH,
                    "QOT_CAND_OCCUPIED": ops.CAND_OCCUPIED, "QOT_CAND_IMPACT_OVERFLOW": ops.CAND_IMPACT_OVERFLOW,
                    "QOT_CAND_BAD_STATE": ops.CAND_BAD_STATE}


def _oracle64():
    from oracle import LightpathGNNOracle
    m = LightpathGNNOracle(5, 32, 3, is_lut_index=1, dropout_p=0.0).double()
    m.load_state_dict(load_golden("ckpt_lightpath_model_1.pt")["model_state_dict"], strict=True)
    return m.eval()


def lightpath_as_candidate(sample, lp_feat, conn):
    """(sample without lightpath `conn`, its links, q0, width, feat) -- the lightpath offered back as a candidate."""
    fi = {k: i for i, k in enumerate(lp_feat)}
    occ = np.any(sample != 0, axis=0)
    mine = occ & (np.trunc(sample[fi["conn_id"]]) == conn)
    ls, qs = np.nonzero(mine)                                   # row-major: (ls[0], qs[0]) is the first channel
    links = sorted(set(ls.tolist()))
    q0, width = int(qs.min()), int(qs.max() - qs.min() + 1)
    assert mine.sum() == len(links) * width                     # same contiguous slots on every link
    feat = [sample[fi[k], ls[0], qs[0]] for k in ("freq", "mod_order", "num_spans", "path_len")]
    rest = sample.copy()
    rest[:, mine] = 0.0
    return rest, links, q0, width, feat


def test_leave_one_out_on_the_oracle_matches_every_node():
    """Remove lightpath j from a sample, offer it back as a candidate: its row is the every-node row of j in the
    original sample, its impact rows are the every-node rows of j's neighbours there."""
    from candidates_ref import candidates_ref
    from every_node_ref import lightpath_every_node_ref
    from gnn_qot_estimation_b200 import synthetic
    from oracle.to_graph_oracle import lightpath_data_ref
    m = _oracle64()
    smp = synthetic.network_status_samples(3, num_links=12, num_freqs=24, seed=8, max_lightpaths=14,
                                           super_channel_p=0.3)
    checked_impact = 0
    for s in range(3):
        sample = smp["data"][s]
        conns, x, _, ei = lightpath_data_ref(sample, np.zeros(3), smp["freqs"], smp["lp_feat"], ["osnr", "snr", "ber"])
        with torch.no_grad():
            every = lightpath_every_node_ref(m, SimpleNamespace(
                x=torch.from_numpy(x).double(), edge_index=torch.from_numpy(ei),
                batch=torch.zeros(x.shape[0], dtype=torch.int64)))
        row_of = {int(c): i for i, c in enumerate(conns)}
        for j, c in enumerate(conns):
            rest, links, q0, width, feat = lightpath_as_candidate(sample, smp["lp_feat"], int(c))
            row, impact = candidates_ref(m, rest, smp["freqs"], smp["lp_feat"], links, q0, width, feat)
            torch.testing.assert_close(row, every[j], rtol=1e-12, atol=1e-12)
            nbr = {int(conns[d]) for s_, d in ei.T if s_ == j and d != j}
            assert set(impact) == nbr
            for cj, r in impact.items():
                torch.testing.assert_close(r, every[row_of[cj]], rtol=1e-12, atol=1e-12)
                checked_impact += 1
    assert checked_impact > 20


def test_candidate_ref_threshold_boundary_follows_numpy():
    """Spacing 0.05 on a 0.05 threshold: the neighbours are exactly what numpy's |df| < 0.05 says (192.2 + k*0.05 in
    fp64 gives differences on both sides of 0.05)."""
    from candidates_ref import candidates_ref, insert_candidate
    from gnn_qot_estimation_b200 import synthetic
    smp = synthetic.network_status_samples(1, num_links=4, num_freqs=16, seed=2, spacing=0.05, max_lightpaths=10)
    freqs = smp["freqs"]
    sample = smp["data"][0]
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    occ = np.any(sample != 0, axis=0)
    m = _oracle64()
    seen_adjacent = 0
    for l in range(4):
        for q in np.flatnonzero(~occ[l]):
            _, impact = candidates_ref(m, sample, freqs, smp["lp_feat"], [l], int(q), 1,
                                       [np.float32(freqs[q]), 16, 10, 100000])
            want = set()
            for qj in np.flatnonzero(occ[l]):
                df = abs(freqs[q] - freqs[qj])
                if 0 < df < 0.05:
                    want.add(int(np.trunc(sample[fi["conn_id"], l, qj])))
            assert set(impact) == want
            seen_adjacent += len(want)
    assert insert_candidate(sample, smp["lp_feat"], [0], 0, 1, [192.2, 4, 1, 24214])[1] > 0
    # at spacing 0.05 some neighbouring slots are adjacent and some are not, depending on fp64 rounding
    d = np.abs(np.diff(freqs))
    assert (d < 0.05).any() and (d >= 0.05).any()
    assert seen_adjacent > 0


def test_synthetic_candidates_use_free_channels_and_are_seeded():
    from gnn_qot_estimation_b200 import synthetic
    smp = synthetic.network_status_samples(6, num_links=20, num_freqs=32, seed=4)
    c = synthetic.lightpath_candidates(smp, 50, seed=3)
    c2 = synthetic.lightpath_candidates(smp, 50, seed=3)
    assert all(torch.equal(a, b) for a, b in zip(c, c2))
    c3 = synthetic.lightpath_candidates(smp, 50, seed=4)
    assert not torch.equal(c.q0, c3.q0)
    K = c.sample.shape[0]
    assert K == 300
    assert (c.sample.dtype, c.link_ptr.dtype, c.links.dtype, c.q0.dtype, c.width.dtype, c.feat.dtype) == \
        (torch.int64, torch.int64, torch.int32, torch.int32, torch.int32, torch.float32)
    assert c.link_ptr.shape == (K + 1,) and int(c.link_ptr[0]) == 0 and int(c.link_ptr[-1]) == c.links.numel()
    n = (c.link_ptr[1:] - c.link_ptr[:-1]).numpy()
    assert n.min() >= 1 and n.max() <= 6
    assert set(c.width.tolist()) <= {1, 2}
    occ = np.any(smp["data"] != 0, axis=1)
    for k in range(K):
        s, q0, w = int(c.sample[k]), int(c.q0[k]), int(c.width[k])
        links = c.links[int(c.link_ptr[k]):int(c.link_ptr[k + 1])].numpy()
        assert len(set(links.tolist())) == len(links)
        assert 0 <= q0 and q0 + w <= 32
        assert not occ[s][np.ix_(links, np.arange(q0, q0 + w))].any()
        assert c.feat[k, 0].item() == np.float32(smp["freqs"][q0])


def _script():
    spec = importlib.util.spec_from_file_location("time_candidates", ROOT / "scripts" / "time_candidates.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_timing_script_arguments_and_bytes():
    mod = _script()
    a = mod.parse_args([])
    assert (a.states, a.links, a.freqs, a.candidates, a.expand, a.max_impact) == (64, 60, 80, 65536, 4096, 64)
    a = mod.parse_args(["--states", "2", "--candidates", "8", "--expand", "3", "--max-impact", "0"])
    assert (a.states, a.candidates, a.expand, a.max_impact) == (2, 8, 3, 0)
    for bad in (["--expand", "0"], ["--states", "4", "--candidates", "3"], ["--max-impact", "-1"]):
        with pytest.raises(SystemExit):
            mod.parse_args(bad)
    # K (40 + 20 + 20 MI) + links (4 + 4 Q) + 36 impact rows + 8 row edges
    assert mod.algorithmic_bytes(2, 5, 80, 7, 30, 4) == 2 * 140 + 5 * 324 + 252 + 240
    assert mod.head_mmas(32) == 480


def test_timing_script_expansion_inputs():
    """The channels the expansion path writes are the candidates' paths x slot ranges, conn_ids new per sample."""
    from gnn_qot_estimation_b200 import synthetic
    mod = _script()
    smp = synthetic.network_status_samples(3, num_links=10, num_freqs=20, seed=1)
    c = synthetic.lightpath_candidates(smp, 4, seed=2)
    smp_k, conn, ck, cl, cq = mod.expansion_inputs(smp, c, 5)
    assert torch.equal(smp_k, c.sample[:5])
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    for k in range(5):
        s = int(smp_k[k])
        assert int(conn[k]) > np.trunc(smp["data"][s, fi["conn_id"]]).max()
        got = {(int(l), int(q)) for l, q in zip(cl[ck == k], cq[ck == k])}
        links = c.links[int(c.link_ptr[k]):int(c.link_ptr[k + 1])].tolist()
        want = {(l, q) for l in links for q in range(int(c.q0[k]), int(c.q0[k]) + int(c.width[k]))}
        assert got == want
    v = mod.channel_vectors(smp["lp_feat"], conn, c.feat[:5])
    assert torch.equal(v[:, fi["conn_id"]], conn.float())
    assert bool((v[:, fi["osnr"]] == -1).all()) and torch.equal(v[:, fi["freq"]], c.feat[:5, 0])
