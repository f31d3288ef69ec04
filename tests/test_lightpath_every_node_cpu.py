"""CPU checks of LightpathGNN's every-node mode: the C ABI declares and binds it, the literal reference definition
(K one-hot copies of every graph) equals a direct evaluation from each node's 1-hop neighbourhood -- the locality the
kernel rests on -- and the timing script's argument parsing and byte / expansion arithmetic."""
import importlib.util
import re
from pathlib import Path
from types import SimpleNamespace

import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]
HEADER = ROOT / "include" / "qot_b200.h"
EVERY_NODE = ("qot_lightpath_every_node_tiles", "qot_lightpath_infer_every_node")


def _header_arity(name):
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", text, flags=re.S)
    assert m, name
    return m.group(1).count(",") + 1


def test_header_declares_and_ctypes_binds_every_node_family():
    from gnn_qot_estimation_b200 import _lib
    for name in EVERY_NODE:
        assert name in _lib.SIGNATURES, name
        assert len(_lib.SIGNATURES[name][1]) == _header_arity(name), name
    assert _header_arity("qot_lightpath_infer_every_node") == 8


def _oracle(seed=0):
    from oracle import LightpathGNNOracle
    torch.manual_seed(seed)
    m = LightpathGNNOracle(5, 32, 3, is_lut_index=1, dropout_p=0.0).double()
    bn = m.norm1.module if hasattr(m.norm1, "module") else m.norm1
    for name, buf in bn.named_buffers():
        if name == "running_mean":
            buf.uniform_(-0.5, 0.5)
        elif name == "running_var":
            buf.uniform_(0.5, 2.0)
    return m.eval()


def _random_batch(g, sizes, flags="random"):
    xs, eis, bts, off = [], [], [], 0
    for gi, n in enumerate(sizes):
        x = torch.rand(n, 5, generator=g, dtype=torch.float64)
        x[:, 1] = torch.rand(n, generator=g, dtype=torch.float64) if flags == "random" else 0.0
        E = 4 * n if gi % 3 else 0 if n < 3 else 2 * n
        src = torch.randint(0, n, (E,), generator=g)
        dst = torch.randint(0, n, (E,), generator=g)      # self loops and duplicates included
        eis.append(torch.stack([src, dst]) + off)
        xs.append(x)
        bts.append(torch.full((n,), gi, dtype=torch.int64))
        off += n
    return SimpleNamespace(x=torch.cat(xs), edge_index=torch.cat(eis, 1), batch=torch.cat(bts))


def _one_hop(model, data, v):
    """Node v as the LUT from its 1-hop in-neighbourhood alone: a star graph j -> v over v's in-edges (self loops
    dropped, duplicates kept, edge order), v's flag 1.0 and every neighbour's 0.0."""
    src, dst = data.edge_index
    nb = src[(dst == v) & (src != v)]
    ids = torch.cat([torch.tensor([v]), nb])
    x = data.x[ids].clone()
    x[:, model.is_lut_index] = 0.0
    x[0, model.is_lut_index] = 1.0
    k = nb.numel()
    ei = torch.stack([torch.arange(1, k + 1), torch.zeros(k, dtype=torch.int64)])
    out, _ = model(SimpleNamespace(x=x, edge_index=ei, batch=torch.zeros(k + 1, dtype=torch.int64)))
    return out[0]


def test_every_node_ref_equals_one_hop_evaluation():
    from every_node_ref import lightpath_every_node_ref
    g = torch.Generator().manual_seed(5)
    m = _oracle()
    data = _random_batch(g, [1, 2, 7, 13, 5, 20])
    with torch.no_grad():
        ref = lightpath_every_node_ref(m, data)
        direct = torch.stack([_one_hop(m, data, v) for v in range(data.x.shape[0])])
    assert ref.shape == (data.x.shape[0], 3)
    torch.testing.assert_close(ref, direct, rtol=1e-12, atol=1e-12)


def test_every_node_ref_ignores_stored_flags():
    from every_node_ref import lightpath_every_node_ref
    g = torch.Generator().manual_seed(6)
    m = _oracle(1)
    data = _random_batch(g, [4, 9, 11])
    zero = SimpleNamespace(x=data.x.clone(), edge_index=data.edge_index, batch=data.batch)
    zero.x[:, 1] = 0.0
    with torch.no_grad():
        torch.testing.assert_close(lightpath_every_node_ref(m, data), lightpath_every_node_ref(m, zero),
                                   rtol=0, atol=0)


def _script():
    spec = importlib.util.spec_from_file_location("time_every_node", ROOT / "scripts" / "time_every_node.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_timing_script_arguments_and_bytes():
    mod = _script()
    a = mod.parse_args([])
    assert (a.batches, a.batch_size, a.expand, a.seed) == (64, 4096, 8, 1)
    a = mod.parse_args(["--batches", "2", "--batch-size", "3", "--expand", "1"])
    assert (a.batches, a.batch_size, a.expand) == (2, 3, 1)
    with pytest.raises(SystemExit):
        mod.parse_args(["--batches", "2", "--expand", "3"])
    # 20N + 8E (+ 8E unverified) + 16(B+1) + 12N
    assert mod.algorithmic_bytes(10, 7, 2, True) == 200 + 56 + 48 + 120
    assert mod.algorithmic_bytes(10, 7, 2, False) == 200 + 112 + 48 + 120
    assert mod.head_flops(16) == 240 * 1024 * 2


def test_timing_script_expansion_matches_oracle_copies():
    """The expansion the script times row for row against equals the oracle's one-hot copies."""
    from every_node_ref import lightpath_every_node_ref
    mod = _script()
    g = torch.Generator().manual_seed(7)
    data = _random_batch(g, [3, 1, 6, 4], flags="zero")
    m = _oracle(2)
    xc, eic, bt, p, ep = mod.one_hot_expansion(data.x, data.edge_index, data.batch, 1)
    N = data.x.shape[0]
    assert p.numel() == N + 1 and int(p[-1]) == xc.shape[0] and int(ep[-1]) == eic.shape[1]
    idx = (xc[:, 1] == 1.0).nonzero().flatten()
    assert torch.equal(bt[idx], torch.arange(N))                          # one flagged node per copy, in copy order
    assert torch.equal(xc[idx][:, [0, 2, 3, 4]], data.x[:, [0, 2, 3, 4]])  # copy c flags node c
    with torch.no_grad():
        out, lb = m(SimpleNamespace(x=xc, edge_index=eic, batch=bt))
        torch.testing.assert_close(out, lightpath_every_node_ref(m, data), rtol=1e-12, atol=1e-12)
    assert torch.equal(lb, torch.arange(N))
