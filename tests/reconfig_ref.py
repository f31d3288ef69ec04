"""Reference for LightpathGNN's reconfiguration QoT (TEST INFRASTRUCTURE, like candidates_ref.py): a lightpath removed
from a numpy copy of its sample and written back literally on its new path and slots (or not at all: a teardown), the
graph rebuilt with the numpy restatement of to_graph (oracle.lightpath_data_ref), one one-hot copy of that graph per
evaluated node, all run through the oracle model."""
from types import SimpleNamespace

import numpy as np
import torch

from candidates_ref import METRIC, insert_candidate
from oracle.to_graph_oracle import lightpath_data_ref


def rewrite_lightpath(sample, lp_feat, conn_id, links, q0, width, feat):
    """sample [F, L, Q] -> copy with every channel of lightpath ``conn_id`` zeroed and, for a non-empty path, one vector
    written on every channel of ``links`` x ``[q0, q0 + width)``: conn_id, ``feat = (freq, mod_order, num_spans,
    path_len)``, and every other row (src/dst, metrics) from the lightpath's first channel (row-major)."""
    fi = {k: i for i, k in enumerate(lp_feat)}
    out = np.array(sample, dtype=np.float32, copy=True)
    mine = np.any(out != 0, axis=0) & (np.trunc(out[fi["conn_id"]]) == conn_id)
    ls, qs = np.nonzero(mine)
    assert ls.size, f"lightpath {conn_id} is not in the sample"
    vec = out[:, ls[0], qs[0]].copy()
    for k, name in enumerate(("freq", "mod_order", "num_spans", "path_len")):
        vec[fi[name]] = np.float32(feat[k])
    out[:, mine] = 0.0
    for l in links:
        out[:, l, q0:q0 + width] = vec[:, None]
    return out


def _rows(model, x, ei, rows, chunk=None, device=None):
    """Eval forward of one one-hot copy of the graph per entry of ``rows`` -> [len(rows), 3] on the CPU.  ``chunk``:
    copies per oracle call (None: all at once; a dense graph's copies can outgrow memory), results concatenated.
    ``device``: where the copies are evaluated (``model`` must be there; None: the CPU)."""
    dt = next(model.parameters()).dtype
    n, R = x.shape[0], len(rows)
    if R == 0:
        return torch.zeros(0, 3, dtype=dt)
    step = R if chunk is None else int(chunk)
    assert step > 0
    outs = []
    for c0 in range(0, R, step):
        part = rows[c0:c0 + step]
        P = len(part)
        xc = torch.from_numpy(np.tile(x, (P, 1))).to(device=device, dtype=dt)
        flag = torch.zeros(P * n, dtype=dt, device=device)
        flag[torch.arange(P, device=device) * n + torch.tensor(part, device=device)] = 1.0
        xc[:, model.is_lut_index] = flag
        e = torch.from_numpy(ei).to(device)
        eic = torch.cat([e + r * n for r in range(P)], 1)
        bt = torch.repeat_interleave(torch.arange(P, device=device), n)
        with torch.no_grad():
            out, lut_batch = model(SimpleNamespace(x=xc, edge_index=eic, batch=bt, num_graphs=P))
        assert torch.equal(lut_batch.cpu(), torch.arange(P)), "every copy has exactly one readout row"
        outs.append(out.cpu())
    return torch.cat(outs)


def _neighbours(conns, ei, c):
    """conn_ids adjacent to lightpath c in a rebuilt graph (self loops aside); empty if c is not in it."""
    hit = np.flatnonzero(conns == c)
    if hit.size == 0:
        return set()
    v = int(hit[0])
    return {int(conns[d]) for s, d in ei.T if s == v and d != v}


def reconfig_ref(model, sample, freqs, lp_feat, conn_id, links, q0, width, feat, freq_threshold=0.05, chunk=None,
                 device=None):
    """Reconfiguration QoT of one change, defined literally.  ``conn_id`` is the moved lightpath (None: an insertion,
    written as candidates_ref.insert_candidate writes it); an empty ``links`` is a teardown.  Returns ``(row [3] or
    None, {conn_id: (kind, row [3])})``: the moved lightpath's row at its new placement (flag one-hot there; None for a
    teardown) and, for every other lightpath that was adjacent to it in the original graph (kind bit 0) or is adjacent
    to it in the rebuilt graph (kind bit 1), that lightpath's row (flag one-hot there).  Runs on ``model``'s dtype, on
    ``device`` (default: the CPU), ``chunk`` copies per oracle call (see ``_rows``); rows come back on the CPU."""
    if conn_id is None:
        s2, c = insert_candidate(sample, lp_feat, links, q0, width, feat)
        old = set()
    else:
        c = int(conn_id)
        s2 = rewrite_lightpath(sample, lp_feat, c, links, q0, width, feat)
        conns0, _, _, ei0 = lightpath_data_ref(sample, np.zeros(3), freqs, lp_feat, METRIC, freq_threshold)
        old = _neighbours(conns0, ei0, c)
    conns, x, _, ei = lightpath_data_ref(s2, np.zeros(3), freqs, lp_feat, METRIC, freq_threshold)
    new = _neighbours(conns, ei, c)
    node_of = {int(v): i for i, v in enumerate(conns)}
    others = sorted(old | new)
    own = [node_of[c]] if len(links) else []
    out = _rows(model, x, ei, own + [node_of[o] for o in others], chunk, device)
    row = out[0] if own else None
    rest = out[len(own):]
    return row, {o: (int(o in old) | int(o in new) << 1, rest[i]) for i, o in enumerate(others)}
