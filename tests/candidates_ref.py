"""Reference for LightpathGNN's candidate QoT (TEST INFRASTRUCTURE, like every_node_ref.py): a candidate lightpath
written literally into a numpy copy of its sample, the graph rebuilt with the numpy restatement of to_graph
(oracle.lightpath_data_ref), one one-hot copy of that graph per evaluated node, all run through the oracle model."""
from types import SimpleNamespace

import numpy as np
import torch

from oracle.to_graph_oracle import lightpath_data_ref

METRIC = ["osnr", "snr", "ber"]


def insert_candidate(sample, lp_feat, links, q0, width, feat):
    """sample [F, L, Q] -> (copy with the candidate on every channel of its path and slot range, its conn_id).  The
    conn_id is one above the sample's largest; features ``feat = (freq, mod_order, num_spans, path_len)``; osnr = snr =
    ber = -1; other rows 0."""
    fi = {k: i for i, k in enumerate(lp_feat)}
    out = np.array(sample, dtype=np.float32, copy=True)
    conn = int(np.trunc(out[fi["conn_id"]]).max(initial=0)) + 1
    vec = np.zeros(out.shape[0], dtype=np.float32)
    vec[fi["conn_id"]] = conn
    for k, name in enumerate(("freq", "mod_order", "num_spans", "path_len")):
        vec[fi[name]] = np.float32(feat[k])
    vec[fi["osnr"]] = vec[fi["snr"]] = vec[fi["ber"]] = -1.0
    for l in links:
        out[:, l, q0:q0 + width] = vec[:, None]
    return out, conn


def candidates_ref(model, sample, freqs, lp_feat, links, q0, width, feat, freq_threshold=0.05):
    """Candidate QoT of one candidate, defined literally.  Returns ``(row [3], {conn_id: row [3]})``: the candidate's
    row (flag one-hot at its node) and, for every existing lightpath adjacent to it in the rebuilt graph, that
    lightpath's row (flag one-hot there).  Runs on ``model``'s dtype, on the CPU."""
    s2, conn = insert_candidate(sample, lp_feat, links, q0, width, feat)
    conns, x, _, ei = lightpath_data_ref(s2, np.zeros(3), freqs, lp_feat, METRIC, freq_threshold)
    c = int(np.flatnonzero(conns == conn)[0])
    nbr = sorted({int(d) for s, d in ei.T if s == c and d != c})
    rows = [c] + nbr
    dt = next(model.parameters()).dtype
    n, R = x.shape[0], len(rows)
    xc = torch.from_numpy(np.tile(x, (R, 1))).to(dt)
    flag = torch.zeros(R * n, dtype=dt)
    flag[torch.arange(R) * n + torch.tensor(rows)] = 1.0
    xc[:, model.is_lut_index] = flag
    e = torch.from_numpy(ei)
    eic = torch.cat([e + r * n for r in range(R)], 1)
    bt = torch.repeat_interleave(torch.arange(R), n)
    with torch.no_grad():
        out, lut_batch = model(SimpleNamespace(x=xc, edge_index=eic, batch=bt, num_graphs=R))
    assert torch.equal(lut_batch, torch.arange(R)), "every copy has exactly one readout row"
    return out[0], {int(conns[j]): out[i + 1] for i, j in enumerate(nbr)}
