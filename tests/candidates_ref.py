"""Reference for LightpathGNN's candidate QoT (TEST INFRASTRUCTURE, like every_node_ref.py): a candidate lightpath
written literally into a numpy copy of its sample, the graph rebuilt with the numpy restatement of to_graph
(oracle.lightpath_data_ref), one one-hot copy of that graph per evaluated node, all run through the oracle model."""
import numpy as np

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


def candidates_ref(model, sample, freqs, lp_feat, links, q0, width, feat, freq_threshold=0.05, chunk=None, device=None):
    """Candidate QoT of one candidate, defined literally.  Returns ``(row [3], {conn_id: row [3]})``: the candidate's
    row (flag one-hot at its node) and, for every existing lightpath adjacent to it in the rebuilt graph, that
    lightpath's row (flag one-hot there).  Runs on ``model``'s dtype, on ``device`` (default: the CPU), ``chunk`` copies
    per oracle call (see ``reconfig_ref._rows``); rows come back on the CPU."""
    from reconfig_ref import _rows
    s2, conn = insert_candidate(sample, lp_feat, links, q0, width, feat)
    conns, x, _, ei = lightpath_data_ref(s2, np.zeros(3), freqs, lp_feat, METRIC, freq_threshold)
    c = int(np.flatnonzero(conns == conn)[0])
    nbr = sorted({int(d) for s, d in ei.T if s == c and d != c})
    out = _rows(model, x, ei, [c] + nbr, chunk, device)
    return out[0], {int(conns[j]): out[i + 1] for i, j in enumerate(nbr)}
