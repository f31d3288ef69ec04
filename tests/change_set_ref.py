"""Reference for LightpathGNN's change-set QoT (TEST INFRASTRUCTURE, like reconfig_ref.py): every lightpath the set moves
or tears down cleared from a numpy copy of its sample, every placement written back literally, the graph rebuilt with
the numpy restatement of to_graph (oracle.lightpath_data_ref), one one-hot copy of that graph per evaluated node, all
run through the oracle model."""
import numpy as np

from candidates_ref import METRIC, insert_candidate
from oracle.to_graph_oracle import lightpath_data_ref
from reconfig_ref import _neighbours, _rows, rewrite_lightpath


def apply_set(sample, lp_feat, changes):
    """sample [F, L, Q] -> (sample', conn_id of each change).  ``changes``: [(conn_id or None, links, q0, width, feat)].
    Step 1 clears every channel of every lightpath a change names; step 2 writes each change with a non-empty path on
    its links x slots: a move with the vector ``rewrite_lightpath`` writes, an insertion with the vector
    ``insert_candidate`` writes and conn_id one above the sample's largest, +1 per insertion in set order."""
    fi = {k: i for i, k in enumerate(lp_feat)}
    top = int(np.trunc(np.asarray(sample)[fi["conn_id"]]).max(initial=0))
    out = np.array(sample, dtype=np.float32, copy=True)
    for c, links, q0, width, feat in changes:
        if c is not None:
            out = rewrite_lightpath(out, lp_feat, int(c), [], 0, 0, feat)
    conns, taken, ins = [], np.zeros(out.shape[1:], dtype=bool), 0
    for c, links, q0, width, feat in changes:
        if len(links) == 0:
            conns.append(None if c is None else int(c))
            continue
        if c is None:
            s2, _ = insert_candidate(sample, lp_feat, links, q0, width, feat)
            ins += 1
            conn = top + ins
        else:
            s2, conn = rewrite_lightpath(sample, lp_feat, int(c), links, q0, width, feat), int(c)
        vec = s2[:, links[0], q0].copy()
        vec[fi["conn_id"]] = conn
        for l in links:
            assert not taken[l, q0:q0 + width].any(), "the placements of a set must be disjoint"
            taken[l, q0:q0 + width] = True
            out[:, l, q0:q0 + width] = vec[:, None]
        conns.append(conn)
    return out, conns


def change_set_ref(model, sample, freqs, lp_feat, changes, freq_threshold=0.05, chunk=None, device=None):
    """Change-set QoT of one set, defined literally.  ``changes``: [(conn_id or None, links, q0, width, feat)], a move
    (conn_id and a path), a teardown (conn_id and an empty path) or an insertion (None).  Returns ``(rows, {conn_id:
    (kind, row [3])})``: per change its row at its new placement (flag one-hot there; None for a teardown) and, for
    every lightpath of the sample the set does not name that was adjacent to a removed one in the original graph (kind
    bit 0) or is adjacent to a changed one in the rebuilt graph (kind bit 1), its row.  Runs on ``model``'s dtype, on
    ``device`` (default: the CPU), ``chunk`` copies per oracle call (see ``reconfig_ref._rows``); rows come back on the CPU."""
    s2, conns = apply_set(sample, lp_feat, changes)
    removed = {int(c) for c, *_ in changes if c is not None}
    changed = {c for c, ch in zip(conns, changes) if c is not None and len(ch[1])}
    conns0, _, _, ei0 = lightpath_data_ref(sample, np.zeros(3), freqs, lp_feat, METRIC, freq_threshold)
    old = set().union(*[_neighbours(conns0, ei0, c) for c in removed]) - removed
    conns1, x, _, ei = lightpath_data_ref(s2, np.zeros(3), freqs, lp_feat, METRIC, freq_threshold)
    new = set().union(*[_neighbours(conns1, ei, c) for c in changed]) - changed - removed
    node_of = {int(v): i for i, v in enumerate(conns1)}
    others = sorted(old | new)
    own = [node_of[c] for c, ch in zip(conns, changes) if len(ch[1])]
    out = _rows(model, x, ei, own + [node_of[o] for o in others], chunk, device)
    rows, r = [], 0
    for ch in changes:
        rows.append(out[r] if len(ch[1]) else None)
        r += int(len(ch[1]) > 0)
    rest = out[len(own):]
    return rows, {o: (int(o in old) | int(o in new) << 1, rest[i]) for i, o in enumerate(others)}
