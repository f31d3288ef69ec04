"""Reference for LightpathGNN's placement search (TEST INFRASTRUCTURE, like candidates_ref.py): every free start slot of
every option of a demand evaluated literally with candidates_ref (the placement written into a numpy copy of its
sample, the graph rebuilt with the oracle's to_graph, one one-hot copy per row), then the margins, the counts and the
policy applied as LightpathGNN.forward_placements defines them.  Margins are taken in the model's dtype (fp64 on the
fp64 oracle)."""
import numpy as np

from candidates_ref import candidates_ref

FIRST_FIT, BEST_QOT, MAX_MARGIN = 0, 1, 2


def free_starts(sample, links, width):
    """Start slots q0 in [0, Q - width] whose channels [q0, q0 + width) are free on every link of the route."""
    occ = np.any(np.asarray(sample) != 0, axis=0)[list(links)].any(axis=0)   # [Q]
    Q = occ.shape[0]
    return [q for q in range(Q - width + 1) if not occ[q:q + width].any()]


def placement_table(model, sample, freqs, lp_feat, options, metric=0, maximize=True, bound=None, freq_threshold=0.05,
                    chunk=None, device=None):
    """{(p, q0): (own row [3], {conn_id: row [3]}, margin)} over every free placement of ``options`` = [(links, width,
    (mod_order, num_spans, path_len), own_bound)].  ``bound``: {conn_id: bound} over the sample's lightpaths, or None
    (impact rows unconstrained).  A margin is v - b (maximize) or b - v, the minimum over the own row and, with a
    bound, every impact row; NaN if any is NaN."""
    table = {}
    for p, (links, width, feat3, own_bound) in enumerate(options):
        for q0 in free_starts(sample, links, width):
            feat = [np.float32(freqs[q0])] + [float(v) for v in feat3]
            row, imp = candidates_ref(model, sample, freqs, lp_feat, links, q0, width, feat, freq_threshold, chunk,
                                      device)
            sign = 1.0 if maximize else -1.0
            ms = [sign * (float(row[metric]) - float(own_bound))]
            if bound is not None:
                ms += [sign * (float(r[metric]) - float(bound[c])) for c, r in imp.items()]
            mg = float("nan") if any(np.isnan(ms)) else min(ms)
            table[(p, q0)] = (row, imp, mg)
    return table


def choose(table, policy, metric=0, maximize=True):
    """(p, q0) the policy picks from a placement table (None if no placement is feasible), n_free, n_feasible."""
    feas = sorted(k for k, (_, _, mg) in table.items() if mg >= 0)        # NaN >= 0 is False
    if not feas:
        return None, len(table), 0
    if policy == FIRST_FIT:
        best = feas[0]
    elif policy == BEST_QOT:
        sign = 1.0 if maximize else -1.0
        best = max(feas, key=lambda k: (sign * float(table[k][0][metric]), -k[0], -k[1]))
    else:
        best = max(feas, key=lambda k: (table[k][2], -k[0], -k[1]))
    return best, len(table), len(feas)


def placement_ref(model, sample, freqs, lp_feat, options, policy, metric=0, maximize=True, bound=None,
                  freq_threshold=0.05, chunk=None, device=None):
    """Placement of one demand, defined literally.  Returns ``(choice, n_free, n_feasible, table)``: the (option, q0)
    the policy picks or None, the counts over every placement, and the per-placement table of ``placement_table``."""
    table = placement_table(model, sample, freqs, lp_feat, options, metric, maximize, bound, freq_threshold, chunk,
                            device)
    best, n_free, n_feas = choose(table, policy, metric, maximize)
    return best, n_free, n_feas, table
