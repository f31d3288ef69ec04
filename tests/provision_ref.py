"""References for LightpathGNN's sequential provisioning (TEST INFRASTRUCTURE, like placement_ref.py).

``provision_ref``: the demands of one sample placed literally, one after another: ``placement_ref`` on the current
numpy sample, the chosen placement written in with ``insert_candidate``, the next demand against the result.

``round_loop``: the same sequence on the device with the library's own pieces, one round per demand index of the
longest sequence: ``forward_placements`` on each sample's next demand, the accepted placements written into the raw
samples, the state rebuilt with ``lightpath_network_state`` and the bound carried over to the new node numbering
through ``lightpath_nodes``.  It is what a caller had to write before ``forward_provision``."""
from types import SimpleNamespace

import numpy as np
import torch

from candidates_ref import insert_candidate
from placement_ref import placement_ref

CAND_IMPACT_OVERFLOW = 8
PROV_FULL = 512
TG_MAX_NODES, TG_MAX_CHANNELS = 256, 6144


def provision_ref(model, sample, freqs, lp_feat, demands, policy, metric=0, maximize=True, bound=None,
                  freq_threshold=0.05, follow=None, chunk=None, device=None):
    """Sequential provisioning of one sample, defined literally.  ``demands``: a list of demands, each the options
    list of ``placement_ref``.  ``bound``: {conn_id: bound} or None.  ``follow``: a list of (option, q0) or None per
    demand, written in place of the reference's own choice (teacher forcing: the rows of each step can then be
    compared with the kernel's even where a near-tie could have gone either way).  Returns ``(steps, sample)``: per
    demand a dict with the reference's ``choice``, ``n_free``, ``n_feasible``, ``table`` (placement_ref's), the
    ``written`` (option, q0) and its ``conn`` (None if nothing was written), and the final sample."""
    cur = np.array(sample, dtype=np.float32, copy=True)
    bnd = dict(bound) if bound is not None else None
    steps = []
    for i, options in enumerate(demands):
        choice, n_free, n_feas, table = placement_ref(model, cur, freqs, lp_feat, options, policy, metric, maximize,
                                                      bnd, freq_threshold, chunk, device)
        written = follow[i] if follow is not None else choice
        conn = None
        if written is not None:
            p, q0 = written
            links, width, feat3, own_bound = options[p]
            cur, conn = insert_candidate(cur, lp_feat, links, q0, width,
                                         [np.float32(freqs[q0])] + [float(v) for v in feat3])
            if bnd is not None:
                bnd[conn] = float(own_bound)
        steps.append(dict(choice=choice, n_free=n_free, n_feasible=n_feas, table=table, written=written, conn=conn))
    return steps, cur


def _select(d, idx):
    """The demands idx (a CPU list) of LightpathDemands d, on d's device."""
    from gnn_qot_estimation_b200.to_graph import LightpathDemands
    optr, lptr = d.opt_ptr.cpu().tolist(), d.link_ptr.cpu().tolist()
    opts = [p for k in idx for p in range(optr[k], optr[k + 1])]
    links = [e for p in opts for e in range(lptr[p], lptr[p + 1])]
    dev = d.sample.device
    t = lambda v: torch.tensor(v, dtype=torch.int64, device=dev)
    return LightpathDemands(d.sample[t(idx)], t(np.cumsum([0] + [optr[k + 1] - optr[k] for k in idx]).tolist()),
                            t(np.cumsum([0] + [lptr[p + 1] - lptr[p] for p in opts]).tolist()), d.links[t(links)],
                            d.width[t(opts)], d.feat[t(opts)], d.own_bound[t(opts)])


def rounds(demands, S):
    """[(demand indices of round r, their LightpathDemands)]: round r holds each sample's r-th demand (index order)."""
    per = {}
    for k, s in enumerate(demands.sample.cpu().tolist()):
        if 0 <= s < S:
            per.setdefault(s, []).append(k)
    out = []
    for r in range(max((len(v) for v in per.values()), default=0)):
        idx = [v[r] for s, v in sorted(per.items()) if r < len(v)]
        out.append((idx, _select(demands, idx)))
    return out


def round_loop(model, data, freqs, lp_feat, demands, policy, metric=0, maximize=True, bound=None, max_impact=64,
               freq_threshold=0.05, plan=None):
    """The round loop on the device.  ``data`` [S, F, L, Q] CUDA float32 is written in place; ``bound`` [N] over the
    first state's nodes or None; ``plan``: ``rounds(demands, S)``, precomputed (it does not depend on the results).
    Returns ``(res, state)``: ``res`` a SimpleNamespace of the ``ProvisionQoT`` fields over all D demands (demands
    outside [0, S) are left as allocated: option -1, conn_id -1, status 0), ``state`` the final state.  A demand whose
    acceptance would overflow the graph builder's capacity is reported with PROV_FULL and not written, as the kernel
    does."""
    from gnn_qot_estimation_b200.to_graph import commit_provision, lightpath_network_state, lightpath_nodes
    dev = data.device
    state = lightpath_network_state(data, freqs, lp_feat, freq_threshold)
    S, D = state.S, int(demands.sample.shape[0])
    res = SimpleNamespace(option=torch.full((D,), -1, dtype=torch.int32, device=dev),
                          q0=torch.full((D,), -1, dtype=torch.int32, device=dev),
                          out=torch.full((D, 3), float("nan"), device=dev),
                          margin=torch.full((D,), float("nan"), device=dev),
                          n_free=torch.zeros(D, dtype=torch.int32, device=dev),
                          n_feasible=torch.zeros(D, dtype=torch.int32, device=dev),
                          status=torch.zeros(D, dtype=torch.int32, device=dev),
                          n_impact=torch.zeros(D, dtype=torch.int32, device=dev),
                          impact_conn=torch.full((D, max_impact), -1, dtype=torch.int64, device=dev),
                          impact_out=torch.full((D, max_impact, 3), float("nan"), device=dev),
                          conn_id=torch.full((D,), -1, dtype=torch.int64, device=dev))
    if bound is not None:                     # the bound by (sample, conn_id), carried over every rebuild
        b_s, b_c, b_v = state.batch.batch.to(torch.int64), state.conn_ids.clone(), bound.clone()
    cur = bound
    for idx, sub in (plan if plan is not None else rounds(demands, S)):
        it = torch.tensor(idx, dtype=torch.int64, device=dev)
        r = model.forward_placements(state, sub, policy, metric, maximize, cur, max_impact)
        ok = ((r.status & ~CAND_IMPACT_OVERFLOW) == 0) & (r.option >= 0)
        # the builder's capacity: lightpaths and occupied channels of each sample after the acceptance
        b = state.batch
        nodes = b.ptr[1:] - b.ptr[:-1]
        chans = (state.chan_node != -1).view(S, -1).sum(1)
        po = sub.opt_ptr[:-1] + r.option.clamp(min=0).to(torch.int64)
        need = (sub.link_ptr[po + 1] - sub.link_ptr[po]) * sub.width[po]
        full = ok & ((nodes[sub.sample] + 1 > TG_MAX_NODES) | (chans[sub.sample] + need > TG_MAX_CHANNELS))
        ok &= ~full
        top = torch.zeros(S, dtype=torch.int64, device=dev).scatter_reduce(0, b.batch.to(torch.int64),
                                                                         state.conn_ids, "amax", include_self=True)
        conn = torch.where(ok, top[sub.sample] + 1, torch.full_like(sub.sample, -1))
        ic = torch.where(r.impact_node >= 0, state.conn_ids[r.impact_node.clamp(min=0)], r.impact_node)
        for name, v in (("option", r.option), ("q0", r.q0), ("out", r.out), ("margin", r.margin),
                        ("n_free", r.n_free), ("n_feasible", r.n_feasible),
                        ("status", r.status | torch.where(full, PROV_FULL, 0).to(torch.int32)),
                        ("n_impact", r.n_impact), ("impact_conn", ic), ("impact_out", r.impact_out),
                        ("conn_id", conn)):
            getattr(res, name)[it] = v
        state = commit_provision(data, state, sub, SimpleNamespace(conn_id=conn, option=r.option, q0=r.q0))
        if bound is not None:
            b_s = torch.cat([b_s, sub.sample[ok]])
            b_c = torch.cat([b_c, conn[ok]])
            b_v = torch.cat([b_v, sub.own_bound[po[ok]]])
            cur = torch.empty(state.batch.x.shape[0], dtype=torch.float32, device=dev)
            cur[lightpath_nodes(state, b_s, b_c)] = b_v
    return res, state
