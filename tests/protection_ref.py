"""References for LightpathGNN's 1+1 protected provisioning (TEST INFRASTRUCTURE, like provision_ref.py).

``partner_eligible`` / ``disjoint_from``: the two option filters, by set disjointness of the routes' links.

``protection_ref``: the demands of one sample taken literally, in order: a protected demand's working path is
``placement_ref`` over its eligible options on the current numpy sample, written in with ``insert_candidate``; its
backup is ``placement_ref`` over the options disjoint from the working route on that sample; no backup: the sample
goes back to what it was before the demand.

``round_loop``: the same sequence on the device with the library's own pieces, two rounds per demand position of the
longest sequence: ``forward_placements`` on each sample's next demand with its eligible options, the working paths
written into a copy of the raw samples and the state rebuilt, the bound carried over by (sample, conn_id),
``forward_placements`` for the backups on that state, then the accepted paths written into the samples (the copy thrown
away and rebuilt when a backup failed).  It is what a caller had to write before ``forward_protection``."""
from types import SimpleNamespace

import numpy as np
import torch

from candidates_ref import insert_candidate
from placement_ref import placement_ref
from provision_ref import CAND_IMPACT_OVERFLOW, PROV_FULL, TG_MAX_CHANNELS, TG_MAX_NODES, rounds

PROT_NO_PARTNER, PROT_NO_BACKUP = 65536, 131072


def partner_eligible(routes):
    """[bool] per option: some option's route shares no link with this one's (link sets compared as sets)."""
    sets = [set(r) for r in routes]
    return [any(not (a & b) for b in sets) for a in sets]


def disjoint_from(routes, working):
    """[bool] per option: its route shares no link with ``working``."""
    w = set(working)
    return [not (set(r) & w) for r in routes]


def protection_ref(model, sample, freqs, lp_feat, demands, protect, policy, metric=0, maximize=True, bound=None,
                   freq_threshold=0.05, follow=None, chunk=None, device=None):
    """Protected provisioning of one sample, defined literally.  ``demands``: a list of demands, each the options list
    of ``placement_ref``; ``protect``: a bool per demand; ``bound``: {conn_id: bound} or None.  ``follow``: per demand
    (working, backup), each an (option, q0) or None, written in place of the reference's own choices (None for the
    demand: the reference's).  Returns ``(steps, sample)``: per demand a dict with the working search's ``choice``,
    ``n_free``, ``n_feasible``, ``table`` (keys in the full option list), ``written`` and ``conn``; the backup search's
    ``b_choice``, ``b_n_free``, ``b_n_feasible``, ``b_table``, ``b_written`` and ``b_conn`` (None / 0 without one); and
    ``status`` (0, PROT_NO_PARTNER or PROT_NO_BACKUP).  ``conn`` is None for a rolled-back demand."""
    cur = np.array(sample, dtype=np.float32, copy=True)
    bnd = dict(bound) if bound is not None else None
    steps = []

    def search(options, keep):
        choice, n_free, n_feas, table = placement_ref(model, cur, freqs, lp_feat, [options[p] for p in keep], policy,
                                                      metric, maximize, bnd, freq_threshold, chunk, device)
        table = {(keep[p], q0): v for (p, q0), v in table.items()}
        return (None if choice is None else (keep[choice[0]], choice[1])), n_free, n_feas, table

    def write(options, placed):
        nonlocal cur
        p, q0 = placed
        links, width, feat3, own_bound = options[p]
        cur, conn = insert_candidate(cur, lp_feat, links, q0, width, [np.float32(freqs[q0])] + [float(v) for v in feat3])
        if bnd is not None:
            bnd[conn] = float(own_bound)
        return conn

    for i, options in enumerate(demands):
        routes = [o[0] for o in options]
        keep = list(range(len(options)))
        if protect[i]:
            keep = [p for p, ok in enumerate(partner_eligible(routes)) if ok]
        st = dict(choice=None, n_free=0, n_feasible=0, table={}, written=None, conn=None, b_choice=None, b_n_free=0,
                  b_n_feasible=0, b_table={}, b_written=None, b_conn=None, status=0)
        steps.append(st)
        if not keep:
            st["status"] = PROT_NO_PARTNER
            continue
        st["choice"], st["n_free"], st["n_feasible"], st["table"] = search(options, keep)
        fw = follow[i] if follow is not None and follow[i] is not None else None
        st["written"] = fw[0] if fw is not None else st["choice"]
        if st["written"] is None:
            continue
        saved = (cur, None if bnd is None else dict(bnd))
        st["conn"] = write(options, st["written"])
        if not protect[i]:
            continue
        bkeep = [p for p, ok in enumerate(disjoint_from(routes, routes[st["written"][0]])) if ok]
        st["b_choice"], st["b_n_free"], st["b_n_feasible"], st["b_table"] = search(options, bkeep)
        st["b_written"] = fw[1] if fw is not None else st["b_choice"]
        if st["b_written"] is not None:
            st["b_conn"] = write(options, st["b_written"])
        else:                                       # no backup: the sample as it was before the demand
            cur, bnd = saved
            st["conn"], st["status"] = None, PROT_NO_BACKUP
    return steps, cur


def conn_ids(top, sample, work_ok, back_ok, protect):
    """The conn_id bookkeeping of one round (each sample at most once): ``(conn, backup_conn, top)``.  An accepted
    demand takes top + 1 and, protected, its backup top + 2; a protected demand without a backup takes nothing and does
    not advance its sample's running top."""
    keep = work_ok & (~protect | back_ok)
    conn = torch.where(keep, top[sample] + 1, torch.full_like(sample, -1))
    bconn = torch.where(keep & protect, top[sample] + 2, torch.full_like(sample, -1))
    return conn, bconn, top.index_add(0, sample, keep.to(torch.int64) + (bconn >= 0).to(torch.int64))


def _routes(d):
    """Per demand of LightpathDemands d, its options' routes (CPU lists)."""
    optr, lptr, lk = d.opt_ptr.cpu().tolist(), d.link_ptr.cpu().tolist(), d.links.cpu().tolist()
    return [[lk[lptr[p]:lptr[p + 1]] for p in range(optr[j], optr[j + 1])] for j in range(len(optr) - 1)]


def _subset(d, picks):
    """LightpathDemands of the demands ``j`` of d, each with only its options ``ks`` (relative), for (j, ks) in
    ``picks``."""
    from gnn_qot_estimation_b200.to_graph import LightpathDemands
    optr, lptr = d.opt_ptr.cpu().tolist(), d.link_ptr.cpu().tolist()
    opts = [optr[j] + k for j, ks in picks for k in ks]
    links = [e for p in opts for e in range(lptr[p], lptr[p + 1])]
    dev = d.sample.device
    t = lambda v: torch.tensor(v, dtype=torch.int64, device=dev)
    return LightpathDemands(d.sample[t([j for j, _ in picks])], t(np.cumsum([0] + [len(ks) for _, ks in picks]).tolist()),
                            t(np.cumsum([0] + [lptr[p + 1] - lptr[p] for p in opts]).tolist()), d.links[t(links)],
                            d.width[t(opts)], d.feat[t(opts)], d.own_bound[t(opts)])


def _remap(state, b_s, b_c, b_v):
    """The bound [N] over ``state``'s nodes from the (sample, conn_id, value) lists."""
    from gnn_qot_estimation_b200.to_graph import lightpath_nodes
    cur = torch.empty(state.batch.x.shape[0], dtype=torch.float32, device=b_v.device)
    cur[lightpath_nodes(state, b_s, b_c)] = b_v
    return cur


def _place(model, state, sub, picks, n, policy, metric, maximize, bound, max_impact):
    """forward_placements of the demands of ``sub`` named by ``picks`` (j, relative options kept), mapped back to
    ``n`` rows of ``sub``: the outputs with the option in the full list, the impact rows by conn_id, PROV_FULL from
    the builder's capacity, and whether each is acceptable."""
    dev = sub.sample.device
    out = SimpleNamespace(option=torch.full((n,), -1, dtype=torch.int32, device=dev),
                          q0=torch.full((n,), -1, dtype=torch.int32, device=dev),
                          out=torch.full((n, 3), float("nan"), device=dev),
                          margin=torch.full((n,), float("nan"), device=dev),
                          n_free=torch.zeros(n, dtype=torch.int32, device=dev),
                          n_feasible=torch.zeros(n, dtype=torch.int32, device=dev),
                          status=torch.zeros(n, dtype=torch.int32, device=dev),
                          n_impact=torch.zeros(n, dtype=torch.int32, device=dev),
                          impact_conn=torch.full((n, max_impact), -1, dtype=torch.int64, device=dev),
                          impact_out=torch.full((n, max_impact, 3), float("nan"), device=dev),
                          ok=torch.zeros(n, dtype=torch.bool, device=dev))
    if not picks:
        return out
    r = model.forward_placements(state, _subset(sub, picks), policy, metric, maximize, bound, max_impact)
    rows = torch.tensor([j for j, _ in picks], dtype=torch.int64, device=dev)
    kmax = max(len(ks) for _, ks in picks)
    lut = torch.tensor([ks + [-1] * (kmax - len(ks)) for _, ks in picks], dtype=torch.int32, device=dev)
    opt = torch.where(r.option >= 0, lut.gather(1, r.option.clamp(min=0).to(torch.int64)[:, None])[:, 0], r.option)
    ok = ((r.status & ~CAND_IMPACT_OVERFLOW) == 0) & (r.option >= 0)
    S, b = state.S, state.batch
    nodes = b.ptr[1:] - b.ptr[:-1]
    chans = (state.chan_node != -1).view(S, -1).sum(1)
    po = sub.opt_ptr[rows] + opt.clamp(min=0).to(torch.int64)
    need = (sub.link_ptr[po + 1] - sub.link_ptr[po]) * sub.width[po]
    s = sub.sample[rows]
    full = ok & ((nodes[s] + 1 > TG_MAX_NODES) | (chans[s] + need > TG_MAX_CHANNELS))
    ic = torch.where(r.impact_node >= 0, state.conn_ids[r.impact_node.clamp(min=0)], r.impact_node)
    for name, v in (("option", opt), ("q0", r.q0), ("out", r.out), ("margin", r.margin), ("n_free", r.n_free),
                    ("n_feasible", r.n_feasible),
                    ("status", r.status | torch.where(full, PROV_FULL, 0).to(torch.int32)),
                    ("n_impact", r.n_impact), ("impact_conn", ic), ("impact_out", r.impact_out), ("ok", ok & ~full)):
        getattr(out, name)[rows] = v
    return out


def round_loop(model, data, freqs, lp_feat, demands, protect, policy, metric=0, maximize=True, bound=None,
               max_impact=64, freq_threshold=0.05, plan=None):
    """The round loop on the device.  ``data`` [S, F, L, Q] CUDA float32 is written in place (the final samples);
    ``protect`` [D] bool; ``bound`` [N] over the first state's nodes or None; ``plan``: ``rounds(demands, S)``.
    Returns ``(res, state)``: ``res`` a SimpleNamespace of the ``ProtectionQoT`` fields over all D demands (demands
    outside [0, S) left as allocated), ``state`` the final state."""
    from gnn_qot_estimation_b200.to_graph import commit_provision, lightpath_network_state
    dev = data.device
    state = lightpath_network_state(data, freqs, lp_feat, freq_threshold)
    S, D = state.S, int(demands.sample.shape[0])
    fields = dict(option=(-1, torch.int32, ()), q0=(-1, torch.int32, ()), out=(float("nan"), torch.float32, (3,)),
                  margin=(float("nan"), torch.float32, ()), n_free=(0, torch.int32, ()),
                  n_feasible=(0, torch.int32, ()), status=(0, torch.int32, ()), n_impact=(0, torch.int32, ()),
                  impact_conn=(-1, torch.int64, (max_impact,)), impact_out=(float("nan"), torch.float32, (max_impact, 3)),
                  conn_id=(-1, torch.int64, ()))
    res = SimpleNamespace(**{pre + k: torch.full((D,) + sh, v, dtype=dt, device=dev)
                             for pre in ("", "backup_") for k, (v, dt, sh) in fields.items()})
    top = torch.zeros(S, dtype=torch.int64, device=dev).scatter_reduce(
        0, state.batch.batch.to(torch.int64), state.conn_ids, "amax", include_self=True)
    if bound is not None:                     # the bound by (sample, conn_id), carried over every rebuild
        b_s, b_c, b_v = state.batch.batch.to(torch.int64), state.conn_ids.clone(), bound.clone()
    cur = bound
    prot_all = protect.cpu().tolist()
    names = [k for k in fields if k != "conn_id"]
    for idx, sub in (plan if plan is not None else rounds(demands, S)):
        n = len(idx)
        it = torch.tensor(idx, dtype=torch.int64, device=dev)
        prot = [bool(prot_all[k]) for k in idx]
        routes = _routes(sub)
        keep = [[p for p, ok in enumerate(partner_eligible(rs)) if ok] if pr else list(range(len(rs)))
                for rs, pr in zip(routes, prot)]
        # ---- the working paths
        w = _place(model, state, sub, [(j, ks) for j, ks in enumerate(keep) if ks], n, policy, metric, maximize, cur,
                   max_impact)
        no_partner = torch.tensor([not ks for ks in keep], device=dev)
        w.status |= torch.where(no_partner, PROT_NO_PARTNER, 0).to(torch.int32)
        tprot = torch.tensor(prot, device=dev)
        s = sub.sample
        wconn = torch.where(w.ok, top[s] + 1, torch.full_like(s, -1))
        # ---- the backups, against the samples with the working paths written in (a copy)
        b = _place(model, state, sub, [], n, policy, metric, maximize, cur, max_impact)
        need_b = [j for j in range(n) if prot[j] and bool(w.ok[j])]
        if need_b:
            data_w = data.clone()
            state_w = commit_provision(data_w, state, sub, SimpleNamespace(conn_id=wconn, option=w.option, q0=w.q0))
            cur_w = None
            if bound is not None:
                po = sub.opt_ptr[:-1] + w.option.clamp(min=0).to(torch.int64)
                cur_w = _remap(state_w, torch.cat([b_s, s[w.ok]]), torch.cat([b_c, wconn[w.ok]]),
                               torch.cat([b_v, sub.own_bound[po[w.ok]]]))
            opt_w = w.option.tolist()
            picks = [(j, [p for p, ok in enumerate(disjoint_from(routes[j], routes[j][opt_w[j]])) if ok])
                     for j in need_b]
            b = _place(model, state_w, sub, picks, n, policy, metric, maximize, cur_w, max_impact)
        conn, bconn, top = conn_ids(top, s, w.ok, b.ok, tprot)
        rolled = tprot & w.ok & ~b.ok
        w.status |= torch.where(rolled, PROT_NO_BACKUP, 0).to(torch.int32)
        for k in names:
            getattr(res, k)[it] = getattr(w, k)
            getattr(res, "backup_" + k)[it] = getattr(b, k)
        res.conn_id[it] = conn
        res.backup_conn_id[it] = bconn
        # ---- the accepted paths into the samples: the copy kept when no backup failed, else rebuilt from the samples
        if need_b and not bool(rolled.any()):
            data.copy_(data_w)
            state = state_w
        else:
            state = commit_provision(data, state, sub, SimpleNamespace(conn_id=conn, option=w.option, q0=w.q0))
        if bool((bconn >= 0).any()):
            state = commit_provision(data, state, sub, SimpleNamespace(conn_id=bconn, option=b.option, q0=b.q0))
        if bound is not None:
            po = sub.opt_ptr[:-1] + w.option.clamp(min=0).to(torch.int64)
            bpo = sub.opt_ptr[:-1] + b.option.clamp(min=0).to(torch.int64)
            a, bb = conn >= 0, bconn >= 0
            b_s, b_c = torch.cat([b_s, s[a], s[bb]]), torch.cat([b_c, conn[a], bconn[bb]])
            b_v = torch.cat([b_v, sub.own_bound[po[a]], sub.own_bound[bpo[bb]]])
            cur = _remap(state, b_s, b_c, b_v)
    return res, state
