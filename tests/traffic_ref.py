"""References for LightpathGNN's dynamic traffic (TEST INFRASTRUCTURE, like provision_ref.py).

``traffic_ref``: the events of one sample taken literally, one after another, on a numpy copy of the sample.  A release
is ``reconfig_ref`` with an empty path for its rows (the former neighbours' rows after the teardown), then the lightpath
zeroed with ``rewrite_lightpath``.  An arrival is ``provision_ref``'s step: ``placement_ref`` on the current sample and
the choice written in, under conn_id top + 1 where top is the largest conn_id the sample has held.

``round_loop``: the same sequences on the device with the library's own pieces, one round per event position (round r
holds each sample's r-th event).  A release is ``forward_reconfigurations`` with a teardown (its rows), then its
channels zeroed in the raw samples.  An arrival is ``forward_placements`` and the accepted placement written in with
``commit_provision``.  The state is rebuilt after every round, the bound carried by (sample, conn_id) through
``lightpath_nodes`` and the conn_ids assigned from a per-sample running top.  It is what a caller writes without
``forward_traffic``."""
from types import SimpleNamespace

import numpy as np
import torch

from candidates_ref import insert_candidate
from placement_ref import placement_ref
from provision_ref import _select
from reconfig_ref import reconfig_ref, rewrite_lightpath

CAND_BAD_SAMPLE, CAND_IMPACT_OVERFLOW = 1, 8
PROV_FULL = 512
TRAF_BAD_REF, TRAF_NOT_ACCEPTED = 2048, 4096
TG_MAX_NODES, TG_MAX_CHANNELS = 256, 6144


def events(demand_sample, rel_sample, rel_before, S):
    """{sample: [("d", d) or ("r", k), ...]}: each sample's demands in index order with its releases before demand d
    when before <= d, ordered by (before, k), and the rest after the last demand."""
    per = {}
    for s in range(S):
        ds = [d for d, x in enumerate(demand_sample) if x == s]
        rs = sorted((b, k) for k, (x, b) in enumerate(zip(rel_sample, rel_before)) if x == s)
        ev, j = [], 0
        for d in ds:
            while j < len(rs) and rs[j][0] <= d:
                ev.append(("r", rs[j][1]))
                j += 1
            ev.append(("d", d))
        ev += [("r", k) for _, k in rs[j:]]
        if ev:
            per[s] = ev
    return per


def traffic_ref(model, sample, freqs, lp_feat, seq, policy, metric=0, maximize=True, bound=None, freq_threshold=0.05,
                follow=None, chunk=None, device=None):
    """Dynamic traffic of one sample, defined literally.  ``seq``: events, each ``("d", options)`` (the options list of
    ``placement_ref``) or ``("r", conn_id)`` or ``("rd", i)`` (release of the lightpath the i-th event, a demand, was
    accepted under).  ``bound``: {conn_id: bound} or None.  ``follow``: per demand event (option, q0) or None, written
    in place of the reference's choice (teacher forcing).  Returns ``(steps, sample)``: per event a dict; a demand's as
    ``provision_ref``'s, a release's with ``conn`` (None if nothing was released), ``rows`` {conn_id: row [3]} of the
    former neighbours after it, and ``margin`` (with a bound, the minimum over them; NaN without)."""
    fi = {k: i for i, k in enumerate(lp_feat)}
    cur = np.array(sample, dtype=np.float32, copy=True)
    top = int(np.trunc(cur[fi["conn_id"]]).max(initial=0))
    present = set(np.unique(np.trunc(cur[fi["conn_id"]][np.any(cur != 0, axis=0)])).astype(int).tolist())
    bnd = dict(bound) if bound is not None else None
    steps, nd = [], 0
    for kind, arg in seq:
        if kind == "d":
            choice, n_free, n_feas, table = placement_ref(model, cur, freqs, lp_feat, arg, policy, metric, maximize,
                                                          bnd, freq_threshold, chunk, device)
            written = follow[nd] if follow is not None else choice
            nd += 1
            conn = None
            if written is not None:
                p, q0 = written
                links, width, feat3, own_bound = arg[p]
                cur, _ = insert_candidate(cur, lp_feat, links, q0, width, [np.float32(freqs[q0])] + list(feat3))
                top += 1
                conn = top
                for l in links:
                    cur[fi["conn_id"], l, q0:q0 + width] = conn
                present.add(conn)
                if bnd is not None:
                    bnd[conn] = float(own_bound)
            steps.append(dict(choice=choice, n_free=n_free, n_feasible=n_feas, table=table, written=written,
                              conn=conn))
            continue
        c = steps[arg]["conn"] if kind == "rd" else int(arg)
        if c is None or c not in present:
            steps.append(dict(conn=None, rows={}, margin=float("nan")))
            continue
        _, imp = reconfig_ref(model, cur, freqs, lp_feat, c, [], 0, 0, [0.0] * 4, freq_threshold, chunk, device)
        rows = {o: r for o, (kd, r) in imp.items()}
        assert all(kd == 1 for kd, _ in imp.values())
        mg = float("nan")
        if bnd is not None and rows:
            sign = 1.0 if maximize else -1.0
            mg = min(sign * (float(r[metric]) - bnd[o]) for o, r in rows.items())
        cur = rewrite_lightpath(cur, lp_feat, c, [], 0, 0, [0.0] * 4)
        present.discard(c)
        if bnd is not None:
            bnd.pop(c, None)
        steps.append(dict(conn=c, rows=rows, margin=mg))
    return steps, cur


def round_loop(model, data, freqs, lp_feat, demands, releases, policy, metric=0, maximize=True, bound=None,
               max_impact=64, freq_threshold=0.05):
    """The round loop on the device.  ``data`` [S, F, L, Q] CUDA float32 is written in place; ``bound`` [N] over the
    first state's nodes or None.  Returns ``(res, state)``: ``res`` a SimpleNamespace of the ``TrafficQoT`` fields
    (events of samples outside [0, S) are left as allocated), ``state`` the final state."""
    from gnn_qot_estimation_b200.to_graph import (LightpathChanges, commit_provision, lightpath_network_state,
                                                  lightpath_nodes)
    dev = data.device
    state = lightpath_network_state(data, freqs, lp_feat, freq_threshold)
    S, D, R = state.S, int(demands.sample.shape[0]), int(releases.sample.shape[0])
    nan = float("nan")
    i32 = lambda n, v: torch.full((n,), v, dtype=torch.int32, device=dev)
    i64 = lambda *s: torch.full(s, -1, dtype=torch.int64, device=dev)
    res = SimpleNamespace(option=i32(D, -1), q0=i32(D, -1), out=torch.full((D, 3), nan, device=dev),
                          margin=torch.full((D,), nan, device=dev), n_free=i32(D, 0), n_feasible=i32(D, 0),
                          status=i32(D, 0), n_impact=i32(D, 0), impact_conn=i64(D, max_impact),
                          impact_out=torch.full((D, max_impact, 3), nan, device=dev), conn_id=i64(D),
                          release_status=i32(R, 0), release_conn_id=i64(R), release_n_impact=i32(R, 0),
                          release_impact_conn=i64(R, max_impact),
                          release_impact_out=torch.full((R, max_impact, 3), nan, device=dev),
                          release_margin=torch.full((R,), nan, device=dev))
    rs, rb = releases.sample.tolist(), releases.before.tolist()
    rd, rc = releases.demand.tolist(), releases.conn_id.tolist()
    ds = demands.sample.tolist()
    per = events(ds, rs, rb, S)
    top = torch.zeros(S, dtype=torch.int64, device=dev).scatter_reduce(
        0, state.batch.batch.to(torch.int64), state.conn_ids, "amax", include_self=True).tolist()
    if bound is not None:
        b_s, b_c, b_v = state.batch.batch.to(torch.int64), state.conn_ids.clone(), bound.clone()
    cur = bound
    conn_of = {}                                           # demand -> conn_id it was accepted under
    lo, span = -(1 << 31), 1 << 32
    for r in range(max((len(v) for v in per.values()), default=0)):
        ev = [(s, v[r]) for s, v in sorted(per.items()) if r < len(v)]
        # ---- releases: what each names, its rows from a teardown against the current state
        rel = []                                           # (k, sample, conn)
        for s, (kind, k) in ev:
            if kind != "r":
                continue
            dm = rd[k]
            st, c = 0, -1
            if not 0 <= rb[k] <= D or dm < -1 or (dm >= 0 and (dm >= D or dm >= rb[k] or ds[dm] != s)):
                st = TRAF_BAD_REF
            elif dm >= 0 and conn_of.get(dm, -1) < 0:
                st = TRAF_NOT_ACCEPTED
            else:
                c = conn_of[dm] if dm >= 0 else rc[k]
            if st:
                res.release_status[k] = st
            else:
                rel.append((k, s, c))
        if rel:
            t = lambda v, dt=torch.int64: torch.tensor(v, dtype=dt, device=dev)
            nodes = lightpath_nodes(state, t([s for _, s, _ in rel]), t([c for _, _, c in rel])).tolist()
            found = [(k, s, c, n) for (k, s, c), n in zip(rel, nodes) if n >= 0]
            for (k, s, c), n in zip(rel, nodes):
                if n < 0:
                    res.release_status[k] = TRAF_BAD_REF
            if found:
                K = len(found)
                ch = LightpathChanges(t([n for *_, n in found]), t([s for _, s, _, _ in found]), t([0] * (K + 1)),
                                      t([], torch.int32), t([0] * K, torch.int32), t([1] * K, torch.int32),
                                      torch.zeros(K, 4, device=dev))
                q = model.forward_reconfigurations(state, ch, TG_MAX_NODES)
                assert bool((q.impact_kind[q.impact_node >= 0] == 1).all())
                ks = t([k for k, *_ in found])
                res.release_status[ks] = torch.where(q.n_impact > max_impact, CAND_IMPACT_OVERFLOW, 0).to(torch.int32)
                res.release_conn_id[ks] = t([c for _, _, c, _ in found])
                res.release_n_impact[ks] = q.n_impact
                ic = torch.where(q.impact_node >= 0, state.conn_ids[q.impact_node.clamp(min=0)], q.impact_node)
                res.release_impact_conn[ks] = ic[:, :max_impact]
                res.release_impact_out[ks] = q.impact_out[:, :max_impact]
                if cur is not None:
                    v = q.impact_out[..., metric]
                    b = cur[q.impact_node.clamp(min=0)]
                    m = torch.where(q.impact_node >= 0, v - b if maximize else b - v, torch.inf)
                    mg = m.min(1).values
                    res.release_margin[ks] = torch.where(q.n_impact > 0, mg, nan)
                # the released channels zeroed
                gone = t([s * span + (c - lo) for _, s, c, _ in found])
                conn = data[:, state.cfg.i_conn].to(torch.int64)
                key = torch.arange(S, device=dev)[:, None, None] * span + (conn - lo)
                data.masked_fill_((torch.isin(key, gone) & (data != 0).any(1))[:, None], 0.0)
        # ---- arrivals: placed against the current state, accepted under the sample's running top + 1
        idx = [k for s, (kind, k) in ev if kind == "d"]
        if idx:
            sub = _select(demands, idx)
            it = torch.tensor(idx, dtype=torch.int64, device=dev)
            p = model.forward_placements(state, sub, policy, metric, maximize, cur, max_impact)
            ok = ((p.status & ~CAND_IMPACT_OVERFLOW) == 0) & (p.option >= 0)
            b = state.batch
            nodes = b.ptr[1:] - b.ptr[:-1]
            chans = (state.chan_node != -1).view(S, -1).sum(1)
            po = sub.opt_ptr[:-1] + p.option.clamp(min=0).to(torch.int64)
            need = (sub.link_ptr[po + 1] - sub.link_ptr[po]) * sub.width[po]
            full = ok & ((nodes[sub.sample] + 1 > TG_MAX_NODES) | (chans[sub.sample] + need > TG_MAX_CHANNELS))
            ok &= ~full
            conn = []
            for k, a in zip(idx, ok.tolist()):
                if a:
                    top[ds[k]] += 1
                conn.append(top[ds[k]] if a else -1)
                conn_of[k] = conn[-1]
            conn = torch.tensor(conn, dtype=torch.int64, device=dev)
            ic = torch.where(p.impact_node >= 0, state.conn_ids[p.impact_node.clamp(min=0)], p.impact_node)
            for name, v in (("option", p.option), ("q0", p.q0), ("out", p.out), ("margin", p.margin),
                            ("n_free", p.n_free), ("n_feasible", p.n_feasible),
                            ("status", p.status | torch.where(full, PROV_FULL, 0).to(torch.int32)),
                            ("n_impact", p.n_impact), ("impact_conn", ic), ("impact_out", p.impact_out),
                            ("conn_id", conn)):
                getattr(res, name)[it] = v
            state = commit_provision(data, state, sub, SimpleNamespace(conn_id=conn, option=p.option, q0=p.q0))
            if bound is not None:
                b_s = torch.cat([b_s, sub.sample[ok]])
                b_c = torch.cat([b_c, conn[ok]])
                b_v = torch.cat([b_v, sub.own_bound[po[ok]]])
        else:
            state = lightpath_network_state(data, freqs, lp_feat, freq_threshold)
        if bound is not None:
            cur = torch.empty(state.batch.x.shape[0], dtype=torch.float32, device=dev)
            n = lightpath_nodes(state, b_s, b_c)
            cur[n[n >= 0]] = b_v[n >= 0]
    return res, state
