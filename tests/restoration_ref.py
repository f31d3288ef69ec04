"""References for LightpathGNN's failure restoration (TEST INFRASTRUCTURE, like traffic_ref.py).

``expand``: the definition of ``forward_restoration`` with the library's own pieces.  Each scenario's sample is
replicated into a batch of its own; the cut set is found in numpy from the raw sample (every lightpath with an occupied
channel on a failed link, independent of ``chan_node``); the cut lightpaths become releases by conn_id at ``before =
0`` and, in ascending node order, demands with their options that avoid the failed links.  One ``forward_traffic`` call
runs every scenario, with the bound carried by node; option indices and conn_ids are mapped back, then
``commit_traffic``, ``lightpath_network_state`` and ``forward_every_node`` give the end rows.  It is what a caller
writes without ``forward_restoration``.

``restoration_ref``: one scenario taken literally in fp64: ``traffic_ref`` on the sequence (the releases, then the
filtered demands, ``follow=`` a given choice per demand), then ``every_node_ref.lightpath_every_node_ref`` on the final
sample's graph."""
from types import SimpleNamespace

import numpy as np
import torch

from traffic_ref import traffic_ref

CAND_BAD_SAMPLE, CAND_BAD_PATH, CAND_BAD_STATE = 1, 2, 16
REST_NO_OPTION, REST_BAD_FAILURE, REST_CUT_OVERFLOW = 8192, 16384, 32768
MAX_OPTIONS, TG_MAX_NODES = 32, 256


def cut_set(sample, lp_feat, failed):
    """The conn_ids of the lightpaths of ``sample`` [F, L, Q] (numpy) with an occupied channel on a failed link."""
    fi = {k: i for i, k in enumerate(lp_feat)}
    x = sample[:, list(failed)]
    occ = np.any(x != 0, axis=0)
    return set(np.trunc(x[fi["conn_id"]][occ]).astype(np.int64).tolist())


def _all_opts(options):
    """Every node's options as lists of (links, width, feat3, own_bound) tuples, from ``LightpathDemands``."""
    optr, lptr = options.opt_ptr.tolist(), options.link_ptr.tolist()
    links, width = options.links.tolist(), options.width.tolist()
    feat, ob = options.feat.tolist(), options.own_bound.tolist()
    one = lambda p: (links[lptr[p]:lptr[p + 1]], width[p], tuple(feat[p]), ob[p])
    return [[one(p) for p in range(optr[v], optr[v + 1])] for v in range(len(optr) - 1)]


def _bad_options(opts, L, Q):
    return len(opts) > MAX_OPTIONS or any(not links or min(links) < 0 or max(links) >= L or not 1 <= w <= Q
                                          for links, w, _, _ in opts)


def scenarios(samples, state, options, failures):
    """Host plan of every scenario: a dict per scenario with ``status`` (scenario-level), ``s``, ``failed``, ``cut``
    (state nodes, ascending) and per cut lightpath ``kind`` ('d': a demand with ``opts`` and ``keep`` (full indices),
    'bad_sample', 'no_option')."""
    L, Q = state.L, state.Q
    ptr = state.batch.ptr.tolist()
    conn = state.conn_ids.tolist()
    every = _all_opts(options)
    osmp = options.sample.tolist()
    fs, lp, fl = failures.sample.tolist(), failures.link_ptr.tolist(), failures.links.tolist()
    plan = []
    for f, s in enumerate(fs):
        if not 0 <= s < state.S:
            plan.append(dict(status=CAND_BAD_SAMPLE))
            continue
        a, b = lp[f], lp[f + 1]
        failed = fl[a:b] if 0 <= a < b <= len(fl) else []
        if not failed or min(failed) < 0 or max(failed) >= L:
            plan.append(dict(status=REST_BAD_FAILURE))
            continue
        cc = cut_set(samples["data"][s], samples["lp_feat"], failed)
        cut = [v for v in range(ptr[s], ptr[s + 1]) if conn[v] in cc]
        per = []
        for v in cut:
            opts = every[v]
            if osmp[v] != s:
                per.append(dict(kind="bad_sample"))
            elif _bad_options(opts, L, Q):
                per.append(dict(kind="d", opts=opts, keep=list(range(len(opts)))))     # forward_traffic: BAD_PATH
            else:
                keep = [i for i, (links, *_) in enumerate(opts) if not set(links) & set(failed)]
                per.append(dict(kind="d", opts=[opts[i] for i in keep], keep=keep) if keep else dict(kind="no_option"))
        plan.append(dict(status=0, s=s, failed=failed, cut=cut, per=per))
    return plan


def expand(model, samples, state, options, failures, policy, metric=0, maximize=True, bound=None, max_cut=64,
           chunk=None):
    """``forward_restoration`` defined through ``forward_traffic`` on replicated samples (see the module docstring).
    ``samples``: the dict the state was built from (``data`` numpy [S, F, L, Q], ``freqs``, ``lp_feat``).  Returns a
    SimpleNamespace of the ``RestorationQoT`` fields with ``end_conn`` / ``end_out``.  ``chunk``: scenarios per
    ``forward_traffic`` call (None: all at once)."""
    from gnn_qot_estimation_b200.to_graph import (LightpathDemands, LightpathReleases, commit_traffic,
                                                  lightpath_network_state)
    dev = state.batch.x.device
    thr = float(state.cfg.freq_threshold)
    plan = scenarios(samples, state, options, failures)
    F = len(plan)
    nan = float("nan")
    t = lambda v, dt=torch.int64: torch.tensor(v, dtype=dt, device=dev)
    full = lambda shape, v, dt: torch.full(shape, v, dtype=dt, device=dev)
    res = SimpleNamespace(cut_node=full((F, max_cut), -1, torch.int64), option=full((F, max_cut), -1, torch.int32),
                          q0=full((F, max_cut), -1, torch.int32), out=full((F, max_cut, 3), nan, torch.float32),
                          margin=full((F, max_cut), nan, torch.float32), n_free=full((F, max_cut), 0, torch.int32),
                          n_feasible=full((F, max_cut), 0, torch.int32), cut_status=full((F, max_cut), 0, torch.int32),
                          status=full((F,), 0, torch.int32), n_cut=full((F,), 0, torch.int32),
                          n_restored=full((F,), 0, torch.int32), end_conn=full((F, TG_MAX_NODES), -1, torch.int64),
                          end_out=full((F, TG_MAX_NODES, 3), nan, torch.float32))
    ptr = state.batch.ptr.tolist()
    conn = state.conn_ids.tolist()
    kind_bits = {"d": 0, "bad_sample": CAND_BAD_SAMPLE, "no_option": REST_NO_OPTION}
    res.status[:] = t([p["status"] | (REST_CUT_OVERFLOW if p["status"] == 0 and len(p["cut"]) > max_cut else 0)
                       for p in plan], torch.int32)
    res.n_cut[:] = t([len(p["cut"]) if p["status"] == 0 else 0 for p in plan], torch.int32)
    cf = [(f, i, v, kind_bits[c["kind"]]) for f, p in enumerate(plan) if p["status"] == 0
          for i, (v, c) in enumerate(zip(p["cut"], p["per"])) if i < max_cut]
    if cf:
        fi_, ii_ = t([x[0] for x in cf]), t([x[1] for x in cf])
        res.cut_node[fi_, ii_] = t([x[2] for x in cf])
        res.cut_status[fi_, ii_] = t([x[3] for x in cf], torch.int32)
    live = [f for f, p in enumerate(plan) if p["status"] == 0]
    step = len(live) if chunk is None else int(chunk)
    for c0 in range(0, len(live), max(step, 1)):
        fs = live[c0:c0 + step]
        data = torch.from_numpy(np.ascontiguousarray(samples["data"][[plan[f]["s"] for f in fs]])).to(dev)
        rep = lightpath_network_state(data, torch.as_tensor(samples["freqs"]), samples["lp_feat"], thr)
        rel, dem, where, keep = [], [], [], []     # where: (replica, scenario, ordinal, original conn) per demand
        for r, f in enumerate(fs):
            p = plan[f]
            for i, (v, c) in enumerate(zip(p["cut"], p["per"])):
                rel.append((r, 0, -1, conn[v]))
                if c["kind"] == "d":
                    dem.append((r, c["opts"]))
                    where.append((r, f, i, conn[v]))
                    keep += c["keep"]
        releases = LightpathReleases(*(t([x[k] for x in rel]) for k in range(4)))
        opts = [o for _, os_ in dem for o in os_]
        optr = t(np.cumsum([0] + [len(os_) for _, os_ in dem]).tolist())
        demands = LightpathDemands(t([r for r, _ in dem]), optr, t(np.cumsum([0] + [len(o[0]) for o in opts]).tolist()),
                                   t([l for o in opts for l in o[0]], torch.int32), t([o[1] for o in opts], torch.int32),
                                   torch.tensor(np.array([o[2] for o in opts], dtype=np.float32).reshape(-1, 3),
                                                device=dev),
                                   torch.tensor(np.array([o[3] for o in opts], dtype=np.float32), device=dev))
        rb = None
        if bound is not None:
            rb = torch.cat([bound[ptr[plan[f]["s"]]:ptr[plan[f]["s"] + 1]] for f in fs]).contiguous()
        tr = model.forward_traffic(rep, demands, releases, policy, metric, maximize, rb, TG_MAX_NODES)
        # per demand: the outputs, the option mapped back to the full list
        if where:
            wr, wf, wi, wc = (t([x[k] for x in where]) for k in range(4))
            acc = tr.conn_id >= 0
            res.n_restored.index_add_(0, wf, acc.to(torch.int32))
            m = wi < max_cut
            kept = t(keep)[optr[:-1] + tr.option.clamp(min=0)]       # every demand has an option
            full_opt = torch.where(tr.option >= 0, kept, -1).to(torch.int32)
            res.option[wf[m], wi[m]] = full_opt[m]
            for name in ("q0", "out", "margin", "n_free", "n_feasible"):
                getattr(res, name)[wf[m], wi[m]] = getattr(tr, name)[m]
            res.cut_status[wf[m], wi[m]] = tr.status[m]
        # the end state: committed, rebuilt, every node's row; the call's conn_ids of restored lightpaths mapped back
        end = commit_traffic(data, rep, demands, releases, tr) if rel else rep
        rows = model.forward_every_node(end.batch)
        span = 1 << 40
        node_r = end.batch.batch.to(torch.int64)
        ec = end.conn_ids.clone()
        if where:
            akey = (wr * span + tr.conn_id)[acc]
            orig = wc[acc]
            nkey = node_r * span + ec
            srt, ix = torch.sort(akey)
            if srt.numel():
                pos = torch.searchsorted(srt, nkey).clamp(max=srt.numel() - 1)
                ec = torch.where(srt[pos] == nkey, orig[ix[pos]], ec)
        local = torch.arange(node_r.numel(), device=dev) - end.batch.ptr[node_r]
        fsel = t(fs)[node_r]
        res.end_out[fsel, local] = rows
        res.end_conn[fsel, local] = ec
    return res


def restoration_ref(model, sample, freqs, lp_feat, conn_of, opts_of, failed, policy, metric=0, maximize=True,
                    bound=None, freq_threshold=0.05, follow=None, device=None, end=True):
    """One scenario, literally, on the fp64 ``model``.  ``sample`` [F, L, Q] numpy; ``conn_of``: the sample's conn_ids
    in node order; ``opts_of[i]``: node i's options (``placement_ref`` tuples); ``failed``: the failed links;
    ``bound``: {conn_id: bound} or None; ``follow``: per demand (filtered option, q0) or None.  Returns ``(cut, steps,
    keep, final, rows)``: the cut nodes (ascending), ``traffic_ref``'s steps of the demands, each demand's kept
    option indices, the final sample and ``(state, rows)`` of its every-node readout in node order (the final sample's
    graph built by ``lightpath_network_state`` as sample 0 of a batch, rows by ``lightpath_every_node_ref`` on
    ``model``; None with ``end=False``, which needs no GPU)."""
    from every_node_ref import lightpath_every_node_ref
    from gnn_qot_estimation_b200.to_graph import lightpath_network_state
    cc = cut_set(sample, lp_feat, failed)
    cut = [i for i, c in enumerate(conn_of) if c in cc]
    seq = [("r", conn_of[i]) for i in cut]
    keep = []
    for i in cut:
        k = [j for j, (links, *_) in enumerate(opts_of[i]) if not set(links) & set(failed)]
        if k:
            keep.append(k)
            seq.append(("d", [opts_of[i][j] for j in k]))
    steps, final = traffic_ref(model, sample, freqs, lp_feat, seq, policy, metric, maximize, bound, freq_threshold,
                               follow=follow, device=device)
    if not end:
        return cut, steps[len(cut):], keep, final, None
    # the final sample is built next to the original one, so that the batch has edges even when the final has none
    st = lightpath_network_state(torch.from_numpy(np.stack([final, sample])).to(device), torch.as_tensor(freqs),
                                 lp_feat, freq_threshold)
    b = st.batch
    rows = lightpath_every_node_ref(model, SimpleNamespace(x=b.x.double(), edge_index=b.edge_index, batch=b.batch))
    return cut, steps[len(cut):], keep, final, (st, rows[:int(b.ptr[1])])
