"""Times LightpathGNN's change-set QoT (qot_lightpath_change_sets, csrc/lightpath_candidates.cu) against the expansion
path producing the same predictions: clear every lightpath a set moves or tears down from a copy of its sample, write
every placement, create_lightpath_graphs over the copies, collate, forward_every_node, pick the changed lightpaths'
rows and the impact rows by conn_id.  In the same call, the single-change sets against forward_reconfigurations on the
same changes, to show what the set machinery costs.

    python scripts/time_change_sets.py [--states 64] [--links 60] [--freqs 80] [--sets-per-state 256] [--expand 512]
                                       [--max-impact 64] [--seed 5] [--out FILE]

States: network_status_samples (seed --seed).  Sets: synthetic.lightpath_change_sets (restoration, batch insertion,
defragmentation with swaps, single changes).  forward_change_sets runs over all sets as ONE CUDA-graph replay after a
read that evicts L2, timed with CUDA events; so do forward_reconfigurations and forward_change_sets over the
single-change sets alone, whose outputs must agree bit for bit.  The expansion path (it synchronises inside
create_lightpath_graphs, so it is timed eagerly with CUDA events, after a warm-up call) runs the first --expand sets;
outputs are compared on them (1e-5 relative, 2e-6 absolute floor).  Prints one JSON line: sets/s, changes/s and rows/s
of each path, the max relative difference, per-change algorithmic bytes and head MMAs, the bound that applies, the
GPU's name and power limit.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from time_candidates import (HBM_BYTES_PER_S, MMA_SYNC_TF32_FLOPS, gpu_identity,  # noqa: E402
                             head_mmas)


def parse_args(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--states", type=int, default=64, help="network states (samples)")
    p.add_argument("--links", type=int, default=60)
    p.add_argument("--freqs", type=int, default=80, help="slots of the frequency grid")
    p.add_argument("--sets-per-state", type=int, default=256)
    p.add_argument("--expand", type=int, default=512, help="sets also run through the expansion path")
    p.add_argument("--max-impact", type=int, default=64)
    p.add_argument("--seed", type=int, default=5)
    p.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = p.parse_args(argv)
    if min(a.states, a.links, a.freqs, a.sets_per_state, a.expand) < 1 or a.max_impact < 0:
        p.error("need states, links, freqs, sets-per-state, expand >= 1 and max-impact >= 0")
    return a


def algorithmic_bytes(K: int, G: int, path_links: int, Q: int, impact_rows: int, row_edges: int, max_impact: int,
                      moved: int, moved_edges: int, pairs: int) -> int:
    """Compulsory traffic of one launch over K changes in G sets: per change its node and change arrays (8 + 40 B)
    and its out row and status (16 B); per set its set_ptr entry, set_status and n_impact (16 B) and 21 B per impact
    slot; time_reconfig's terms for links, impact rows and moved lightpaths; and 16 B (two link_ptr pairs) per pair
    of placed changes of a set whose paths are compared."""
    return (K * (8 + 40 + 16) + G * (16 + 21 * max_impact) + path_links * (4 + 4 * Q) + 36 * impact_rows +
            8 * row_edges + 16 * moved + 8 * moved_edges + 16 * pairs)


def expansion_inputs(samples, changes, set_ptr, conn_ids, count: int):
    """Host-side part of the expansion path for the first `count` sets: the sample of each copy, the (copy, conn_id)
    pairs to clear, each change's conn_id (an insertion's one above the sample's largest, +1 per insertion in set
    order) and written vector, and the (change, link, slot) channels to write.  Returns (sample [c], clear_copy,
    clear_conn, change_copy [k], conn [k], vec [k, F] float32, ck, cl, cq)."""
    import numpy as np
    fi = {k: i for i, k in enumerate(samples["lp_feat"])}
    data = samples["data"]
    conn_rows = np.trunc(data[:, fi["conn_id"]])
    occ = np.any(data != 0, axis=1)
    top = conn_rows.reshape(data.shape[0], -1).max(axis=1).astype(np.int64)
    sp = set_ptr.numpy()
    nk = int(sp[count])
    node, smp = changes.node.numpy(), changes.sample.numpy()
    lp, lk = changes.link_ptr.numpy(), changes.links.numpy()
    q0, w, feat = changes.q0.numpy(), changes.width.numpy(), changes.feat.numpy()
    copy_smp = smp[sp[:count]]
    clear_copy, clear_conn = [], []
    copy_of = np.zeros(nk, dtype=np.int64)
    conn = np.zeros(nk, dtype=np.int64)
    vec = np.zeros((nk, data.shape[1]), dtype=np.float32)
    ck, cl, cq = [], [], []
    for g in range(count):
        ins = 0
        for k in range(sp[g], sp[g + 1]):
            s = int(smp[k])
            copy_of[k] = g
            if node[k] < 0:
                ins += 1
                conn[k] = top[s] + ins
                vec[k, fi["conn_id"]] = conn[k]
                vec[k, [fi["osnr"], fi["snr"], fi["ber"]]] = -1.0
            else:
                conn[k] = int(conn_ids[node[k]])
                clear_copy.append(g)
                clear_conn.append(conn[k])
                ls, qs = np.nonzero(occ[s] & (conn_rows[s] == conn[k]))
                vec[k] = data[s, :, ls[0], qs[0]]
            for i, name in enumerate(("freq", "mod_order", "num_spans", "path_len")):
                vec[k, fi[name]] = feat[k, i]
            for l in lk[lp[k]:lp[k + 1]]:
                for q in range(q0[k], q0[k] + w[k]):
                    ck.append(k)
                    cl.append(int(l))
                    cq.append(q)
    t = lambda v: torch.tensor(np.asarray(v), dtype=torch.int64)
    return (t(copy_smp), t(clear_copy), t(clear_conn), t(copy_of), t(conn), torch.from_numpy(vec), t(ck), t(cl),
            t(cq))


def _graph_time(fn, l2_flush):
    """fn captured as one CUDA graph, replayed once untimed, then once after an L2-evicting read: (result, us)."""
    s = torch.cuda.Stream()
    holder = {}
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        fn()
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            holder["r"] = fn()
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l2_flush.sum()
        e0.record(s)
        g.replay()
        e1.record(s)
        torch.cuda.synchronize()
    return holder["r"], e0.elapsed_time(e1) * 1e3


def main(argv=None):
    a = parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("time_change_sets.py measures on a CUDA device; none is available")
    from gnn_qot_estimation_b200 import LightpathGNN, ops, synthetic
    from gnn_qot_estimation_b200.to_graph import LightpathChanges, create_lightpath_graphs, lightpath_network_state
    dev = torch.device("cuda:0")
    root = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
    sd = torch.load(os.path.join(root, "tests/golden/ckpt_lightpath_model_1.pt"), map_location="cpu",
                    weights_only=False)["model_state_dict"]
    m = LightpathGNN(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    m.load_state_dict(sd)
    m.to(dev).eval()
    smp = synthetic.network_status_samples(a.states, num_links=a.links, num_freqs=a.freqs, seed=a.seed)
    data = torch.from_numpy(smp["data"]).to(dev)
    freqs = torch.from_numpy(smp["freqs"])
    state = lightpath_network_state(data, freqs, smp["lp_feat"])
    ch_h, sp_h = synthetic.lightpath_change_sets(smp, state, a.sets_per_state, seed=a.seed + 1)
    K, G = int(ch_h.sample.shape[0]), int(sp_h.shape[0]) - 1
    ch, sp = ch_h.to(dev), sp_h.to(dev)
    MI = a.max_impact
    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    r, t_set = _graph_time(lambda: m.forward_change_sets(state, ch, sp, MI), l2_flush)

    # ---- the single-change sets: forward_reconfigurations vs forward_change_sets on the same changes
    size = sp[1:] - sp[:-1]
    one = sp[:-1][size == 1]
    ch1 = LightpathChanges(*(t[one] for t in (ch.node, ch.sample)),
                           *_sub_paths(ch, one), *(t[one] for t in (ch.q0, ch.width, ch.feat)))
    sp1 = torch.arange(one.numel() + 1, device=dev)
    rr, t_rec = _graph_time(lambda: m.forward_reconfigurations(state, ch1, MI), l2_flush)
    r1, t_one = _graph_time(lambda: m.forward_change_sets(state, ch1, sp1, MI), l2_flush)
    same = lambda x, y: bool(torch.equal(x.nan_to_num(7.0) if x.is_floating_point() else x,
                                         y.nan_to_num(7.0) if y.is_floating_point() else y))
    single_identical = all(same(getattr(rr, f), getattr(r1, f)) for f in
                           ("out", "status", "n_impact", "impact_node", "impact_kind", "impact_out"))

    # ---- expansion path on the first --expand sets
    X = min(a.expand, G)
    (esmp, clr_copy, clr_conn, copy_of, econn, vec, ck, cl, cq) = (
        t.to(dev) for t in expansion_inputs(smp, ch_h, sp_h, state.conn_ids.cpu().numpy(), X))
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    metric = ["osnr", "snr", "ber"]

    def expand():
        ex = data[esmp].clone()
        crow = torch.trunc(ex[clr_copy, fi["conn_id"]])
        hit = (ex[clr_copy] != 0).any(dim=1) & (crow == clr_conn[:, None, None].to(ex.dtype))
        mine = torch.zeros(ex.shape[0], *hit.shape[1:], dtype=torch.int32, device=dev)
        mine.index_add_(0, clr_copy, hit.to(torch.int32))
        ex.masked_fill_((mine > 0)[:, None], 0.0)
        ex[copy_of[ck], :, cl, cq] = vec[ck]
        st, conn = create_lightpath_graphs(ex, torch.zeros(X, 3, dtype=torch.float64, device=dev), freqs,
                                           smp["lp_feat"], metric, return_conn_ids=True)
        st.sym_by_src = True
        b = st.collate(range(X))
        return b, conn, m.forward_every_node(b)

    expand()
    torch.cuda.synchronize()
    l2_flush.sum()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eb, econn_ids, eout = expand()
    e1.record()
    torch.cuda.synchronize()
    t_exp = e0.elapsed_time(e1) * 1e3

    # ---- parity on the expanded sets, rows matched by (copy, conn_id)
    XK = int(sp_h[X])
    big = int(max(int(econn_ids.max()) if econn_ids.numel() else 0, int(econn.max()) if econn.numel() else 0)) + 2
    key = eb.batch * big + econn_ids
    order = torch.argsort(key)
    skey = key[order]

    def lookup(copy, conn):
        q = copy * big + conn
        i = torch.searchsorted(skey, q).clamp(max=max(skey.numel() - 1, 0))
        assert bool((skey[i] == q).all()), "a lightpath is missing from the expanded graph"
        return order[i]

    placed = ch.link_ptr[1:XK + 1] > ch.link_ptr[:XK]
    kk = torch.arange(XK, device=dev)[placed]
    got = [r.out[:XK][placed]]
    ref = [eout[lookup(copy_of[kk], econn[kk])]]
    rows_g = torch.minimum(r.n_impact[:X].long(), torch.tensor(MI, device=dev))
    sel = torch.arange(MI, device=dev)[None, :] < rows_g[:, None]
    gr, ir = sel.nonzero(as_tuple=True)
    if gr.numel():
        got.append(r.impact_out[:X][gr, ir])
        ref.append(eout[lookup(gr, state.conn_ids[r.impact_node[:X][gr, ir]])])
    got, ref = torch.cat(got), torch.cat(ref)
    d = (got - ref).abs()
    worst_rel = float(d.max()) / max(float(ref.abs().max()), 1e-30)
    ok = bool((d <= 2e-6 + 1e-5 * ref.abs()).all()) and bool(torch.isfinite(got).all())
    fatal = ~ops.CAND_IMPACT_OVERFLOW
    ok &= int((r.set_status[:X] & fatal).max()) == 0 and bool(torch.isnan(r.out[:XK][~placed]).all())
    ok &= single_identical

    # ---- work and bounds
    ok_sets = (r.set_status & fatal) == 0
    ok_chg = torch.repeat_interleave(ok_sets, size)
    lpk = ch.link_ptr[1:] > ch.link_ptr[:-1]
    own_rows = int((ok_chg & lpk).sum())
    rows_all = torch.minimum(r.n_impact.long(), torch.tensor(MI, device=dev))
    impact_rows = int(rows_all[ok_sets].sum())
    rows_total = own_rows + impact_rows
    rp = state.rowptr
    sel = torch.arange(MI, device=dev)[None, :] < rows_all[:, None]
    nodes = r.impact_node[sel]
    row_edges = int((rp[nodes + 1] - rp[nodes]).sum())
    mv = ch.node[ok_chg & (ch.node >= 0)]
    moved_edges = int((rp[mv + 1] - rp[mv]).sum())
    placed_per_set = torch.zeros(G, dtype=torch.int64, device=dev).index_add_(
        0, torch.repeat_interleave(torch.arange(G, device=dev), size), lpk.long())
    pairs = int((placed_per_set * (placed_per_set - 1) // 2).sum())
    alg = algorithmic_bytes(K, G, int(ch.link_ptr[-1]), a.freqs, impact_rows, row_edges, MI, int(mv.numel()),
                            moved_edges, pairs)
    mmas = head_mmas(rows_total)
    bound_hbm = alg / HBM_BYTES_PER_S * 1e6
    bound_tc = mmas * 1024 * 2 / MMA_SYNC_TF32_FLOPS * 1e6
    bound = max(bound_hbm, bound_tc)
    exp_rows = int(placed.sum()) + int(rows_g.sum())
    nd = ch.node
    name, pl = gpu_identity()
    res = {
        "gpu": name, "power_limit": pl, "states": a.states, "links": a.links, "freqs": a.freqs, "sets": G,
        "changes": K, "moves": int(((nd >= 0) & lpk).sum()), "teardowns": int(((nd >= 0) & ~lpk).sum()),
        "insertions": int((nd < 0).sum()), "single_change_sets": int(one.numel()), "max_set": int(size.max()),
        "expanded_sets": X, "expanded_changes": XK, "max_impact": MI,
        "sets_us": t_set, "expansion_us": t_exp,
        "sets_per_s": G / (t_set * 1e-6), "changes_per_s": K / (t_set * 1e-6), "rows_per_s": rows_total / (t_set * 1e-6),
        "expansion_sets_per_s": X / (t_exp * 1e-6), "expansion_changes_per_s": XK / (t_exp * 1e-6),
        "expansion_rows_per_s": exp_rows / (t_exp * 1e-6),
        "speedup_changes_per_s": (K / t_set) / (XK / t_exp),
        "single_sets_us": t_one, "single_reconfig_us": t_rec,
        "single_set_changes_per_s": one.numel() / (t_one * 1e-6),
        "single_reconfig_changes_per_s": one.numel() / (t_rec * 1e-6),
        "single_bit_identical": single_identical,
        "mean_impact_rows_per_set": impact_rows / max(int(ok_sets.sum()), 1),
        "overflow_sets": int(((r.set_status & ops.CAND_IMPACT_OVERFLOW) != 0).sum()),
        "rejected_sets": int((~ok_sets).sum()),
        "alg_bytes_per_change": alg / K, "head_mmas_per_change": mmas / K,
        "hbm_bound_us": bound_hbm, "tensor_pipe_bound_us": bound_tc,
        "bound": "hbm" if bound_hbm >= bound_tc else "tensor_pipe", "bound_fraction": bound / t_set,
        "parity_ok": ok, "parity_rel_err": worst_rel,
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not ok:
        raise SystemExit("forward_change_sets disagrees with the expansion path or with forward_reconfigurations")


def _sub_paths(ch, idx):
    """(link_ptr, links) of the changes `idx` of `ch`, in that order."""
    a, b = ch.link_ptr[idx], ch.link_ptr[idx + 1]
    n = b - a
    lp = torch.zeros(idx.numel() + 1, dtype=torch.int64, device=idx.device)
    lp[1:] = torch.cumsum(n, 0)
    pos = torch.repeat_interleave(a - lp[:-1], n) + torch.arange(int(lp[-1]), device=idx.device)
    return lp, ch.links[pos]


if __name__ == "__main__":
    main()
