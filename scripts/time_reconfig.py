"""Times LightpathGNN's reconfiguration QoT (qot_lightpath_reconfigure, csrc/lightpath_candidates.cu) against the
expansion path producing the same predictions: clear the moved lightpath from a copy of its sample, write it on its new
path and slots, create_lightpath_graphs over the copies, collate, forward_every_node, pick the moved lightpath's row and
its old and new neighbours' rows by conn_id.

    python scripts/time_reconfig.py [--states 64] [--links 60] [--freqs 80] [--changes 65536] [--expand 4096]
                                    [--max-impact 64] [--seed 5] [--out FILE]

States: network_status_samples (seed --seed).  Changes: synthetic.lightpath_changes (retunes, reroutes, teardowns and
insertions), spread evenly over the states.  forward_reconfigurations runs over all --changes as ONE CUDA-graph replay
after a read that evicts L2, timed with CUDA events; the expansion path (it synchronises inside
create_lightpath_graphs, so it is timed eagerly with CUDA events, after a warm-up call) runs the first --expand changes.
Outputs are compared on those changes (1e-5 relative, 2e-6 absolute floor), and the kind bits against the moved
lightpath's degree before and after.  Prints one JSON line: changes/s and rows/s of both paths, their ratio, the max
relative difference, per-change algorithmic bytes and head MMAs, the bound that applies, the GPU's name and power
limit.
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
    p.add_argument("--changes", type=int, default=65536, help="changes, spread evenly over the states")
    p.add_argument("--expand", type=int, default=4096, help="changes also run through the expansion path")
    p.add_argument("--max-impact", type=int, default=64)
    p.add_argument("--seed", type=int, default=5)
    p.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = p.parse_args(argv)
    if min(a.states, a.links, a.freqs) < 1 or a.changes < a.states or not 1 <= a.expand <= a.changes \
            or a.max_impact < 0:
        p.error("need states, links, freqs >= 1, changes >= states, 1 <= expand <= changes, max-impact >= 0")
    return a


def algorithmic_bytes(K: int, path_links: int, Q: int, impact_rows: int, row_edges: int, max_impact: int,
                      moved: int, moved_edges: int) -> int:
    """Compulsory traffic of one launch over K changes: time_candidates.algorithmic_bytes' terms (40 B of change
    arrays and 4 B per link, 4 B per chan_node slot of each link, 36 B per impact row plus 8 B per edge of its
    out-run, 20 B of outputs plus 20 B per impact slot), plus what a change adds: the node entry (8 B) and one
    impact_kind byte per impact slot, and for each moved lightpath its rowptr pair (16 B) and its out-run's
    destinations (8 B per edge)."""
    return (K * (40 + 8 + 20 + 21 * max_impact) + path_links * (4 + 4 * Q) + 36 * impact_rows + 8 * row_edges +
            16 * moved + 8 * moved_edges)


def expansion_inputs(samples, changes, conn_ids, count: int):
    """Host-side part of the expansion path for the first `count` changes: the sample of each copy, the conn_id of the
    lightpath it moves (a new one, one above the sample's largest, for an insertion), the vector written on its new
    channels and the (copy, link, slot) channels to write.  ``conn_ids``: the state's [N] conn_ids.  Returns
    (sample [c], conn [c], vec [c, F] float32, ck, cl, cq)."""
    import numpy as np
    fi = {k: i for i, k in enumerate(samples["lp_feat"])}
    data = samples["data"]
    conn_rows = np.trunc(data[:, fi["conn_id"]])
    occ = np.any(data != 0, axis=1)
    top = conn_rows.reshape(data.shape[0], -1).max(axis=1).astype(np.int64)
    smp = changes.sample[:count].numpy()
    node = changes.node[:count].numpy()
    lp, lk = changes.link_ptr.numpy(), changes.links.numpy()
    q0, w, feat = changes.q0.numpy(), changes.width.numpy(), changes.feat.numpy()
    conn = np.zeros(count, dtype=np.int64)
    vec = np.zeros((count, data.shape[1]), dtype=np.float32)
    ck, cl, cq = [], [], []
    for k in range(count):
        s = int(smp[k])
        if node[k] < 0:                                      # an insertion: candidates_ref.insert_candidate's vector
            conn[k] = top[s] + 1
            vec[k, fi["conn_id"]] = conn[k]
            vec[k, [fi["osnr"], fi["snr"], fi["ber"]]] = -1.0
        else:                                                # the lightpath's first channel
            conn[k] = int(conn_ids[node[k]])
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
    return t(smp), t(conn), torch.from_numpy(vec), t(ck), t(cl), t(cq)


def main(argv=None):
    a = parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("time_reconfig.py measures on a CUDA device; none is available")
    from gnn_qot_estimation_b200 import LightpathGNN, synthetic
    from gnn_qot_estimation_b200.to_graph import create_lightpath_graphs, lightpath_network_state
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
    ch_h = synthetic.lightpath_changes(smp, state, a.changes // a.states, seed=a.seed + 1)
    K = int(ch_h.sample.shape[0])
    ch = ch_h.to(dev)
    MI = a.max_impact
    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    s = torch.cuda.Stream()
    holder = {}

    def run():
        holder["r"] = m.forward_reconfigurations(state, ch, MI)

    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        run()
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            run()
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l2_flush.sum()
        e0.record(s)
        g.replay()
        e1.record(s)
        torch.cuda.synchronize()
    t_chg = e0.elapsed_time(e1) * 1e3                                         # us
    r = holder["r"]

    # ---- expansion path on the first --expand changes
    X = min(a.expand, K)
    esmp, econn, vec, ck, cl, cq = (t.to(dev) for t in expansion_inputs(smp, ch_h, state.conn_ids.cpu().numpy(), X))
    fi = {k: i for i, k in enumerate(smp["lp_feat"])}
    metric = ["osnr", "snr", "ber"]

    def expand():
        ex = data[esmp].clone()
        mine = (ex != 0).any(dim=1) & (torch.trunc(ex[:, fi["conn_id"]]) == econn[:, None, None].to(ex.dtype))
        ex.masked_fill_(mine[:, None], 0.0)
        ex[ck, :, cl, cq] = vec[ck]
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

    # ---- parity on the expanded changes, rows matched by (copy, conn_id)
    n_imp = r.n_impact[:X].long()
    rows_k = torch.minimum(n_imp, torch.tensor(MI, device=dev))
    big = int(econn_ids.max().item() if econn_ids.numel() else 0) + int(econn.max().item()) + 2
    key = eb.batch * big + econn_ids
    order = torch.argsort(key)
    skey = key[order]

    def lookup(copy, conn):
        q = copy * big + conn
        i = torch.searchsorted(skey, q).clamp(max=max(skey.numel() - 1, 0))
        assert bool((skey[i] == q).all()), "a lightpath is missing from the expanded graph"
        return order[i]

    kk = torch.arange(X, device=dev)
    placed = ch.link_ptr[1:X + 1] > ch.link_ptr[:X]                          # not a teardown
    kp = kk[placed]
    got = [r.out[:X][placed]]
    ref = [eout[lookup(kp, econn[placed])]]
    sel = torch.arange(MI, device=dev)[None, :] < rows_k[:, None]
    kr, ir = sel.nonzero(as_tuple=True)
    if kr.numel():
        got.append(r.impact_out[:X][kr, ir])
        ref.append(eout[lookup(kr, state.conn_ids[r.impact_node[:X][kr, ir]])])
    got, ref = torch.cat(got), torch.cat(ref)
    d = (got - ref).abs()
    worst_rel = float(d.max()) / max(float(ref.abs().max()), 1e-30)
    ok = bool((d <= 2e-6 + 1e-5 * ref.abs()).all())
    status = r.status
    ok &= int(status[:X].max()) == 0 and bool(torch.isfinite(got).all())    # legal changes, <= MI rows each
    ok &= bool(torch.isnan(r.out[:X][~placed]).all())
    # kind bits: bit 1 counts the moved lightpath's neighbours in the expanded graph, bit 0 those in the state
    kind = r.impact_kind[:X].long()
    n_new, n_old = ((kind >> 1) & 1).sum(1), (kind & 1).sum(1)
    ei = eb.edge_index
    deg_e = torch.bincount(ei[0][ei[0] != ei[1]], minlength=eb.x.shape[0])
    exp_new = torch.zeros(X, dtype=torch.int64, device=dev)
    exp_new[placed] = deg_e[lookup(kp, econn[placed])]
    si = state.batch.edge_index
    deg_s = torch.bincount(si[0][si[0] != si[1]], minlength=state.batch.x.shape[0])
    moved = ch.node[:X] >= 0
    exp_old = torch.where(moved, deg_s[ch.node[:X].clamp(min=0)], torch.zeros_like(exp_new))
    ok &= bool(torch.equal(n_new, exp_new)) and bool(torch.equal(n_old, exp_old))

    # ---- work and bounds
    ok_rows = (status & (1 | 2 | 4 | 16 | 32)) == 0
    own_rows = int((ok_rows & (ch.link_ptr[1:] > ch.link_ptr[:-1])).sum())
    rows_all = torch.minimum(r.n_impact.long(), torch.tensor(MI, device=dev))
    impact_rows = int(rows_all[ok_rows].sum())
    rows_total = own_rows + impact_rows
    rp = state.rowptr
    sel = torch.arange(MI, device=dev)[None, :] < rows_all[:, None]
    nodes = r.impact_node[sel]
    row_edges = int((rp[nodes + 1] - rp[nodes]).sum())
    mv = ch.node[ok_rows & (ch.node >= 0)]
    moved_edges = int((rp[mv + 1] - rp[mv]).sum())
    path_links = int(ch.link_ptr[-1])
    alg = algorithmic_bytes(K, path_links, a.freqs, impact_rows, row_edges, MI, int(mv.numel()), moved_edges)
    mmas = head_mmas(rows_total)
    bound_hbm = alg / HBM_BYTES_PER_S * 1e6
    bound_tc = mmas * 1024 * 2 / MMA_SYNC_TF32_FLOPS * 1e6
    bound = max(bound_hbm, bound_tc)
    exp_rows = int(placed.sum()) + int(rows_k.sum())
    nd, lpk = ch.node, ch.link_ptr[1:] > ch.link_ptr[:-1]
    name, pl = gpu_identity()
    res = {
        "gpu": name, "power_limit": pl, "states": a.states, "links": a.links, "freqs": a.freqs, "changes": K,
        "moves": int(((nd >= 0) & lpk).sum()), "teardowns": int(((nd >= 0) & ~lpk).sum()),
        "insertions": int((nd < 0).sum()), "expanded_changes": X, "max_impact": MI,
        "changes_us": t_chg, "expansion_us": t_exp,
        "changes_per_s": K / (t_chg * 1e-6), "expansion_changes_per_s": X / (t_exp * 1e-6),
        "rows_per_s": rows_total / (t_chg * 1e-6), "expansion_rows_per_s": exp_rows / (t_exp * 1e-6),
        "speedup_changes_per_s": (K / t_chg) / (X / t_exp),
        "mean_impact_rows": impact_rows / max(int(ok_rows.sum()), 1),
        "overflow_changes": int(((status & 8) != 0).sum()),
        "alg_bytes_per_change": alg / K, "head_mmas_per_change": mmas / K,
        "hbm_bound_us": bound_hbm, "tensor_pipe_bound_us": bound_tc,
        "bound": "hbm" if bound_hbm >= bound_tc else "tensor_pipe", "bound_fraction": bound / t_chg,
        "parity_ok": ok, "parity_rel_err": worst_rel,
        "rejected_changes": int((~ok_rows).sum()),
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not ok:
        raise SystemExit("forward_reconfigurations disagrees with the expansion path")


if __name__ == "__main__":
    main()
