"""Times LightpathGNN's candidate QoT (csrc/lightpath_candidates.cu) against the expansion path producing the same
predictions: write each candidate into a copy of its sample, create_lightpath_graphs over the copies, collate,
forward_every_node, pick the candidate's row and its neighbours' rows by conn_id.

    python scripts/time_candidates.py [--states 64] [--links 60] [--freqs 80] [--candidates 65536] [--expand 4096]
                                      [--max-impact 64] [--seed 5] [--out FILE]

States: network_status_samples (seed --seed).  Candidates: synthetic.lightpath_candidates, spread evenly over the
states.  forward_candidates runs over all --candidates as ONE CUDA-graph replay after a read that evicts L2, timed
with CUDA events; the expansion path (it synchronises inside create_lightpath_graphs, so it is timed eagerly with CUDA
events, after a warm-up call) runs the first --expand candidates.  Outputs are compared on those candidates (1e-5
relative, 2e-6 absolute floor).  Prints one JSON line: candidates/s and rows/s of both paths, their ratio, the max
relative difference, per-candidate algorithmic bytes and head MMAs, the bound that applies, the GPU's name and power
limit.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

MMA_SYNC_TF32_FLOPS = 295e12    # profiles/r1_mma_sync_rate.txt: mma.sync m16n8k8 TF32, 148 SMs, B200
HEAD_MMAS_PER_16_ROWS = 240     # head_rows16_tf32x3: 4 heads x 4 (3 projection + 4 x 3 mlp.0) m16n8k8 MMAs
HBM_BYTES_PER_S = 6.5e12        # measured stream bandwidth of the B200 (DESIGN.md)


def parse_args(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--states", type=int, default=64, help="network states (samples)")
    p.add_argument("--links", type=int, default=60)
    p.add_argument("--freqs", type=int, default=80, help="slots of the frequency grid")
    p.add_argument("--candidates", type=int, default=65536, help="candidates, spread evenly over the states")
    p.add_argument("--expand", type=int, default=4096, help="candidates also run through the expansion path")
    p.add_argument("--max-impact", type=int, default=64)
    p.add_argument("--seed", type=int, default=5)
    p.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = p.parse_args(argv)
    if min(a.states, a.links, a.freqs) < 1 or a.candidates < a.states or not 1 <= a.expand <= a.candidates \
            or a.max_impact < 0:
        p.error("need states, links, freqs >= 1, candidates >= states, 1 <= expand <= candidates, max-impact >= 0")
    return a


def algorithmic_bytes(K: int, path_links: int, Q: int, impact_rows: int, row_edges: int, max_impact: int) -> int:
    """Compulsory traffic of one launch over K candidates: their arrays (sample, link_ptr, q0, width, feat: 40 B; 4 B
    per link), the chan_node rows of their links (4 B per slot), per impact row the neighbour's x row (20 B), its
    rowptr pair (16 B) and its out-run's destinations (8 B per edge), and the outputs (out, status, n_impact: 20 B; 20 B
    per impact slot).  Message sources' x rows are other neighbours' rows (cache hits) and are not counted."""
    return K * (40 + 20 + 20 * max_impact) + path_links * (4 + 4 * Q) + 36 * impact_rows + 8 * row_edges


def head_mmas(rows: int) -> float:
    """m16n8k8 MMAs of the readout head over `rows` z rows (3xTF32 split, rows go 16 at a time)."""
    return rows / 16 * HEAD_MMAS_PER_16_ROWS


def expansion_inputs(samples, cands, count: int):
    """Host-side part of the expansion path for the first `count` candidates: the sample of each copy, the new
    conn_id, and the (copy, link, slot) channels to write.  Returns (sample [c], conn [c], ck, cl, cq) int64 tensors."""
    import numpy as np
    fi = {k: i for i, k in enumerate(samples["lp_feat"])}
    data = samples["data"]
    top = np.trunc(data[:, fi["conn_id"]]).reshape(data.shape[0], -1).max(axis=1).astype(np.int64)
    smp = cands.sample[:count].numpy()
    lp, lk = cands.link_ptr.numpy(), cands.links.numpy()
    q0, w = cands.q0.numpy(), cands.width.numpy()
    ck, cl, cq = [], [], []
    for k in range(count):
        for l in lk[lp[k]:lp[k + 1]]:
            for q in range(q0[k], q0[k] + w[k]):
                ck.append(k)
                cl.append(int(l))
                cq.append(q)
    t = lambda v: torch.tensor(np.asarray(v), dtype=torch.int64)
    return t(smp), t(top[smp] + 1), t(ck), t(cl), t(cq)


def channel_vectors(lp_feat, conn, feat):
    """[c, F] float32: what the candidate writes on each of its channels (new conn_id, feat, osnr = snr = ber = -1)."""
    fi = {k: i for i, k in enumerate(lp_feat)}
    v = torch.zeros(conn.shape[0], len(lp_feat), dtype=torch.float32, device=feat.device)
    v[:, fi["conn_id"]] = conn.to(torch.float32)
    for k, name in enumerate(("freq", "mod_order", "num_spans", "path_len")):
        v[:, fi[name]] = feat[:, k]
    v[:, fi["osnr"]] = v[:, fi["snr"]] = v[:, fi["ber"]] = -1.0
    return v


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def main(argv=None):
    a = parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("time_candidates.py measures on a CUDA device; none is available")
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
    cands_h = synthetic.lightpath_candidates(smp, a.candidates // a.states, seed=a.seed + 1)
    K = int(cands_h.sample.shape[0])
    data = torch.from_numpy(smp["data"]).to(dev)
    freqs = torch.from_numpy(smp["freqs"])
    state = lightpath_network_state(data, freqs, smp["lp_feat"])
    cands = cands_h.to(dev)
    MI = a.max_impact
    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    s = torch.cuda.Stream()
    holder = {}

    def run():
        holder["r"] = m.forward_candidates(state, cands, MI)

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
    t_cand = e0.elapsed_time(e1) * 1e3                                        # us
    r = holder["r"]

    # ---- expansion path on the first --expand candidates
    X = min(a.expand, K)
    esmp, econn, ck, cl, cq = (t.to(dev) for t in expansion_inputs(smp, cands_h, X))
    vec = channel_vectors(smp["lp_feat"], econn, cands.feat[:X])
    metric = ["osnr", "snr", "ber"]

    def expand():
        ex = data[esmp].clone()
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

    # ---- parity on the expanded candidates, rows matched by (copy, conn_id)
    n_imp = r.n_impact[:X].long()
    rows_k = torch.minimum(n_imp, torch.tensor(MI, device=dev))
    big = int(econn_ids.max().item() if econn_ids.numel() else 0) + int(econn.max().item()) + 2
    key = eb.batch * big + econn_ids
    order = torch.argsort(key)
    skey = key[order]

    def lookup(copy, conn):
        q = copy * big + conn
        i = torch.searchsorted(skey, q).clamp(max=skey.numel() - 1)
        assert bool((skey[i] == q).all()), "a lightpath is missing from the expanded graph"
        return order[i]

    kk = torch.arange(X, device=dev)
    got = [r.out[:X]]
    ref = [eout[lookup(kk, econn)]]
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
    ok &= int(status[:X].max()) == 0 and bool(torch.isfinite(got).all())    # free channels, <= MI neighbours
    # the expansion's neighbour count equals n_impact: every row the expanded graph adds for a candidate is matched
    exp_deg = torch.bincount(eb.batch[eb.edge_index[0][eb.edge_index[0] != eb.edge_index[1]]], minlength=X)
    base_deg = torch.bincount(state.batch.batch[state.batch.edge_index[0][state.batch.edge_index[0] !=
                                                                          state.batch.edge_index[1]]],
                              minlength=a.states)
    ok &= bool(torch.equal(exp_deg - base_deg[esmp], 2 * n_imp))

    # ---- work and bounds
    ok_rows = (status & 7) == 0
    impact_rows = int(torch.minimum(r.n_impact.long(), torch.tensor(MI, device=dev))[ok_rows].sum())
    rows_total = int(ok_rows.sum()) + impact_rows
    rp = state.rowptr
    sel = torch.arange(MI, device=dev)[None, :] < torch.minimum(r.n_impact.long(), torch.tensor(MI, device=dev))[:, None]
    nodes = r.impact_node[sel]
    row_edges = int((rp[nodes + 1] - rp[nodes]).sum())
    path_links = int(cands.link_ptr[-1])
    alg = algorithmic_bytes(K, path_links, a.freqs, impact_rows, row_edges, MI)
    mmas = head_mmas(rows_total)
    bound_hbm = alg / HBM_BYTES_PER_S * 1e6
    bound_tc = mmas * 1024 * 2 / MMA_SYNC_TF32_FLOPS * 1e6
    bound = max(bound_hbm, bound_tc)
    exp_rows = X + int(rows_k.sum())
    name, pl = gpu_identity()
    res = {
        "gpu": name, "power_limit": pl, "states": a.states, "links": a.links, "freqs": a.freqs, "candidates": K,
        "expanded_candidates": X, "max_impact": MI,
        "candidates_us": t_cand, "expansion_us": t_exp,
        "candidates_per_s": K / (t_cand * 1e-6), "expansion_candidates_per_s": X / (t_exp * 1e-6),
        "rows_per_s": rows_total / (t_cand * 1e-6), "expansion_rows_per_s": exp_rows / (t_exp * 1e-6),
        "speedup_candidates_per_s": (K / t_cand) / (X / t_exp),
        "mean_impact_rows": impact_rows / max(int(ok_rows.sum()), 1),
        "overflow_candidates": int(((status & 8) != 0).sum()),
        "alg_bytes_per_candidate": alg / K, "head_mmas_per_candidate": mmas / K,
        "hbm_bound_us": bound_hbm, "tensor_pipe_bound_us": bound_tc,
        "bound": "hbm" if bound_hbm >= bound_tc else "tensor_pipe", "bound_fraction": bound / t_cand,
        "parity_ok": ok, "parity_rel_err": worst_rel,
        "rejected_candidates": int(((status & 7) != 0).sum()),
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not ok:
        raise SystemExit("forward_candidates disagrees with the expansion path")


if __name__ == "__main__":
    main()
