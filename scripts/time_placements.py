"""Times LightpathGNN's placement search (qot_lightpath_placements, csrc/lightpath_candidates.cu) against the expansion
path producing the same choices: every free placement of every demand enumerated on the device with torch ops, all of
them through forward_candidates (max_impact large enough that none overflows), the margins and the choice taken in
torch.

    python scripts/time_placements.py [--states 64] [--links 60] [--freqs 80] [--demands 8192] [--max-impact 64]
                                      [--seed 5] [--out FILE]

States: network_status_samples (seed --seed).  Demands: synthetic.lightpath_demands, spread evenly over the states.
Both paths answer PLACE_MAX_MARGIN on output column 0 (maximised) with a per-lightpath bound (each lightpath's
every-node value minus 0.01), so every impact row of every placement counts.  forward_placements runs as ONE
CUDA-graph replay after a read that evicts L2, timed with CUDA events; the expansion synchronises inside (nonzero), so
it is timed eagerly with CUDA events after a warm-up call and an L2-evicting read.  Prints one JSON line: demands/s and
placements/s of both paths, whether the choices match exactly, the max relative difference of the chosen rows,
per-demand algorithmic bytes and head MMAs, the bound that applies and the fraction of it reached, the GPU's name and
power limit.
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
EXPAND_MAX_IMPACT = 256         # a sample holds at most 256 lightpaths: no placement overflows


def parse_args(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--states", type=int, default=64, help="network states (samples)")
    p.add_argument("--links", type=int, default=60)
    p.add_argument("--freqs", type=int, default=80, help="slots of the frequency grid")
    p.add_argument("--demands", type=int, default=8192, help="demands, spread evenly over the states")
    p.add_argument("--max-impact", type=int, default=64)
    p.add_argument("--seed", type=int, default=5)
    p.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = p.parse_args(argv)
    if min(a.states, a.links, a.freqs) < 1 or a.freqs > 1024 or a.demands < a.states or a.max_impact < 0:
        p.error("need states, links >= 1, 1 <= freqs <= 1024, demands >= states, max-impact >= 0")
    return a


def algorithmic_bytes(D: int, P: int, route_links: int, Q: int, impact_rows: int, row_edges: int,
                      max_impact: int) -> int:
    """Compulsory traffic of one launch over D demands with P options: the demand arrays (sample, opt_ptr: 16 B), the
    option arrays (link_ptr, width, feat, own_bound: 28 B; 4 B per link), the chan_node rows of every route link (4 B
    per slot), per impact row of a chosen placement its lightpath's x row (20 B), rowptr pair (16 B), bound (4 B) and
    out-run destinations (8 B per edge), and the outputs (option, q0, margin, n_free, n_feasible, status, n_impact,
    out: 40 B; 20 B per impact slot).  The impact rows a bound adds during the search read the same sample's rows
    again (cache hits) and are not counted."""
    return D * (16 + 40 + 20 * max_impact) + P * 28 + route_links * (4 + 4 * Q) + 40 * impact_rows + 8 * row_edges


def head_mmas(rows: int) -> float:
    """m16n8k8 MMAs of the readout head over `rows` z rows (3xTF32 split, rows go 16 at a time)."""
    return rows / 16 * HEAD_MMAS_PER_16_ROWS


def expand(state, d):
    """Every free placement of every demand, on the device: (option index p [X], q0 [X], LightpathCandidates)."""
    from gnn_qot_estimation_b200.to_graph import LightpathCandidates
    dev = d.sample.device
    P, Q = int(d.width.shape[0]), state.Q
    n_opt = d.opt_ptr[1:] - d.opt_ptr[:-1]
    opt_dem = torch.repeat_interleave(torch.arange(d.sample.shape[0], device=dev), n_opt)        # [P]
    rlen = d.link_ptr[1:] - d.link_ptr[:-1]
    link_opt = torch.repeat_interleave(torch.arange(P, device=dev), rlen)                      # [n]
    busy = (state.chan_node[d.sample[opt_dem[link_opt]], d.links.long()] != -1).to(torch.int32)   # [n, Q]
    occ = torch.zeros(P, Q, dtype=torch.int32, device=dev).index_add_(0, link_opt, busy)      # [P, Q]
    cs = torch.nn.functional.pad(torch.cumsum((occ > 0).to(torch.int32), 1), (1, 0))          # [P, Q+1]
    q = torch.arange(Q, device=dev)
    end = q[None, :] + d.width[:, None].long()
    ok = (end <= Q) & ((cs.gather(1, end.clamp(max=Q)) - cs[:, :Q]) == 0)
    p, q0 = ok.nonzero(as_tuple=True)
    rl = rlen[p]
    lptr = torch.nn.functional.pad(torch.cumsum(rl, 0), (1, 0))
    pos = torch.arange(int(lptr[-1]), device=dev) - torch.repeat_interleave(lptr[:-1], rl)
    links = d.links[torch.repeat_interleave(d.link_ptr[p], rl) + pos]
    feat = torch.cat([state.freqs[q0].to(torch.float32)[:, None], d.feat[p]], 1)
    c = LightpathCandidates(d.sample[opt_dem[p]], lptr, links, q0.to(torch.int32), d.width[p], feat)
    return p, q0, opt_dem, c


def select(p, q0, opt_dem, d, r, bound, max_impact):
    """PLACE_MAX_MARGIN (column 0, maximised) over the expansion: option, q0, n_free, n_feasible, chosen rows."""
    D = int(d.sample.shape[0])
    dem = opt_dem[p]
    mg = r.out[:, 0] - d.own_bound[p]
    rows = torch.arange(r.impact_out.shape[1], device=p.device)[None, :] < r.n_impact[:, None]
    im = torch.where(rows, r.impact_out[:, :, 0] - bound[r.impact_node.clamp(min=0)], float("inf"))
    mg = torch.minimum(mg, im.min(1).values)
    feas = mg >= 0
    key = torch.where(feas, mg, -float("inf"))
    top = torch.full((D,), -float("inf"), device=p.device).scatter_reduce(0, dem, key, "amax")
    X = p.shape[0]
    idx = torch.arange(X, device=p.device)
    cand = torch.where(feas & (key == top[dem]), idx, X)
    best = torch.full((D,), X, device=p.device).scatter_reduce(0, dem, cand, "amin")
    has = best < X
    b = best.clamp(max=max(X - 1, 0))
    option = torch.where(has, (p[b] - d.opt_ptr[:-1]).to(torch.int32), -1)
    qq = torch.where(has, q0[b].to(torch.int32), -1)
    n_free = torch.bincount(dem, minlength=D).to(torch.int32)
    n_feas = torch.bincount(dem[feas], minlength=D).to(torch.int32)
    return option, qq, n_free, n_feas, has, b, mg


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def _graphed(fn, s, l2_flush):
    """Captures fn in a CUDA graph; returns (its result, replay time in us after an L2-evicting read)."""
    g = torch.cuda.CUDAGraph()
    holder = {}
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
        raise SystemExit("time_placements.py measures on a CUDA device; none is available")
    from gnn_qot_estimation_b200 import LightpathGNN, ops, synthetic
    from gnn_qot_estimation_b200.to_graph import lightpath_network_state
    dev = torch.device("cuda:0")
    root = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
    sd = torch.load(os.path.join(root, "tests/golden/ckpt_lightpath_model_1.pt"), map_location="cpu",
                    weights_only=False)["model_state_dict"]
    m = LightpathGNN(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    m.load_state_dict(sd)
    m.to(dev).eval()
    smp = synthetic.network_status_samples(a.states, num_links=a.links, num_freqs=a.freqs, seed=a.seed)
    d = synthetic.lightpath_demands(smp, a.demands // a.states, seed=a.seed + 1).to(dev)
    D, P = int(d.sample.shape[0]), int(d.width.shape[0])
    state = lightpath_network_state(torch.from_numpy(smp["data"]).to(dev), torch.from_numpy(smp["freqs"]),
                                    smp["lp_feat"])
    bound = (m.forward_every_node(state.batch)[:, 0] - 0.01).contiguous()
    MI = a.max_impact
    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    s = torch.cuda.Stream()
    r, t_pl = _graphed(lambda: m.forward_placements(state, d, ops.PLACE_MAX_MARGIN, 0, True, bound, MI), s, l2_flush)

    def expansion():
        p, q0, opt_dem, c = expand(state, d)
        rc = m.forward_candidates(state, c, EXPAND_MAX_IMPACT)
        return (p, q0, opt_dem, rc) + select(p, q0, opt_dem, d, rc, bound, MI)

    # the expansion synchronises (its sizes are data-dependent), so it is timed eagerly with CUDA events after a
    # warm-up call
    expansion()
    torch.cuda.synchronize()
    l2_flush.sum()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ex = expansion()
    e1.record()
    torch.cuda.synchronize()
    t_exp = e0.elapsed_time(e1) * 1e3
    p, q0, opt_dem, rc, option, qq, n_free, n_feas, has, b, mg = ex
    X = int(p.shape[0])
    assert int((rc.status & ops.CAND_IMPACT_OVERFLOW).sum()) == 0, "the expansion must not overflow"

    # ---- the choices, counts and rows
    ok = bool(torch.equal(r.option, option) and torch.equal(r.q0, qq) and torch.equal(r.n_free, n_free) and
              torch.equal(r.n_feasible, n_feas))
    ok &= int((r.status & ~ops.CAND_IMPACT_OVERFLOW).sum()) == 0
    got, ref = r.out[has], rc.out[b[has]]
    d_ = (got - ref).abs()
    worst = float(d_.max()) / max(float(ref.abs().max()), 1e-30) if got.numel() else 0.0
    ok &= bool(torch.equal(r.margin[has], mg[b[has]])) and bool(torch.isnan(r.out[~has]).all())
    nimp = rc.n_impact[b[has]].long()
    ok &= bool(torch.equal(r.n_impact[has].long(), nimp))
    rows_k = torch.minimum(nimp, torch.tensor(MI, device=dev))
    sel = torch.arange(MI, device=dev)[None, :] < rows_k[:, None]
    ok &= bool(torch.equal(r.impact_node[has][sel], rc.impact_node[b[has]][:, :MI][sel]))
    ok &= bool(torch.equal(r.impact_out[has][sel], rc.impact_out[b[has]][:, :MI][sel]))

    # ---- work and bounds
    search_rows = X + int(rc.n_impact.long().sum())               # every own and every impact row (a bound is given)
    chosen_rows = int(rows_k.sum())
    rp = state.rowptr
    nodes = r.impact_node[has][sel]
    row_edges = int((rp[nodes + 1] - rp[nodes]).sum())
    alg = algorithmic_bytes(D, P, int(d.link_ptr[-1]), a.freqs, chosen_rows, row_edges, MI)
    mmas = head_mmas(search_rows + chosen_rows)
    bound_hbm = alg / HBM_BYTES_PER_S * 1e6
    bound_tc = mmas * 1024 * 2 / MMA_SYNC_TF32_FLOPS * 1e6
    bnd = max(bound_hbm, bound_tc)
    name, pl = gpu_identity()
    res = {
        "gpu": name, "power_limit": pl, "states": a.states, "links": a.links, "freqs": a.freqs, "demands": D,
        "options": P, "placements": X, "max_impact": MI, "policy": "max_margin",
        "placements_us": t_pl, "expansion_us": t_exp,
        "demands_per_s": D / (t_pl * 1e-6), "expansion_demands_per_s": D / (t_exp * 1e-6),
        "placements_per_s": X / (t_pl * 1e-6), "expansion_placements_per_s": X / (t_exp * 1e-6),
        "speedup": t_exp / t_pl,
        "feasible_demands": int(has.sum()), "mean_impact_rows_per_placement": (search_rows - X) / max(X, 1),
        "alg_bytes_per_demand": alg / D, "head_mmas_per_demand": mmas / D,
        "hbm_bound_us": bound_hbm, "tensor_pipe_bound_us": bound_tc,
        "bound": "hbm" if bound_hbm >= bound_tc else "tensor_pipe", "bound_fraction": bnd / t_pl,
        "choices_match": ok, "rows_max_rel_diff": worst,
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not ok:
        raise SystemExit("forward_placements disagrees with the expansion path")


if __name__ == "__main__":
    main()
