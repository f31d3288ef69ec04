"""Times LightpathGNN's dynamic traffic (qot_lightpath_traffic, csrc/lightpath_candidates.cu) against the round loop
producing the same outputs: per event position, forward_reconfigurations teardowns for the releases (their channels
then zeroed in the samples) and forward_placements for the arrivals (the accepted placements written in with
commit_provision), the state rebuilt with lightpath_network_state and the bound carried over through lightpath_nodes
(tests/traffic_ref.py:round_loop).

    python scripts/time_traffic.py [--states 1024] [--links 60] [--freqs 80] [--per-sample 16] [--load 8]
                                   [--release-existing 0.2] [--max-impact 64] [--seed 5] [--blocking-loads 64,256,1024]
                                   [--blocking-arrivals 1024] [--out FILE]

States: network_status_samples (seed --seed, spacing 0.0375).  Traffic: synthetic.lightpath_traffic, --per-sample
arrivals per sample at --load Erlang with unit-mean holding times, and a --release-existing share of the states'
lightpaths released by conn_id.  Both paths answer PLACE_MAX_MARGIN on output column 0 (maximised) with a per-lightpath
bound (each lightpath's every-node value minus 0.01).  forward_traffic runs as ONE CUDA-graph replay after a read that
evicts L2, timed with CUDA events; the round loop synchronises with the host every round, so it is timed eagerly with
CUDA events after a warm-up run.  Prints one JSON line: events/s of both paths, whether every output matches bit for
bit, the algorithmic bytes and head MMAs of the run's counts, the bound that applies and the fraction of it reached,
the blocking probability at each of --blocking-loads (forward_traffic alone, --blocking-arrivals per sample, first fit
with no QoT bound: a demand is blocked by the spectrum or by the sample's capacity, PROV_FULL, whose share is reported
too), the GPU's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))          # traffic_ref: the round loop

MMA_SYNC_TF32_FLOPS = 295e12    # profiles/r1_mma_sync_rate.txt: mma.sync m16n8k8 TF32, 148 SMs, B200
HEAD_MMAS_PER_16_ROWS = 240     # head_rows16_tf32x3: 4 heads x 4 (3 projection + 4 x 3 mlp.0) m16n8k8 MMAs
HBM_BYTES_PER_S = 6.5e12        # measured stream bandwidth of the B200 (DESIGN.md)
FIELDS = ("option", "q0", "out", "margin", "n_free", "n_feasible", "status", "n_impact", "impact_conn", "impact_out",
          "conn_id", "release_status", "release_conn_id", "release_n_impact", "release_impact_conn",
          "release_impact_out", "release_margin")


def parse_args(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--states", type=int, default=1024, help="network states (samples)")
    p.add_argument("--links", type=int, default=60)
    p.add_argument("--freqs", type=int, default=80, help="slots of the frequency grid")
    p.add_argument("--per-sample", type=int, default=16, help="demands per sample (on average)")
    p.add_argument("--load", type=float, default=8.0, help="offered load per sample (Erlang)")
    p.add_argument("--release-existing", type=float, default=0.2, help="share of the states' lightpaths released")
    p.add_argument("--blocking-loads", default="64,256,1024", help="loads of the blocking-probability sweep")
    p.add_argument("--blocking-arrivals", type=int, default=1024, help="arrivals per sample in the sweep")
    p.add_argument("--max-impact", type=int, default=64)
    p.add_argument("--seed", type=int, default=5)
    p.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = p.parse_args(argv)
    if min(a.states, a.links, a.freqs, a.per_sample) < 1 or a.freqs > 1024 or a.max_impact < 0:
        p.error("need states, links, per-sample >= 1, 1 <= freqs <= 1024, max-impact >= 0")
    return a


def algorithmic_bytes(D: int, R: int, S: int, L: int, Q: int, N: int, E: int, P: int, route_links: int,
                      max_impact: int) -> int:
    """Compulsory traffic of one call: the chan_node copy (read and write, 8 B per channel) and the kernel's one read
    of each sample's channels (4 B), the state's x rows (20 B), conn_ids and rowptr (16 B), bound (4 B) and edges (8 B),
    the demand and option arrays (16 B per demand, 28 B per option, 4 B per link), the route rows of every option
    (4 B per slot per link), the accepted channels written (counted with the copy) and the outputs (48 B per demand,
    20 B per impact slot); per release its four inputs (32 B), its grouping entry (8 B), one read and write of its
    sample's channels (8 B per channel) and its outputs (20 B + 20 B per impact slot); impact rows' messages come from
    shared memory."""
    return (12 * S * L * Q + 40 * N + 8 * E + D * (16 + 48 + 20 * max_impact) + P * 28 + route_links * (4 + 4 * Q) +
            R * (60 + 8 * L * Q + 20 * max_impact))


def head_mmas(rows: int) -> float:
    return rows / 16.0 * HEAD_MMAS_PER_16_ROWS


def _gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, lim = (v.strip() for v in q.split(","))
        return name, lim
    except Exception:
        return torch.cuda.get_device_name(), "unknown"


def main(argv=None):
    a = parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("time_traffic.py needs a CUDA device: there is nothing to time without one")
    from gnn_qot_estimation_b200 import LightpathGNN, ops, synthetic
    from gnn_qot_estimation_b200.to_graph import lightpath_network_state
    from traffic_ref import round_loop
    dev = torch.device("cuda")
    from conftest import load_golden
    m = LightpathGNN(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    m.load_state_dict(load_golden("ckpt_lightpath_model_1.pt")["model_state_dict"], strict=True)
    m = m.to(dev).eval()
    smp = synthetic.network_status_samples(a.states, num_links=a.links, num_freqs=a.freqs, seed=a.seed,
                                           spacing=0.0375, super_channel_p=0.3)
    data0 = torch.from_numpy(smp["data"]).to(dev).contiguous()
    freqs = torch.from_numpy(smp["freqs"]).to(dev)
    state = lightpath_network_state(data0, freqs, smp["lp_feat"])
    d, r = synthetic.lightpath_traffic(smp, a.per_sample, a.load, seed=a.seed + 1,
                                       release_existing=a.release_existing)
    d, r = d.to(dev), r.to(dev)
    bound = (m.forward_every_node(state.batch)[:, 0] - 0.01).contiguous()
    D, R = int(d.sample.shape[0]), int(r.sample.shape[0])
    evict = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # 256 MB > 126 MB of L2

    # ---- forward_traffic: one CUDA-graph replay after an L2-evicting read
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        m.forward_traffic(state, d, r, ops.PLACE_MAX_MARGIN, 0, True, bound, a.max_impact)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        res = m.forward_traffic(state, d, r, ops.PLACE_MAX_MARGIN, 0, True, bound, a.max_impact)
    times = []
    for _ in range(5):
        evict.add_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) / 1e3)
    t_traf = sorted(times)[len(times) // 2]

    # ---- the round loop, eager, after a warm-up run
    round_loop(m, data0.clone(), freqs, smp["lp_feat"], d, r, ops.PLACE_MAX_MARGIN, 0, True, bound, a.max_impact)
    data = data0.clone()
    evict.add_(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    ref, _ = round_loop(m, data, freqs, smp["lp_feat"], d, r, ops.PLACE_MAX_MARGIN, 0, True, bound, a.max_impact)
    e1.record()
    torch.cuda.synchronize()
    t_loop = e0.elapsed_time(e1) / 1e3

    def same(x, y):
        if x.is_floating_point():
            return bool(torch.equal(x.nan_to_num(7.0), y.nan_to_num(7.0)) and torch.equal(x.isnan(), y.isnan()))
        return bool(torch.equal(x, y))
    match = {f: same(getattr(res, f), getattr(ref, f)) for f in FIELDS}

    # ---- counts of the run: bytes and head rows (own rows of every free placement, impact rows with the bound, and
    # every release's neighbour rows)
    P = int(d.width.shape[0])
    route_links = int(d.links.shape[0])
    n_free = int(res.n_free.sum())
    n_imp = int(res.n_impact.clamp(max=a.max_impact).sum())
    deg = float(res.n_impact[res.option >= 0].float().mean()) if bool((res.option >= 0).any()) else 0.0
    rows = n_free * (1.0 + deg) + n_imp + int(res.release_n_impact.sum())
    nbytes = algorithmic_bytes(D, R, state.S, state.L, state.Q, int(state.batch.x.shape[0]),
                               int(state.batch.edge_index.shape[1]), P, route_links, a.max_impact)
    mmas = head_mmas(rows)
    t_mem = nbytes / HBM_BYTES_PER_S
    t_mma = mmas * 16 * 8 * 8 * 2 / MMA_SYNC_TF32_FLOPS
    bound_t = max(t_mem, t_mma)

    # ---- blocking probability per load (forward_traffic alone, first fit without QoT bounds, so that a demand is
    # blocked by the spectrum alone: --blocking-arrivals per sample)
    blocking = {}
    for load in (float(v) for v in a.blocking_loads.split(",") if v):
        db, rb = synthetic.lightpath_traffic(smp, a.blocking_arrivals, load, seed=a.seed + 1,
                                             release_existing=a.release_existing)
        db = db._replace(own_bound=torch.full_like(db.own_bound, float("-inf")))
        tb = m.forward_traffic(state, db.to(dev), rb.to(dev), ops.PLACE_FIRST_FIT, 0, True, None, 0)
        ok = (tb.status & ~(ops.CAND_IMPACT_OVERFLOW | ops.PROV_FULL)) == 0     # blocked: no slot, or the sample full
        n = max(int(ok.sum()), 1)
        blocking[str(load)] = {"blocked": float(((tb.conn_id < 0) & ok).sum()) / n,
                               "of_which_full": float(((tb.status & ops.PROV_FULL) != 0).sum()) / n, "demands": n}
    name, lim = _gpu_info()
    line = {"what": "forward_traffic vs round loop", "states": state.S, "L": state.L, "Q": state.Q,
            "load_erlang": a.load, "demands": D, "releases": R, "accepted": int((res.conn_id >= 0).sum()),
            "released": int((res.release_conn_id >= 0).sum()),
            "blocked_fraction": float((res.conn_id < 0).float().mean()), "free_placements": n_free,
            "traffic_s": t_traf, "round_loop_s": t_loop, "traffic_events_per_s": (D + R) / t_traf,
            "round_loop_events_per_s": (D + R) / t_loop, "speedup": t_loop / t_traf,
            "bit_identical": all(match.values()), "mismatched_fields": [f for f, v in match.items() if not v],
            "algorithmic_bytes": nbytes, "head_rows_est": rows, "head_mmas_est": mmas,
            "bound": "memory" if t_mem >= t_mma else "tensor pipe (mma.sync TF32)", "bound_s": bound_t,
            "fraction_of_bound": bound_t / t_traf, "blocking_by_load": blocking, "gpu": name, "power_limit": lim}
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
