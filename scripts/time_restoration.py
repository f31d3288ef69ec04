"""Times LightpathGNN's failure restoration (qot_lightpath_restore, csrc/lightpath_candidates.cu) against the expansion
producing the same outputs (tests/restoration_ref.py:expand): every scenario's sample replicated, the cut set found in
numpy, the cut lightpaths released and their filtered options provisioned by one forward_traffic call per chunk of
scenarios, then commit_traffic, lightpath_network_state and forward_every_node for the end rows.

    python scripts/time_restoration.py [--states 64,1024] [--links 60] [--freqs 80] [--chunk 4096] [--max-cut 64]
                                       [--seed 5] [--out FILE]

States: network_status_samples (seed --seed, spacing 0.0375); failures: every single-link failure that cuts something
(to_graph.single_link_failures); options: synthetic.lightpath_restoration_options (1..4 per lightpath, option 0 the
current route).  Both paths answer PLACE_MAX_MARGIN on output column 0 (maximised) with a per-lightpath bound (each
lightpath's every-node value minus 0.01) and return the end rows.  forward_restoration runs as ONE CUDA-graph replay
after a read that evicts L2, timed with CUDA events (median of 5); expand() is timed once with CUDA events around the
whole call after a warm-up on the first chunk, its chunks summed in that one window.  Prints one JSON line per state
count: scenarios/s of both paths, whether every per-cut and count output matches bit for bit and the end rows'
largest relative difference (and how many are bit-identical), the algorithmic bytes and head MMAs of the run's counts,
the bound that applies and the fraction of it reached, the GPU's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))          # restoration_ref: the expansion

MMA_SYNC_TF32_FLOPS = 295e12    # profiles/r1_mma_sync_rate.txt: mma.sync m16n8k8 TF32, 148 SMs, B200
HEAD_MMAS_PER_16_ROWS = 240     # head_rows16_tf32x3: 4 heads x 4 (3 projection + 4 x 3 mlp.0) m16n8k8 MMAs
HBM_BYTES_PER_S = 6.5e12        # measured stream bandwidth of the B200 (DESIGN.md)
FIELDS = ("cut_node", "option", "q0", "out", "margin", "n_free", "n_feasible", "cut_status", "status", "n_cut",
          "n_restored", "end_conn")


def parse_args(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--states", default="64,1024", help="network state counts, one run each")
    p.add_argument("--links", type=int, default=60)
    p.add_argument("--freqs", type=int, default=80, help="slots of the frequency grid")
    p.add_argument("--chunk", type=int, default=4096, help="scenarios per forward_traffic call of the expansion")
    p.add_argument("--max-cut", type=int, default=64)
    p.add_argument("--seed", type=int, default=5)
    p.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = p.parse_args(argv)
    a.states = [int(v) for v in a.states.split(",") if v]
    if min(a.states + [a.links, a.freqs, a.chunk]) < 1 or a.freqs > 1024 or a.max_cut < 0:
        p.error("need states, links, chunk >= 1, 1 <= freqs <= 1024, max-cut >= 0")
    return a


def algorithmic_bytes(n_s, e_s, L, Q, cut, kept_links, failed_links):
    """Compulsory traffic of one call, from the scenarios' counts: per scenario its sample's chan_node row read and
    copied into the block's slab (12 B per channel: read, write, one read back through L2 for the end state's keys
    counted with the read), the failed links' rows (4 B per slot), the sample's x rows, conn_ids, rowptr and bound
    (48 B per node) and edges (8 B), the outputs (20 B + 20 B per end row slot, 256 slots); per cut lightpath its
    options (28 B each, counted with the route rows) and outputs (48 B); per kept option's route link its chan_work row
    (4 B per slot); messages and attention come from shared memory."""
    F = len(n_s)
    return (F * (12 * L * Q + 20 + 256 * 20) + 4 * Q * failed_links + 48 * sum(n_s) + 8 * sum(e_s) + 48 * cut +
            kept_links * (4 * Q + 28))


def head_mmas(rows: float) -> float:
    return rows / 16.0 * HEAD_MMAS_PER_16_ROWS


def _gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, lim = (v.strip() for v in q.split(","))
        return name, lim
    except Exception:
        return torch.cuda.get_device_name(), "unknown"


def run(a, S, m, dev):
    from gnn_qot_estimation_b200 import ops, synthetic
    from gnn_qot_estimation_b200.to_graph import lightpath_network_state, single_link_failures
    from restoration_ref import expand, scenarios
    smp = synthetic.network_status_samples(S, num_links=a.links, num_freqs=a.freqs, seed=a.seed, spacing=0.0375,
                                           super_channel_p=0.3)
    data0 = torch.from_numpy(smp["data"]).to(dev).contiguous()
    state = lightpath_network_state(data0, torch.from_numpy(smp["freqs"]), smp["lp_feat"])
    options = synthetic.lightpath_restoration_options(smp, state, seed=a.seed + 1).to(dev)
    fails = single_link_failures(state)
    F = int(fails.sample.shape[0])
    bound = (m.forward_every_node(state.batch)[:, 0] - 0.01).contiguous()
    evict = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # 256 MB > 126 MB of L2
    args = (state, options, fails, ops.PLACE_MAX_MARGIN, 0, True, bound, a.max_cut, True)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        m.forward_restoration(*args)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        res = m.forward_restoration(*args)
    times = []
    for _ in range(5):
        evict.add_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) / 1e3)
    t_rest = sorted(times)[len(times) // 2]

    first = fails._replace(sample=fails.sample[:a.chunk], link_ptr=fails.link_ptr[:min(a.chunk, F) + 1])
    expand(m, smp, state, options, first, ops.PLACE_MAX_MARGIN, 0, True, bound, a.max_cut, a.chunk)   # warm-up
    evict.add_(1)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ref = expand(m, smp, state, options, fails, ops.PLACE_MAX_MARGIN, 0, True, bound, a.max_cut, a.chunk)
    e1.record()
    torch.cuda.synchronize()
    t_exp = e0.elapsed_time(e1) / 1e3

    def same(x, y):
        if x.is_floating_point():
            return bool(torch.equal(x.nan_to_num(7.0), y.nan_to_num(7.0)) and torch.equal(x.isnan(), y.isnan()))
        return bool(torch.equal(x, y))
    match = {f: same(getattr(res, f), getattr(ref, f)) for f in FIELDS}
    live = res.end_conn >= 0
    x, y = res.end_out[live].double(), ref.end_out[live].double()
    end_rel = float((x - y).abs().max() / y.abs().max().clamp(min=1e-30)) if x.numel() else 0.0
    end_same = int((res.end_out[live] == ref.end_out[live]).all(1).sum())

    # counts of the run, for the bound
    plan = scenarios(smp, state, options, fails)
    ptr = state.batch.ptr.tolist()
    deg = torch.bincount(state.batch.edge_index[0], minlength=int(state.batch.x.shape[0])).tolist()
    n_s = [ptr[p["s"] + 1] - ptr[p["s"]] for p in plan]
    e_s = [sum(deg[ptr[p["s"]]:ptr[p["s"] + 1]]) for p in plan]
    cut = sum(len(p["cut"]) for p in plan)
    kept_links = sum(len(o[0]) for p in plan for c in p["per"] if c["kind"] == "d" for o in c["opts"])
    failed_links = sum(len(p["failed"]) for p in plan)
    mean_deg = float(state.batch.edge_index.shape[1]) / max(int(state.batch.x.shape[0]), 1)
    n_free = int(res.n_free.sum())
    end_rows = int(live.sum())
    rows = n_free * (1.0 + mean_deg) + end_rows            # own row + every impact row against the bound, end rows
    nbytes = algorithmic_bytes(n_s, e_s, state.L, state.Q, cut, kept_links, failed_links)
    mmas = head_mmas(rows)
    t_mem = nbytes / HBM_BYTES_PER_S
    t_mma = mmas * 16 * 8 * 8 * 2 / MMA_SYNC_TF32_FLOPS
    bound_t = max(t_mem, t_mma)
    name, lim = _gpu_info()
    return {"what": "forward_restoration vs expand (forward_traffic on replicated samples)", "states": state.S,
            "L": state.L, "Q": state.Q, "scenarios": F, "cut": int(res.n_cut.sum()),
            "restored": int(res.n_restored.sum()), "no_option": int(((res.cut_status & ops.REST_NO_OPTION) != 0).sum()),
            "below_at_end": int(res.n_below.sum()), "free_placements": n_free, "restoration_s": t_rest,
            "expand_s": t_exp, "restoration_scenarios_per_s": F / t_rest, "expand_scenarios_per_s": F / t_exp,
            "speedup": t_exp / t_rest, "bit_identical": all(match.values()),
            "mismatched_fields": [f for f, v in match.items() if not v], "end_rows": end_rows,
            "end_rows_bit_identical": end_same, "end_rows_max_rel_diff": end_rel,
            "work_bytes": int(chan_bytes(state, dev)), "expand_replica_bytes": int(smp["data"][0].nbytes) * F,
            "algorithmic_bytes": nbytes, "head_rows_est": rows, "head_mmas_est": mmas,
            "bound": "memory" if t_mem >= t_mma else "tensor pipe (mma.sync TF32)", "bound_s": bound_t,
            "fraction_of_bound": bound_t / t_rest, "gpu": name, "power_limit": lim}


def chan_bytes(state, dev):
    """The kernel's scratch: one chan_node slab and one bound slab per SM."""
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    return sms * (state.L * state.Q * 4 + 256 * 4)


def main(argv=None):
    a = parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("time_restoration.py needs a CUDA device: there is nothing to time without one")
    from gnn_qot_estimation_b200 import LightpathGNN
    from conftest import load_golden
    dev = torch.device("cuda")
    m = LightpathGNN(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    m.load_state_dict(load_golden("ckpt_lightpath_model_1.pt")["model_state_dict"], strict=True)
    m = m.to(dev).eval()
    for S in a.states:
        s = json.dumps(run(a, S, m, dev))
        print(s, flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "a") as f:
                f.write(s + "\n")


if __name__ == "__main__":
    main()
