"""Times LightpathGNN's 1+1 protected provisioning (qot_lightpath_protect, csrc/lightpath_candidates.cu) against the
round loop producing the same outputs: per demand position of the longest sequence, forward_placements for the working
paths over their eligible options, the working paths written into a copy of the samples and the state rebuilt, the
bound carried over, forward_placements for the backups over the options disjoint from the working route, then the
accepted paths written in (tests/protection_ref.py:round_loop).  Optionally also times forward_provision on
time_provision.py's seeded inputs with a parent build of the library against this one, alternating.

    python scripts/time_protection.py [--states 1024] [--links 60] [--freqs 80] [--per-sample 16]
                                      [--shares 0.5,1.0] [--max-impact 64] [--seed 5] [--parent-lib FILE]
                                      [--runs 3] [--out FILE]

States: network_status_samples (seed --seed, spacing 0.0375).  Demands: synthetic.lightpath_demands with 2..4
options, --per-sample per sample on average, interleaved; each protected with probability --shares (a seeded torch
generator).  Both paths answer PLACE_MAX_MARGIN on output column 0 (maximised) with a per-lightpath bound (each
lightpath's every-node value minus 0.01).  forward_protection runs as ONE CUDA-graph replay after a read that evicts
L2, timed with CUDA events (median of 5); the round loop synchronises with the host every round, so it is timed
eagerly after a warm-up run.  Prints one JSON line per share: demands/s of both paths, whether every output matches
bit for bit, accepted / NO_PARTNER / NO_BACKUP counts, algorithmic bytes and head MMAs, the bound that applies and the
fraction reached, the GPU's name and power limit.  With --parent-lib, one more line: forward_provision with each
library (subprocesses, alternating, --runs each, seven CUDA-graph replays after an L2-evicting read per run) and
whether their outputs are equal bit for bit.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))          # protection_ref: the round loop
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from time_provision import (FIELDS, HBM_BYTES_PER_S, MMA_SYNC_TF32_FLOPS, _gpu_info, algorithmic_bytes,  # noqa: E402
                            head_mmas)

BFIELDS = FIELDS + tuple("backup_" + f for f in FIELDS)


def parse_args(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--states", type=int, default=1024, help="network states (samples)")
    p.add_argument("--links", type=int, default=60)
    p.add_argument("--freqs", type=int, default=80, help="slots of the frequency grid")
    p.add_argument("--per-sample", type=int, default=16, help="demands per sample (on average)")
    p.add_argument("--shares", default="0.5,1.0", help="protected shares of the demands, comma-separated")
    p.add_argument("--max-impact", type=int, default=64)
    p.add_argument("--seed", type=int, default=5)
    p.add_argument("--parent-lib", default=None, help="a parent build of libqot_b200.so: forward_provision against it")
    p.add_argument("--runs", type=int, default=3, help="alternating runs per library with --parent-lib")
    p.add_argument("--provision-only", default=None, help=argparse.SUPPRESS)   # subprocess: time, dump outputs here
    p.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = p.parse_args(argv)
    a.shares = [float(v) for v in a.shares.split(",") if v]
    if min(a.states, a.links, a.freqs, a.per_sample, a.runs) < 1 or a.freqs > 1024 or a.max_impact < 0 or \
            not all(0.0 <= v <= 1.0 for v in a.shares):
        p.error("need states, links, per-sample, runs >= 1, 1 <= freqs <= 1024, max-impact >= 0, shares in [0, 1]")
    return a


def _setup(a, options):
    from conftest import load_golden
    from gnn_qot_estimation_b200 import LightpathGNN, synthetic
    from gnn_qot_estimation_b200.to_graph import lightpath_network_state
    dev = torch.device("cuda")
    m = LightpathGNN(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    m.load_state_dict(load_golden("ckpt_lightpath_model_1.pt")["model_state_dict"], strict=True)
    m = m.to(dev).eval()
    smp = synthetic.network_status_samples(a.states, num_links=a.links, num_freqs=a.freqs, seed=a.seed,
                                           spacing=0.0375, super_channel_p=0.3)
    data0 = torch.from_numpy(smp["data"]).to(dev).contiguous()
    freqs = torch.from_numpy(smp["freqs"]).to(dev)
    state = lightpath_network_state(data0, freqs, smp["lp_feat"])
    kw = {} if options is None else {"options": options}
    d = synthetic.lightpath_demands(smp, a.per_sample, seed=a.seed + 1, **kw).to(dev)
    bound = (m.forward_every_node(state.batch)[:, 0] - 0.01).contiguous()
    return m, smp, data0, freqs, state, d, bound


def _replays(fn, n):
    """(median seconds of n CUDA-graph replays of fn, each after an L2-evicting read, the captured result)."""
    dev = torch.device("cuda")
    evict = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # 256 MB > 126 MB of L2
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        res = fn()
    times = []
    for _ in range(n):
        evict.add_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) / 1e3)
    return sorted(times)[len(times) // 2], times, res


def _same(x, y):
    if x.is_floating_point():
        return bool(torch.equal(x.nan_to_num(7.0), y.nan_to_num(7.0)) and torch.equal(x.isnan(), y.isnan()))
    return bool(torch.equal(x, y))


def provision_only(a):
    """The subprocess of --parent-lib: forward_provision on time_provision.py's inputs with the library QOT_B200_LIB
    names; its times on stdout, its outputs into the file a.provision_only."""
    from gnn_qot_estimation_b200 import _lib, ops
    _lib.SIGNATURES.pop("qot_lightpath_protect")         # a parent build predates it; both builds bind the same set
    m, _, _, _, state, d, bound = _setup(a, None)
    t, times, res = _replays(lambda: m.forward_provision(state, d, ops.PLACE_MAX_MARGIN, 0, True, bound,
                                                         a.max_impact), 7)
    torch.save({f: getattr(res, f).cpu() for f in FIELDS}, a.provision_only)
    print(json.dumps({"median_s": t, "times_s": times}))


def provision_vs_parent(a):
    libs = [("parent", os.path.abspath(a.parent_lib)),
            ("this", os.path.abspath(os.path.join(ROOT, "gnn_qot_estimation_b200", "libqot_b200.so")))]
    out = {name: [] for name, _ in libs}
    dumps = {}
    with tempfile.TemporaryDirectory() as tmp:
        for run in range(a.runs):
            for name, lib in libs:
                dump = os.path.join(tmp, f"{name}.pt")
                cmd = [sys.executable, os.path.abspath(__file__), "--states", str(a.states), "--links", str(a.links),
                       "--freqs", str(a.freqs), "--per-sample", str(a.per_sample), "--max-impact",
                       str(a.max_impact), "--seed", str(a.seed), "--provision-only", dump]
                p = subprocess.run(cmd, env=dict(os.environ, QOT_B200_LIB=lib), capture_output=True, text=True)
                if p.returncode:
                    raise SystemExit(f"forward_provision with {lib} failed:\n{p.stderr}")
                out[name].append(json.loads(p.stdout.strip().splitlines()[-1]))
                dumps[name] = torch.load(dump)
        same = all(_same(dumps["parent"][f], dumps["this"][f]) for f in FIELDS)
    name, lim = _gpu_info()
    return {"what": "forward_provision, parent library vs this one (alternating)", "states": a.states,
            "per_sample": a.per_sample, "bit_identical": same,
            "parent_median_ms": [round(r["median_s"] * 1e3, 3) for r in out["parent"]],
            "this_median_ms": [round(r["median_s"] * 1e3, 3) for r in out["this"]],
            "parent_times_ms": [[round(t * 1e3, 3) for t in r["times_s"]] for r in out["parent"]],
            "this_times_ms": [[round(t * 1e3, 3) for t in r["times_s"]] for r in out["this"]],
            "gpu": name, "power_limit": lim}


def main(argv=None):
    a = parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("time_protection.py needs a CUDA device: there is nothing to time without one")
    if a.provision_only:
        provision_only(a)
        return
    from gnn_qot_estimation_b200 import ops
    from protection_ref import round_loop
    from provision_ref import rounds
    m, smp, data0, freqs, state, d, bound = _setup(a, (2, 4))
    D = int(d.sample.shape[0])
    lines = []
    for share in a.shares:
        g = torch.Generator(device="cpu").manual_seed(a.seed + 2)
        prot = (torch.rand(D, generator=g) < share).to(d.sample.device)
        t_prot, _, res = _replays(lambda: m.forward_protection(state, d, prot, ops.PLACE_MAX_MARGIN, 0, True, bound,
                                                               a.max_impact), 5)
        plan = rounds(d, state.S)
        round_loop(m, data0.clone(), freqs, smp["lp_feat"], d, prot, ops.PLACE_MAX_MARGIN, 0, True, bound,
                   a.max_impact, plan=plan)
        data = data0.clone()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        ref, _ = round_loop(m, data, freqs, smp["lp_feat"], d, prot, ops.PLACE_MAX_MARGIN, 0, True, bound,
                            a.max_impact, plan=plan)
        e1.record()
        torch.cuda.synchronize()
        t_loop = e0.elapsed_time(e1) / 1e3
        match = {f: _same(getattr(res, f), getattr(ref, f)) for f in BFIELDS}
        # ---- counts of the run: bytes and head rows (both searches' own rows, impact rows with the bound)
        P = int(d.width.shape[0])
        route_links = int(d.links.shape[0])
        n_free = int(res.n_free.sum() + res.backup_n_free.sum())
        n_imp = int(res.n_impact.clamp(max=a.max_impact).sum() + res.backup_n_impact.clamp(max=a.max_impact).sum())
        chosen = torch.cat([res.n_impact[res.option >= 0], res.backup_n_impact[res.backup_option >= 0]]).float()
        deg = float(chosen.mean()) if chosen.numel() else 0.0
        rows = n_free * (1.0 + deg) + n_imp
        # the backup search reads its option routes a second time and writes a second set of outputs
        nbytes = algorithmic_bytes(D, state.S, state.L, state.Q, int(state.batch.x.shape[0]),
                                   int(state.batch.edge_index.shape[1]), P, route_links, a.max_impact) + \
            D * (48 + 20 * a.max_impact) + route_links * (4 + 4 * state.Q)
        mmas = head_mmas(rows)
        t_mem = nbytes / HBM_BYTES_PER_S
        t_mma = mmas * 16 * 8 * 8 * 2 / MMA_SYNC_TF32_FLOPS
        bound_t = max(t_mem, t_mma)
        name, lim = _gpu_info()
        st = res.status
        line = {"what": "forward_protection vs round loop", "states": state.S, "L": state.L, "Q": state.Q,
                "demands": D, "protected_share": share, "protected": int(prot.sum()),
                "accepted": int((res.conn_id >= 0).sum()),
                "accepted_protected": int((res.backup_conn_id >= 0).sum()),
                "no_partner": int(((st & ops.PROT_NO_PARTNER) != 0).sum()),
                "no_backup": int(((st & ops.PROT_NO_BACKUP) != 0).sum()), "rounds": 2 * len(plan),
                "free_placements": n_free, "protection_s": t_prot, "round_loop_s": t_loop,
                "protection_demands_per_s": D / t_prot, "round_loop_demands_per_s": D / t_loop,
                "speedup": t_loop / t_prot, "bit_identical": all(match.values()),
                "mismatched_fields": [f for f, v in match.items() if not v],
                "algorithmic_bytes": nbytes, "head_rows_est": rows, "head_mmas_est": mmas,
                "bound": "memory" if t_mem >= t_mma else "tensor pipe (mma.sync TF32)", "bound_s": bound_t,
                "fraction_of_bound": bound_t / t_prot, "gpu": name, "power_limit": lim}
        lines.append(line)
        print(json.dumps(line), flush=True)
    if a.parent_lib:
        line = provision_vs_parent(a)
        lines.append(line)
        print(json.dumps(line), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
