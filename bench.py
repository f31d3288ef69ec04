#!/usr/bin/env python
"""Benchmark of the B200 message-passing hot path (contract: see DESIGN.md "Measurement").

Default workload = BASELINE.json configs[1]: LightpathGNN inference (shipped weights
lightpath_training/models/model_1.pth) over 1,000,000 synthetic lightpath graphs per GPU in
batches of 4096.  One STEP = one pass of the fused eval kernel chain over one batch.

  value   graphs/s, whole job, batches already resident in HBM (reference tensor layout:
          fp32 x, int64 edge_index), evaluated by LightpathGNN.forward_stream (one launch of the
          persistent kernel per run of batches), --steps steps replayed from one CUDA graph, timed
          with CUDA events
  e2e     graphs/s through the public host-facing API (LightpathInferencePipeline): pinned HOST
          batches (compact wire format) -> H2D -> kernels -> D2H of (out, lut_batch) every step
  secondary  time-boxed cfg 3 (DDP training step) and cfg 5 (stress graph) blocks
  roofline  algorithmic bytes of the dominant kernel / its measured duration vs MEASURED_PEAKS.json
  cpu_baseline  the CPU oracle (pure-PyTorch port of the reference's PyG path) on the host cores

`--impl reference` times that CPU oracle alone, all host threads, same config and metric.
N>1 (torchrun): every rank owns a disjoint shard of graphs (weak scaling, no collective on the
data path); time = max over ranks.
`--dump-outputs DIR` writes what the last timed step returned (rank 0) as DIR/out.npy (float32) and
DIR/lut_batch.npy (float64); the inputs are seeded, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

CKPT = ROOT / "tests" / "golden" / "ckpt_lightpath_model_1.pt"
METRIC = "lightpath_infer_graphs_per_sec"
UNIT = "graphs/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=24500)
    ap.add_argument("--warmup", type=int, default=245)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--graphs", type=int, default=1_000_000, help="graphs per GPU shard")
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--e2e-steps", type=int, default=490)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU-baseline sample budget")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-depth", type=int, default=6, help="batches in flight in the host pipeline (measured: 3 -> 6.5e7, 4 -> 7.2e7, 6 -> 7.4e7, 8 -> 7.4e7 graphs/s)")
    ap.add_argument("--no-graph", action="store_true", help="topo_train: eager step instead of the CUDA-graphed step")
    ap.add_argument("--workload", default="lightpath_infer", choices=["lightpath_infer", "topo_train", "topo_stress", "lightpath_train"],
                    help="lightpath_infer = BASELINE configs[1] (the headline line); topo_train = configs[2] "
                         "(TopologicalGNN DDP training, batch 1024/GPU); topo_stress = configs[4] (10k nodes, hidden 256)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (lightpath_infer only)")
    ap.add_argument("--secondary-box-s", type=float, default=150.0,
                    help="wall-clock box of the secondary blocks; past it the headline line is printed without them")
    ap.add_argument("--no-secondary", action="store_true",
                    help="skip the time-boxed cfg 3 (DDP training) and cfg 5 (stress graph) blocks of the default line")
    args = ap.parse_args()
    if args.dump_outputs and args.workload != "lightpath_infer":
        ap.error("--dump-outputs is implemented for --workload lightpath_infer only")
    return args


def workload_config(args, world: int) -> dict:
    """`config` of the JSON line: a function of the command line only, so both arms print the same dict."""
    nb = (args.graphs + args.batch - 1) // args.batch
    return {"workload": "BASELINE cfg2: LightpathGNN eval (GAT->BN->ReLU->LUT->MLP), "
                        f"{args.graphs} synthetic lightpath graphs per GPU, n~U{{8..56}}, batch {args.batch}",
            "batch": args.batch, "graphs_per_gpu": args.graphs, "weights": "lightpath_training/models/model_1.pth",
            "l2": f"evicted before the timed region; the timed steps walk the shard's {nb} distinct batches in order "
                  "(~1.7 KB/graph; the bytes actually cycled are reported as l2_cycled_bytes)",
            "parallelism": f"graph-sharded x{world}, no collective"}


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock + throttle reasons of one GPU through NVML while a timed region runs."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap", 0x80: "hw_power_brake", 0x2: "applications_clocks_setting"}

    def __init__(self, index: int, period: float = 0.01):
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# --------------------------------------------------------------------------- helpers
def load_state():
    return torch.load(CKPT, map_location="cpu", weights_only=False)["model_state_dict"]


def algorithmic_bytes(batch) -> int:
    """Compulsory traffic of the fused eval kernel for one batch (DESIGN.md, 'lp_infer'):
    x (20 B/node) + destination row of edge_index (8 B/edge) + gptr/eptr/lut_ptr (24 B/graph) +
    out/lut_batch/lut_node rows (24 B/LUT row, L = lut_ptr[B])."""
    N, E, B = batch.num_nodes, batch.num_edges, batch.num_graphs
    L = B if batch.lut_ptr is None else int(batch.lut_ptr[-1])
    return 20 * N + 8 * E + 24 * (B + 1) + 24 * L + 4


def dump_outputs(out_dir: str, arrays: dict, cap: int = 60 << 20) -> None:
    """Writes tensors that share their first dimension as out_dir/<name>.npy: float32 and float64 as they are,
    anything else as float64.  Past `cap` bytes in all, the same seeded sample of rows is taken from every
    tensor and the sampled row indices are written as rows.npy."""
    import numpy as np
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    arrays = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    total = sum(v.nbytes for v in arrays.values())
    if total > cap:
        rows = np.sort(np.random.default_rng(0).choice(n, int(n * cap / (total + 8 * n)), replace=False))
        arrays = {**{k: v[rows] for k, v in arrays.items()}, "rows": rows.astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def cpu_oracle_rate(host_batches, seconds: float, threads: int):
    """graphs/s of the CPU oracle (oracle.LightpathGNNOracle, fp32, eval) on a bounded sample."""
    from oracle import LightpathGNNOracle
    torch.set_num_threads(threads)
    m = LightpathGNNOracle(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    m.load_state_dict(load_state(), strict=True)
    m.eval()
    done, t_used, i = 0, 0.0, 0
    with torch.no_grad():
        m(host_batches[0])                                   # warm-up
        while t_used < seconds:
            b = host_batches[i % len(host_batches)]
            t0 = time.perf_counter()
            m(b)
            t_used += time.perf_counter() - t0
            done += b.num_graphs
            i += 1
    return done / t_used, i, done


# --------------------------------------------------------------------------- reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from gnn_qot_estimation_b200 import synthetic
    threads = os.cpu_count() or 1
    n_b = 4
    store = synthetic.lightpath_store(args.batch * n_b, seed=1, device="cpu")
    hbs = [store.host_batch(i * args.batch, (i + 1) * args.batch) for i in range(n_b)]
    from oracle import LightpathGNNOracle
    torch.set_num_threads(threads)
    m = LightpathGNNOracle(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    m.load_state_dict(load_state(), strict=True)
    m.eval()
    # bounded sample: a step (one 4096-graph batch) is ~0.1 s of CPU work; the caps only bite on the
    # long default run (24 500 steps) and are stated in `steps` / `warmup` / `cpu_baseline.sample`
    steps = max(1, min(args.steps, 200))
    warm = max(1, min(args.warmup, 50))
    with torch.no_grad():
        for i in range(warm):
            m(hbs[i % n_b])
        t0 = time.perf_counter()
        g = 0
        for i in range(steps):
            out, lut_batch = m(hbs[i % n_b])
            g += hbs[i % n_b].num_graphs
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"out": out, "lut_batch": lut_batch})
    v = g / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": dt / steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{steps} batches of {args.batch} graphs, pure-PyTorch oracle (PyG absent)"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- B200 arm
class ResidentRunner:
    """The K timed steps as one CUDA graph over batches resident in HBM.

    A step = one 4096-graph batch through the persistent eval kernel (LightpathGNN.forward_stream: ONE launch
    of lp_stream_kernel covers a whole run of consecutive batches).  Step s evaluates batch s modulo the shard:
    the W warm-up steps run eagerly, the K timed steps that follow them are captured as one graph, and that
    graph is replayed once before the timed region, so no cold replay is ever timed."""

    def __init__(self, model, plan, K: int, W: int):
        self.model, self.plan = model, plan
        self.nb, self.K, self.W = len(plan), K, W
        self.side = torch.cuda.Stream()
        self.graph = None
        self.launches = 0

    def run_steps(self, first: int, count: int) -> int:
        """Enqueues steps [first, first + count) (batch index modulo the shard); returns the launches made."""
        n = 0
        while count > 0:
            i = first % self.nb
            c = min(count, self.nb - i)
            self.model.forward_stream(self.plan, i, c)
            first, count, n = first + c, count - c, n + 1
        return n

    def capture(self):
        with torch.cuda.stream(self.side):
            self.run_steps(0, self.W)                              # eager warm-up on the stream captured below
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=self.side):
                self.launches = self.run_steps(self.W, self.K)
            self.graph.replay()                                    # upload + first replay outside the timed region
            torch.cuda.synchronize()

    def timed(self, ev0, ev1, l2_flush):
        with torch.cuda.stream(self.side):
            # reading a buffer larger than L2 evicts the batches the untimed replay left there, and keeps the GPU
            # busy while the host enqueues the replay: the region starts with the first kernel, not a launch gap
            l2_flush.sum()
            ev0.record(self.side)
            self.graph.replay()
            ev1.record(self.side)

    def batches(self) -> list:
        """Batch index of every timed step, in order."""
        return [s % self.nb for s in range(self.W, self.W + self.K)]


def run_b200(args):
    import torch.distributed as dist
    from gnn_qot_estimation_b200 import LightpathGNN, synthetic
    from gnn_qot_estimation_b200.pipeline import LightpathInferencePipeline

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    t_start = time.perf_counter()

    def mark(what):                                   # progress on stderr: where a stuck run was, per rank
        print(f"[bench rank {rank} +{time.perf_counter() - t_start:6.1f}s] {what}", file=sys.stderr, flush=True)

    wd = float(os.environ.get("QOT_BENCH_STACKS_AFTER_S", "0"))
    if wd > 0:                                        # debugging aid: dump every thread's stack and exit
        import faulthandler
        faulthandler.dump_traceback_later(wd, exit=True)
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from gnn_qot_estimation_b200.distributed import bind_to_gpu_numa_node
    all_cpus = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa = bind_to_gpu_numa_node(local)          # before any pinned allocation: host buffers land next to the GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_ranks(v: float):
        """[v of rank 0, ..., v of rank world-1] on every rank."""
        t = torch.zeros(world, dtype=torch.float64, device=dev)
        t[rank] = v
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(a) for a in t.tolist()]

    model = LightpathGNN(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    model.load_state_dict(load_state(), strict=True)
    model.to(dev).eval()

    # ---- shard of graphs owned by this rank, generated on the device (seed 1 + rank)
    G, Bsz = args.graphs, args.batch
    store = synthetic.lightpath_store(G, seed=1 + rank, device=dev)
    # one-time check of the from_networkx layout (grouped by source, symmetric, simple): batches collated from a
    # verified store carry the mark that lets the kernel derive the sources of a row from the destination row alone
    layout_ok = store.verify_layout()
    nb = (G + Bsz - 1) // Bsz
    batches = [store.collate(range(i * Bsz, min((i + 1) * Bsz, G))) for i in range(nb)]
    plan = model.stream_plan(batches)                            # pooled outputs + the device array of batch descriptors
    torch.cuda.synchronize()

    K, W = max(1, args.steps), max(args.warmup, 3)
    mark("shard resident; capturing")
    runner = ResidentRunner(model, plan, K, W)
    runner.capture()
    steps = runner.batches()
    graphs_done = sum(plan.batches[i].num_graphs for i in steps)
    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    prof = bool(os.environ.get("QOT_PROFILE_TIMED_REGION"))      # `ncu --profile-from-start off`: only the timed launches
    if prof:
        torch.cuda.profiler.start()
    with ClockSampler(local) as clk:
        runner.timed(ev0, ev1, l2_flush)
        torch.cuda.synchronize()
    if prof:
        torch.cuda.profiler.stop()
    barrier()
    mark("timed region done")
    if args.dump_outputs and rank == 0:
        last = plan.result(steps[-1])
        n = int(last.n_lut.item())
        dump_outputs(args.dump_outputs, {"out": last.out[:n], "lut_batch": last.lut_batch[:n]})
    del l2_flush
    ms = ev0.elapsed_time(ev1)
    per_rank_ms = all_ranks(ms)
    ms_max = max(per_rank_ms)
    graphs_all = sum(all_ranks(float(graphs_done)))
    value = graphs_all / (ms_max * 1e-3)
    cycled = sorted(set(steps))
    l2_cycled_bytes = sum(batches[i].nbytes(("x", "ptr", "edge_ptr", "lut_ptr")) + batches[i].num_edges * 8 for i in cycled)

    # ---- the replays against an eager run through the oracle-checked module path (one launch per batch): same rows
    # in the same order, values to the 1e-5 bar (the two kernels sum the readout head in different orders)
    n_chk = min(nb, 3)
    assert int(plan.status.max().item()) == 0, "a batch's lut_ptr does not describe its x"
    for i in range(n_chk):
        with torch.no_grad():
            ref, ref_lb = model(batches[i])
        r = plan.result(i)
        n = int(r.n_lut.item())
        assert n == ref.shape[0] and torch.equal(r.lut_batch[:n], ref_lb), "stream kernel rows differ from the module path"
        torch.testing.assert_close(r.out[:n], ref, rtol=1e-5, atol=2e-6)

    # ---- roofline of the dominant kernel: its average duration over the timed region, measured live
    # (CUDA events on the launching stream; the region is nothing but launches of that kernel)
    alg = sum(algorithmic_bytes(batches[i]) for i in cycled) / len(cycled)
    step_s = ms * 1e-3 / K
    peak, peak_kind = peaks()
    achieved = alg / step_s / 1e9
    n_launch = runner.launches
    per_launch = K / n_launch                                    # batches one launch of the persistent kernel covers
    traffic = None
    tp = ROOT / "profiles" / "lp_infer_traffic.json"             # dram__bytes_{read,write}.sum of one ncu --set full capture
    if tp.exists() and Bsz == 4096:
        tj = json.loads(tp.read_text())
        if tj.get("kernel", "").startswith("lp_stream_kernel"):
            traffic = tj["dram_bytes_read_per_batch"] + tj["dram_bytes_write_per_batch"]
    kernel_name = "lp_stream_kernel<tcgen05 head, %s>" % ("verified layout" if plan.flags & 1 else "source row read")
    if traffic is not None:
        traffic *= per_launch                                    # the capture is per batch; a launch covers per_launch batches
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": kernel_name, "alg_bytes_per_launch": alg * per_launch,
                "avg_launch_us": step_s * 1e6 * per_launch, "batches_per_launch": per_launch,
                "alg_bytes_per_batch": alg, "us_per_batch": step_s * 1e6, "verified_layout": bool(layout_ok),
                "peak_kind": f"{peak_kind} (MEASURED_PEAKS.json hbm_gbs)"}

    # ---- end to end: pinned host batches -> H2D -> kernels -> D2H, through the public pipeline API
    e2e = None
    if not args.no_e2e:
        n_host = min(nb, 64)
        cpu_store = synthetic.lightpath_store(n_host * Bsz, seed=101 + rank, device=dev)
        cpu_store = cpu_store.to("cpu")
        assert cpu_store.verify_layout()                       # the wire format carries no source row
        hbs = [cpu_store.host_wire_batch(i * Bsz, (i + 1) * Bsz, pin=True) for i in range(n_host)]
        ref0 = cpu_store.host_batch(0, Bsz)                    # reference tensors of batch 0 for the parity check below
        pipe = LightpathInferencePipeline(model, max_nodes=max(b.num_nodes for b in hbs),
                                          max_edges=max(b.num_edges for b in hbs), max_graphs=Bsz, depth=args.e2e_depth)
        # the K-step sequence repeated until the region is long enough to time (>= ~0.15 s of copies)
        Ke = max(1, min(args.e2e_steps, K))
        Ke = Ke * max(1, -(-1500 // Ke))
        seq = [hbs[i % n_host] for i in range(Ke)]
        mark("e2e warm-up")
        pipe.run(seq)                                          # warm-up: same length, so the pinned result buffer of the timed run exists
        mark("e2e timed")
        h2d0, zc0, d2h0, st0 = pipe.h2d_bytes, pipe.zero_copy_bytes, pipe.d2h_bytes, pipe.steps
        barrier()
        t0 = time.perf_counter()
        res = pipe.run(seq)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        dt_max = max(all_ranks(dt))
        ge = sum(all_ranks(float(sum(b.num_graphs for b in seq))))
        # parity of the pipeline against the module path on one batch
        with torch.no_grad():
            o_ref, l_ref = model(ref0.to(dev))
        assert torch.equal(res[0][0], o_ref.cpu()) and torch.equal(res[0][1], l_ref.cpu())
        n_st = max(pipe.steps - st0, 1)
        e2e = {"value": ge / dt_max, "unit": UNIT,
               "h2d_bytes_per_step": (pipe.h2d_bytes - h2d0 + pipe.zero_copy_bytes - zc0) / n_st,
               "h2d_bytes_per_graph": (pipe.h2d_bytes - h2d0) / max(sum(b.num_graphs for b in seq), 1),
               "d2h_bytes_per_step": (pipe.d2h_bytes - d2h0) / n_st, "steps": Ke, "ms_per_step": dt_max / Ke * 1e3,
               "h2d_note": pipe.wire_note}

    cpu_base = None
    if all_cpus is not None:
        os.sched_setaffinity(0, all_cpus)        # the CPU baseline gets every host core back
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        cs = synthetic.lightpath_store(4 * Bsz, seed=1, device="cpu")
        chb = [cs.host_batch(i * Bsz, (i + 1) * Bsz) for i in range(4)]
        v, n_it, n_g = cpu_oracle_rate(chb, args.cpu_seconds, threads)
        cpu_base = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                    "sample": f"{n_it} batches of {Bsz} graphs ({n_g} graphs), pure-PyTorch oracle of the "
                              f"PyG path (torch_geometric absent), fp32, {threads} threads"}

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args, world),
            "timed_steps": K, "timed_region_ms": ms_max,
            "per_rank_ms": per_rank_ms, "l2_cycled_bytes": l2_cycled_bytes, "host": numa,
            "roofline": roofline, "cpu_baseline": cpu_base, "e2e": e2e,
            "gpu_launches": n_launch, "clocks": clk.summary(), "secondary": None,
        }

    # ---- secondary, time-boxed: BASELINE cfg 3 (DDP training step, exercises the gradient exchange at N > 1)
    # and cfg 5 (stress graph, rank 0 only: replicas).  Not part of `value`.  The headline line is complete at this
    # point: if the secondary blocks do not finish inside their box (a rank that never reaches a collective), rank 0
    # prints the line without them and every rank leaves -- a secondary block never costs the headline.
    secondary = None
    if not args.no_secondary:
        printed = threading.Lock()

        def give_up():
            if not printed.acquire(blocking=False):
                return
            mark(f"secondary blocks exceeded {args.secondary_box_s:.0f} s: leaving without them")
            if rank == 0:
                line["secondary"] = {"error": f"not finished within {args.secondary_box_s:.0f} s"}
                print(json.dumps(line), flush=True)
            os._exit(0)

        box = threading.Timer(args.secondary_box_s, give_up)
        box.daemon = True
        box.start()
        del runner, plan, batches, store
        torch.cuda.empty_cache()
        import bench_topological
        secondary = {}
        mark("secondary: cfg3")
        try:
            secondary["cfg3_topo_train"] = bench_topological.measure_train(world, rank, dev, steps=300, warmup=20)
            mark("secondary: cfg3 dropout")
            # the reference trains with dropout 0.5 (topological_training/train.py:54-60): same step, masks drawn per step
            d5 = bench_topological.measure_train(world, rank, dev, steps=300, warmup=20, dropout_p=0.5, min_timed_ms=30.0)
            secondary["cfg3_topo_train"]["dropout_0.5"] = {k: d5[k] for k in ("value", "ms_per_step", "steps")}
        except Exception as e:                                    # noqa: BLE001 -- a secondary block never kills the headline
            secondary["cfg3_topo_train"] = {"error": f"{type(e).__name__}: {e}"[:300]}
        mark("secondary: rank-0 blocks")
        if rank == 0:
            try:
                secondary["lightpath_train_step"] = bench_topological.measure_lightpath_train(dev, 512, 200, 5)
            except Exception as e:                                # noqa: BLE001
                secondary["lightpath_train_step"] = {"error": f"{type(e).__name__}: {e}"[:300]}
            try:
                secondary["cfg5_topo_stress"] = bench_topological.measure_stress(dev, reps=10)
            except Exception as e:                                # noqa: BLE001
                secondary["cfg5_topo_stress"] = {"error": f"{type(e).__name__}: {e}"[:300]}
        barrier()
        mark("secondary done")
        if not printed.acquire(blocking=False):                   # the box fired while the last block was finishing
            time.sleep(3600)
        box.cancel()

    if rank == 0:
        line["secondary"] = secondary
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.workload != "lightpath_infer":
        import bench_topological
        bench_topological.run(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
