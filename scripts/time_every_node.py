"""Times LightpathGNN's every-node mode (csrc/lightpath_every_node.cu) against the existing path producing the same
predictions: forward_stream over the materialised one-hot expansion (one copy of a graph per node, that node flagged).

    python scripts/time_every_node.py [--batches 64] [--batch-size 4096] [--expand 8] [--seed 1] [--out FILE]

BASELINE cfg-2 store (seed 1), batches of 4096 graphs; the every-node plan walks all --batches batches (more than
L2 holds) as ONE CUDA-graph replay after a read that evicts L2, timed with CUDA events.  The expansion path runs the
first --expand of those batches the same way.  Both outputs are compared (1e-5 relative, 2e-6 absolute floor).
Prints one JSON line: us per source batch, predictions/s of both paths, algorithmic bytes per batch, the
tensor-pipe bound of the readout head, the GPU's name and power limit.
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
    p.add_argument("--batches", type=int, default=64, help="source batches in the every-node plan (>= 64 cycles > L2)")
    p.add_argument("--batch-size", type=int, default=4096, help="graphs per source batch")
    p.add_argument("--expand", type=int, default=8, help="source batches run through the one-hot expansion path")
    p.add_argument("--seed", type=int, default=1)
    p.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = p.parse_args(argv)
    if a.batches < 1 or a.batch_size < 1 or not 1 <= a.expand <= a.batches:
        p.error("need batches >= 1, batch-size >= 1 and 1 <= expand <= batches")
    return a


def algorithmic_bytes(N: int, E: int, B: int, verified: bool) -> int:
    """Compulsory traffic of one every-node launch over a batch: x (20 B/node), the destination row (8 B/edge; the
    source row too, 8 B/edge, on an unverified layout), ptr and edge_ptr (16 B/graph + 16), out (12 B/node)."""
    return 20 * N + 8 * E + (0 if verified else 8 * E) + 16 * (B + 1) + 12 * N


def head_flops(N: int) -> float:
    """Tensor-core work of the readout head over N rows (3xTF32 split, m16n8k8 = 1024 MAC)."""
    return N / 16 * HEAD_MMAS_PER_16_ROWS * 1024 * 2


def one_hot_expansion(x, edge_index, batch, col: int):
    """One copy of every graph per node, that node's flag column 1.0 and every other 0.0 (graphs contiguous in node
    order, edges grouped by graph).  Returns x, edge_index, batch, ptr, edge_ptr of the expanded batch; copy c is
    node c's, so the expansion's readout rows come out in node order."""
    dev, N = x.device, x.shape[0]
    B = int(batch.max()) + 1
    n = torch.bincount(batch, minlength=B)
    gstart = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    gstart[1:] = torch.cumsum(n, 0)
    csize = n[batch]
    coff = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    coff[1:] = torch.cumsum(csize, 0)
    copy_row = torch.repeat_interleave(torch.arange(N, device=dev), csize)
    node = gstart[batch[copy_row]] + torch.arange(int(coff[-1]), device=dev) - coff[copy_row]
    xc = x[node].clone()
    xc[:, col] = (node == copy_row).to(x.dtype)
    eg = batch[edge_index[0]]
    ecount = torch.bincount(eg, minlength=B)
    estart = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    estart[1:] = torch.cumsum(ecount, 0)
    emult = ecount[batch]
    eoff = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    eoff[1:] = torch.cumsum(emult, 0)
    copy_e = torch.repeat_interleave(torch.arange(N, device=dev), emult)
    e = estart[batch[copy_e]] + torch.arange(int(eoff[-1]), device=dev) - eoff[copy_e]
    shift = coff[copy_e] - gstart[batch[copy_e]]
    eic = edge_index[:, e] + shift
    return xc, eic, copy_row, coff, eoff


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def _graph_time(fn, l2_flush, stream):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        fn()
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=stream):
            fn()
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l2_flush.sum()                                  # evicts what the untimed replay left in L2
        e0.record(stream)
        g.replay()
        e1.record(stream)
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3                    # us


def main(argv=None):
    a = parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("time_every_node.py measures on a CUDA device; none is available")
    from gnn_qot_estimation_b200 import Batch, LightpathGNN, ops, synthetic
    dev = torch.device("cuda:0")
    root = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
    sd = torch.load(os.path.join(root, "tests/golden/ckpt_lightpath_model_1.pt"), map_location="cpu",
                    weights_only=False)["model_state_dict"]
    m = LightpathGNN(5, 32, 3, is_lut_index=1, dropout_p=0.0)
    m.load_state_dict(sd)
    m.to(dev).eval()
    bs_ = a.batch_size
    store = synthetic.lightpath_store(a.batches * bs_, seed=a.seed, device=dev)
    verified = store.verify_layout()
    bs = [store.collate(range(i * bs_, (i + 1) * bs_)) for i in range(a.batches)]
    plan = m.stream_plan(bs, every_node=True)
    ex = []
    for b in bs[:a.expand]:
        xc, eic, bt, p, ep = one_hot_expansion(b.x, b.edge_index, b.batch, 1)
        eb = Batch(x=xc, edge_index=eic, batch=bt, ptr=p, edge_ptr=ep, num_graphs=int(p.numel() - 1), lut_col=1,
                   sym_by_src=verified)
        eb.lut_ptr = ops.lightpath_lut_ptr(eb.x, eb.ptr, 1)
        ex.append(eb)
    eplan = m.stream_plan(ex)
    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    s = torch.cuda.Stream()
    t_every = _graph_time(lambda: m.forward_stream(plan), l2_flush, s)
    t_expand = _graph_time(lambda: m.forward_stream(eplan), l2_flush, s)
    # parity on the expanded batches: row c of the expansion is node c as the LUT
    worst_rel, ok = 0.0, True
    for i in range(a.expand):
        got = plan.result(i).out
        ref = eplan.result(i).out[:got.shape[0]]
        d = (got - ref).abs()
        worst_rel = max(worst_rel, float(d.max()) / max(float(ref.abs().max()), 1e-30))
        ok &= bool((d <= 2e-6 + 1e-5 * ref.abs()).all())
    N_all = sum(b.num_nodes for b in bs)
    alg = sum(algorithmic_bytes(b.num_nodes, b.num_edges, b.num_graphs, verified) for b in bs) / a.batches
    pred_every = N_all / (t_every * 1e-6)
    pred_expand = sum(b.num_nodes for b in bs[:a.expand]) / (t_expand * 1e-6)
    bound_tc_us = head_flops(N_all) / MMA_SYNC_TF32_FLOPS * 1e6 / a.batches
    bound_hbm_us = alg / HBM_BYTES_PER_S * 1e6
    name, pl = gpu_identity()
    res = {
        "gpu": name, "power_limit": pl, "batches": a.batches, "batch_size": bs_, "verified_layout": verified,
        "every_node_us_per_batch": t_every / a.batches,
        "expansion_us_per_source_batch": t_expand / a.expand,
        "every_node_predictions_per_s": pred_every, "expansion_predictions_per_s": pred_expand,
        "speedup": pred_every / pred_expand,
        "alg_bytes_per_batch": alg, "hbm_bound_us_per_batch": bound_hbm_us,
        "tensor_pipe_bound_us_per_batch": bound_tc_us,
        "tensor_pipe_bound_fraction": bound_tc_us / (t_every / a.batches),
        "parity_ok": ok, "parity_rel_err": worst_rel,
        "status": int(plan.status.max().item()) | int(eplan.status.max().item()),
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not ok:
        raise SystemExit("every-node output disagrees with the expansion path")


if __name__ == "__main__":
    main()
