"""Device-side graph construction: the B200 counterpart of the reference's ``to_graph.py``.

``create_lightpath_graphs`` turns a batch of raw network-status samples ``[S, lp_feat, link, freq]``
(what ``xr.open_dataset(...)["data"]`` holds, to_graph.py:216-223) straight into the
:class:`PackedGraphStore` the collate kernel consumes -- i.e. it replaces, for all samples at once,
``to_graph.create_lightpath_graph`` (to_graph.py:187-312) -> pickle (store_graphs.py:73-76) ->
``LightpathDataset.__getitem__`` (lightpath_training/dataset.py:53-123).  The arithmetic runs in
``csrc/to_graph.cu`` (qot_lightpath_graph_count / _fill); there is no CPU path.

Node order, node features, labels and the edge SET equal the reference's (tests/test_to_graph_gpu.py
against golden vectors made by the reference's own code); edges are emitted sorted by (source, target)
-- the reference's edge order follows CPython set iteration (to_graph.py:278) and carries no meaning.
"""
from __future__ import annotations

import ctypes as C
from typing import NamedTuple, Optional, Sequence

import torch

from . import _lib
from .batch import PackedGraphStore
from .ops import _track_status, check, ptr, stream

# constants.py:1-12 of the reference
FEATURE_RANGES = {"mod_order": (0.0, 64.0), "path_len": (24214.0, 7834746.0), "num_spans": (1.0, 106.0),
                  "freq": (192.2, 195.8)}
TARGET_RANGES = {"osnr": (12.47, 33.49), "snr": (8.96, 29.98), "ber": (1.70e-12, 1.98e-2)}
NODE_FEATURES = ["freq", "is_lut", "mod_order", "num_spans", "path_len"]     # sorted names, dataset.py:45-48


def _cfg(lp_feat: Sequence[str], metric: Sequence[str], F: int, L: int, Q: int, T: int, freq_threshold: float):
    fi = {k: i for i, k in enumerate(lp_feat)}
    mi = {k: i for i, k in enumerate(metric)}
    for k in ("conn_id", "osnr", "snr", "ber", "freq", "mod_order", "num_spans", "path_len"):
        if k not in fi:
            raise KeyError(f"lp_feat has no '{k}' entry (to_graph.py:27-33 needs it)")
    cfg = _lib.QotLpGraphCfg()
    cfg.F, cfg.L, cfg.Q, cfg.T = F, L, Q, T
    cfg.i_conn, cfg.i_osnr, cfg.i_snr, cfg.i_ber = fi["conn_id"], fi["osnr"], fi["snr"], fi["ber"]
    for q, name in enumerate(("freq", "mod_order", "num_spans", "path_len")):
        cfg.i_feat[q] = fi[name]
        cfg.feat_lo[q], cfg.feat_hi[q] = FEATURE_RANGES[name]
    for q, name in enumerate(("osnr", "snr", "ber")):
        cfg.i_tgt[q] = mi[name]
        cfg.tgt_lo[q], cfg.tgt_hi[q] = TARGET_RANGES[name]
    cfg.freq_threshold = float(freq_threshold)
    return cfg


@_lib.on_tensor_device
def create_lightpath_graphs(data: torch.Tensor, target: torch.Tensor, freqs: torch.Tensor, lp_feat: Sequence[str],
                            metric: Sequence[str], freq_threshold: float = 0.05,
                            return_conn_ids: bool = False):
    """data [S, F, L, Q] float32 (CUDA), target [S, T] float64, freqs [Q] float64 -> PackedGraphStore with
    node_feat [N,5] (``NODE_FEATURES`` order, min-max scaled), y [S,3], lut_col = 1.  The sample tensor is read
    once (scan launch -> per-sample records), then packed; one host sync (the per-sample counts are scanned on
    the device, their totals size the output)."""
    if not data.is_cuda:
        raise RuntimeError("create_lightpath_graphs needs CUDA tensors (gnn_qot_estimation_b200 has no CPU path)")
    dev = data.device
    data = data.to(torch.float32).contiguous()
    target = target.to(dev, torch.float64).contiguous()
    freqs = freqs.to(dev, torch.float64).contiguous()
    S, F, L, Q = (int(v) for v in data.shape)
    if freqs.numel() != Q or target.shape[0] != S:
        raise ValueError("freqs must have data.shape[3] entries and target data.shape[0] rows")
    cfg = _cfg(lp_feat, metric, F, L, Q, int(target.shape[1]), freq_threshold)
    lib = _lib.lib()
    counts = torch.zeros(S, 2, dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    y = torch.empty(S, 3, dtype=torch.float32, device=dev)
    scratch = torch.empty(lib.qot_lightpath_graph_scratch_bytes(S), dtype=torch.uint8, device=dev)
    check(lib.qot_lightpath_graph_count(ptr(data), ptr(freqs), ptr(target), S, C.byref(cfg), ptr(counts), ptr(y),
                                        ptr(scratch), scratch.numel(), ptr(status), stream()),
          "qot_lightpath_graph_count")
    ptrs = torch.zeros(2, S + 1, dtype=torch.int64, device=dev)
    ptrs[:, 1:] = torch.cumsum(counts.to(torch.int64).t(), dim=1)
    n_tot, e_tot, st = (int(v) for v in torch.stack([ptrs[0, -1], ptrs[1, -1], status[0].to(torch.int64)]).tolist())
    if st & 1:
        raise RuntimeError("create_lightpath_graphs: a sample exceeds the per-block capacity "
                           "(QOT_TG_MAX_CHANNELS occupied channels / QOT_TG_MAX_NODES lightpaths / QOT_TG_MAX_LINKS links)")
    node_feat = torch.empty(max(n_tot, 1), 5, dtype=torch.float32, device=dev)[:n_tot]
    conn_ids = torch.empty(max(n_tot, 1), dtype=torch.int64, device=dev)[:n_tot]
    edge_src = torch.empty(max(e_tot, 1), dtype=torch.int32, device=dev)[:e_tot]
    edge_dst = torch.empty(max(e_tot, 1), dtype=torch.int32, device=dev)[:e_tot]
    node_ptr, edge_ptr = ptrs[0].contiguous(), ptrs[1].contiguous()
    check(lib.qot_lightpath_graph_fill(ptr(scratch), S, ptr(node_ptr), ptr(edge_ptr), ptr(node_feat), ptr(conn_ids),
                                       ptr(edge_src), ptr(edge_dst), ptr(status), stream()), "qot_lightpath_graph_fill")
    store = PackedGraphStore(node_ptr, edge_ptr, edge_src, edge_dst, node_feat, None, y, lut_col=1)
    return (store, conn_ids) if return_conn_ids else store


@_lib.on_tensor_device
def create_topological_graphs(data: torch.Tensor, target: torch.Tensor, lp_feat: Sequence[str], metric: Sequence[str],
                              num_nodes: int = 75) -> PackedGraphStore:
    """The topological representation for all samples at once: ``to_graph.create_topological_graph``
    (to_graph.py:62-184) -> pickle -> ``TopologicalDataset.__getitem__`` (topological_training/dataset.py:46-123).
    data [S, F, L, Q] float32 (CUDA), target [S, T] float64 -> PackedGraphStore with ``num_nodes`` nodes per
    graph (no node features: the model embeds ``node_ids``), edges in the reference's order, edge_feat [E,4] in
    sorted-name order [freq, mod_order, num_spans, path_len] (min-max scaled), y [S,3]."""
    if not data.is_cuda:
        raise RuntimeError("create_topological_graphs needs CUDA tensors (gnn_qot_estimation_b200 has no CPU path)")
    dev = data.device
    data = data.to(torch.float32).contiguous()
    target = target.to(dev, torch.float64).contiguous()
    S, F, L, Q = (int(v) for v in data.shape)
    if target.shape[0] != S:
        raise ValueError("target must have data.shape[0] rows")
    fi = {k: i for i, k in enumerate(lp_feat)}
    for k in ("src_id", "dst_id"):
        if k not in fi:
            raise KeyError(f"lp_feat has no '{k}' entry (to_graph.py:152-153 needs it)")
    cfg = _cfg(lp_feat, metric, F, L, Q, int(target.shape[1]), 0.05)
    lib = _lib.lib()
    counts = torch.zeros(S, dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    y = torch.empty(S, 3, dtype=torch.float32, device=dev)
    scratch = torch.empty(lib.qot_topological_graph_scratch_bytes(S), dtype=torch.uint8, device=dev)
    check(lib.qot_topological_graph_count(ptr(data), ptr(target), S, C.byref(cfg), int(num_nodes), fi["src_id"],
                                          fi["dst_id"], ptr(counts), ptr(y), ptr(scratch), scratch.numel(),
                                          ptr(status), stream()), "qot_topological_graph_count")
    edge_ptr = torch.zeros(S + 1, dtype=torch.int64, device=dev)
    edge_ptr[1:] = torch.cumsum(counts.to(torch.int64), dim=0)
    e_tot, st = (int(v) for v in torch.stack([edge_ptr[-1], status[0].to(torch.int64)]).tolist())
    if st & 1:
        raise RuntimeError("create_topological_graphs: a sample exceeds the per-block capacity or names a network "
                           f"node outside 1..{num_nodes}")
    edge_src = torch.empty(max(e_tot, 1), dtype=torch.int32, device=dev)[:e_tot]
    edge_dst = torch.empty(max(e_tot, 1), dtype=torch.int32, device=dev)[:e_tot]
    edge_feat = torch.empty(max(e_tot, 1), 4, dtype=torch.float32, device=dev)[:e_tot]
    check(lib.qot_topological_graph_fill(ptr(scratch), S, ptr(edge_ptr), ptr(edge_src), ptr(edge_dst), ptr(edge_feat),
                                         ptr(status), stream()), "qot_topological_graph_fill")
    node_ptr = torch.arange(S + 1, dtype=torch.int64, device=dev) * int(num_nodes)
    return PackedGraphStore(node_ptr, edge_ptr, edge_src, edge_dst, None, edge_feat, y)


class LightpathNetworkState(NamedTuple):
    """A resident network state: raw samples turned into graphs once, plus the index structures candidate QoT needs
    (``lightpath_network_state``; ``LightpathGNN.forward_candidates``)."""
    batch: "object"               # Batch of all S graphs in sample order (works with forward_every_node)
    conn_ids: torch.Tensor        # [N] int64: lightpath of each node of ``batch``
    chan_node: torch.Tensor       # [S, L, Q] int32: node of ``batch`` on each channel, -1 = free
    rowptr: torch.Tensor          # [N+1] int64: node v's out-edges are [rowptr[v], rowptr[v+1]) of batch.edge_index
    freqs: torch.Tensor           # [Q] float64
    cfg: "object"                 # the QotLpGraphCfg the graphs were built with (scaling ranges, threshold)
    S: int
    L: int
    Q: int


class LightpathCandidates(NamedTuple):
    """Candidate lightpaths (device tensors).  Candidate k: sample ``sample[k]`` of the state, the path
    ``links[link_ptr[k]:link_ptr[k+1]]``, slots ``[q0[k], q0[k] + width[k])`` on every link of the path, raw channel
    vector ``feat[k] = (freq, mod_order, num_spans, path_len)``."""
    sample: torch.Tensor          # [K] int64
    link_ptr: torch.Tensor        # [K+1] int64
    links: torch.Tensor           # [sum of path lengths] int32
    q0: torch.Tensor              # [K] int32
    width: torch.Tensor           # [K] int32
    feat: torch.Tensor            # [K, 4] float32

    def to(self, device) -> "LightpathCandidates":
        return LightpathCandidates(*(t.to(device) for t in self))


class LightpathChanges(NamedTuple):
    """Changes to a network state (device tensors): change k moves lightpath ``node[k]`` (a node of ``state.batch`` in
    sample ``sample[k]``, see ``lightpath_nodes``; -1 = a new lightpath, as a candidate) onto the path
    ``links[link_ptr[k]:link_ptr[k+1]]`` and slots ``[q0[k], q0[k] + width[k])`` with raw channel vector ``feat[k] =
    (freq, mod_order, num_spans, path_len)``.  An empty path with ``node[k] >= 0`` tears the lightpath down."""
    node: torch.Tensor            # [K] int64
    sample: torch.Tensor          # [K] int64
    link_ptr: torch.Tensor        # [K+1] int64
    links: torch.Tensor           # [sum of path lengths] int32
    q0: torch.Tensor              # [K] int32
    width: torch.Tensor           # [K] int32
    feat: torch.Tensor            # [K, 4] float32

    def to(self, device) -> "LightpathChanges":
        return LightpathChanges(*(t.to(device) for t in self))


class LightpathDemands(NamedTuple):
    """Lightpath demands to place (device tensors; ``LightpathGNN.forward_placements``).  Demand d goes into sample
    ``sample[d]`` of the state and offers options ``[opt_ptr[d], opt_ptr[d+1])`` (1..32).  Option p is the route
    ``links[link_ptr[p]:link_ptr[p+1]]`` with slot width ``width[p]``, channel features ``feat[p] = (mod_order,
    num_spans, path_len)`` and a bound ``own_bound[p]`` on its own predicted metric.  The same route with another
    modulation format is another option."""
    sample: torch.Tensor          # [D] int64
    opt_ptr: torch.Tensor         # [D+1] int64
    link_ptr: torch.Tensor        # [P+1] int64
    links: torch.Tensor           # [sum of route lengths] int32
    width: torch.Tensor           # [P] int32
    feat: torch.Tensor            # [P, 3] float32
    own_bound: torch.Tensor       # [P] float32

    def to(self, device) -> "LightpathDemands":
        return LightpathDemands(*(t.to(device) for t in self))


def lightpath_nodes(state: LightpathNetworkState, sample: torch.Tensor, conn_id: torch.Tensor) -> torch.Tensor:
    """[K] int64: the node of ``state.batch`` that holds lightpath ``conn_id[k]`` in sample ``sample[k]``, -1 where the
    sample has no such lightpath (or ``sample[k]`` is outside the state).  Device tensor ops, no host synchronisation:
    one sort of the state's (sample, conn_id) keys and a binary search per query."""
    b = state.batch
    dev = b.x.device
    sample = sample.to(dev, torch.int64)
    conn_id = conn_id.to(dev, torch.int64)
    lo, span = -(1 << 31), 1 << 32                           # conn_ids are int32 values (a float32 row truncated)
    key = b.batch.to(torch.int64) * span + (state.conn_ids - lo)
    skey, order = torch.sort(key)
    ok = (sample >= 0) & (sample < state.S) & (conn_id >= lo) & (conn_id < lo + span)
    q = torch.where(ok, sample * span + (conn_id - lo), torch.full_like(sample, -1))
    if skey.numel() == 0:
        return torch.full_like(sample, -1)
    i = torch.searchsorted(skey, q).clamp(max=skey.numel() - 1)
    return torch.where(ok & (skey[i] == q), order[i], torch.full_like(sample, -1))


@_lib.on_tensor_device
def lightpath_network_state(data: torch.Tensor, freqs: torch.Tensor, lp_feat: Sequence[str],
                            freq_threshold: float = 0.05) -> LightpathNetworkState:
    """data [S, F, L, Q] float32 (CUDA, 0 = free channel), freqs [Q] float64 -> the network state candidate lightpaths
    are evaluated against.  Builds the S graphs with ``create_lightpath_graphs`` (its one host synchronisation; no
    targets needed), collates them in sample order, and maps every channel to its node (qot_lightpath_channel_map).
    ``state.batch`` goes straight into ``LightpathGNN.forward_every_node`` (the QoT of the lightpaths already set up)."""
    if not data.is_cuda:
        raise RuntimeError("lightpath_network_state needs CUDA tensors (gnn_qot_estimation_b200 has no CPU path)")
    dev = data.device
    data = data.to(torch.float32).contiguous()
    freqs = freqs.to(dev, torch.float64).contiguous()
    S, F, L, Q = (int(v) for v in data.shape)
    metric = ["osnr", "snr", "ber"]
    store, conn_ids = create_lightpath_graphs(data, torch.zeros(S, 3, dtype=torch.float64, device=dev), freqs, lp_feat,
                                              metric, freq_threshold, return_conn_ids=True)
    # edges come out sorted by (source, target), both directions of every interaction, no repeated pair: the layout
    # verify_layout() checks, by construction
    store.sym_by_src = True
    batch = store.collate(range(S))
    N = int(batch.x.shape[0])
    rowptr = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    rowptr[1:] = torch.cumsum(torch.bincount(batch.edge_index[0], minlength=N), 0)
    cfg = _cfg(lp_feat, metric, F, L, Q, 3, freq_threshold)
    chan_node = torch.empty(S, L, Q, dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    check(_lib.lib().qot_lightpath_channel_map(ptr(data), S, C.byref(cfg), ptr(batch.ptr), ptr(conn_ids), N,
                                               ptr(chan_node), ptr(status), stream()), "qot_lightpath_channel_map")
    _track_status("qot_lightpath_channel_map (an occupied channel's conn_id is not among its sample's lightpaths)",
                  status)
    return LightpathNetworkState(batch, conn_ids, chan_node, rowptr, freqs, cfg, S, L, Q)


def commit_provision(data: torch.Tensor, state: LightpathNetworkState, demands: LightpathDemands,
                     res) -> LightpathNetworkState:
    """Writes the demands ``LightpathGNN.forward_provision`` accepted (``res.conn_id >= 0``) into ``data`` [S, F, L, Q]
    (float32, CUDA, the samples ``state`` was built from) in place, on the device, and returns
    ``lightpath_network_state`` of the written samples: the state the next demand of each sample would be placed
    against.  Each accepted demand goes onto its chosen route x ``[q0, q0 + width)`` with conn_id ``res.conn_id[d]``,
    freq ``float32(state.freqs[q0])``, the option's (mod_order, num_spans, path_len), osnr = snr = ber = -1 and every
    other row 0.  The new state is the builder's by construction (node order by first channel, so a new lightpath
    lands among the existing nodes).  Not capturable: one host synchronisation gathers the written channels, and the
    rebuild keeps the builder's own."""
    if not (data.is_cuda and data.dtype == torch.float32 and data.is_contiguous()):
        raise TypeError("commit_provision: data must be a contiguous float32 CUDA tensor (it is written in place)")
    S, F, L, Q = (int(v) for v in data.shape)
    if (S, L, Q) != (state.S, state.L, state.Q):
        raise ValueError("commit_provision: data must be the [S, F, L, Q] samples the state was built from")
    cfg, d, dev = state.cfg, demands, data.device
    # chosen[p] = the accepted demand whose chosen option is p (an option belongs to one demand), else -1
    P = int(d.width.shape[0])
    acc = res.conn_id >= 0
    po = d.opt_ptr[:-1] + res.option.to(torch.int64)
    chosen = torch.full((P + 1,), -1, dtype=torch.int64, device=dev)
    chosen.scatter_(0, torch.where(acc, po, torch.full_like(po, P)), torch.arange(po.shape[0], device=dev))
    chosen[P] = -1
    # every (route entry, slot) an accepted demand occupies; accepted placements of a sample are disjoint
    opt = torch.searchsorted(d.link_ptr, torch.arange(d.links.shape[0], device=dev), right=True) - 1
    dm = chosen[opt]
    q0 = res.q0[dm.clamp(min=0)].to(torch.int64)
    q = torch.arange(Q, device=dev)
    on = (dm >= 0)[:, None] & (q[None, :] >= q0[:, None]) & (q[None, :] < (q0 + d.width[opt])[:, None])
    e, c = on.nonzero(as_tuple=True)                            # the host synchronisation
    dm, p = dm[e], opt[e]
    vec = torch.zeros(int(e.shape[0]), F, dtype=torch.float32, device=dev)
    vec[:, cfg.i_conn] = res.conn_id[dm].to(torch.float32)
    vec[:, cfg.i_feat[0]] = state.freqs[q0[e]].to(torch.float32)
    for k in range(3):
        vec[:, cfg.i_feat[k + 1]] = d.feat[p, k]
    vec[:, cfg.i_osnr] = vec[:, cfg.i_snr] = vec[:, cfg.i_ber] = -1.0
    data[d.sample[dm], :, d.links[e].to(torch.int64), c] = vec
    names = [f"row{f}" for f in range(F)]                       # the builder reads only the rows cfg names
    names[cfg.i_conn], names[cfg.i_osnr], names[cfg.i_snr], names[cfg.i_ber] = "conn_id", "osnr", "snr", "ber"
    for k, name in enumerate(("freq", "mod_order", "num_spans", "path_len")):
        names[cfg.i_feat[k]] = name
    return lightpath_network_state(data, state.freqs, names, float(cfg.freq_threshold))
