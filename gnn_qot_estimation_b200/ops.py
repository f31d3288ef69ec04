"""Thin Python layer over the C ABI: tensor-in/tensor-out wrappers and the
``torch.autograd.Function``s the two modules are assembled from.

Every function here launches hand-written sm_100a kernels from libqot_b200.so on
torch's current stream.  Nothing falls back to PyTorch ops for the arithmetic;
torch only allocates the tensors.
"""
from __future__ import annotations

import ctypes as C
import weakref
from typing import Sequence, NamedTuple, Optional

import torch

from . import _lib
from ._lib import check, ptr, stream

EDGE_HID = 8          # QOT_EDGE_HID
CSR_DROP_SELF = 1
CSR_ADD_SELF = 2


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("gnn_qot_estimation_b200 runs on CUDA tensors only (no CPU fallback): "
                               "move the batch and the model to a B200 with .to('cuda')")


def _f32(t):
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.to(torch.float32).contiguous()


def _edge_attr(t):
    """fp32 contiguous edge_attr; a zero-edge batch gets one dummy row so the pointer is not NULL."""
    t = _f32(t)
    return t if t.shape[0] else t.new_zeros(1, t.shape[1])


def _i64(t):
    return t if (t.dtype == torch.int64 and t.is_contiguous()) else t.to(torch.int64).contiguous()


# --------------------------------------------------------------------------- #
# device status words
# --------------------------------------------------------------------------- #
# Kernels never synchronise; when an input violates a contract the reference would raise on (an edge
# endpoint or node id out of range, edges not grouped by graph, a graph larger than the sizes a fused
# launch was made for, a tensor-core barrier timeout) they set a bit in a one-word device buffer, write
# NaN (never stale memory) where a result is missing, and carry on.  check_status() is the explicit sync
# point: ONE device->host read of every word produced since the last call; raises naming the ops.
_status_words = {}          # data_ptr -> (what, tensor): a long-lived word (e.g. one per device) is tracked once
_STATUS_CAP = 4096


def _track_status(what: str, t: torch.Tensor) -> torch.Tensor:
    if len(_status_words) >= _STATUS_CAP:
        for k in list(_status_words)[:_STATUS_CAP // 2]:
            del _status_words[k]
    _status_words[t.data_ptr()] = (what, t)
    return t


def check_status(clear: bool = True) -> None:
    """Raises RuntimeError if any kernel launched through this module since the last call flagged its
    input (see above).  Costs one small device->host copy (a synchronisation): call it where the loop
    already reads the loss, or once per epoch."""
    if not _status_words:
        return
    words = list(_status_words.values())
    if clear:
        _status_words.clear()
    by_dev = {}
    for what, t in words:
        by_dev.setdefault(t.device, []).append((what, t))
    bad = []
    for dev, items in by_dev.items():
        vals = iter(torch.cat([t.reshape(-1) for _, t in items]).tolist())
        for what, t in items:                     # a tracked tensor may hold several words (one per batch): OR them
            v = 0
            for _ in range(t.numel()):
                v |= next(vals)
            if v:
                bad.append(f"{what} (status {v})")
    if bad:
        raise RuntimeError("libqot_b200: input contract violated in: " + "; ".join(sorted(set(bad))[:8]) +
                           " -- out-of-range node ids / edge endpoints, edges not grouped by graph, or a graph "
                           "larger than the captured launch was sized for")


# --------------------------------------------------------------------------- #
# integer side
# --------------------------------------------------------------------------- #
class CSR(NamedTuple):
    rowptr: torch.Tensor   # [N+1] int32
    nbr: torch.Tensor      # [E'] int32 (source for by=1, destination for by=0)
    eid: torch.Tensor      # [E'] int32 original edge id (E + node for appended self loops)
    status: torch.Tensor   # [1] int32, non-zero on device when an index was out of range


def build_csr(edge_index: torch.Tensor, num_nodes: int, by: int = 1, flags: int = 0) -> CSR:
    """Stable CSR of ``edge_index`` grouped by row ``by`` (1 = destination)."""
    _require_cuda(edge_index)
    edge_index = _i64(edge_index)
    E = int(edge_index.shape[1])
    N = int(num_nodes)
    dev = edge_index.device
    Ep = E + (N if flags & CSR_ADD_SELF else 0)
    rowptr = torch.empty(N + 1, dtype=torch.int32, device=dev)
    nbr = torch.empty(max(Ep, 1), dtype=torch.int32, device=dev)[:Ep]    # never a NULL pointer
    eid = torch.empty(max(Ep, 1), dtype=torch.int32, device=dev)[:Ep]
    status = torch.empty(1, dtype=torch.int32, device=dev)
    L = _lib.lib()
    nb = L.qot_csr_workspace_bytes(N, E)
    ws = _lib.workspace(nb, dev)
    check(L.qot_build_csr(ptr(edge_index), E, N, by, flags, ptr(rowptr), ptr(nbr), ptr(eid), ptr(status),
                          ptr(ws), ws.numel(), stream()), "qot_build_csr")
    return CSR(rowptr, nbr, eid, _track_status("qot_build_csr (edge_index entry outside [0, num_nodes))", status))


def graph_ptr(batch: torch.Tensor, num_graphs: int) -> torch.Tensor:
    _require_cuda(batch)
    batch = _i64(batch)
    out = torch.empty(num_graphs + 1, dtype=torch.int64, device=batch.device)
    check(_lib.lib().qot_graph_ptr(ptr(batch), batch.numel(), num_graphs, ptr(out), stream()), "qot_graph_ptr")
    return out


def edge_ptr(edge_index: torch.Tensor, batch: torch.Tensor, num_graphs: int):
    """Edge offsets per graph + a device status flag (non-zero when the edges are not
    grouped by graph)."""
    _require_cuda(edge_index, batch)
    edge_index, batch = _i64(edge_index), _i64(batch)
    out = torch.empty(num_graphs + 1, dtype=torch.int64, device=batch.device)
    status = torch.empty(1, dtype=torch.int32, device=batch.device)
    check(_lib.lib().qot_edge_ptr(ptr(edge_index), edge_index.shape[1], ptr(batch), batch.numel(),
                                  num_graphs, ptr(out), ptr(status), stream()), "qot_edge_ptr")
    return out, status          # read by the caller (LightpathGNN._forward_eval): chooses the general path


def batch_num_graphs(data) -> int:
    """``data.num_graphs`` when the batch object carries it (PyG's and ours do), else
    ``batch.max()+1`` as the reference's global_mean_pool does (one host sync)."""
    B = getattr(data, "num_graphs", None)
    if B is None:
        B = int(data.batch.max().item()) + 1 if data.batch.numel() else 0
    return int(B)


def batch_cache(data) -> dict:
    """Per-batch cache of derived index structures (graph offsets, CSR, transposed
    CSR) -- built once per batch object, shared by both conv layers and the backward."""
    cache = getattr(data, "_cache", None)
    if cache is None:
        cache = {}
        try:
            setattr(data, "_cache", cache)
        except Exception:   # foreign batch object refusing attributes: rebuild each call
            pass
    return cache


def batch_graph_ptr(data) -> torch.Tensor:
    cache = batch_cache(data)
    if "gptr" in cache:
        return cache["gptr"]
    p = getattr(data, "ptr", None)
    if p is None or not p.is_cuda or p.dtype != torch.int64:
        p = graph_ptr(data.batch, batch_num_graphs(data))
    cache["gptr"] = p.contiguous()
    return cache["gptr"]


# --------------------------------------------------------------------------- #
# LightpathGNN fused inference
# --------------------------------------------------------------------------- #
def lightpath_prepare(params: dict, bn_eps: float, is_lut_index: int) -> torch.Tensor:
    """Folds the eval-mode parameters (see qot_lightpath_prepare)."""
    L = _lib.lib()
    ts = {k: _f32(v.detach()) for k, v in params.items()}
    _require_cuda(*ts.values())
    st = _lib.QotLightpathParams(
        ptr(ts["lin_w"]), ptr(ts["att_src"]), ptr(ts["att_dst"]), ptr(ts["conv_bias"]),
        ptr(ts["bn_w"]), ptr(ts["bn_b"]), ptr(ts["bn_mean"]), ptr(ts["bn_var"]),
        ptr(ts["mlp_w1"]), ptr(ts["mlp_b1"]), ptr(ts["mlp_w2"]), ptr(ts["mlp_b2"]),
        float(bn_eps), int(is_lut_index))
    out = torch.empty(L.qot_lightpath_prepared_floats(), dtype=torch.float32, device=ts["lin_w"].device)
    check(L.qot_lightpath_prepare(C.byref(st), ptr(out), stream()), "qot_lightpath_prepare")
    return out


class LightpathInferOut(NamedTuple):
    out: torch.Tensor         # [cap,3]; rows [0,L) valid
    lut_batch: torch.Tensor   # [cap] int64
    lut_node: torch.Tensor    # [cap] int32
    n_lut: torch.Tensor       # [1] int32 on device (= lut_ptr[B])
    status: torch.Tensor      # [1] int32 on device; non-zero: lut_ptr did not match x


def lightpath_lut_ptr(x, gptr, is_lut_index: int) -> torch.Tensor:
    """lut_ptr [B+1] int64: exclusive prefix of the per-graph LUT-node counts (device, no sync)."""
    _require_cuda(x, gptr)
    x = _f32(x)
    N, B = int(x.shape[0]), int(gptr.numel() - 1)
    out = torch.empty(B + 1, dtype=torch.int64, device=x.device)
    L = _lib.lib()
    ws = _lib.workspace(L.qot_lightpath_lut_ptr_workspace_bytes(B), x.device)
    check(L.qot_lightpath_lut_ptr(ptr(x), ptr(gptr), N, B, int(is_lut_index), ptr(out), ptr(ws), ws.numel(),
                                  stream()), "qot_lightpath_lut_ptr")
    return out


# --------------------------------------------------------------------------- #
# graph index shared by the layers of one forward/backward
# --------------------------------------------------------------------------- #
class LightpathStreamPlan:
    """Many resident batches evaluated by ONE launch of the persistent kernel (qot_lightpath_infer_stream).

    Built once for a list of batches (each carrying ptr / edge_ptr / lut_ptr): pooled output buffers sized by
    the batches' readout-row counts (one device->host read of the nb counts here, none afterwards), one
    status word and one row count per batch, and the DEVICE array of batch descriptors the kernel walks.
    ``launch(prepared, first, count)`` enqueues batches [first, first+count) on the current stream: no
    synchronisation, CUDA-graph capturable.  ``result(i)`` gives views of batch i's outputs.

    ``every_node=True`` (qot_lightpath_infer_every_node): every node of every graph is evaluated as the LUT.  Row i of
    batch b's output [N_b, 3] is what the reference forward under eval() returns for node i's graph with node i's flag
    column set to 1.0 and every other node's to 0.0; the stored flag column has no effect.  Rows are in node order, the
    graph of row i is ``batch[i]``.  Buffers are sized by N: no lut_ptr is needed and nothing is read from the device."""

    def __init__(self, batches, is_lut_index: int, split_head: bool = False, every_node: bool = False):
        """``split_head``: QOT_LP_SPLIT_HEAD -- the readout head as a second launch instead of inside the kernel."""
        L = _lib.lib()
        if not batches:
            raise ValueError("LightpathStreamPlan: no batches")
        if every_node and split_head:
            raise ValueError("LightpathStreamPlan: split_head does not apply to every_node mode")
        dev = batches[0].x.device
        for b in batches:
            if every_node:
                if b.ptr is None or b.edge_ptr is None:
                    raise RuntimeError("LightpathStreamPlan(every_node=True) needs batches carrying ptr and edge_ptr "
                                       "(PackedGraphStore.collate provides them)")
                _require_cuda(b.x, b.edge_index, b.ptr, b.edge_ptr)
                continue
            if b.ptr is None or b.edge_ptr is None or b.lut_ptr is None or getattr(b, "lut_col", None) != is_lut_index:
                raise RuntimeError("LightpathStreamPlan needs batches carrying ptr, edge_ptr and lut_ptr for "
                                   "is_lut_index (PackedGraphStore.collate provides them)")
            _require_cuda(b.x, b.edge_index, b.ptr, b.edge_ptr, b.lut_ptr)
        self.batches = list(batches)                 # keeps the input tensors alive
        self.device = dev                            # (_lib.on_tensor_device makes it current around forward_stream)
        self.is_lut_index = int(is_lut_index)
        self.every_node = bool(every_node)
        # QOT_LP_SYMMETRIC_BY_SOURCE only when EVERY batch carries the verified-layout mark
        self.flags = (1 if all(getattr(b, "sym_by_src", False) for b in batches) else 0) | (2 if split_head else 0)
        nb = len(batches)
        if every_node:
            self.rows = [int(b.x.shape[0]) for b in batches]
        else:
            rows = torch.stack([b.lut_ptr[-1] for b in batches]).tolist()      # the one sync
            self.rows = [int(r) for r in rows]
        cap = [max(r, 1) for r in self.rows]
        off = [0]
        for c in cap:
            off.append(off[-1] + c)
        tot = off[-1]
        self.out = torch.empty(tot, 3, dtype=torch.float32, device=dev)
        if every_node:                               # the kernel writes `out` only
            self.lut_batch = self.lut_node = self.z = None
        else:
            self.lut_batch = torch.empty(tot, dtype=torch.int64, device=dev)
            self.lut_node = torch.empty(tot, dtype=torch.int32, device=dev)
            self.z = torch.empty(tot, 20, dtype=torch.float32, device=dev)
        self.n_lut = torch.zeros(nb, dtype=torch.int32, device=dev)
        self.status = torch.zeros(nb, dtype=torch.int32, device=dev)
        self.off = off
        self.keep = []
        descs = (_lib.QotLpBatch * nb)()
        tile0 = [0]
        for i, b in enumerate(batches):
            x, ei = _f32(b.x), _i64(b.edge_index)
            gp, ep = _i64(b.ptr), _i64(b.edge_ptr)
            self.keep += [x, ei, gp, ep]
            d = descs[i]
            d.x, d.edge_index, d.ptr, d.edge_ptr = ptr(x), ptr(ei), ptr(gp), ptr(ep)
            d.N, d.E, d.B = int(x.shape[0]), int(ei.shape[1]), int(gp.numel() - 1)
            o = off[i]
            d.out = self.out.data_ptr() + o * 12
            d.n_lut = self.n_lut.data_ptr() + i * 4
            d.status = self.status.data_ptr() + i * 4
            d.tile0 = tile0[-1]
            if every_node:
                tile0.append(tile0[-1] + int(L.qot_lightpath_every_node_tiles(d.B)))
                continue
            lp = _i64(b.lut_ptr)
            self.keep.append(lp)
            d.lut_ptr = ptr(lp)
            d.lut_batch = self.lut_batch.data_ptr() + o * 8
            d.lut_node = self.lut_node.data_ptr() + o * 4
            d.z = self.z.data_ptr() + o * 80
            tile0.append(tile0[-1] + int(L.qot_lightpath_stream_tiles(d.B)))
        self.tile0 = tile0
        self.desc_size = C.sizeof(_lib.QotLpBatch)
        raw = torch.frombuffer(bytearray(bytes(descs)), dtype=torch.uint8)
        self.descs = raw.to(dev)
        _track_status("qot_lightpath_infer_every_node (malformed graph offsets)" if every_node else
                      "qot_lightpath_infer_stream (lut_ptr does not describe x, or a pipeline barrier timed out)",
                      self.status)

    def __len__(self):
        return len(self.batches)

    def launch(self, prepared: torch.Tensor, first: int = 0, count: Optional[int] = None) -> None:
        nb = len(self.batches)
        count = nb - first if count is None else count
        if first < 0 or count <= 0 or first + count > nb:
            raise ValueError(f"LightpathStreamPlan.launch: range [{first}, {first + count}) outside [0, {nb})")
        tiles = [self.tile0[i + 1] - self.tile0[i] for i in range(first, first + count)]
        uniform = tiles[0] if all(t == tiles[0] for t in tiles[:-1]) and tiles[-1] <= tiles[0] else 0
        self.status[first:first + count].zero_()
        if self.every_node:
            check(_lib.lib().qot_lightpath_infer_every_node(
                self.descs.data_ptr() + first * self.desc_size, count, self.tile0[first + count] - self.tile0[first],
                uniform, ptr(prepared), self.is_lut_index, self.flags, stream()), "qot_lightpath_infer_every_node")
            return
        check(_lib.lib().qot_lightpath_infer_stream(
            self.descs.data_ptr() + first * self.desc_size, count, self.tile0[first + count] - self.tile0[first],
            uniform, max(self.rows[first:first + count]), ptr(prepared), self.is_lut_index, self.flags, stream()),
            "qot_lightpath_infer_stream")

    def result(self, i: int) -> LightpathInferOut:
        """every_node: ``out`` holds batch i's N rows, ``lut_batch`` is the batch's ``batch`` vector (or None),
        ``lut_node`` / ``n_lut`` are None."""
        a, b = self.off[i], self.off[i + 1]
        if self.every_node:
            return LightpathInferOut(self.out[a:a + self.rows[i]], getattr(self.batches[i], "batch", None), None, None,
                                     self.status[i:i + 1])
        return LightpathInferOut(self.out[a:b], self.lut_batch[a:b], self.lut_node[a:b], self.n_lut[i:i + 1],
                                 self.status[i:i + 1])


# status bits of qot_lightpath_candidates / qot_lightpath_reconfigure (include/qot_b200.h)
CAND_BAD_SAMPLE, CAND_BAD_PATH, CAND_OCCUPIED, CAND_IMPACT_OVERFLOW, CAND_BAD_STATE = 1, 2, 4, 8, 16
CAND_BAD_NODE = 32
# impact_kind bits of qot_lightpath_reconfigure
KIND_LOST, KIND_GAINED, KIND_KEPT = 1, 2, 3
# status bits of qot_lightpath_change_sets, on top of the CAND_* bits; a set holds at most SET_MAX_CHANGES changes
SET_BAD_SET, SET_DUPLICATE, SET_CONFLICT = 64, 128, 256
SET_MAX_CHANGES = 64


class CandidateQoT(NamedTuple):
    out: torch.Tensor            # [K,3]: the candidate's own QoT (NaN with status bits 0-2)
    status: torch.Tensor         # [K] int32, CAND_* bits
    n_impact: torch.Tensor       # [K] int32: existing lightpaths the candidate interferes with (may exceed max_impact)
    impact_node: torch.Tensor    # [K, max_impact] int64: their nodes in the state batch, ascending; -1 past the rows
    impact_out: torch.Tensor     # [K, max_impact, 3]: their QoT with the candidate set up; NaN past the rows


class ReconfigQoT(NamedTuple):
    out: torch.Tensor            # [K,3]: the moved lightpath's QoT at its new placement (NaN for a teardown)
    status: torch.Tensor         # [K] int32, CAND_* bits
    n_impact: torch.Tensor       # [K] int32: lightpaths that lose, gain or keep the moved one (may exceed max_impact)
    impact_node: torch.Tensor    # [K, max_impact] int64: their nodes in the state batch, ascending; -1 past the rows
    impact_kind: torch.Tensor    # [K, max_impact] int8: KIND_LOST / KIND_GAINED / KIND_KEPT; 0 past the rows
    impact_out: torch.Tensor     # [K, max_impact, 3]: their QoT after the change; NaN past the rows


class ChangeSetQoT(NamedTuple):
    out: torch.Tensor            # [K,3]: each changed lightpath's QoT at its new placement (NaN: teardown, fatal set)
    status: torch.Tensor         # [K] int32, CAND_* | SET_* bits of each change
    set_status: torch.Tensor     # [G] int32, the OR over the set's changes
    n_impact: torch.Tensor       # [G] int32: lightpaths the set disturbs (may exceed max_impact)
    impact_node: torch.Tensor    # [G, max_impact] int64: their nodes in the state batch, ascending; -1 past the rows
    impact_kind: torch.Tensor    # [G, max_impact] int8: KIND_LOST / KIND_GAINED / KIND_KEPT; 0 past the rows
    impact_out: torch.Tensor     # [G, max_impact, 3]: their QoT after the set; NaN past the rows


_CAND_DTYPES = {"sample": torch.int64, "link_ptr": torch.int64, "links": torch.int32, "q0": torch.int32,
                "width": torch.int32, "feat": torch.float32}


def _check_state_tensor(who: str, name: str, t, dev, dt) -> None:
    """An input of a network-state query: a CUDA tensor on the state's device, of dtype dt."""
    if not torch.is_tensor(t) or not t.is_cuda:
        raise RuntimeError(f"{who}: {name} must be a CUDA tensor (no CPU path)")
    if t.device != dev:
        raise ValueError(f"{who}: {name} is on {t.device}, the state on {dev}")
    if t.dtype != dt:
        raise TypeError(f"{who}: {name} must be {dt}, got {t.dtype}")


def _cptr(t):
    """Pointer of a contiguous t, None for an absent or empty tensor."""
    return ptr(t.contiguous()) if t is not None and t.numel() else None


def _check_candidate_args(state, c, prepared, max_impact, who: str, arg: str, want: dict) -> int:
    """Host-side checks shared by forward_candidates and forward_reconfigurations; returns K."""
    if int(max_impact) != max_impact or max_impact < 0:
        raise ValueError(f"{who}: max_impact must be a non-negative integer")
    dev = state.batch.x.device
    for name, dt in want.items():
        _check_state_tensor(who, f"{arg}.{name}", getattr(c, name), dev, dt)
    if prepared.device != dev:
        raise ValueError(f"{who}: the model is on {prepared.device}, the state on {dev}")
    K = int(c.sample.shape[0]) if c.sample.dim() == 1 else -1
    shapes_ok = (K >= 0 and c.link_ptr.shape == (K + 1,) and c.links.dim() == 1 and
                 c.q0.shape == (K,) and c.width.shape == (K,) and c.feat.shape == (K, 4))
    if not shapes_ok:
        raise ValueError(f"{who}: need sample [K], link_ptr [K+1], links [n], q0 [K], width [K], feat [K,4]")
    if "node" in want and c.node.shape != (K,):
        raise ValueError(f"{who}: need node [K] with K = sample.shape[0]")
    return K


def _state_desc(state, keep: list) -> "_lib.QotLpState":
    """The qot_lp_state_t of a ``LightpathNetworkState``; converted tensors go into `keep`.  Built on every call, never
    cached on the state: a state made with ``_replace`` must not reuse another state's pointers."""
    b = state.batch
    x, ei = _f32(b.x), _i64(b.edge_index)
    keep += [x, ei]
    return _lib.QotLpState(state.cfg, state.S, int(x.shape[0]), int(ei.shape[1]), ptr(state.freqs), ptr(x), ptr(b.ptr),
                           ptr(state.rowptr), ptr(ei) if ei.numel() else None, ptr(state.chan_node),
                           ptr(state.conn_ids) if state.conn_ids.numel() else None)


def _changes_desc(c, K: int, keep: list) -> "_lib.QotLpChanges":
    """The qot_lp_changes_t of ``LightpathChanges`` or ``LightpathCandidates`` (node NULL); contiguous tensors go into
    `keep`."""
    node = getattr(c, "node", None)
    ts = [None if t is None else t.contiguous() for t in (node, c.sample, c.link_ptr, c.links, c.q0, c.width, c.feat)]
    keep += ts
    return _lib.QotLpChanges(K, int(c.links.numel()), *(_cptr(t) for t in ts))


def lightpath_candidates(state, cands, prepared: torch.Tensor, is_lut_index: int, max_impact: int) -> CandidateQoT:
    """One launch of qot_lightpath_candidates; nothing is read back (CUDA-graph capturable).  Refuses CPU tensors and
    mismatched devices, dtypes or shapes; what can only be judged on the device comes back as status bits."""
    K = _check_candidate_args(state, cands, prepared, max_impact, "forward_candidates", "cands", _CAND_DTYPES)
    max_impact = int(max_impact)
    dev = state.batch.x.device
    out = torch.empty(K, 3, dtype=torch.float32, device=dev)
    status = torch.empty(K, dtype=torch.int32, device=dev)
    n_impact = torch.empty(K, dtype=torch.int32, device=dev)
    impact_node = torch.empty(K, max_impact, dtype=torch.int64, device=dev)
    impact_out = torch.empty(K, max_impact, 3, dtype=torch.float32, device=dev)
    if K == 0:
        return CandidateQoT(out, status, n_impact, impact_node, impact_out)
    keep = []                                        # alive until the launch is enqueued
    with torch.cuda.device(dev):                     # stream() of the state's device
        check(_lib.lib().qot_lightpath_candidates(
            C.byref(_state_desc(state, keep)), C.byref(_changes_desc(cands, K, keep)), ptr(prepared),
            int(is_lut_index), max_impact, ptr(out), ptr(status), ptr(n_impact), _cptr(impact_node),
            _cptr(impact_out), stream()), "qot_lightpath_candidates")
    return CandidateQoT(out, status, n_impact, impact_node, impact_out)


def lightpath_reconfigure(state, changes, prepared: torch.Tensor, is_lut_index: int, max_impact: int) -> ReconfigQoT:
    """One launch of qot_lightpath_reconfigure (moves, teardowns and insertions of lightpaths, each against the state
    alone); nothing is read back (CUDA-graph capturable).  Same host-side checks as ``lightpath_candidates``."""
    want = dict(_CAND_DTYPES, node=torch.int64)
    K = _check_candidate_args(state, changes, prepared, max_impact, "forward_reconfigurations", "changes", want)
    max_impact = int(max_impact)
    dev = state.batch.x.device
    out = torch.empty(K, 3, dtype=torch.float32, device=dev)
    status = torch.empty(K, dtype=torch.int32, device=dev)
    n_impact = torch.empty(K, dtype=torch.int32, device=dev)
    impact_node = torch.empty(K, max_impact, dtype=torch.int64, device=dev)
    impact_kind = torch.empty(K, max_impact, dtype=torch.int8, device=dev)
    impact_out = torch.empty(K, max_impact, 3, dtype=torch.float32, device=dev)
    if K == 0:
        return ReconfigQoT(out, status, n_impact, impact_node, impact_kind, impact_out)
    keep = []
    with torch.cuda.device(dev):
        check(_lib.lib().qot_lightpath_reconfigure(
            C.byref(_state_desc(state, keep)), C.byref(_changes_desc(changes, K, keep)), ptr(prepared),
            int(is_lut_index), max_impact, ptr(out), ptr(status), ptr(n_impact), _cptr(impact_node),
            _cptr(impact_kind), _cptr(impact_out), stream()), "qot_lightpath_reconfigure")
    return ReconfigQoT(out, status, n_impact, impact_node, impact_kind, impact_out)


def lightpath_change_sets(state, changes, set_ptr: torch.Tensor, prepared: torch.Tensor, is_lut_index: int,
                          max_impact: int) -> "ChangeSetQoT":
    """One launch of qot_lightpath_change_sets (sets of changes to one sample each, evaluated jointly); nothing is read
    back (CUDA-graph capturable).  The host checks of ``lightpath_reconfigure`` plus set_ptr's device, dtype and shape;
    set_ptr's values are judged on the device (``SET_BAD_SET``)."""
    who = "forward_change_sets"
    want = dict(_CAND_DTYPES, node=torch.int64)
    K = _check_candidate_args(state, changes, prepared, max_impact, who, "changes", want)
    max_impact = int(max_impact)
    dev = state.batch.x.device
    _check_state_tensor(who, "set_ptr", set_ptr, dev, torch.int64)
    if set_ptr.dim() != 1 or set_ptr.shape[0] < 1:
        raise ValueError(f"{who}: need set_ptr [G+1] with G >= 0")
    G = int(set_ptr.shape[0]) - 1
    out = torch.empty(K, 3, dtype=torch.float32, device=dev)
    status = torch.empty(K, dtype=torch.int32, device=dev)
    set_status = torch.empty(G, dtype=torch.int32, device=dev)
    n_impact = torch.empty(G, dtype=torch.int32, device=dev)
    impact_node = torch.empty(G, max_impact, dtype=torch.int64, device=dev)
    impact_kind = torch.empty(G, max_impact, dtype=torch.int8, device=dev)
    impact_out = torch.empty(G, max_impact, 3, dtype=torch.float32, device=dev)
    res = ChangeSetQoT(out, status, set_status, n_impact, impact_node, impact_kind, impact_out)
    if K == 0 and G == 0:
        return res
    keep = [set_ptr.contiguous()]
    with torch.cuda.device(dev):
        check(_lib.lib().qot_lightpath_change_sets(
            C.byref(_state_desc(state, keep)), C.byref(_changes_desc(changes, K, keep)), G, ptr(keep[0]),
            ptr(prepared), int(is_lut_index), max_impact, _cptr(out), _cptr(status), _cptr(set_status),
            _cptr(n_impact), _cptr(impact_node), _cptr(impact_kind), _cptr(impact_out), stream()),
            "qot_lightpath_change_sets")
    return res


# placement policies of qot_lightpath_placements; a demand offers at most PLACE_MAX_OPTIONS options, Q is at most
# PLACE_MAX_SLOTS
PLACE_FIRST_FIT, PLACE_BEST_QOT, PLACE_MAX_MARGIN = 0, 1, 2
PLACE_MAX_OPTIONS = 32
PLACE_MAX_SLOTS = 1024


class PlacementQoT(NamedTuple):
    option: torch.Tensor         # [D] int32: the chosen option, relative to opt_ptr[d] (-1: no feasible placement)
    q0: torch.Tensor             # [D] int32: its start slot (-1: none)
    out: torch.Tensor            # [D,3]: the chosen placement's own QoT (NaN: none)
    margin: torch.Tensor         # [D]: its margin (NaN: none)
    n_free: torch.Tensor         # [D] int32: free placements over the demand's options
    n_feasible: torch.Tensor     # [D] int32: feasible placements among them
    status: torch.Tensor         # [D] int32, CAND_* bits
    n_impact: torch.Tensor       # [D] int32: lightpaths the chosen placement interferes with (may exceed max_impact)
    impact_node: torch.Tensor    # [D, max_impact] int64: their nodes in the state batch, ascending; -1 past the rows
    impact_out: torch.Tensor     # [D, max_impact, 3]: their QoT with the placement set up; NaN past the rows
    all_out: Optional[torch.Tensor] = None     # [P, Q, 3] (return_all): every free placement's own QoT, NaN elsewhere
    all_margin: Optional[torch.Tensor] = None  # [P, Q] (return_all): every free placement's margin, NaN elsewhere


_DEMAND_DTYPES = {"sample": torch.int64, "opt_ptr": torch.int64, "link_ptr": torch.int64, "links": torch.int32,
                  "width": torch.int32, "feat": torch.float32, "own_bound": torch.float32}


def _check_demand_args(who: str, state, demands, policy: int, metric: int, bound, prepared, max_impact):
    """Host-side checks shared by forward_placements and forward_provision; returns (D, P)."""
    if int(max_impact) != max_impact or max_impact < 0:
        raise ValueError(f"{who}: max_impact must be a non-negative integer")
    if policy not in (PLACE_FIRST_FIT, PLACE_BEST_QOT, PLACE_MAX_MARGIN):
        raise ValueError(f"{who}: policy must be PLACE_FIRST_FIT, PLACE_BEST_QOT or PLACE_MAX_MARGIN")
    if metric not in (0, 1, 2):
        raise ValueError(f"{who}: metric must be an output column 0, 1 or 2")
    if state.Q > PLACE_MAX_SLOTS:
        raise ValueError(f"{who}: Q = {state.Q} slots, at most {PLACE_MAX_SLOTS} (one 32-bit free word per lane)")
    dev = state.batch.x.device
    want = dict(_DEMAND_DTYPES)
    named = [(n, getattr(demands, n), dt) for n, dt in want.items()]
    if bound is not None:
        named.append(("bound", bound, torch.float32))
    for name, t, dt in named:
        _check_state_tensor(who, name if name == "bound" else f"demands.{name}", t, dev, dt)
    if prepared.device != dev:
        raise ValueError(f"{who}: the model is on {prepared.device}, the state on {dev}")
    d = demands
    D = int(d.sample.shape[0]) if d.sample.dim() == 1 else -1
    P = int(d.width.shape[0]) if d.width.dim() == 1 else -1
    if not (D >= 0 and P >= 0 and d.opt_ptr.shape == (D + 1,) and d.link_ptr.shape == (P + 1,) and
            d.links.dim() == 1 and d.feat.shape == (P, 3) and d.own_bound.shape == (P,)):
        raise ValueError(f"{who}: need sample [D], opt_ptr [D+1], link_ptr [P+1], links [n], width [P], feat [P,3], "
                         "own_bound [P]")
    N = int(state.batch.x.shape[0])
    if bound is not None and bound.shape != (N,):
        raise ValueError(f"{who}: need bound [N] with N = {N} nodes of the state batch")
    return D, P


def _demands_desc(d, D: int, P: int, keep: list) -> "_lib.QotLpDemands":
    """The qot_lp_demands_t of ``LightpathDemands``; contiguous tensors go into `keep`."""
    ts = [t.contiguous() for t in (d.sample, d.opt_ptr, d.link_ptr, d.links, d.width, d.feat, d.own_bound)]
    keep += ts
    return _lib.QotLpDemands(D, P, int(d.links.numel()), *(_cptr(t) for t in ts))


def _demand_outputs(D: int, max_impact: int, dev) -> list:
    """Uninitialised outputs of a demand query, in PlacementQoT / ProvisionQoT field order: option, q0, out, margin,
    n_free, n_feasible, status, n_impact, the impact rows' ids [D, max_impact] int64 and impact_out."""
    i32 = lambda *s: torch.empty(*s, dtype=torch.int32, device=dev)
    f32 = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)
    return [i32(D), i32(D), f32(D, 3), f32(D), i32(D), i32(D), i32(D), i32(D),
            torch.empty(D, max_impact, dtype=torch.int64, device=dev), f32(D, max_impact, 3)]


def lightpath_placements(state, demands, policy: int, metric: int, maximize: bool, bound, prepared: torch.Tensor,
                         is_lut_index: int, max_impact: int, return_all: bool = False) -> PlacementQoT:
    """One launch of qot_lightpath_placements (the placement of each demand chosen over every free slot of its
    options); nothing is read back (CUDA-graph capturable).  Refuses CPU tensors and mismatched devices, dtypes or
    shapes, an unknown policy or metric and Q over PLACE_MAX_SLOTS; what can only be judged on the device comes back
    as status bits."""
    who = "forward_placements"
    D, P = _check_demand_args(who, state, demands, policy, metric, bound, prepared, max_impact)
    dev = state.batch.x.device
    max_impact = int(max_impact)
    f32 = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)
    res = PlacementQoT(*_demand_outputs(D, max_impact, dev), f32(P, state.Q, 3) if return_all else None,
                       f32(P, state.Q) if return_all else None)
    if D == 0:
        return res
    bound = None if bound is None else bound.contiguous()
    keep = []
    with torch.cuda.device(dev):
        check(_lib.lib().qot_lightpath_placements(
            C.byref(_state_desc(state, keep)), C.byref(_demands_desc(demands, D, P, keep)), _cptr(bound),
            int(metric), int(bool(maximize)), int(policy), ptr(prepared), int(is_lut_index), max_impact,
            ptr(res.option), ptr(res.q0), ptr(res.out), ptr(res.margin), ptr(res.n_free), ptr(res.n_feasible),
            ptr(res.status), ptr(res.n_impact), _cptr(res.impact_node), _cptr(res.impact_out), _cptr(res.all_out),
            _cptr(res.all_margin), stream()), "qot_lightpath_placements")
    return res


# status bits of qot_lightpath_provision, on top of the CAND_* bits
PROV_FULL, PROV_BAD_GROUPING = 512, 1024
TG_MAX_NODES, TG_MAX_CHANNELS = 256, 6144      # QOT_TG_MAX_NODES / QOT_TG_MAX_CHANNELS: a sample's graph capacity


class ProvisionQoT(NamedTuple):
    option: torch.Tensor         # [D] int32: the chosen option, relative to opt_ptr[d] (-1: no feasible placement)
    q0: torch.Tensor             # [D] int32: its start slot (-1: none)
    out: torch.Tensor            # [D,3]: the chosen placement's own QoT (NaN: none)
    margin: torch.Tensor         # [D]: its margin (NaN: none)
    n_free: torch.Tensor         # [D] int32: free placements over the demand's options
    n_feasible: torch.Tensor     # [D] int32: feasible placements among them
    status: torch.Tensor         # [D] int32, CAND_* | PROV_* bits
    n_impact: torch.Tensor       # [D] int32: lightpaths the chosen placement interferes with (may exceed max_impact)
    impact_conn: torch.Tensor    # [D, max_impact] int64: their conn_ids, ascending in node order; -1 past the rows
    impact_out: torch.Tensor     # [D, max_impact, 3]: their QoT with the placement set up; NaN past the rows
    conn_id: torch.Tensor        # [D] int64: the conn_id the demand was accepted under (-1: not accepted)


def provision_grouping(sample: torch.Tensor, S: int):
    """(order [D], sample_ptr [S+1]) int64: the demands grouped by sample, ascending within a sample (a stable sort),
    samples outside [0, S) after the last range.  Device tensor ops, no host synchronisation."""
    key = torch.where((sample >= 0) & (sample < S), sample, torch.full_like(sample, S))
    skey, order = torch.sort(key, stable=True)
    sample_ptr = torch.searchsorted(skey, torch.arange(S + 1, dtype=torch.int64, device=sample.device))
    return order, sample_ptr


def lightpath_provision(state, demands, policy: int, metric: int, maximize: bool, bound, prepared: torch.Tensor,
                        is_lut_index: int, max_impact: int) -> ProvisionQoT:
    """qot_lightpath_provision: each sample's demands placed in index order, each against the state with the earlier
    accepted ones set up.  The grouping is computed on the device and the work arrays allocated here; one copy and one
    launch, nothing read back (CUDA-graph capturable).  The host checks of ``lightpath_placements``."""
    who = "forward_provision"
    D, P = _check_demand_args(who, state, demands, policy, metric, bound, prepared, max_impact)
    dev = state.batch.x.device
    max_impact = int(max_impact)
    res = ProvisionQoT(*_demand_outputs(D, max_impact, dev), torch.empty(D, dtype=torch.int64, device=dev))
    if D == 0:
        return res
    order, sample_ptr = provision_grouping(demands.sample, state.S)
    chan_work = torch.empty_like(state.chan_node)
    bound_work = torch.empty(state.S, TG_MAX_NODES, dtype=torch.float32, device=dev) if bound is not None else None
    bound = None if bound is None else bound.contiguous()
    keep = []
    with torch.cuda.device(dev):
        check(_lib.lib().qot_lightpath_provision(
            C.byref(_state_desc(state, keep)), C.byref(_demands_desc(demands, D, P, keep)), ptr(order),
            ptr(sample_ptr), _cptr(bound), int(metric), int(bool(maximize)), int(policy), ptr(prepared),
            int(is_lut_index), max_impact, _cptr(chan_work), _cptr(bound_work), ptr(res.option), ptr(res.q0),
            ptr(res.out), ptr(res.margin), ptr(res.n_free), ptr(res.n_feasible), ptr(res.status), ptr(res.n_impact),
            ptr(res.conn_id), _cptr(res.impact_conn), _cptr(res.impact_out), stream()), "qot_lightpath_provision")
    return res


class GraphIndex:
    """Lazily built, cached index structures of one batch: the destination-sorted CSR
    (forward), its GAT variant (self loops replaced) and the source-sorted transposed
    CSR (deterministic scatter of the backward)."""

    def __init__(self, edge_index: torch.Tensor, num_nodes: int):
        _require_cuda(edge_index)
        self.edge_index = _i64(edge_index)
        self.num_nodes = int(num_nodes)
        self.num_edges = int(edge_index.shape[1])
        self._csr = self._csr_gat = self._csr_t = None

    @property
    def csr(self) -> CSR:
        if self._csr is None:
            self._csr = build_csr(self.edge_index, self.num_nodes, by=1, flags=0)
        return self._csr

    @property
    def csr_gat(self) -> CSR:
        if self._csr_gat is None:
            self._csr_gat = build_csr(self.edge_index, self.num_nodes, by=1,
                                      flags=CSR_DROP_SELF | CSR_ADD_SELF)
        return self._csr_gat

    @property
    def csr_t(self) -> CSR:
        if self._csr_t is None:
            self._csr_t = build_csr(self.edge_index, self.num_nodes, by=0, flags=0)
        return self._csr_t


def batch_graph(data, num_nodes: int) -> GraphIndex:
    cache = batch_cache(data)
    g = cache.get("graph")
    if g is None or g.num_nodes != num_nodes or g.edge_index.data_ptr() != data.edge_index.data_ptr():
        g = GraphIndex(data.edge_index, num_nodes)
        cache["graph"] = g
    return g


def _ws(nbytes, dev):
    return _lib.workspace(nbytes, dev)


# --------------------------------------------------------------------------- #
# GATConv (general path)
# --------------------------------------------------------------------------- #
class _GatConvFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, lin_w, att_src, att_dst, bias, graph: GraphIndex):
        L = _lib.lib()
        x = _f32(x)
        N, dev = x.shape[0], x.device
        csr = graph.csr_gat
        need = any(t.requires_grad for t in (lin_w, att_src, att_dst, bias))
        h = torch.empty(N, 128, dtype=torch.float32, device=dev)
        z = torch.empty(N, 20, dtype=torch.float32, device=dev) if need else None
        smax = torch.empty(N, 4, dtype=torch.float32, device=dev) if need else None
        sden = torch.empty(N, 4, dtype=torch.float32, device=dev) if need else None
        w, a_s, a_d, b = _f32(lin_w.detach()), _f32(att_src.detach()), _f32(att_dst.detach()), _f32(bias.detach())
        check(L.qot_gat_fwd(ptr(x), ptr(csr.rowptr), ptr(csr.nbr), N, ptr(w), ptr(a_s), ptr(a_d), ptr(b),
                            ptr(h), ptr(z), ptr(smax), ptr(sden), stream()), "qot_gat_fwd")
        if need:
            ctx.save_for_backward(x, w, a_s, a_d, z, smax, sden)
            ctx.csr = csr
        return h

    @staticmethod
    def backward(ctx, dh):
        L = _lib.lib()
        x, w, a_s, a_d, z, smax, sden = ctx.saved_tensors
        csr = ctx.csr
        N, dev = x.shape[0], x.device
        dh = _f32(dh)
        dW = torch.empty_like(w)
        das = torch.empty_like(a_s)
        dad = torch.empty_like(a_d)
        db = torch.empty(128, dtype=torch.float32, device=dev)
        ws = _ws(L.qot_gat_bwd_workspace_bytes(N), dev)
        check(L.qot_gat_bwd(ptr(x), ptr(csr.rowptr), ptr(csr.nbr), N, ptr(w), ptr(a_s), ptr(a_d), ptr(z),
                            ptr(smax), ptr(sden), ptr(dh), ptr(dW), ptr(das), ptr(dad), ptr(db),
                            ptr(ws), ws.numel(), stream()), "qot_gat_bwd")
        return None, dW, das, dad, db, None


def gat_conv(x, graph: GraphIndex, lin_w, att_src, att_dst, bias) -> torch.Tensor:
    """GATConv with gradients for its parameters only: x is data (the lightpath features of
    lightpath_training/models.py:30), so an x that requires grad raises instead of getting a silent zero."""
    _require_cuda(x, lin_w)
    if torch.is_grad_enabled() and x.requires_grad:
        raise NotImplementedError("libqot_b200 GATConv: no gradient with respect to x (the input features are data); "
                                  "pass x.detach()")
    return _GatConvFn.apply(x, lin_w, att_src, att_dst, bias, graph)


# --------------------------------------------------------------------------- #
# BatchNorm statistics, LUT readout + MLP head
# --------------------------------------------------------------------------- #
def _bn_train_stats(h, bn: torch.nn.BatchNorm1d):
    """Batch statistics of ``bn`` in train(), with torch's running-stat update: ``num_batches_tracked`` counts the
    batch first, and ``momentum=None`` takes the cumulative average ``1 / num_batches_tracked`` -- a read of the
    counter, like torch's own BatchNorm, so only a fixed momentum is capturable in a CUDA graph.  One row raises
    torch's ValueError (its variance is 0); N is on the host, so that check costs nothing."""
    if h.shape[0] == 1:
        raise ValueError(f"Expected more than 1 value per channel when training, got input size {h.shape}")
    with torch.no_grad():
        bn.num_batches_tracked += 1
    momentum = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked)
    return bn_batch_stats(h.detach(), bn.running_mean, bn.running_var, momentum)


def bn_batch_stats(h, running_mean=None, running_var=None, momentum: float = 0.1):
    L = _lib.lib()
    h = _f32(h)
    N, C = h.shape
    mean = torch.empty(C, dtype=torch.float32, device=h.device)
    var = torch.empty(C, dtype=torch.float32, device=h.device)
    ws = _ws(L.qot_bn_stats_workspace_bytes(N, C), h.device)
    check(L.qot_bn_stats(ptr(h), N, C, ptr(mean), ptr(var), ptr(running_mean), ptr(running_var),
                         float(momentum), ptr(ws), ws.numel(), stream()), "qot_bn_stats")
    return mean, var


def lut_select(x, batch, is_lut_index: int, n_known: Optional[int] = None):
    """Ordered LUT compaction; one host sync for the row count (the reference's boolean indexing synchronises
    twice) -- none when the caller knows it (`n_known`: collates of this package record it on the host as
    ``batch.lut_rows``), which is what makes the training step CUDA-graph capturable."""
    L = _lib.lib()
    x = _f32(x)
    N, F = x.shape
    dev = x.device
    node = torch.empty(max(N, 1), dtype=torch.int32, device=dev)
    lb = torch.empty(max(N, 1), dtype=torch.int64, device=dev)
    n_lut = torch.empty(1, dtype=torch.int32, device=dev)
    ws = _ws(L.qot_lut_select_workspace_bytes(N), dev)
    check(L.qot_lut_select(ptr(x), N, F, int(is_lut_index), ptr(_i64(batch)), ptr(node), ptr(lb), ptr(n_lut),
                           ptr(ws), ws.numel(), stream()), "qot_lut_select")
    n = int(n_lut.item()) if n_known is None else int(n_known)
    return node[:n], lb[:n], n


class _LutHeadFn(torch.autograd.Function):
    """BN(given statistics) -> ReLU -> LUT rows -> Linear -> LeakyReLU -> (dropout) -> Linear."""

    @staticmethod
    def forward(ctx, h, lut_node, mean, var, eps, bn_w, bn_b, W1, b1, W2, b2, hmask, batch_stats):
        L = _lib.lib()
        nL, dev = lut_node.numel(), h.device
        y = torch.empty(nL, 128, dtype=torch.float32, device=dev)
        hid = torch.empty(nL, 32, dtype=torch.float32, device=dev)
        out = torch.empty(nL, 3, dtype=torch.float32, device=dev)
        ts = [_f32(t.detach()) for t in (bn_w, bn_b, W1, b1, W2, b2)]
        check(L.qot_lut_head_fwd(ptr(h), ptr(lut_node), nL, ptr(mean), ptr(var), float(eps), ptr(ts[0]), ptr(ts[1]),
                                 ptr(ts[2]), ptr(ts[3]), ptr(ts[4]), ptr(ts[5]), ptr(hmask), ptr(y), ptr(hid),
                                 ptr(out), stream()), "qot_lut_head_fwd")
        ctx.save_for_backward(h, lut_node, mean, var, ts[0], ts[2], ts[4], y, hid, hmask)
        ctx.eps, ctx.batch_stats = float(eps), bool(batch_stats)
        return out

    @staticmethod
    def backward(ctx, dout):
        L = _lib.lib()
        h, lut_node, mean, var, bn_w, W1, W2, y, hid, hmask = ctx.saved_tensors
        dev = h.device
        nL, (N, C) = lut_node.numel(), h.shape
        dout = _f32(dout)
        dy = torch.empty(nL, 128, dtype=torch.float32, device=dev)
        dW1, db1 = torch.empty_like(W1), torch.empty(32, dtype=torch.float32, device=dev)
        dW2, db2 = torch.empty_like(W2), torch.empty(3, dtype=torch.float32, device=dev)
        ws = _ws(L.qot_lut_head_bwd_workspace_bytes(nL), dev)
        check(L.qot_lut_head_bwd(ptr(dout), ptr(y), ptr(hid), ptr(hmask), nL, ptr(W1), ptr(W2), ptr(dy),
                                 ptr(dW1), ptr(db1), ptr(dW2), ptr(db2), ptr(ws), ws.numel(), stream()),
              "qot_lut_head_bwd")
        dh = torch.empty_like(h)
        dbn_w = torch.empty(C, dtype=torch.float32, device=dev)
        dbn_b = torch.empty(C, dtype=torch.float32, device=dev)
        ws = _ws(L.qot_bn_bwd_workspace_bytes(N, nL, C), dev)
        check(L.qot_bn_bwd_sparse(ptr(h), ptr(mean), ptr(var), ctx.eps, ptr(bn_w), ptr(dy), ptr(lut_node),
                                  nL, N, C, int(ctx.batch_stats), ptr(dh), ptr(dbn_w), ptr(dbn_b),
                                  ptr(ws), ws.numel(), stream()), "qot_bn_bwd_sparse")
        return dh, None, None, None, None, dbn_w, dbn_b, dW1, db1, dW2, db2, None, None


def lut_bn_head(h, x_feat, batch, is_lut_index, bn: torch.nn.BatchNorm1d, W1, b1, W2, b2,
                training: bool, dropout_p: float = 0.0, n_known: Optional[int] = None):
    """norm1 -> relu -> LUT readout -> mlp of lightpath_training/models.py:31-43.
    Raises ``ValueError("No LUT node found in the batch.")`` like the reference."""
    _require_cuda(h, x_feat, batch)
    # norm1 before the readout, as in the reference: a 1-node batch raises BatchNorm's error, not the LUT one
    if training:
        mean, var = _bn_train_stats(h, bn)
    else:
        mean, var = bn.running_mean, bn.running_var
    lut_node, lut_batch, n = lut_select(x_feat, batch, is_lut_index, n_known)
    if n == 0:
        raise ValueError("No LUT node found in the batch.")
    hmask = None
    if training and dropout_p > 0.0:
        keep = 1.0 - dropout_p
        hmask = (torch.rand(n, 32, device=h.device) < keep).to(torch.float32) / keep
    out = _LutHeadFn.apply(_f32(h), lut_node, mean, var, bn.eps, bn.weight, bn.bias, W1, b1, W2, b2,
                           hmask, training)
    return out, lut_batch


class _BatchNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, mean, var, eps, w, b, batch_stats):
        L = _lib.lib()
        x = _f32(x)
        N, C_ = x.shape
        w_, b_ = _f32(w.detach()), _f32(b.detach())
        y = torch.empty_like(x)
        check(L.qot_bn_apply(ptr(x), N, C_, ptr(mean), ptr(var), float(eps), ptr(w_), ptr(b_), ptr(y), stream()),
              "qot_bn_apply")
        ctx.save_for_backward(x, mean, var, w_)
        ctx.eps, ctx.batch_stats = float(eps), bool(batch_stats)
        return y

    @staticmethod
    def backward(ctx, dy):
        L = _lib.lib()
        x, mean, var, w = ctx.saved_tensors
        N, C_ = x.shape
        dy = _f32(dy)
        dx = torch.empty_like(x)
        dw = torch.empty(C_, dtype=torch.float32, device=x.device)
        db = torch.empty(C_, dtype=torch.float32, device=x.device)
        ws = _ws(L.qot_bn_bwd_dense_workspace_bytes(N, C_), x.device)
        check(L.qot_bn_bwd_dense(ptr(x), ptr(mean), ptr(var), ctx.eps, ptr(w), ptr(dy), N, C_, int(ctx.batch_stats),
                                 ptr(dx), ptr(dw), ptr(db), ptr(ws), ws.numel(), stream()), "qot_bn_bwd_dense")
        return dx, None, None, None, dw, db, None


def batch_norm(x, bn: torch.nn.BatchNorm1d, training: bool):
    """BatchNorm1d over the node dimension as its own layer (PyG ``BatchNorm.forward``):
    batch statistics + running-stat update in train(), running statistics in eval()."""
    _require_cuda(x)
    if x.shape[0] == 0:
        return x
    if training:
        mean, var = _bn_train_stats(x, bn)
    else:
        mean, var = bn.running_mean, bn.running_var
    return _BatchNormFn.apply(x, mean, var, bn.eps, bn.weight, bn.bias, training)


class _MeanPoolFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gptr):
        L = _lib.lib()
        x = _f32(x)
        N, H = x.shape
        B = gptr.numel() - 1
        pooled = torch.empty(B, H, dtype=torch.float32, device=x.device)
        ws = _ws(L.qot_mean_pool_workspace_bytes(N, B, H), x.device)
        check(L.qot_mean_pool_fwd(ptr(x), ptr(gptr), N, B, H, ptr(pooled), ptr(ws), ws.numel(), stream()),
              "qot_mean_pool_fwd")
        ctx.save_for_backward(gptr)
        ctx.N = N
        return pooled

    @staticmethod
    def backward(ctx, dpooled):
        L = _lib.lib()
        (gptr,) = ctx.saved_tensors
        dpooled = _f32(dpooled)
        B, H = dpooled.shape
        dx = torch.empty(ctx.N, H, dtype=torch.float32, device=dpooled.device)
        ws = _ws(L.qot_mean_pool_workspace_bytes(ctx.N, B, H), dpooled.device)
        check(L.qot_mean_pool_bwd(ptr(dpooled), ptr(gptr), ctx.N, B, H, ptr(dx), ptr(ws), ws.numel(), stream()),
              "qot_mean_pool_bwd")
        return dx, None


# --------------------------------------------------------------------------- #
# dense node-wise projection  y = x[ids] W^T + b   (exact fp32)
# --------------------------------------------------------------------------- #
def _ids_csr(ids: torch.Tensor, num_rows: int) -> CSR:
    """CSR of positions grouped by id (deterministic embedding backward)."""
    n = ids.numel()
    pair = torch.stack([torch.arange(n, dtype=torch.int64, device=ids.device), ids])
    # rows are ids (by=1 groups by the second row); the CSR may have more nodes than rows
    return build_csr(pair, max(num_rows, n), by=1, flags=0)


TC_MIN_ROWS = 1024        # below this the 128-row tensor-core tiles cannot fill the machine


def _tc_ok(M: int, Nc: int, K: int) -> bool:
    """Tensor-core path (qot_gemm_tf32x3): only where the projection is a real contraction."""
    return K % 32 == 0 and K >= 64 and M >= TC_MIN_ROWS and Nc >= 64 and Nc % 4 == 0


_tc_status = {}


def gemm_tf32x3(A, W, bias=None, gather=None):
    """C = A[gather] @ W^T (+ bias) on tcgen05 tensor cores with split-fp32 (3 x TF32) operands."""
    L = _lib.lib()
    M = gather.numel() if gather is not None else A.shape[0]
    K, Nc = A.shape[1], W.shape[0]
    dev = A.device
    st = _tc_status.get(dev)
    if st is None:
        st = _tc_status[dev] = torch.zeros(1, dtype=torch.int32, device=dev)
    _track_status("qot_gemm_tf32x3 (tcgen05 barrier timeout)", st)
    C_ = torch.empty(M, Nc, dtype=torch.float32, device=dev)
    ws = _lib.workspace(L.qot_gemm_tf32x3_workspace_bytes(M, Nc, K), dev)
    check(L.qot_gemm_tf32x3(ptr(A), K, ptr(gather), ptr(W), K, ptr(bias), ptr(C_), Nc, M, Nc, K, ptr(st),
                            ptr(ws), ws.numel(), stream()), "qot_gemm_tf32x3")
    return C_


def wgrad_tf32x3(dy, x, gather=None):
    """dW [Nc,K] = dy^T @ x[gather] on the tensor cores (split-K, fixed-order sum)."""
    L = _lib.lib()
    R, Nc = dy.shape
    K = x.shape[1]
    dev = dy.device
    st = _tc_status.get(dev)
    if st is None:
        st = _tc_status[dev] = torch.zeros(1, dtype=torch.int32, device=dev)
    _track_status("qot_wgrad_tf32x3 (tcgen05 barrier timeout)", st)
    dW = torch.empty(Nc, K, dtype=torch.float32, device=dev)
    ws = _lib.workspace(L.qot_wgrad_tf32x3_workspace_bytes(R, Nc, K), dev)
    check(L.qot_wgrad_tf32x3(ptr(dy), Nc, ptr(x), K, ptr(gather), R, Nc, K, ptr(dW), K, ptr(st),
                             ptr(ws), ws.numel(), stream()), "qot_wgrad_tf32x3")
    return dW


class _NodeLinearFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, ids, W, b):
        L = _lib.lib()
        x = _f32(x)
        W_ = _f32(W.detach())
        b_ = _f32(b.detach()) if b is not None else None
        M = ids.numel() if ids is not None else x.shape[0]
        K, Nc = x.shape[1], W_.shape[0]
        if _tc_ok(M, Nc, K):
            y = gemm_tf32x3(x, W_, b_, ids)
        else:
            y = torch.empty(M, Nc, dtype=torch.float32, device=x.device)
            check(L.qot_gemm(ptr(x), K, 1, ptr(ids), ptr(W_), 1, K, ptr(b_), ptr(y), Nc, M, Nc, K, stream()),
                  "qot_gemm")
        ctx.save_for_backward(x, ids, W_)
        ctx.has_bias = b is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        L = _lib.lib()
        x, ids, W = ctx.saved_tensors
        dy = _f32(dy)
        dev = dy.device
        M, Nc = dy.shape
        K = W.shape[1]
        dx = dW = db = None
        need_x, _, need_w, need_b = ctx.needs_input_grad
        if need_x:
            if _tc_ok(M, K, Nc):                                             # dy @ W = dy @ (W^T)^T
                dxr = gemm_tf32x3(dy, W.t().contiguous())
            else:
                dxr = torch.empty(M, K, dtype=torch.float32, device=dev)    # dy @ W
                check(L.qot_gemm(ptr(dy), Nc, 1, None, ptr(W), K, 1, None, ptr(dxr), K, M, K, Nc, stream()),
                      "qot_gemm")
            if ids is None:
                dx = dxr
            else:
                V = x.shape[0]
                csr = _ids_csr(ids, V)
                dx = torch.empty(V, K, dtype=torch.float32, device=dev)
                ws = _ws(L.qot_segment_sum_workspace_bytes(M, V, K), dev)
                check(L.qot_segment_sum(ptr(dxr), ptr(csr.rowptr), ptr(csr.eid), M, V, K, ptr(dx),
                                        ptr(ws), ws.numel(), stream()), "qot_segment_sum")
        if need_w and M >= TC_MIN_ROWS and Nc >= 64 and K >= 64:
            dW = wgrad_tf32x3(dy, x, ids)                                    # dy^T @ x[ids], tensor cores
        elif need_w:
            xr = x if ids is None else _gather_rows(x, ids)
            dW = torch.empty(Nc, K, dtype=torch.float32, device=dev)         # dy^T @ x
            ws = _ws(L.qot_wgrad_workspace_bytes(M, Nc, K), dev)
            check(L.qot_wgrad(ptr(dy), Nc, ptr(xr), K, M, Nc, K, ptr(dW), K, ptr(ws), ws.numel(), stream()),
                  "qot_wgrad")
        if need_b and ctx.has_bias:
            db = torch.empty(Nc, dtype=torch.float32, device=dev)
            ws = _ws(L.qot_colsum_workspace_bytes(M, Nc), dev)
            check(L.qot_colsum(ptr(dy), Nc, M, Nc, ptr(db), ptr(ws), ws.numel(), stream()), "qot_colsum")
        return dx, None, dW, db


def _gather_rows(x, ids):
    """x[ids] through the gemm kernel's gather path with an identity right operand would
    waste flops; a [K,K] identity product is still tiny at K<=256, and keeps the arithmetic
    in libqot_b200."""
    L = _lib.lib()
    K = x.shape[1]
    eye = torch.eye(K, dtype=torch.float32, device=x.device)
    out = torch.empty(ids.numel(), K, dtype=torch.float32, device=x.device)
    check(L.qot_gemm(ptr(x), K, 1, ptr(ids), ptr(eye), K, 1, None, ptr(out), K, ids.numel(), K, K, stream()),
          "qot_gemm")
    return out


def node_linear(x, W, b=None, ids=None):
    _require_cuda(x, W)
    return _NodeLinearFn.apply(x, _i64(ids) if ids is not None else None, W, b)


# --------------------------------------------------------------------------- #
# TransformerConv / NNConv edge phases
# --------------------------------------------------------------------------- #
class _TConvEdgeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, qkvs, edge_attr, We, graph: GraphIndex, slope: float):
        L = _lib.lib()
        N, H4 = qkvs.shape
        H = H4 // 4
        dev = qkvs.device
        csr = graph.csr
        edge_attr = _edge_attr(edge_attr)
        We_ = _f32(We.detach())
        need = qkvs.requires_grad or We.requires_grad
        out = torch.empty(N, H, dtype=torch.float32, device=dev)
        E = graph.num_edges
        logit = torch.empty(max(E, 1), dtype=torch.float32, device=dev) if need else None
        rmax = torch.empty(max(N, 1), dtype=torch.float32, device=dev) if need else None
        rden = torch.empty(max(N, 1), dtype=torch.float32, device=dev) if need else None
        check(L.qot_tconv_fwd(ptr(qkvs), ptr(csr.rowptr), ptr(csr.nbr), ptr(csr.eid), ptr(edge_attr), ptr(We_),
                              N, H, float(slope), ptr(out), ptr(logit), ptr(rmax), ptr(rden), stream()),
              "qot_tconv_fwd")
        if need:
            ctx.save_for_backward(qkvs, edge_attr, We_, out, logit, rmax, rden)
            ctx.graph, ctx.slope = graph, float(slope)
        return out

    @staticmethod
    def backward(ctx, dout):
        L = _lib.lib()
        qkvs, edge_attr, We, out, logit, rmax, rden = ctx.saved_tensors
        g = ctx.graph
        csr, csr_t = g.csr, g.csr_t
        N, H4 = qkvs.shape
        H, E, dev = H4 // 4, g.num_edges, qkvs.device
        dout = _f32(dout)
        dqkvs = torch.empty_like(qkvs)
        dWe = torch.empty_like(We)
        ws = _ws(L.qot_tconv_bwd_workspace_bytes(N, E, H), dev)
        check(L.qot_tconv_bwd(ptr(qkvs), ptr(csr.rowptr), ptr(csr.nbr), ptr(csr.eid), ptr(csr_t.rowptr),
                              ptr(csr_t.nbr), ptr(csr_t.eid), ptr(edge_attr), ptr(We), ptr(out), ptr(dout),
                              ptr(logit), ptr(rmax), ptr(rden), N, E, H, ctx.slope, ptr(dqkvs), ptr(dWe),
                              ptr(ws), ws.numel(), stream()), "qot_tconv_bwd")
        return dqkvs, None, dWe, None, None


_derived_cache = {}


def _derived(tag: str, srcs, make):
    """A tensor that depends on parameters only (concatenated / re-laid-out weights).  While autograd records, it is
    rebuilt every call (autograd routes its gradient back to the parameters); otherwise -- eval under no_grad, the
    serving case -- it is cached: keyed by the sources' storage, shape and version counter (optimizer steps,
    load_state_dict and .to() all change one of them) and validated against weak references to the source tensors,
    so a recycled address never aliases an old entry."""
    if torch.is_grad_enabled() and any(t.requires_grad for t in srcs):
        return make()
    key = (tag,) + tuple((t.data_ptr(), t._version, tuple(t.shape)) for t in srcs)
    hit = _derived_cache.get(key)
    if hit is not None and all(r() is t for r, t in zip(hit[0], srcs)):
        return hit[1]
    if len(_derived_cache) >= 64:
        _derived_cache.clear()
    with torch.no_grad():
        val = make()
    _derived_cache[key] = (tuple(weakref.ref(t) for t in srcs), val)
    return val


def transformer_conv(x, node_ids, graph: GraphIndex, edge_attr, Wq, bq, Wk, bk, Wv, bv, We, Ws, bs,
                     slope: float = 1.0):
    """TransformerConv (+ fused embedding lookup when ``node_ids`` is given and ``x`` is
    the embedding table; + fused leaky_relu when slope != 1)."""
    Wcat = _derived("tconv.W", (Wq, Wk, Wv, Ws), lambda: torch.cat([Wq, Wk, Wv, Ws], dim=0))   # [4H,H]; autograd splits the gradient
    bcat = _derived("tconv.b", (bq, bk, bv, bs), lambda: torch.cat([bq, bk, bv, bs], dim=0))
    qkvs = node_linear(x, Wcat, bcat, ids=node_ids)
    return _TConvEdgeFn.apply(qkvs, edge_attr, We, graph, slope)


class _NNConvEdgeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, yr, edge_attr, W1, b1, bias, graph: GraphIndex, slope: float):
        L = _lib.lib()
        N = yr.shape[0]
        H = yr.shape[1] // (EDGE_HID + 2)
        dev = yr.device
        csr = graph.csr
        edge_attr = _edge_attr(edge_attr)
        W1_, b1_, bias_ = _f32(W1.detach()), _f32(b1.detach()), _f32(bias.detach())
        out = torch.empty(N, H, dtype=torch.float32, device=dev)
        check(L.qot_nnconv_fwd(ptr(yr), ptr(csr.rowptr), ptr(csr.nbr), ptr(csr.eid), ptr(edge_attr), ptr(W1_),
                               ptr(b1_), ptr(bias_), N, H, float(slope), ptr(out), stream()), "qot_nnconv_fwd")
        ctx.save_for_backward(yr, edge_attr, W1_, b1_, out)
        ctx.graph, ctx.slope = graph, float(slope)
        return out

    @staticmethod
    def backward(ctx, dout):
        L = _lib.lib()
        yr, edge_attr, W1, b1, out = ctx.saved_tensors
        g = ctx.graph
        csr, csr_t = g.csr, g.csr_t
        N = yr.shape[0]
        H = yr.shape[1] // (EDGE_HID + 2)
        E, dev = g.num_edges, yr.device
        dout = _f32(dout)
        dyr = torch.empty_like(yr)
        dW1, db1 = torch.empty_like(W1), torch.empty_like(b1)
        dbias = torch.empty(H, dtype=torch.float32, device=dev)
        ws = _ws(L.qot_nnconv_bwd_workspace_bytes(N, E, H), dev)
        check(L.qot_nnconv_bwd(ptr(yr), ptr(csr.rowptr), ptr(csr.nbr), ptr(csr.eid), ptr(csr_t.rowptr),
                               ptr(csr_t.nbr), ptr(csr_t.eid), ptr(edge_attr), ptr(W1), ptr(b1), ptr(out),
                               ptr(dout), N, E, H, ctx.slope, ptr(dyr), ptr(dW1), ptr(db1), ptr(dbias),
                               ptr(ws), ws.numel(), stream()), "qot_nnconv_bwd")
        return dyr, None, dW1, db1, dbias, None, None


def nnconv_mean(x, graph: GraphIndex, edge_attr, W1, b1, W2, b2, Wroot, bias, slope: float = 1.0):
    """NNConv(aggr='mean') in factorised form: one node-wise projection
    yr = x [P_0 .. P_7 | P_b | Wroot^T]  then the edge kernel (SURVEY.md A.2)."""
    H = x.shape[1]
    K = EDGE_HID
    # Pcat[i, k*H+o] = W2[i*H+o, k];  slab K: b2[i*H+o];  slab K+1: Wroot[o,i]   (tensor
    # reshuffles only -- autograd routes dPcat back to W2 / b2 / Wroot)
    PcatT = _derived("nnconv.P", (W2, b2, Wroot), lambda: torch.cat(
        [W2.view(H, H, K).permute(0, 2, 1).reshape(H, K * H), b2.view(H, H), Wroot.t()], dim=1).t().contiguous())
    yr = node_linear(x, PcatT, None)                      # W argument is [out,in]
    return _NNConvEdgeFn.apply(yr, edge_attr, W1, b1, bias, graph, slope)


# --------------------------------------------------------------------------- #
# TopologicalGNN, one block per graph (csrc/topo_fused.cu)
# --------------------------------------------------------------------------- #
def batch_max_sizes(data):
    """(largest node count, largest edge count) of a graph in the batch.  Collates of this package record
    them from host arrays; a foreign batch costs one device->host read, cached on the batch."""
    if getattr(data, "max_nodes", None) is not None and getattr(data, "max_edges", None) is not None:
        return int(data.max_nodes), int(data.max_edges)
    cache = batch_cache(data)
    if "max_sizes" not in cache:
        gptr = batch_graph_ptr(data)
        eptr = getattr(data, "edge_ptr", None)
        if eptr is None:
            if "eptr" not in cache:
                cache["eptr"] = edge_ptr(data.edge_index, data.batch, gptr.numel() - 1)
            eptr = cache["eptr"][0]
        if gptr.numel() < 2:
            cache["max_sizes"] = (0, 0)
        else:
            v = torch.stack([(gptr[1:] - gptr[:-1]).max(), (eptr[1:] - eptr[:-1]).max()]).tolist()
            cache["max_sizes"] = (int(v[0]), int(v[1]))
    return cache["max_sizes"]


class _TopoFusedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, flat, emb, node_ids, edge_index, edge_attr, gptr, eptr, nmax: int, emax: int,
                drop_mask=None, drop_scale: float = 1.0, drop_scale_head: float = 1.0):
        L = _lib.lib()
        B = int(gptr.numel() - 1)
        dev = flat.device
        flat_, emb_ = _f32(flat.detach()), _f32(emb.detach())
        node_ids, edge_index, edge_attr = _i64(node_ids), _i64(edge_index), _edge_attr(edge_attr)
        out = torch.empty(B, 3, dtype=torch.float32, device=dev)
        status = _track_status("qot_topo_fused (graph over the launch's node/edge caps, or ids out of range)",
                               torch.zeros(1, dtype=torch.int32, device=dev))
        prep = torch.empty(L.qot_topo_fused_prepared_floats(), dtype=torch.float32, device=dev)
        check(L.qot_topo_fused_prepare(ptr(flat_), ptr(prep), stream()), "qot_topo_fused_prepare")
        N, E = int(node_ids.shape[0]), int(edge_index.shape[1])
        saved = None                                     # forward state for the backward (training only)
        if any(ctx.needs_input_grad[:2]):
            saved = torch.empty(L.qot_topo_fused_saved_floats(N, E, B), dtype=torch.float32, device=dev)
        check(L.qot_topo_fused_fwd(ptr(prep), ptr(emb_), ptr(node_ids), ptr(edge_index), E,
                                   ptr(edge_attr), ptr(gptr), ptr(eptr), B, N, int(nmax), int(emax), int(emb_.shape[0]),
                                   ptr(out), ptr(saved), ptr(status), ptr(drop_mask), float(drop_scale),
                                   float(drop_scale_head), stream()), "qot_topo_fused_fwd")
        ctx.save_for_backward(prep, emb_, node_ids, edge_index, edge_attr, gptr, eptr, status, saved, drop_mask)
        ctx.sizes = (int(nmax), int(emax), float(drop_scale), float(drop_scale_head))
        return out

    @staticmethod
    def backward(ctx, dout):
        L = _lib.lib()
        prep, emb, node_ids, edge_index, edge_attr, gptr, eptr, status, saved, drop_mask = ctx.saved_tensors
        nmax, emax, drop_scale, drop_scale_head = ctx.sizes
        B = int(gptr.numel() - 1)
        dev = prep.device
        gflat = torch.empty(L.qot_topo_fused_params(), dtype=torch.float32, device=dev)
        gemb = torch.empty_like(emb)
        ws = _ws(L.qot_topo_fused_bwd_workspace_bytes(int(emb.shape[0])), dev)
        check(L.qot_topo_fused_bwd(ptr(prep), ptr(emb), ptr(node_ids), ptr(edge_index), int(edge_index.shape[1]),
                                   ptr(edge_attr), ptr(gptr), ptr(eptr), B, int(node_ids.shape[0]), nmax, emax,
                                   int(emb.shape[0]), ptr(_f32(dout)), ptr(saved), ptr(gflat), ptr(gemb), ptr(ws),
                                   ws.numel(), ptr(status), ptr(drop_mask), drop_scale, drop_scale_head, stream()),
              "qot_topo_fused_bwd")
        return gflat, gemb, None, None, None, None, None, None, None, None, None, None


TOPO_FUSED_SMEM_LIMIT = 227 * 1024


def topo_fused_fits(nmax: int, emax: int, num_nodes: int) -> bool:
    """Whether one graph of the batch fits one block's shared memory in the BACKWARD kernel (the larger one)."""
    P = _lib.lib().qot_topo_fused_params()
    floats = P + num_nodes * 16 + nmax * (16 * 10 + 144) + emax * (4 + 8 + 2 + 8) + 96
    nbytes = floats * 4 + 2 * (nmax + 1) * 4 + 4 * emax * 2 + 16
    return nmax <= 4096 and emax <= 512 and nbytes <= TOPO_FUSED_SMEM_LIMIT


def topo_fused_dropout_mask(num_nodes: int, num_graphs: int, p: float, p_head: float, device):
    """Masks for the fused training step, one byte per element: [N,16] after conv1 | [N,16] after conv2 | [B,16] in
    the head (1 = keep), drawn with torch's generator (graph-capture safe); returns (mask, scale, scale_head)."""
    n1 = 2 * num_nodes * 16
    mask = torch.empty(n1 + num_graphs * 16, dtype=torch.uint8, device=device)
    if p == p_head:
        mask.bernoulli_(1.0 - p)
    else:
        mask[:n1].bernoulli_(1.0 - p)
        mask[n1:].bernoulli_(1.0 - p_head)
    inv = lambda q: 0.0 if q >= 1.0 else 1.0 / (1.0 - q)
    return mask, inv(p), inv(p_head)


def topological_fused(params: Sequence[torch.Tensor], emb, node_ids, edge_index, edge_attr, gptr, eptr,
                      nmax: int, emax: int, drop_mask=None, drop_scale: float = 1.0, drop_scale_head: float = 1.0):
    """out [B,3] of TopologicalGNN (reference shape) with one launch forward / two backward.  `params` in the
    order of include/qot_b200.h (qot_topo_fused_fwd).  `drop_mask` (see topo_fused_dropout_mask): training-mode
    dropout inside the kernels."""
    flat = torch.cat([p.reshape(-1) for p in params] + [params[0].new_zeros(1)])
    return _TopoFusedFn.apply(flat, emb, node_ids, edge_index, edge_attr, gptr, eptr, nmax, emax,
                              drop_mask, drop_scale, drop_scale_head)


# --------------------------------------------------------------------------- #
# global_mean_pool + MLP head
# --------------------------------------------------------------------------- #
class _PoolMlpFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gptr, W1, b1, W2, b2, hmask):
        L = _lib.lib()
        x = _f32(x)
        N, H = x.shape
        B, dev = gptr.numel() - 1, x.device
        ts = [_f32(t.detach()) for t in (W1, b1, W2, b2)]
        pooled = torch.empty(B, H, dtype=torch.float32, device=dev)
        hid = torch.empty(B, H, dtype=torch.float32, device=dev)
        out = torch.empty(B, 3, dtype=torch.float32, device=dev)
        ws = _ws(L.qot_pool_mlp_fwd_workspace_bytes(N, B, H), dev)
        check(L.qot_pool_mlp_fwd(ptr(x), ptr(gptr), N, B, H, ptr(ts[0]), ptr(ts[1]), ptr(ts[2]), ptr(ts[3]),
                                 ptr(hmask), ptr(pooled), ptr(hid), ptr(out), ptr(ws), ws.numel(), stream()),
              "qot_pool_mlp_fwd")
        ctx.save_for_backward(gptr, ts[0], ts[2], pooled, hid, hmask)
        ctx.N = N
        return out

    @staticmethod
    def backward(ctx, dout):
        L = _lib.lib()
        gptr, W1, W2, pooled, hid, hmask = ctx.saved_tensors
        B, H = pooled.shape
        dev, N = pooled.device, ctx.N
        dout = _f32(dout)
        dx = torch.empty(N, H, dtype=torch.float32, device=dev)
        dW1, db1 = torch.empty_like(W1), torch.empty(H, dtype=torch.float32, device=dev)
        dW2, db2 = torch.empty_like(W2), torch.empty(3, dtype=torch.float32, device=dev)
        ws = _ws(L.qot_pool_mlp_bwd_workspace_bytes(B, H), dev)
        check(L.qot_pool_mlp_bwd(ptr(dout), ptr(pooled), ptr(hid), ptr(hmask), ptr(gptr), N, B, H, ptr(W1),
                                 ptr(W2), ptr(dx), ptr(dW1), ptr(db1), ptr(dW2), ptr(db2), ptr(ws), ws.numel(),
                                 stream()), "qot_pool_mlp_bwd")
        return dx, None, dW1, db1, dW2, db2, None


def pool_mlp(x, gptr, W1, b1, W2, b2, training: bool = False, dropout_p: float = 0.0):
    """global_mean_pool -> Linear -> LeakyReLU -> Dropout -> Linear
    (topological_training/models.py:61-63)."""
    _require_cuda(x, gptr)
    hmask = None
    if training and dropout_p > 0.0:
        keep = 1.0 - dropout_p
        hmask = (torch.rand(gptr.numel() - 1, x.shape[1], device=x.device) < keep).to(torch.float32) / keep
    if W2.shape[0] != 3:
        raise RuntimeError("libqot_b200 pool_mlp: out_channels must be 3 (osnr, snr, ber)")
    return _PoolMlpFn.apply(x, gptr, W1, b1, W2, b2, hmask)


def mean_pool(x, gptr):
    """global_mean_pool as its own layer (the fused form is ops.pool_mlp)."""
    _require_cuda(x, gptr)
    return _MeanPoolFn.apply(x, gptr)


# --------------------------------------------------------------------------- #
# fused SmoothL1 loss + running regression metrics
# --------------------------------------------------------------------------- #
class RegressionMetrics:
    """Device-side accumulator of the sums behind the reference's per-epoch numbers
    (topological_training/train.py:117-129): average loss and sklearn ``r2_score`` (uniform average
    over the three outputs).  Nothing is read on the host until :meth:`result`."""

    def __init__(self, device):
        self.sums = torch.zeros(3, 5, dtype=torch.float64, device=device)

    def reset(self) -> None:
        self.sums.zero_()

    def result(self) -> dict:
        s = self.sums.cpu()
        n, sy, syy, ssr, sl = (s[:, i] for i in range(5))
        ss_tot = syy - sy * sy / n.clamp(min=1)
        r2 = 1.0 - ssr / ss_tot
        return {"count": int(n[0]), "loss": float(sl.sum() / (n[0] * 3).clamp(min=1)),
                "mse": (ssr / n.clamp(min=1)).tolist(), "r2": r2.tolist(), "r2_uniform_average": float(r2.mean())}


class _SmoothL1Fn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, target, target_rows, beta, metrics):
        L = _lib.lib()
        pred, target = _f32(pred), _f32(target)
        n, dev = pred.shape[0], pred.device
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        dpred = torch.empty_like(pred)
        ws = _ws(L.qot_smooth_l1_workspace_bytes(n), dev)
        check(L.qot_smooth_l1(ptr(pred), ptr(target), ptr(target_rows), n, float(beta), ptr(loss), ptr(dpred),
                              ptr(metrics), ptr(ws), ws.numel(), stream()), "qot_smooth_l1")
        ctx.save_for_backward(dpred)
        return loss.view(())

    @staticmethod
    def backward(ctx, g):
        (dpred,) = ctx.saved_tensors
        return dpred * g, None, None, None, None


def smooth_l1_loss(pred, target, target_rows=None, beta: float = 1.0, metrics: Optional[RegressionMetrics] = None):
    """``torch.nn.SmoothL1Loss()(pred, target[target_rows])`` with the gradient computed in the same
    kernel and, optionally, the epoch metrics accumulated on the device."""
    _require_cuda(pred, target)
    if pred.dim() != 2 or pred.shape[1] != 3:
        raise RuntimeError("libqot_b200 smooth_l1_loss: predictions must be [n, 3] (osnr, snr, ber)")
    target = target.reshape(-1, 3)
    rows = _i64(target_rows) if target_rows is not None else None
    if rows is None and target.shape[0] != pred.shape[0]:
        raise RuntimeError("smooth_l1_loss: target rows do not match the predictions")
    return _SmoothL1Fn.apply(pred, target, rows, beta, metrics.sums if metrics is not None else None)
