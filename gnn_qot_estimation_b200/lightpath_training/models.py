"""LightpathGNN on the B200 kernels -- drop-in for lightpath_training/models.py:7-45.

Same constructor, ``forward(data) -> (out [L,3], lut_batch [L])``, same
``ValueError("No LUT node found in the batch.")`` and the same state_dict names as
the shipped checkpoints (``conv1.lin.weight``, ``conv1.att_src``, ``conv1.att_dst``,
``conv1.bias``, ``norm1.module.*``, ``mlp.0.*``, ``mlp.3.*``), so
``lightpath_training/test.py:63`` loads ``models/model_N.pth`` with strict=True.

eval(): one launch of the persistent kernel (csrc/lightpath_stream.cu) per batch -- or per MANY
batches through ``stream_plan`` / ``forward_stream``.  ``forward_every_node`` / ``stream_plan(..., every_node=True)``:
every node of a graph evaluated as the LUT in one pass (csrc/lightpath_every_node.cu).
train(): GAT forward -> batch statistics -> LUT head, with the matching backward
kernels (csrc/lightpath_train.cu) through ``torch.autograd.Function``.
"""
from __future__ import annotations

import torch
from torch.nn import Dropout, LeakyReLU, Linear

from .. import _lib, ops
from ..nn import BatchNorm, GATConv


class LightpathGNN(torch.nn.Module):
    dominant_kernel = "lp_stream_kernel"   # csrc/lightpath_stream.cu: eval forward, one launch for any number of batches

    def __init__(self, in_channels, hidden_channels, output_dim, is_lut_index, dropout_p=0.5):
        super().__init__()
        self.conv1 = GATConv(in_channels, hidden_channels, heads=4, concat=True)
        self.norm1 = BatchNorm(hidden_channels * 4)
        self.mlp = torch.nn.Sequential(
            Linear(hidden_channels * 4, hidden_channels),
            LeakyReLU(),
            Dropout(p=dropout_p),
            Linear(hidden_channels, output_dim),
        )
        self.is_lut_index = is_lut_index
        self._prepared = None
        self._prepared_key = None

    # ------------------------------------------------------------------ eval
    def _eval_params(self):
        bn = self.norm1.module
        return {
            "lin_w": self.conv1.lin.weight, "att_src": self.conv1.att_src, "att_dst": self.conv1.att_dst,
            "conv_bias": self.conv1.bias, "bn_w": bn.weight, "bn_b": bn.bias,
            "bn_mean": bn.running_mean, "bn_var": bn.running_var,
            "mlp_w1": self.mlp[0].weight, "mlp_b1": self.mlp[0].bias,
            "mlp_w2": self.mlp[3].weight, "mlp_b2": self.mlp[3].bias,
        }

    def prepared(self) -> torch.Tensor:
        """Folded eval-mode parameters, rebuilt only when a tensor changed."""
        ps = self._eval_params()
        key = tuple((t.data_ptr(), t._version) for t in ps.values())
        if self._prepared is None or key != self._prepared_key:
            self._prepared = ops.lightpath_prepare(ps, self.norm1.module.eps, self.is_lut_index)
            self._prepared_key = key
        return self._prepared

    @_lib.on_tensor_device
    def forward_device(self, data) -> ops.LightpathInferOut:
        """Eval forward of ONE batch without reading anything back: one launch of the persistent kernel
        (qot_lightpath_infer_stream, n_batches = 1) when the batch carries ``ptr`` / ``edge_ptr`` / ``lut_ptr``
        (every collate of this package provides them; a foreign batch gets them from qot_graph_ptr / qot_edge_ptr /
        qot_lightpath_lut_ptr first).  The plan (output buffers + device descriptor) is cached on the batch object."""
        from ..batch import Batch
        cache = ops.batch_cache(data)
        key = ("stream_plan", self.is_lut_index, data.x.data_ptr(), data.edge_index.data_ptr(),
               tuple(data.x.shape), tuple(data.edge_index.shape))
        plan = cache.get(key)
        if plan is None:
            gptr = ops.batch_graph_ptr(data)
            eptr = getattr(data, "edge_ptr", None)
            if eptr is None:
                if "eptr" not in cache:
                    cache["eptr"] = ops.edge_ptr(data.edge_index, data.batch, gptr.numel() - 1)
                eptr = cache["eptr"][0]
            lut_ptr = getattr(data, "lut_ptr", None)
            if lut_ptr is None or getattr(data, "lut_col", None) != self.is_lut_index:
                lut_ptr = ops.lightpath_lut_ptr(data.x, gptr, self.is_lut_index)
            view = Batch(x=data.x, edge_index=data.edge_index, ptr=gptr, edge_ptr=eptr, lut_ptr=lut_ptr,
                         num_graphs=int(gptr.numel() - 1), lut_col=self.is_lut_index,
                         sym_by_src=bool(getattr(data, "sym_by_src", False)))
            plan = cache[key] = ops.LightpathStreamPlan([view], self.is_lut_index)
        plan.launch(self.prepared())
        return plan.result(0)

    def stream_plan(self, batches, split_head: bool = False, every_node: bool = False) -> "ops.LightpathStreamPlan":
        """Plan for evaluating many resident batches with one launch of the persistent kernel each time
        ``forward_stream`` is called (the streaming form of lightpath_training/test.py:77-94).
        ``every_node``: every node of every graph as the LUT (see ``forward_every_node``)."""
        self._check_supported()
        return ops.LightpathStreamPlan(batches, self.is_lut_index, split_head, every_node)

    @_lib.on_tensor_device
    def forward_every_node(self, data) -> torch.Tensor:
        """QoT of every lightpath of every graph of ONE batch, one pass over each graph (eval mode only).

        Returns ``out [N, 3]``: row i is what ``forward`` under ``eval()`` returns for node i's graph, given a copy of
        that graph in which node i's flag column ``x[:, is_lut_index]`` is 1.0 and every other node's flag column is
        0.0.  Whatever the stored flag column holds (0, 1, several ones, any value) has no effect.  Rows are in node
        order; the graph of row i is ``data.batch[i]``.  From raw samples: ``to_graph.create_lightpath_graphs(...,
        return_conn_ids=True)``, then ``collate``, then this call -- row i is lightpath ``conn_ids[i]`` of sample
        ``batch[i]``.  Foreign batches (PyG / pyg_compat) get ``ptr`` / ``edge_ptr`` derived; their edges must be
        grouped by graph.  The plan (output buffer + device descriptor) is cached on the batch object; the call reads
        one status word back (a synchronisation) and raises on malformed input."""
        if self.training:
            raise RuntimeError("LightpathGNN.forward_every_node is eval-only (in training mode BatchNorm couples the "
                               "nodes): call model.eval()")
        if not data.x.is_cuda or not data.edge_index.is_cuda:
            raise RuntimeError("LightpathGNN (B200) needs the batch on a CUDA device; there is no CPU path")
        self._check_supported()
        from ..batch import Batch
        cache = ops.batch_cache(data)
        key = ("every_node_plan", self.is_lut_index, data.x.data_ptr(), data.edge_index.data_ptr(),
               tuple(data.x.shape), tuple(data.edge_index.shape))
        plan = cache.get(key)
        if plan is None:
            gptr = ops.batch_graph_ptr(data)
            eptr = getattr(data, "edge_ptr", None)
            if eptr is None:
                if "eptr" not in cache:
                    cache["eptr"] = ops.edge_ptr(data.edge_index, data.batch, gptr.numel() - 1)
                eptr = cache["eptr"][0]
            view = Batch(x=data.x, edge_index=data.edge_index, batch=getattr(data, "batch", None), ptr=gptr,
                         edge_ptr=eptr, num_graphs=int(gptr.numel() - 1),
                         sym_by_src=bool(getattr(data, "sym_by_src", False)))
            plan = cache[key] = ops.LightpathStreamPlan([view], self.is_lut_index, every_node=True)
        plan.launch(self.prepared())
        flags = [plan.status[:1]]
        if getattr(data, "edge_ptr", None) is None:
            flags.append(cache["eptr"][1])                         # "edges grouped by graph" check
        vals = torch.cat(flags).tolist()                          # the one D2H of this call
        if len(vals) > 1 and vals[1]:
            raise RuntimeError("LightpathGNN.forward_every_node: the batch's edges are not grouped by graph "
                               "(every-node mode reads each graph's edges as one contiguous range)")
        if vals[0]:
            raise RuntimeError("LightpathGNN.forward_every_node: malformed graph offsets (ptr / edge_ptr outside "
                               "the batch)")
        return plan.result(0).out.clone()                         # the plan's buffer is reused by the next call

    @_lib.on_tensor_device
    def forward_candidates(self, state, cands, max_impact: int = 64) -> "ops.CandidateQoT":
        """QoT of candidate lightpaths against a network state, and what each candidate does to the lightpaths
        already set up (eval mode only; csrc/lightpath_candidates.cu).

        ``state``: ``to_graph.lightpath_network_state(data, freqs, lp_feat)``; ``cands``: ``to_graph.LightpathCandidates``
        on the state's device.  For candidate k, let sample' be sample ``cands.sample[k]`` with the candidate written
        into every channel of its path and slot range (a new conn_id, features ``cands.feat[k]``, unknown metrics).  In
        sample''s lightpath graph with the flag column ``x[:, is_lut_index]`` one-hot:
        ``out[k]`` is ``forward`` under ``eval()`` with the flag at the candidate; ``impact_out[k, i]`` is the same with
        the flag at the i-th lightpath the candidate interferes with (``impact_node[k, i]``, a node of ``state.batch``,
        ascending) -- compare it with ``forward_every_node(state.batch)`` for the "before" value.  Candidates are
        evaluated independently, each against the state alone.  ``status`` holds ``ops.CAND_*`` bits: a bad sample,
        a bad path or slot range, or an occupied channel gives a NaN row and no impact rows; more than ``max_impact``
        neighbours keeps the first ``max_impact`` rows and reports the true count in ``n_impact``.
        One launch, nothing read back: capturable in a CUDA graph.  Malformed arguments raise on the host."""
        self._check_state_query("forward_candidates", state)
        return ops.lightpath_candidates(state, cands, self.prepared(), self.is_lut_index, max_impact)

    @_lib.on_tensor_device
    def forward_reconfigurations(self, state, changes, max_impact: int = 64) -> "ops.ReconfigQoT":
        """QoT after moving, retuning, rerouting or tearing down a lightpath of a network state, and what each change
        does to the other lightpaths (eval mode only; csrc/lightpath_candidates.cu, qot_lightpath_reconfigure).

        ``changes``: ``to_graph.LightpathChanges`` on the state's device (``to_graph.lightpath_nodes`` turns conn_ids
        into its ``node`` entries).  For change k with moved lightpath j (conn_id c), let sample' be sample
        ``changes.sample[k]`` with every channel of c cleared and, unless the path is empty (a teardown), j written on
        every channel of the new path and slot range with features ``changes.feat[k]`` (its other rows as on its first
        channel).  In sample''s lightpath graph with the flag column one-hot: ``out[k]`` is ``forward`` under ``eval()``
        with the flag at j (NaN for a teardown); ``impact_out[k, r]`` is the same with the flag at ``impact_node[k, r]``,
        each lightpath that was or is adjacent to j, ascending, and ``impact_kind[k, r]`` says which (``ops.KIND_LOST``
        1, ``KIND_GAINED`` 2, ``KIND_KEPT`` 3).  Every other lightpath's QoT is unchanged:
        ``forward_every_node(state.batch)`` gives it.  ``node[k] = -1`` is an insertion, bit-identical to
        ``forward_candidates``.  Changes are evaluated independently, each against the state alone.  ``status`` holds
        ``ops.CAND_*`` bits (``CAND_BAD_NODE``: the node is not in the sample; j's own channels are not OCCUPIED).
        One launch, nothing read back: capturable in a CUDA graph.  Malformed arguments raise on the host."""
        self._check_state_query("forward_reconfigurations", state)
        return ops.lightpath_reconfigure(state, changes, self.prepared(), self.is_lut_index, max_impact)

    @_lib.on_tensor_device
    def forward_change_sets(self, state, changes, set_ptr, max_impact: int = 64) -> "ops.ChangeSetQoT":
        """QoT after several changes to one sample applied together -- batch provisioning, defragmentation with swaps,
        failure restoration -- and what each set does to the other lightpaths (eval mode only;
        csrc/lightpath_candidates.cu, qot_lightpath_change_sets).

        ``changes``: ``to_graph.LightpathChanges`` as for ``forward_reconfigurations``; ``set_ptr`` [G+1] int64 on the
        state's device: set g is changes ``[set_ptr[g], set_ptr[g+1])``, all naming one sample, at most
        ``ops.SET_MAX_CHANGES``.  sample' = the sample with every lightpath the set moves or tears down cleared, then
        every non-teardown change written on its path and slots (a move keeps its conn_id and other rows; an insertion
        gets a new conn_id, one above the sample's largest, +1 per insertion in set order).  In sample''s lightpath graph
        with the flag column one-hot: ``out[k]`` is the changed lightpath's row (NaN for a teardown);
        ``impact_out[g, r]`` is the row of ``impact_node[g, r]``, each lightpath the set does not move that is adjacent
        to a changed lightpath before or after it, ascending, with ``impact_kind[g, r]`` bit 0 (it loses a neighbour)
        | bit 1 (a changed lightpath is its neighbour now).  Every other lightpath's QoT is unchanged:
        ``forward_every_node(state.batch)`` gives it.  A channel is occupied only by a lightpath the set does not move,
        so swaps are legal.  ``status`` holds ``ops.CAND_*`` and ``ops.SET_*`` bits per change, ``set_status`` their
        OR; any bit but ``CAND_IMPACT_OVERFLOW`` makes the whole set NaN with ``n_impact`` 0.  A set of one change is
        bit-identical to ``forward_reconfigurations``.  One launch, nothing read back: capturable in a CUDA graph.
        Malformed arguments raise on the host."""
        self._check_state_query("forward_change_sets", state)
        return ops.lightpath_change_sets(state, changes, set_ptr, self.prepared(), self.is_lut_index, max_impact)

    @_lib.on_tensor_device
    def forward_placements(self, state, demands, policy: int, metric: int = 0, maximize: bool = True, bound=None,
                           max_impact: int = 64, return_all: bool = False) -> "ops.PlacementQoT":
        """QoT-aware placement of lightpath demands: for each demand, the free slot range on one of its routes that a
        policy picks among those whose predicted QoT meets its bounds (eval mode only; csrc/lightpath_candidates.cu,
        qot_lightpath_placements).

        ``demands``: ``to_graph.LightpathDemands`` on the state's device.  A placement of demand d is an option p
        (route, width, features) with a start slot q0 such that ``[q0, q0 + width)`` is free on every link of the
        route; its rows are, by definition, what ``forward_candidates`` returns for the candidate (sample, route, q0,
        width, feat = (float32(state.freqs[q0]), mod_order, num_spans, path_len)).  A row's margin on output column
        ``metric`` is ``v - b`` if ``maximize`` (OSNR, SNR) and ``b - v`` otherwise (BER), in fp32, with b the
        option's ``own_bound`` for the own row and ``bound[node]`` (``bound`` [N] float32 over ``state.batch``'s
        nodes, or None: impact rows unconstrained) for every impact row, whatever ``max_impact`` is.  The placement's
        margin is the minimum over its rows, and it is feasible iff that is >= 0 (never when NaN).  ``policy``:
        ``ops.PLACE_FIRST_FIT`` (the first feasible placement in (option, q0) order), ``ops.PLACE_BEST_QOT`` (the best
        own value) or ``ops.PLACE_MAX_MARGIN`` (the largest margin); ties go to the lower option, then the lower q0.
        Returns ``ops.PlacementQoT``: ``option`` (relative to the demand's first option) and ``q0`` (-1 if none is
        feasible), the chosen own row ``out`` and ``margin`` (NaN if none), ``n_free`` / ``n_feasible`` over every
        placement of the demand, ``status`` (``ops.CAND_*``: a bad sample, a bad route, width or option range, or a
        bad state give -1 / NaN and zero counts; ``CAND_IMPACT_OVERFLOW`` applies to the chosen placement) and the
        chosen placement's impact rows laid out as in ``forward_candidates``.  ``return_all``: also ``all_out`` [P, Q,
        3] and ``all_margin`` [P, Q], every free placement's own row and margin, NaN at the other slots of the demands'
        options.  Q is at most ``ops.PLACE_MAX_SLOTS``.  One launch, nothing read back: capturable in a CUDA graph.
        Malformed arguments raise on the host."""
        self._check_state_query("forward_placements", state)
        return ops.lightpath_placements(state, demands, policy, metric, maximize, bound, self.prepared(),
                                        self.is_lut_index, max_impact, return_all)

    @_lib.on_tensor_device
    def forward_provision(self, state, demands, policy: int, metric: int = 0, maximize: bool = True, bound=None,
                          max_impact: int = 64) -> "ops.ProvisionQoT":
        """Sequential provisioning of lightpath demands (eval mode only; csrc/lightpath_candidates.cu,
        qot_lightpath_provision): the demands of each sample are placed in increasing index, each against the state
        with the sample's earlier accepted demands set up.  Samples are independent; their demands may be interleaved.

        Demand d is placed exactly as ``forward_placements`` places it against ``state_d`` =
        ``lightpath_network_state(data_d, ...)``, where ``data_d`` is the raw samples with every earlier accepted demand
        of d's sample written in as ``forward_candidates`` writes a candidate: the chosen route x ``[q0, q0 + width)``,
        conn_id one above the sample's largest (top + 1, top + 2, ... for successive acceptances), ``freq =
        float32(freqs[q0])``, the option's (mod_order, num_spans, path_len), osnr = snr = ber = -1, other rows 0.
        With a ``bound`` ([N] float32 over ``state.batch``'s nodes), an accepted demand is bound from then on by its
        option's ``own_bound``: a later placement that would take it below is infeasible; with ``bound=None`` impact
        rows are unconstrained.  A demand is accepted when it has a feasible placement and no status bit but
        ``CAND_IMPACT_OVERFLOW``; otherwise it commits nothing and the sample's later demands go on.

        Returns ``ops.ProvisionQoT``: the fields of ``ops.PlacementQoT`` but ``all_out`` / ``all_margin``,
        bit-identical to ``forward_placements(state_d, ...)`` for that demand, with the impact rows named by conn_id
        (``impact_conn``, since node numbers change as lightpaths are added) and ``conn_id`` [D], the id the demand
        was accepted under (-1 if not).  Status bits on top of ``ops.CAND_*``: ``ops.PROV_FULL`` (accepting would take
        the sample past 256 lightpaths or 6144 occupied channels, which the graph builder refuses: not accepted, the
        placement still reported).  ``state`` is not modified; ``to_graph.commit_provision`` writes the accepted
        demands into the samples.  One copy and one launch, nothing read back: capturable in a CUDA graph.  Malformed
        arguments raise on the host."""
        self._check_state_query("forward_provision", state)
        return ops.lightpath_provision(state, demands, policy, metric, maximize, bound, self.prepared(),
                                       self.is_lut_index, max_impact)

    @_lib.on_tensor_device
    def forward_stream(self, plan, first: int = 0, count=None) -> None:
        """Enqueues batches [first, first+count) of ``plan`` (eval mode; no host synchronisation)."""
        if self.training:
            raise RuntimeError("LightpathGNN.forward_stream is the eval-mode forward: call model.eval()")
        plan.launch(self.prepared(), first, count)

    def _forward_eval(self, data):
        self._check_supported()
        res = self.forward_device(data)
        flags = [res.n_lut, res.status]
        if getattr(data, "edge_ptr", None) is None:
            flags.append(ops.batch_cache(data)["eptr"][1])      # "edges grouped by graph" check
        vals = torch.cat(flags).tolist()                          # the one D2H of this forward
        n_lut, stale = vals[0], vals[1]
        if len(vals) > 2 and vals[2]:
            return self._forward_general(data)                    # CSR path handles any edge order
        if stale:
            raise RuntimeError("LightpathGNN: the batch's lut_ptr does not match x[:, is_lut_index] "
                               "(stale or foreign index array)")
        if n_lut == 0:
            raise ValueError("No LUT node found in the batch.")
        return res.out[:n_lut].clone(), res.lut_batch[:n_lut].clone()   # the plan's buffers are reused by the next call

    def _check_state_query(self, who: str, state):
        """The checks every network-state query makes first: eval mode, the state on CUDA, the supported shape."""
        if self.training:
            raise RuntimeError(f"LightpathGNN.{who} is eval-only (in training mode BatchNorm couples the nodes): "
                               "call model.eval()")
        if not state.batch.x.is_cuda:
            raise RuntimeError("LightpathGNN (B200) needs the network state on a CUDA device; there is no CPU path")
        self._check_supported()

    def _check_supported(self):
        c = self.conv1
        if (c.in_channels, c.out_channels, c.heads) != (5, 32, 4) or self.mlp[0].out_features != 32 \
                or self.mlp[3].out_features != 3:
            raise RuntimeError("libqot_b200 implements the reference LightpathGNN shape only: "
                               "in_channels=5, hidden_channels=32, heads=4, output_dim=3")

    # ----------------------------------------------------------- train/general
    def _forward_general(self, data):
        self._check_supported()
        h = self.conv1(data.x, data.edge_index)
        out, lut_batch = ops.lut_bn_head(
            h, data.x, data.batch, self.is_lut_index, self.norm1.module,
            self.mlp[0].weight, self.mlp[0].bias, self.mlp[3].weight, self.mlp[3].bias,
            self.training, self.mlp[2].p if self.training else 0.0,
            getattr(data, "lut_rows", None) if getattr(data, "lut_col", None) == self.is_lut_index else None)
        return out, lut_batch

    @_lib.on_tensor_device
    def forward(self, data):
        if not data.x.is_cuda:
            raise RuntimeError("LightpathGNN (B200) needs the batch on a CUDA device; there is no CPU path")
        needs_grad = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        if self.training or needs_grad:
            return self._forward_general(data)
        return self._forward_eval(data)
