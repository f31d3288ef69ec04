"""GPU parity of the TopologicalGNN training step at the shapes it trains on (DESIGN §4.13).

The fused kernels (csrc/topo_fused.cu) are persistent: graph g runs in block g % grid, and the grid is smaller than the
batch whenever shared memory allows fewer blocks than graphs (tests/topo_batches.grids).  test_topological_gpu.py
gives every block at most one graph; here a block takes two or more, so the gradient accumulators carried from graph
to graph, the saved-state offsets and dropout masks of later graphs, a small graph after a large one in the same
shared memory and a partial reduction over 740 block partials all run.  Every fused case is compared with the fp64
TopologicalGNNOracle (run on the GPU: it is device-agnostic) -- out, loss and every gradient including the embedding
table -- with the layer-by-layer kernels (at dropout 0: at 0.5 the layer path draws its own masks), and with a second
fused run, which must be bit-identical.  The fused SGD update (csrc/ddp_step.cu) is compared with torch.optim.SGD bit
for bit over its whole option matrix.  Tolerance: 1e-5 relative (BASELINE.json north_star), RTOL below."""
import copy

import pytest
import torch

import topo_batches as TB
from conftest import grad_errs, rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-5
ZERO = ("conv1.lin_key.bias",)      # exactly-zero gradient (softmax shift invariance), see conftest.grad_errs


def _models(cuda, num_nodes, p, seed):
    from gnn_qot_estimation_b200 import TopologicalGNN
    from oracle import TopologicalGNNOracle
    torch.manual_seed(seed)
    m = TopologicalGNN(num_nodes, 16, 3, edge_dim=4, dropout_p=p)
    with torch.no_grad():
        m.conv2.bias.normal_(0, 0.1)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    oracles = []
    for dt in (torch.float64, torch.float32):
        o = TopologicalGNNOracle(num_nodes, 16, 3, 4, dropout_p=p).to(dt)
        o.load_state_dict(sd, strict=True)
        oracles.append(o.to(cuda).eval())            # masks, when any, are replayed explicitly
    return m.to(cuda).train(), oracles[0], oracles[1]


def _run(m, b, fused=True):
    m.use_fused = fused
    m.zero_grad(set_to_none=True)
    out = m(b)
    loss = torch.nn.SmoothL1Loss()(out, b.y.view(-1, 3))
    loss.backward()
    return out.detach().clone(), loss.detach().clone(), {k: q.grad.detach().clone() for k, q in m.named_parameters()}


def _oracle(o, b, masks=None):
    dt = next(o.parameters()).dtype
    ob = copy.copy(b)
    ob.edge_attr = b.edge_attr.to(dt)
    o.zero_grad(set_to_none=True)
    out = o(ob, masks=masks)
    loss = torch.nn.SmoothL1Loss()(out, b.y.view(-1, 3).to(dt))
    loss.backward()
    return out.detach(), loss.detach(), {k: q.grad.detach() for k, q in o.named_parameters()}


@pytest.fixture
def fused_calls(monkeypatch):
    """Records every call of ops.topological_fused (the model's fused path), so a test can assert which path ran."""
    from gnn_qot_estimation_b200 import ops
    calls, real = [], ops.topological_fused

    def counting(*a, **k):
        calls.append((a, k))
        return real(*a, **k)
    monkeypatch.setattr(ops, "topological_fused", counting)
    return calls


def _grad_check(grads, ref64, ref32, hatch=()):
    """Every gradient within RTOL of the fp64 oracle; a tensor named in `hatch` may instead be no worse than twice the
    fp32 oracle (conftest.grad_parity's rule, applied to that tensor only)."""
    ours = grad_errs(grads, ref64, exact_zero=ZERO)
    fp32 = grad_errs(ref32, ref64, exact_zero=ZERO)
    for k, e in ours.items():
        bar = max(RTOL, 2.0 * fp32[k]) if k in hatch else RTOL
        assert e <= bar, (k, e, fp32[k])
    return ours, fp32


def _check_fused_case(label, m, o64, o32, b, p, calls, hatch=()):
    """The three comparisons of a fused training step (see the module docstring); returns the worst gradient errors."""
    n0 = len(calls)
    of, lf, gf = _run(m, b)
    assert len(calls) == n0 + 1, "the fused path did not run"
    masks = None
    if p > 0:
        mask, N, B, s = m.last_dropout_mask, b.num_nodes, b.num_graphs, 1.0 / (1.0 - p)
        assert mask.numel() == 2 * N * 16 + B * 16
        masks = (mask[:N * 16].view(N, 16), mask[N * 16:2 * N * 16].view(N, 16), mask[2 * N * 16:].view(B, 16), s, s)
        b.dropout_mask = (mask, s, s)                # the second run replays the same masks
    of2, lf2, gf2 = _run(m, b)
    if p > 0:
        del b.dropout_mask
    assert torch.equal(of, of2) and torch.equal(lf, lf2)
    for k in gf:
        assert torch.equal(gf[k], gf2[k]), k
    eo, el, eg = _oracle(o64, b, masks)
    _, _, fg = _oracle(o32, b, masks)
    assert rel_err(of, eo) <= RTOL and rel_err(lf, el) <= RTOL
    ours, fp32 = _grad_check(gf, eg, fg, hatch)
    if p == 0:
        ol, ll, gl = _run(m, b, fused=False)
        m.use_fused = True
        assert len(calls) == n0 + 2, "the layer path called the fused kernels"
        assert rel_err(of, ol) <= RTOL and rel_err(lf, ll) <= RTOL
        for k, e in grad_errs(gf, gl, exact_zero=ZERO).items():
            assert e <= RTOL, ("layer path", k, e)
    worst = max(ours, key=ours.get)
    print(f"\n{label}: worst gradient error vs fp64 {ours[worst]:.2e} ({worst}); fp32 oracle {max(fp32.values()):.2e}")
    return ours


def _nsfnet(cuda, B, seed):
    from gnn_qot_estimation_b200 import synthetic
    return synthetic.nsfnet_store(B, seed=seed).to(cuda).collate(range(0, B))


@pytest.mark.parametrize("p", [0.0, 0.5])
def test_cfg3_train_step(cuda, fused_calls, p):
    """BASELINE cfg 3 exactly: 1 024 NSFNET graphs in train(); the backward grid is 740 blocks, 284 of which take
    two graphs, and the partial reduction sums 740 partials."""
    assert TB.grids(1024, 14, 42, 14) == (1024, 740)
    m, o64, o32 = _models(cuda, 14, p, seed=31)
    _check_fused_case(f"cfg3 p={p}", m, o64, o32, _nsfnet(cuda, 1024, seed=12), p, fused_calls)


def test_4096_nsfnet_train_step(cuda, fused_calls):
    """4 096 NSFNET graphs: more than 2 x 8 x 148, so both kernels give every block at least two graphs for any
    per-SM block count up to 8."""
    assert 4096 > 2 * 8 * 148
    m, o64, o32 = _models(cuda, 14, 0.0, seed=32)
    _check_fused_case("4096 NSFNET", m, o64, o32, _nsfnet(cuda, 4096, seed=13), 0.0, fused_calls)


@pytest.mark.parametrize("p", [0.0, 0.5])
def test_ragged_75_node_train_step(cuda, fused_calls, p):
    """600 graphs of 1..75 nodes in mixed order (tests/topo_batches.ragged75: hubs, isolated nodes, self loops,
    repeated edges and node ids, 1-node graphs without edges) on the 75-row table: 148 blocks of 4-5 graphs each,
    larger graphs followed by smaller ones and the reverse."""
    assert TB.grids(600, 75, 300, 75) == (296, 148)
    m, o64, o32 = _models(cuda, TB.RAGGED_TABLE, p, seed=33)
    _check_fused_case(f"ragged75 p={p}", m, o64, o32, TB.ragged75().to(cuda), p, fused_calls)


def test_512_edge_graph_at_the_fits_edge(cuda, fused_calls):
    """A 128-node graph of 512 edges (a destination and a source of degree >= 420) on a 128-row table is the largest
    the fused path admits: the CSR's fourth edge slot (edges 384..511) and 420-edge in- and out-rows run.  The same
    batch with one more edge in that graph takes the layer path and still matches the oracle."""
    from gnn_qot_estimation_b200 import ops
    m, o64, o32 = _models(cuda, TB.EDGE512_TABLE, 0.0, seed=34)
    b = TB.edge512().to(cuda)
    assert (b.max_nodes, b.max_edges) == (128, 512) and ops.topo_fused_fits(128, 512, TB.EDGE512_TABLE)
    _check_fused_case("512 edges", m, o64, o32, b, 0.0, fused_calls)
    b = TB.edge512(extra_edges=1).to(cuda)
    assert not ops.topo_fused_fits(128, 513, TB.EDGE512_TABLE)
    n0 = len(fused_calls)
    out, loss, grads = _run(m, b)
    assert len(fused_calls) == n0, "a 513-edge graph took the fused path"
    eo, el, eg = _oracle(o64, b)
    _, _, fg = _oracle(o32, b)
    assert rel_err(out, eo) <= RTOL and rel_err(loss, el) <= RTOL
    _grad_check(grads, eg, fg)


def _direct_fused(args, use_saved, dout):
    """qot_topo_fused_fwd + qot_topo_fused_bwd called directly with the arguments the model passed to
    ops.topological_fused; the backward restores the forward's saved state or, given saved = NULL, recomputes it."""
    from gnn_qot_estimation_b200 import _lib, ops
    from gnn_qot_estimation_b200._lib import check, ptr, stream
    (params, emb, node_ids, edge_index, edge_attr, gptr, eptr, nmax, emax, drop_mask, ds, dsh), _ = args
    L = _lib.lib()
    dev = emb.device
    flat = torch.cat([q.detach().reshape(-1) for q in params] + [params[0].new_zeros(1)])
    emb, node_ids, edge_index, edge_attr = emb.detach().contiguous(), ops._i64(node_ids), ops._i64(edge_index), \
        ops._edge_attr(edge_attr)
    gptr, eptr = ops._i64(gptr), ops._i64(eptr)
    B, N, E, T = int(gptr.numel() - 1), int(node_ids.numel()), int(edge_index.shape[1]), int(emb.shape[0])
    prep = torch.empty(L.qot_topo_fused_prepared_floats(), dtype=torch.float32, device=dev)
    check(L.qot_topo_fused_prepare(ptr(flat), ptr(prep), stream()), "prepare")
    out = torch.empty(B, 3, dtype=torch.float32, device=dev)
    saved = torch.empty(L.qot_topo_fused_saved_floats(N, E, B), dtype=torch.float32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    check(L.qot_topo_fused_fwd(ptr(prep), ptr(emb), ptr(node_ids), ptr(edge_index), E, ptr(edge_attr), ptr(gptr),
                               ptr(eptr), B, N, nmax, emax, T, ptr(out), ptr(saved), ptr(status), ptr(drop_mask),
                               ds, dsh, stream()), "fwd")
    gflat = torch.empty(L.qot_topo_fused_params(), dtype=torch.float32, device=dev)
    gemb = torch.empty_like(emb)
    ws = torch.empty(L.qot_topo_fused_bwd_workspace_bytes(T), dtype=torch.uint8, device=dev)
    check(L.qot_topo_fused_bwd(ptr(prep), ptr(emb), ptr(node_ids), ptr(edge_index), E, ptr(edge_attr), ptr(gptr),
                               ptr(eptr), B, N, nmax, emax, T, ptr(dout), ptr(saved) if use_saved else None,
                               ptr(gflat), ptr(gemb), ptr(ws), ws.numel(), ptr(status), ptr(drop_mask), ds, dsh,
                               stream()), "bwd")
    assert int(status) == 0
    return out, gflat, gemb


@pytest.mark.parametrize("p", [0.0, 0.5])
@pytest.mark.parametrize("batch", ["cfg3", "ragged75"])
def test_recomputed_backward_equals_restored(cuda, fused_calls, batch, p):
    """qot_topo_fused_bwd with saved = NULL recomputes the forward of every graph (dropout masks included) instead
    of restoring it: the gradients must be bit-identical to the restoring backward's."""
    num_nodes = 14 if batch == "cfg3" else TB.RAGGED_TABLE
    m, _, _ = _models(cuda, num_nodes, p, seed=35)
    b = _nsfnet(cuda, 1024, seed=14) if batch == "cfg3" else TB.ragged75().to(cuda)
    out_model = m(b).detach()
    args = fused_calls[-1]
    dout = torch.randn(b.num_graphs, 3, generator=torch.Generator(device=cuda).manual_seed(5), device=cuda) * 1e-3
    o1, gf1, ge1 = _direct_fused(args, True, dout)
    o2, gf2, ge2 = _direct_fused(args, False, dout)
    assert torch.equal(o1, out_model) and torch.equal(o1, o2)
    assert torch.equal(gf1, gf2) and torch.equal(ge1, ge2)
    assert bool(gf1.abs().max() > 0) and bool(ge1.abs().max() > 0)


def test_eval_no_grad_forward_4096(cuda, fused_calls):
    """eval() + no_grad at 4 096 NSFNET graphs: the forward kernel alone (no saved state), 1 036 blocks."""
    m, o64, _ = _models(cuda, 14, 0.5, seed=36)
    m.eval()
    b = _nsfnet(cuda, 4096, seed=15)
    with torch.no_grad():
        out = m(b)
        ob = copy.copy(b)
        ob.edge_attr = b.edge_attr.double()
        eo = o64(ob)
    assert len(fused_calls) == 1
    assert rel_err(out, eo) <= RTOL


def test_understated_caps_are_reported_and_leave_nan(cuda, fused_calls, monkeypatch):
    """A batch whose max_nodes / max_edges understate its largest graph: the fused kernels skip the graphs over the
    caps, set the status word ops.check_status() raises on, and write NaN (not stale memory) into their output rows;
    every other row still matches the oracle."""
    from gnn_qot_estimation_b200 import ops
    # only this test's status words: earlier tests feed malformed inputs on purpose and leave their words set
    monkeypatch.setattr(ops, "_status_words", {})
    m, o64, _ = _models(cuda, TB.RAGGED_TABLE, 0.0, seed=37)
    m.eval()
    b = TB.ragged75().to(cuda)
    n = (b.ptr[1:] - b.ptr[:-1]).cpu()
    e = (b.edge_ptr[1:] - b.edge_ptr[:-1]).cpu()
    b.max_nodes, b.max_edges = 60, 200
    over = (n > 60) | (e > 200)
    assert bool(((n > 60) & (e <= 200)).any()) and bool(((n <= 60) & (e > 200)).any()) and bool((~over).any())
    torch.full((b.num_graphs, 3), 7.0, device=cuda)           # leaves finite values in the allocator's free block
    with torch.no_grad():
        out = m(b).cpu()
        ob = copy.copy(b)
        ob.edge_attr = b.edge_attr.double()
        eo = o64(ob).cpu()
    assert len(fused_calls) == 1
    assert torch.isnan(out[over]).all() and torch.isfinite(out[~over]).all()
    assert rel_err(out[~over], eo[~over]) <= RTOL
    with pytest.raises(RuntimeError, match="qot_topo_fused"):
        ops.check_status()


# ---- fused SGD update (ddp_sgd_step_kernel at world 1) against torch.optim.SGD's default (foreach) implementation
_WD = (0.0, 5e-4, 1e-2)
SGD_CASES = ([dict(momentum=0.0, weight_decay=wd) for wd in _WD]
             + [dict(momentum=0.9, dampening=d, weight_decay=wd) for d in (0.0, 0.1, 0.9, 0.99, 1 / 3) for wd in _WD]
             + [dict(momentum=0.9, nesterov=True, weight_decay=wd) for wd in _WD]
             + [dict(momentum=mo, maximize=True, weight_decay=wd) for mo in (0.0, 0.9) for wd in (0.0, 5e-4)]
             + [dict(momentum=0.9, nesterov=True, weight_decay=5e-4, maximize=True)])


def _sgd_id(h):
    return "-".join(f"{k}={v:.3g}" if isinstance(v, float) else k for k, v in h.items())


@pytest.mark.parametrize("resumed", [False, True], ids=["fresh", "resumed"])
@pytest.mark.parametrize("hyper", SGD_CASES, ids=_sgd_id)
def test_fused_sgd_matches_torch_bit_for_bit(cuda, hyper, resumed):
    """FusedSGDStep on the TopologicalGNN parameter list, 5 steps of gradients spanning 1e-8..1e2 (either sign), with
    an lr change through sync_hyper() before step 4: parameters and momentum buffers torch.equal to torch.optim.SGD's
    after every step.  `resumed`: both optimizers start from the state of two earlier torch steps."""
    from gnn_qot_estimation_b200 import TopologicalGNN
    from gnn_qot_estimation_b200.distributed import FlatGradBuffer, FusedSGDStep
    torch.manual_seed(0)
    m1 = TopologicalGNN(14, 16, 3, edge_dim=4, dropout_p=0.0).to(cuda)
    o1 = torch.optim.SGD(m1.parameters(), lr=0.1, **hyper)
    gen = torch.Generator(device=cuda).manual_seed(1)

    def draw():
        return [torch.pow(10.0, torch.rand(q.shape, generator=gen, device=cuda) * 10 - 8) *
                torch.where(torch.rand(q.shape, generator=gen, device=cuda) < 0.5, -1.0, 1.0) for q in m1.parameters()]
    if resumed:
        for _ in range(2):
            for q, g in zip(m1.parameters(), draw()):
                q.grad = g
            o1.step()
    m2 = copy.deepcopy(m1)
    o2 = torch.optim.SGD(m2.parameters(), lr=0.1, **hyper)
    if resumed:
        o2.load_state_dict(copy.deepcopy(o1.state_dict()))
    flat = FlatGradBuffer(m2.parameters())
    fused = FusedSGDStep(o2, flat, distributed=False)
    assert fused.had_state == (resumed and hyper["momentum"] != 0)
    for step in range(5):
        if step == 3:
            for o in (o1, o2):
                o.param_groups[0]["lr"] = 0.037
            fused.sync_hyper()
        gs = draw()
        for q1, q2, g in zip(m1.parameters(), m2.parameters(), gs):
            q1.grad, q2.grad = g.clone(), g.clone()
        flat.gather()
        o1.step()
        fused.step()
        for (k, q1), q2 in zip(m1.named_parameters(), m2.parameters()):
            assert torch.equal(q1, q2), (step, k)
            if hyper["momentum"] != 0:
                assert torch.equal(o1.state[q1]["momentum_buffer"], o2.state[q2]["momentum_buffer"]), (step, k)
    assert int(fused.status) == 0


@pytest.mark.parametrize("hyper", [dict(momentum=0.9, dampening=0.9),
                                   dict(momentum=0.9, nesterov=True, weight_decay=5e-4, maximize=True)], ids=_sgd_id)
def test_graphed_cfg3_step_matches_eager_sgd(cuda, hyper):
    """GraphedTrainStep (fused update inside the captured step) at the cfg-3 shape, 6 steps from a fresh optimizer:
    every loss and every parameter bit-identical to the eager loop with torch.optim.SGD."""
    from gnn_qot_estimation_b200 import TopologicalGNN, synthetic
    from gnn_qot_estimation_b200.graphed import GraphedTrainStep
    torch.manual_seed(3)
    m1 = TopologicalGNN(14, 16, 3, edge_dim=4, dropout_p=0.0).to(cuda)
    m2 = copy.deepcopy(m1)
    crit = torch.nn.SmoothL1Loss()
    o1 = torch.optim.SGD(m1.parameters(), lr=0.1, **hyper)
    o2 = torch.optim.SGD(m2.parameters(), lr=0.1, **hyper)
    store = synthetic.nsfnet_store(1024 * 6, seed=16).to(cuda)
    batches = [store.collate(range(i * 1024, (i + 1) * 1024)) for i in range(6)]
    g = GraphedTrainStep(m2, o2, crit, batches[0], warmup=2)
    assert g.fused is not None
    for b in batches:
        o1.zero_grad()
        l1 = crit(m1(b), b.y.view(-1, 3))
        l1.backward()
        o1.step()
        l2 = g.step(b)
        assert torch.equal(l1.detach(), l2), (float(l1), float(l2))
    for (k, p1), (_, p2) in zip(m1.named_parameters(), m2.named_parameters()):
        assert torch.equal(p1, p2), k
