"""GPU parity of the LightpathGNN training path where test_lightpath_train_gpu.py does not reach: the reference's
dropout (the head's mask replayed into the oracles), a full 4096-graph training batch (more LUT rows than one
grid-stride pass of the head kernels, hundreds of chunks in every multi-stage reduction), hand-built irregular graphs,
attention logits near +-100, BatchNorm's momentum=None / eps / one-row contract, GATConv with an input that requires
grad, and dropout through the CUDA-graphed step.

"All of it" below: the output, lut_batch (exact), the loss, every gradient (grad_parity), the running mean and
variance, and num_batches_tracked, against the fp64 oracle (fp32 oracle for grad_parity's allowance)."""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import grad_parity, load_golden, rel_err
from test_lightpath_train_gpu import RTOL, _b64, _kink_free_batch, _kink_margin, _pair, _step

pytestmark = pytest.mark.gpu
CKPT = "ckpt_lightpath_model_1.pt"
HEAD_ROWS_PER_PASS = 148 * 4 * 8        # head kernels: grid capped at kNumSMs * 4 blocks of 8 warps, one row per warp


class _FixedDropout(torch.nn.Module):
    """The oracles' stand-in for mlp[2]: dropout with a given keep mask, x * mask / (1 - p)."""

    def __init__(self, mask, p):
        super().__init__()
        self.mask, self.p = mask, p

    def forward(self, x):
        return x * (self.mask.to(x.dtype) / (1.0 - self.p))


def _drawn_mask(rng_before, n, p, dev):
    """The keep mask the step drew, recovered by replaying the CUDA generator from its state before the step.
    The generator must end where the step left it: the head's torch.rand was the step's only draw."""
    after = torch.cuda.get_rng_state(dev)
    torch.cuda.set_rng_state(rng_before, dev)
    mask = torch.rand(n, 32, device=dev) < 1.0 - p
    assert torch.equal(torch.cuda.get_rng_state(dev), after), "the step drew more than the head's dropout mask"
    return mask.cpu()


def _check_step(m, o, o32, hb, dev, p=0.0):
    """One step of m (train, or eval with grad) against the fp64 and fp32 oracles on host batch hb; with dropout p
    the mask m drew goes into both oracles.  Asserts all of it; returns the mask (None without dropout)."""
    before = torch.cuda.get_rng_state(dev)
    out, lb, loss, grads = _step(m, hb.to(dev))
    mask = None
    if m.training and p > 0.0:
        mask = _drawn_mask(before, lb.numel(), p, dev)
        o.mlp[2], o32.mlp[2] = _FixedDropout(mask, p), _FixedDropout(mask, p)
    eo, el, eloss, eg = _step(o, _b64(hb), torch.float64)
    _, _, _, eg32 = _step(o32, hb.to("cpu"))
    assert torch.equal(lb.cpu(), el)
    assert rel_err(out, eo) <= RTOL, rel_err(out, eo)
    assert rel_err(loss, eloss) <= RTOL, rel_err(loss, eloss)
    # conv1.bias feeds a batch-statistics BatchNorm: its exact gradient is 0 in training
    grad_parity(grads, eg, eg32, RTOL, exact_zero=("conv1.bias",) if m.training else ())
    bn, obn = m.norm1.module, o.norm1.module
    assert rel_err(bn.running_mean, obn.running_mean) <= RTOL
    assert rel_err(bn.running_var, obn.running_var) <= RTOL
    assert int(bn.num_batches_tracked) == int(obn.num_batches_tracked)
    return mask


def _models(dev, ckpt=CKPT, p=0.0, train=True, seed=0):
    m, o, o32 = _pair(dev, load_golden(ckpt)["model_state_dict"] if ckpt else None, seed=seed)
    m.mlp[2].p = p                                  # LightpathGNN reads its dropout rate from mlp[2]
    for mod in (m, o, o32):
        mod.train(train)
    return m, o, o32


# --------------------------------------------------------------------------- dropout
@pytest.mark.parametrize("ckpt", [CKPT, None])
@pytest.mark.parametrize("p", [0.5, 0.2])
def test_dropout_mask_replayed_through_the_oracle(cuda, p, ckpt):
    """512 ragged graphs (the bench step's shape) at the reference's dropout: the mask enters the head forward (act *=
    mask) and both factors of its backward (dh, and act into dW2); a missing factor changes the gradients."""
    m, o, o32 = _models(cuda, ckpt, p, seed=5)
    hb = _kink_free_batch(o, 512, 1, seed=40)
    torch.cuda.manual_seed(7)
    mask = _check_step(m, o, o32, hb, cuda, p)
    assert mask.shape == (512, 32)
    assert abs(float(mask.double().mean()) - (1.0 - p)) < 0.02       # 16384 draws: sd 0.004
    mask2 = _check_step(m, o, o32, hb, cuda, p)
    assert not torch.equal(mask, mask2)


# --------------------------------------------------------------------------- full training batch
@pytest.mark.parametrize("mode", ["train", "train_dropout", "eval_with_grad"])
def test_full_training_batch(cuda, mode):
    """4096 graphs with 2 LUTs each: ~8000 LUT rows (the head kernels' grid-stride loops take a second pass), ~130k
    nodes (~510 bn_stats chunks, ~2050 GAT backward block partials, a 130k-row qot_wgrad), ~125 chunks of the sparse
    BN backward.  eval() with grad: the running-statistics branch of the dense BN backward at that size."""
    p = 0.5 if mode == "train_dropout" else 0.0
    m, o, o32 = _models(cuda, CKPT, p, train=mode != "eval_with_grad")
    hb = _kink_free_batch(o, 4096, 2, seed=0)
    N, L = hb.x.shape[0], int((hb.x[:, 1] == 1.0).sum())
    assert L > HEAD_ROWS_PER_PASS and -(-L // 64) > 120
    assert -(-N // 256) > 500 and -(-N // 64) > 2000
    torch.cuda.manual_seed(11)
    mask = _check_step(m, o, o32, hb, cuda, p)
    if p > 0.0:
        assert mask.shape == (L, 32)
        # dropped units in the rows of the second grid-stride pass
        assert not bool(mask[HEAD_ROWS_PER_PASS:].all())


# --------------------------------------------------------------------------- irregular graphs
def _irregular_batch(seed=0):
    """One hand-built CPU Batch of structures the generator never makes, in this order:
    0. a boundary graph of 256 nodes whose node 0 has in-degree 255, two explicit self loops, 5 LUTs -- at its first
       node (the hub, the batch's first node) and its last;
    1. a 1-node graph carrying a LUT (no edges: its only message is the self loop GATConv adds);
    2. 40 nodes: 30 with random edges plus explicit self loops (one listed twice) and duplicated edges, 10 isolated;
       one LUT, on an isolated node; flags 0.99999994 and 1.0000001 (not LUTs);
    3. a 128-node boundary graph with no LUT and flags one ulp from 1.0;
    4. a 12-node ring with one LUT, at its last node (the batch's last node)."""
    from gnn_qot_estimation_b200 import Batch
    from dense_samples import boundary_graph
    rng = np.random.default_rng(seed)
    below, above = np.nextafter(np.float32(1), np.float32(0)), np.nextafter(np.float32(1), np.float32(2))
    graphs = []
    x, ei = boundary_graph(256, 1024, rng, hub_degree=255)
    assert int(((ei[1] == 0) & (ei[0] != 0)).sum()) == 255
    x[[0, 60, 128, 200, 255], 1] = 1.0
    graphs.append((x, ei))
    x = rng.random((1, 5), dtype=np.float32)
    x[0, 1] = 1.0
    graphs.append((x, np.zeros((2, 0), np.int64)))
    x = rng.random((40, 5), dtype=np.float32)
    x[:, 1] = 0.0
    x[35, 1], x[5, 1], x[6, 1] = 1.0, below, above
    rand = rng.integers(0, 30, size=(2, 80))
    loops = np.array([[3, 7, 7], [3, 7, 7]])
    ei = np.concatenate([rand, loops, rand[:, :10]], axis=1)
    graphs.append((x, ei))
    x, ei = boundary_graph(128, 512, rng)
    x[[0, 127], 1] = below
    x[64, 1] = above
    graphs.append((x, ei))
    x = rng.random((12, 5), dtype=np.float32)
    x[:, 1] = 0.0
    x[11, 1] = 1.0
    ring = np.arange(12)
    ei = np.concatenate([np.stack([ring, (ring + 1) % 12]), np.stack([(ring + 1) % 12, ring])], axis=1)
    graphs.append((x, ei))
    off = np.cumsum([0] + [g[0].shape[0] for g in graphs])
    xs = torch.from_numpy(np.concatenate([g[0] for g in graphs]))
    ei = torch.from_numpy(np.concatenate([g[1] + o for g, o in zip(graphs, off[:-1])], axis=1).astype(np.int64))
    batch = torch.repeat_interleave(torch.arange(len(graphs)), torch.from_numpy(np.diff(off)))
    y = torch.from_numpy(rng.random((len(graphs), 3), dtype=np.float32))
    return Batch(x=xs, edge_index=ei, batch=batch, y=y, num_graphs=len(graphs))


@pytest.mark.parametrize("p", [0.0, 0.5])
def test_irregular_graphs(cuda, p):
    m, o, o32 = _models(cuda, CKPT, p)
    hb = _irregular_batch()
    assert hb.batch[hb.x[:, 1] == 1.0].tolist() == [0] * 5 + [1, 2, 4]    # flags one ulp from 1.0 are not LUTs
    assert _kink_margin(o, hb) > 2e-6
    torch.cuda.manual_seed(13)
    _check_step(m, o, o32, hb, cuda, p)


# --------------------------------------------------------------------------- large attention logits
def _gat_logits(o, x, edge_index):
    """fp64 attention logits [E', 4] of every GATConv message in the kernel's row order (destination rows, edge
    order, the added self loop last), with each message's row, its position in the row and the row's length."""
    from oracle.qot_oracle import gat_edges_ref
    N = x.shape[0]
    ei = gat_edges_ref(edge_index, N)
    order = torch.argsort(ei[1], stable=True)
    src, dst = ei[0][order], ei[1][order]
    xp = (x.double() @ o.conv1.lin.weight.detach().double().T).view(N, 4, 32)
    s = (xp * o.conv1.att_src.detach().double()).sum(-1)
    d = (xp * o.conv1.att_dst.detach().double()).sum(-1)
    deg = torch.bincount(dst, minlength=N)
    pos = torch.arange(dst.numel()) - (torch.cumsum(deg, 0) - deg)[dst]
    return F.leaky_relu(s[src] + d[dst], 0.2), dst, pos, deg[dst]


def _large_logit_batch(o, scale_to=100.0, margin=1e-4):
    """64 generated graphs whose features (all but the flag column) are centred and scaled so that the largest
    attention logit is ~scale_to; the first seed whose LUT pre-activations keep `margin` from the ReLU kinks (fp32
    exp at these logits costs ~1e-5 of h on its own)."""
    from gnn_qot_estimation_b200 import synthetic
    cols = [0, 2, 3, 4]
    for seed in range(50, 90):
        hb = synthetic.lightpath_store(64, seed=seed).host_batch(0, 64)
        hb.x[:, cols] -= 0.5
        for _ in range(4):                              # the flag column is not scaled: the logits are affine in it
            hb.x[:, cols] *= scale_to / float(_gat_logits(o, hb.x, hb.edge_index)[0].max())
        if _kink_margin(o, hb) > margin:
            return hb
    raise AssertionError("no kink-free large-logit batch found")


def test_large_attention_logits(cuda):
    """Logits up to ~100 (fp32 exp overflows above 88 without the online-softmax rescale), the row maximum first in
    some rows and last in others.  Output and gradients against fp64 under grad_parity's 2x fp32-oracle allowance."""
    m, o, o32 = _models(cuda, CKPT)
    hb = _large_logit_batch(o)
    a, row, pos, deg = _gat_logits(o, hb.x, hb.edge_index)
    assert 88.0 < float(a.max()) < 130.0 and float(a.min()) < -15.0
    rmax = torch.zeros(int(row.max()) + 1, 4, dtype=a.dtype).scatter_reduce(
        0, row[:, None].expand_as(a), a, reduce="amax", include_self=False)
    rmin = torch.zeros_like(rmax).scatter_reduce(0, row[:, None].expand_as(a), a, reduce="amin", include_self=False)
    is_max = (a == rmax[row]) & (deg >= 3)[:, None]
    assert int((is_max & (pos == 0)[:, None]).sum()) >= 20            # maximum first: every later term rescales
    assert int((is_max & (pos == deg - 1)[:, None]).sum()) >= 20      # maximum last: every earlier term rescales
    assert int(((rmax - rmin) > 60.0).sum()) >= 100
    out, lb, loss, grads = _step(m, hb.to(cuda))
    eo, el, eloss, eg = _step(o, _b64(hb), torch.float64)
    o32_out, _, o32_loss, eg32 = _step(o32, hb.to("cpu"))
    assert torch.equal(lb.cpu(), el)
    assert torch.isfinite(out).all()
    assert rel_err(out, eo) <= max(RTOL, 2.0 * rel_err(o32_out, eo)), (rel_err(out, eo), rel_err(o32_out, eo))
    assert rel_err(loss, eloss) <= max(RTOL, 2.0 * rel_err(o32_loss, eloss))
    grad_parity(grads, eg, eg32, RTOL, exact_zero=("conv1.bias",))
    bn, obn = m.norm1.module, o.norm1.module
    assert rel_err(bn.running_mean, obn.running_mean) <= RTOL
    assert rel_err(bn.running_var, obn.running_var) <= RTOL


# --------------------------------------------------------------------------- BatchNorm / GATConv contract
BN_SETTINGS = [pytest.param(None, 1e-5, id="momentum_None"), pytest.param(0.01, 1e-3, id="momentum_0.01_eps_1e-3")]


@pytest.mark.parametrize("momentum,eps", BN_SETTINGS)
def test_lightpath_norm1_momentum_and_eps(cuda, momentum, eps):
    """Three training steps; momentum=None is torch's cumulative average 1/num_batches_tracked."""
    m, o, o32 = _models(cuda, CKPT)
    for mod in (m, o, o32):
        mod.norm1.module.momentum, mod.norm1.module.eps = momentum, eps
    start = int(m.norm1.module.num_batches_tracked)
    for k in range(3):
        _check_step(m, o, o32, _kink_free_batch(o, 64 + 32 * k, 1, seed=60 + k), cuda)
    assert int(m.norm1.module.num_batches_tracked) == start + 3


@pytest.mark.parametrize("momentum,eps", BN_SETTINGS)
def test_standalone_batchnorm_momentum_and_eps(cuda, momentum, eps):
    from gnn_qot_estimation_b200 import nn as qnn
    g = torch.Generator().manual_seed(3)
    bn = qnn.BatchNorm(128, eps=eps, momentum=momentum)
    ref = torch.nn.BatchNorm1d(128, eps=eps, momentum=momentum).double()
    with torch.no_grad():
        bn.module.weight.uniform_(0.5, 1.5, generator=g)
        bn.module.bias.normal_(0.0, 0.1, generator=g)
        ref.weight.copy_(bn.module.weight)
        ref.bias.copy_(bn.module.bias)
    bn.to(cuda).train()
    ref.train()
    for k in range(3):
        x = torch.randn(300 + 200 * k, 128, generator=g) * (1.0 + k) + 5.0
        w = torch.randn(300 + 200 * k, 128, generator=g)
        bn.zero_grad()
        ref.zero_grad()
        xd = x.to(cuda)
        y = bn(xd)
        (y * w.to(cuda)).sum().backward()
        y64 = ref(x.double())
        (y64 * w.double()).sum().backward()
        assert rel_err(y, y64) <= RTOL
        for name in ("weight", "bias"):
            assert rel_err(getattr(bn.module, name).grad, getattr(ref, name).grad) <= RTOL, name
        assert rel_err(bn.module.running_mean, ref.running_mean) <= RTOL
        assert rel_err(bn.module.running_var, ref.running_var) <= RTOL
        assert int(bn.module.num_batches_tracked) == int(ref.num_batches_tracked) == k + 1


def test_one_node_training_batch_raises(cuda):
    from gnn_qot_estimation_b200 import Batch, nn as qnn
    msg = "Expected more than 1 value per channel when training"
    with pytest.raises(ValueError, match=msg):
        torch.nn.BatchNorm1d(128).train()(torch.randn(1, 128))                 # what torch does
    bn = qnn.BatchNorm(128).to(cuda).train()
    with pytest.raises(ValueError, match=msg):
        bn(torch.randn(1, 128, device=cuda))
    assert int(bn.module.num_batches_tracked) == 0
    m, _, _ = _models(cuda, CKPT)
    x = torch.rand(1, 5)
    x[0, 1] = 1.0
    b = Batch(x=x, edge_index=torch.zeros(2, 0, dtype=torch.int64), batch=torch.zeros(1, dtype=torch.int64),
              y=torch.rand(1, 3), num_graphs=1).to(cuda)
    with pytest.raises(ValueError, match=msg):
        m(b)
    m.eval()                                           # running statistics: one node is fine
    out, lb = m(b)
    assert out.shape == (1, 3) and lb.tolist() == [0]


def test_gatconv_input_requiring_grad_raises(cuda):
    """The kernels give no gradient for x (the reference's x is data): an x that requires grad raises rather than
    receiving a silent zero."""
    from gnn_qot_estimation_b200 import nn as qnn, synthetic
    conv = qnn.GATConv(5, 32, heads=4, concat=True).to(cuda)
    b = synthetic.lightpath_store(4, seed=1).host_batch(0, 4).to(cuda)
    x = b.x.clone().requires_grad_(True)
    with pytest.raises(NotImplementedError, match="no gradient with respect to x"):
        conv(x, b.edge_index)
    with torch.no_grad():
        h0 = conv(x, b.edge_index)
    h1 = conv(b.x, b.edge_index)
    assert h1.requires_grad and torch.equal(h0, h1.detach())


# --------------------------------------------------------------------------- graphed step with dropout
def test_graphed_dropout_steps_equal_eager(cuda):
    """GraphedStepCache at dropout 0.5 over ragged batches.  Only replays are compared (the warm-up steps of a capture
    draw from the generator): before each, the eager model m1 takes m2's parameters, buffers and optimizer state and
    both steps start from the same generator seed -- the captured torch.rand reads seed and offset at replay, so the
    two steps are bit-identical.  Two replays of one batch from one starting state draw different masks unless the
    generator is reseeded."""
    from gnn_qot_estimation_b200 import LightpathGNN, synthetic
    from gnn_qot_estimation_b200.graphed import GraphedStepCache
    torch.manual_seed(4)
    m1 = LightpathGNN(5, 32, 3, is_lut_index=1, dropout_p=0.5).to(cuda).train()
    m2 = copy.deepcopy(m1)
    crit = torch.nn.SmoothL1Loss()
    o1 = torch.optim.SGD(m1.parameters(), lr=0.05, momentum=0.9)
    o2 = torch.optim.SGD(m2.parameters(), lr=0.05, momentum=0.9)
    store = synthetic.lightpath_store(3 * 128, seed=8).to(cuda)
    batches = [store.collate(range(i * 128, (i + 1) * 128)) for i in range(3)]
    assert len({b.num_nodes for b in batches}) == 3

    def loss_of(model, b):
        out, lb = model(b)
        return crit(out, b.y[lb])
    cache = GraphedStepCache(m2, o2, loss_of)
    for b in batches:                                  # captures
        cache.step(b)
    for epoch in (1, 2):
        for i, b in enumerate(batches):
            m1.load_state_dict(m2.state_dict())
            o1.load_state_dict(copy.deepcopy(o2.state_dict()))
            seed = 100 * epoch + i
            torch.cuda.manual_seed(seed)
            o1.zero_grad()
            l1 = loss_of(m1, b)
            l1.backward()
            o1.step()
            torch.cuda.manual_seed(seed)
            l2 = cache.step(b)
            assert torch.equal(l1.detach(), l2), (epoch, i, float(l1), float(l2))
            for (k, v1), (_, v2) in zip(m1.state_dict().items(), m2.state_dict().items()):
                assert torch.equal(v1, v2), (epoch, i, k)
    assert cache.captures == 3 and cache.replays == 9

    model_sd = {k: v.clone() for k, v in m2.state_dict().items()}
    opt_sd = copy.deepcopy(o2.state_dict())

    def restore():
        with torch.no_grad():
            for k, v in m2.state_dict().items():
                v.copy_(model_sd[k])
            cur = o2.state_dict()["state"]
            for idx, st in opt_sd["state"].items():
                cur[idx]["momentum_buffer"].copy_(st["momentum_buffer"])
    torch.cuda.manual_seed(7)
    la = cache.step(batches[0]).clone()
    restore()
    lb = cache.step(batches[0]).clone()                # generator advanced by the previous replay
    restore()
    torch.cuda.manual_seed(7)
    lc = cache.step(batches[0]).clone()
    assert not torch.equal(la, lb)
    assert torch.equal(la, lc)
