"""Reference for LightpathGNN's every-node mode (TEST INFRASTRUCTURE, like tg_cases.py): the readout of every node as
the LUT, defined literally through one-hot copies of every graph and the oracle model (oracle.LightpathGNNOracle)."""
from types import SimpleNamespace

import torch


def lightpath_every_node_ref(model, batch, chunk=None) -> torch.Tensor:
    """Every-node readout of a LightpathGNN, defined literally: for every node c of the batch, a copy of c's graph
    (its nodes, the edges with both endpoints in it, in edge order) whose flag column ``x[:, model.is_lut_index]`` is
    1.0 at c and 0.0 elsewhere; all copies are run through ``model`` at once and each copy's single readout row is
    taken.  Returns ``out [N, 3]`` in node order.  ``batch`` needs ``x``, ``edge_index`` and ``batch``; runs on their
    device and dtype.  ``chunk``: copies per oracle call (None: all at once; the copies of dense graphs can outgrow
    memory), results concatenated in node order."""
    x, ei, b = batch.x, batch.edge_index.to(torch.int64), batch.batch.to(torch.int64)
    dev, N = x.device, x.shape[0]
    col = model.is_lut_index
    if N == 0:
        return x.new_zeros(0, 3)
    B = int(b.max()) + 1
    n = torch.bincount(b, minlength=B)
    gstart = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    gstart[1:] = torch.cumsum(n, 0)
    order = torch.argsort(b, stable=True)                          # nodes grouped by graph
    pos = torch.empty(N, dtype=torch.int64, device=dev)
    pos[order] = torch.arange(N, device=dev)
    local = pos - gstart[b]                                        # position of a node inside its graph
    # edges of graph g (both endpoints in g, edge order): eorder[estart[g]:estart[g + 1]]
    keep = b[ei[0]] == b[ei[1]]
    ek = ei[:, keep]
    eg = b[ek[0]]
    eorder = torch.argsort(eg, stable=True)
    ecount = torch.bincount(eg, minlength=B)
    estart = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    estart[1:] = torch.cumsum(ecount, 0)
    outs = []
    step = N if chunk is None else int(chunk)
    assert step > 0
    for c0 in range(0, N, step):
        cs = torch.arange(c0, min(c0 + step, N), device=dev)        # the nodes whose copies this call evaluates
        P = cs.numel()
        # nodes of the copies: copy c holds graph b[c]'s nodes in order
        csize = n[b[cs]]
        coff = torch.zeros(P + 1, dtype=torch.int64, device=dev)
        coff[1:] = torch.cumsum(csize, 0)
        copy_row = torch.repeat_interleave(torch.arange(P, device=dev), csize)
        t = torch.arange(int(coff[-1]), device=dev) - coff[copy_row]
        node = order[gstart[b[cs[copy_row]]] + t]
        xc = x[node].clone()
        xc[:, col] = (node == cs[copy_row]).to(x.dtype)
        # edges of the copies: graph g's edges relabelled into each copy of g
        emult = ecount[b[cs]]
        eoff = torch.zeros(P + 1, dtype=torch.int64, device=dev)
        eoff[1:] = torch.cumsum(emult, 0)
        copy_e = torch.repeat_interleave(torch.arange(P, device=dev), emult)
        te = torch.arange(int(eoff[-1]), device=dev) - eoff[copy_e]
        e = eorder[estart[b[cs[copy_e]]] + te]
        eic = torch.stack([coff[copy_e] + local[ek[0, e]], coff[copy_e] + local[ek[1, e]]])
        data = SimpleNamespace(x=xc, edge_index=eic, batch=copy_row, num_graphs=P)
        out, lut_batch = model(data)
        assert torch.equal(lut_batch.cpu(), torch.arange(P)), "every copy has exactly one readout row"
        outs.append(out)
    return torch.cat(outs)
