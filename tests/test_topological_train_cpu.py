"""CPU checks behind tests/test_topological_train_parity_gpu.py: the batch builders give the shapes the GPU tests
claim, the fused kernels' grid (restated from csrc/topo_fused.cu) gives some block two or more graphs in every
multi-graph case, and the fused SGD update is handed torch's rounding of 1 - dampening."""
import numpy as np
import pytest
import torch

import topo_batches as TB


def _sizes(b):
    return (b.ptr[1:] - b.ptr[:-1]), (b.edge_ptr[1:] - b.edge_ptr[:-1])


def _graph(b, g):
    n0, n1 = int(b.ptr[g]), int(b.ptr[g + 1])
    e0, e1 = int(b.edge_ptr[g]), int(b.edge_ptr[g + 1])
    return b.node_ids[n0:n1], b.edge_index[0, e0:e1] - n0, b.edge_index[1, e0:e1] - n0


def test_shared_memory_and_grid_arithmetic():
    """The byte counts DESIGN §4.4 quotes, and the grid each case of the GPU file launches."""
    assert TB.tf_smem_bytes(14, 42, 14, False) == 17360 and TB.tf_smem_bytes(14, 42, 14, True) == 38832
    assert TB.tf_smem_bytes(75, 300, 75, False) == 95792 and TB.tf_smem_bytes(75, 300, 75, True) == 142160
    assert TB.tf_smem_bytes(128, 512, 128, True) == 230784 <= TB.MAX_SMEM
    assert TB.grids(1024, 14, 42, 14) == (1024, 740)              # fwd 7 blocks per SM, bwd 5
    assert TB.grids(4096, 14, 42, 14) == (1036, 740)
    assert TB.grids(600, 75, 300, 75) == (296, 148)
    assert TB.grids(160, 128, 512, 128) == (148, 148)


@pytest.mark.parametrize("B,nmax,emax,table,every", [(1024, 14, 42, 14, False), (4096, 14, 42, 14, True),
                                                      (600, 75, 300, 75, True), (160, 128, 512, 128, False)])
def test_every_multi_graph_case_gives_a_block_two_graphs(B, nmax, emax, table, every):
    """Graph g and g + grid share a block: the backward grid is smaller than the batch in every case, and with
    `every` both grids are at most half the batch, so every block of both kernels takes two or more graphs."""
    fwd, bwd = TB.grids(B, nmax, emax, table)
    assert B > bwd
    if every:
        assert B >= 2 * bwd and B >= 2 * fwd
    if B == 4096:                                                  # and for any per-SM block count up to 8
        assert B >= 2 * 8 * TB.NUM_SMS


def test_ragged75_batch():
    b = TB.ragged75()
    n, e = _sizes(b)
    assert b.num_graphs == 600 and set(n.tolist()) == set(range(1, 76))
    assert (b.max_nodes, b.max_edges) == (int(n.max()), int(e.max())) == (75, 300)
    assert bool((e <= 4 * n).all()) and bool((e[n == 1] == 0).all())
    assert int(b.node_ids.min()) >= 0 and int(b.node_ids.max()) < TB.RAGGED_TABLE
    grid = TB.grids(600, 75, 300, 75)[1]
    assert any(n[g] > n[g + grid] for g in range(600 - grid)) and any(n[g] < n[g + grid] for g in range(600 - grid))
    hubs = isolated = loops = dup_edges = dup_ids = 0
    for g in range(600):
        ids, src, dst = _graph(b, g)
        k = ids.numel()
        dup_ids += ids.unique().numel() < k
        if src.numel() == 0:
            continue
        hubs += int(torch.bincount(dst, minlength=k).max()) * 3 >= src.numel() >= 40
        isolated += torch.bincount(torch.cat([src, dst]), minlength=k).eq(0).any().item()
        loops += bool((src == dst).any())
        dup_edges += (src * k + dst).unique().numel() < src.numel()
    assert min(hubs, isolated, loops, dup_edges, dup_ids) >= 20, (hubs, isolated, loops, dup_edges, dup_ids)
    # the understated caps of the GPU file cut graphs by node count alone, by edge count alone, and leave others
    over_n, over_e = n > 60, e > 200
    assert bool((over_n & ~over_e).any()) and bool((~over_n & over_e).any()) and bool((~(over_n | over_e)).any())


@pytest.mark.parametrize("extra", [0, 1])
def test_edge512_batch(extra):
    from gnn_qot_estimation_b200 import ops
    b = TB.edge512(extra_edges=extra)
    n, e = _sizes(b)
    assert (b.max_nodes, b.max_edges) == (128, 512 + extra)
    assert int(n[TB.EDGE512_BIG]) == 128 and int(e[TB.EDGE512_BIG]) == 512 + extra
    assert int(torch.cat([e[:TB.EDGE512_BIG], e[TB.EDGE512_BIG + 1:]]).max()) <= 500
    _, src, dst = _graph(b, TB.EDGE512_BIG)
    assert int(torch.bincount(dst).max()) >= 400 and int(torch.bincount(src).max()) >= 400
    assert ops.topo_fused_fits(b.max_nodes, b.max_edges, TB.EDGE512_TABLE) == (extra == 0)


DAMPENING = (0.0, 0.1, 0.6, 0.8, 0.9, 0.99, 1 / 3)


@pytest.mark.parametrize("d", DAMPENING)
def test_sgd_hyper_packs_torchs_dampening_factor(d):
    """torch.optim.SGD passes alpha = 1 - dampening (Python double) to a foreach kernel that rounds it to fp32 once;
    the packed struct carries exactly that value, which for 0.6, 0.8, 0.9, 0.99 and 1/3 is one ulp away from
    float(1) - float(dampening)."""
    from gnn_qot_estimation_b200.distributed import pack_sgd_hyper
    h = pack_sgd_hyper(0.1, 0.9, d, 5e-4, False, True)
    assert np.float32(h.one_minus_dampening) == np.float32(1 - d)
    assert np.float32(h.dampening) == np.float32(d) and np.float32(h.lr) == np.float32(0.1)
    assert (h.nesterov, h.maximize) == (0, 1)
    naive = np.float32(1) - np.float32(d)
    assert (naive != np.float32(1 - d)) == (d in (0.6, 0.8, 0.9, 0.99, 1 / 3))
