"""Batches for the TopologicalGNN training-step tests at production shapes (tests/test_topological_train_*), and a
restatement of how csrc/topo_fused.cu sizes its persistent grid, so a test can say how many graphs a block takes.

Everything here is host-side and seeded: the GPU file moves the batches to the device, the CPU file checks their
shapes and the occupancy arithmetic."""
import torch

# csrc/topo_fused.cu: tf_smem_bytes / tf_blocks
TF_PARAMS, TF_H, TF_T, TF_D, TF_K = 4092, 16, 144, 4, 8
NUM_SMS, SMEM_PER_SM, MAX_SMEM = 148, 228 * 1024, 227 * 1024


def tf_smem_bytes(nmax, emax, num_nodes, bwd):
    f = (TF_PARAMS + num_nodes * TF_H) if bwd else 0
    f += nmax * (TF_H * (10 if bwd else 7) + TF_T)
    f += emax * (TF_D + TF_K + (2 + TF_K if bwd else 1))
    f += 96
    b = f * 4 + 2 * (nmax + 1) * 4 + 4 * emax * 2
    return (b + 15) & ~15


def tf_blocks(B, smem):
    per_sm = max(1, min(7, SMEM_PER_SM // (smem + 1024)))
    return min(B, per_sm * NUM_SMS)


def grids(B, nmax, emax, num_nodes):
    """(forward blocks, backward blocks) of a fused launch; graph g runs in block g % blocks."""
    return (tf_blocks(B, tf_smem_bytes(nmax, emax, num_nodes, False)),
            tf_blocks(B, tf_smem_bytes(nmax, emax, num_nodes, True)))


def assemble(graphs, seed):
    """graphs: list of (node_ids [n], src [E], dst [E]) with graph-local endpoints -> a host Batch that records its
    offsets (ptr, edge_ptr) and largest graph (max_nodes, max_edges), as PackedGraphStore.collate does; y [B,3]."""
    from gnn_qot_estimation_b200 import Batch
    g = torch.Generator().manual_seed(seed)
    ids, eis, bts, ptr, eptr = [], [], [], [0], [0]
    for gi, (nid, src, dst) in enumerate(graphs):
        off = ptr[-1]
        ids.append(nid)
        eis.append(torch.stack([src, dst]) + off)
        bts.append(torch.full((nid.numel(),), gi, dtype=torch.int64))
        ptr.append(off + nid.numel())
        eptr.append(eptr[-1] + src.numel())
    E = eptr[-1]
    b = Batch(edge_index=torch.cat(eis, 1), edge_attr=torch.rand(E, 4, generator=g), batch=torch.cat(bts),
              node_ids=torch.cat(ids), y=torch.rand(len(graphs), 3, generator=g) * 3 - 1, ptr=torch.tensor(ptr),
              edge_ptr=torch.tensor(eptr), num_graphs=len(graphs))
    b.max_nodes = max(nid.numel() for nid, _, _ in graphs)
    b.max_edges = max(src.numel() for _, src, _ in graphs)
    return b


RAGGED_TABLE = 75


def ragged75(num_graphs=600, seed=3):
    """Graphs of the real 75-node topology's size range in mixed order: n = 1..75 (every size at least 7 times), E up
    to 4n with one graph at (75, 300); every third graph has a hub taking half its edges as destination, every fifth
    an isolated node, every graph with edges self loops and (from 3 edges on) repeated edges, every fourth graph with
    n >= 2 a repeated node id; 1-node graphs have no edges."""
    g = torch.Generator().manual_seed(seed)
    sizes = [1 + i % RAGGED_TABLE for i in range(num_graphs)]
    sizes = [sizes[i] for i in torch.randperm(num_graphs, generator=g).tolist()]
    sizes[sizes.index(RAGGED_TABLE)] = -RAGGED_TABLE          # marks the (75, 300) graph
    graphs = []
    for gi, s in enumerate(sizes):
        n = abs(s)
        ids = torch.randperm(RAGGED_TABLE, generator=g)[:n]
        if n >= 2 and gi % 4 == 0:
            ids[-1] = ids[0]
        if n == 1:
            graphs.append((ids, torch.zeros(0, dtype=torch.int64), torch.zeros(0, dtype=torch.int64)))
            continue
        E = 4 * n if s < 0 else int(torch.randint(1, 4 * n + 1, (1,), generator=g))
        src = torch.randint(0, n, (E,), generator=g)
        dst = torch.randint(0, n, (E,), generator=g)
        if gi % 3 == 0:
            dst[torch.randperm(E, generator=g)[:E // 2]] = int(torch.randint(0, n, (1,), generator=g))
        if gi % 5 == 0 and n >= 3:                               # node n-1 isolated: no edge touches it
            src[src == n - 1] = 0
            dst[dst == n - 1] = 1
        k = max(1, E // 8)
        dst[:k] = src[:k]                                        # self loops
        if E >= 3 * k:                                           # repeated edges
            src[-k:], dst[-k:] = src[k:2 * k].clone(), dst[k:2 * k].clone()
        graphs.append((ids, src, dst))
    return assemble(graphs, seed)


EDGE512_TABLE, EDGE512_BIG = 128, 5


def edge512(extra_edges=0, num_graphs=160, seed=4):
    """The largest graph topo_fused_fits admits: graph EDGE512_BIG has 128 nodes and 512 + extra_edges edges, 420 of
    them into node 7 and 420 out of node 9 (so at least 328 are 9 -> 7), on a 128-row table: 230 784 B of the
    backward kernel's 232 448.  The other graphs are random (n <= 128, E <= min(4n, 500)); with 148 blocks, block 5
    takes the big graph first and graph 153 after it."""
    g = torch.Generator().manual_seed(seed)
    graphs = []
    for gi in range(num_graphs):
        if gi == EDGE512_BIG:
            n, E = EDGE512_TABLE, 512 + extra_edges
            src = torch.randint(0, n, (E,), generator=g)
            dst = torch.randint(0, n, (E,), generator=g)
            dst[torch.randperm(E, generator=g)[:420]] = 7
            src[torch.randperm(E, generator=g)[:420]] = 9
        else:
            n = int(torch.randint(1, EDGE512_TABLE + 1, (1,), generator=g))
            E = 0 if n == 1 else int(torch.randint(0, min(4 * n, 500) + 1, (1,), generator=g))
            src = torch.randint(0, n, (E,), generator=g)
            dst = torch.randint(0, n, (E,), generator=g)
        graphs.append((torch.randperm(EDGE512_TABLE, generator=g)[:n], src, dst))
    return assemble(graphs, seed)
