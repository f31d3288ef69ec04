"""lp_stream_kernel (csrc/lightpath_stream.cu) at every cap it branches on, against the fp64 oracle.

The kernel stages a tile of kTG graphs only when the tile spans at most kTNodes nodes and kTEdges edges; inside a
staged tile a graph takes the fast path only with n <= kMaxN, E <= kTMaxE, exactly one LUT node, a LUT row of at
most kSubMsg - 1 in-edges and no source inside [0, N) but outside the graph.  Everything else goes to the generic
path, which reads global memory.  Both paths give the oracle's answer to 1e-5, so parity alone cannot see a cap that
moved by one.  Each case below therefore also checks WHICH path every graph at a boundary took: a graph's fast-path
row is a function of the graph alone (bit for bit, wherever its tile sits), and so is its generic-path row, and the
two differ in the last bits (other sum orders, another readout head).  `path_refs` evaluates every such graph once in
a tile that is surely staged and once in a tile that surely is not; the case's row must equal, bit for bit, the
reference of the path `kernel_paths` (the kernel's rules restated on the host) names.

The caps are read from the sources, so a changed constant moves the cases with it.  The builders are checked on the
CPU by test_lightpath_stream_caps_cpu.py: each case sits on the boundary it names."""
import functools
import re
from dataclasses import dataclass, field
from pathlib import Path

import numpy as np
import pytest
import torch

from conftest import ABS_FLOOR, load_golden, rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-5
CSRC = Path(__file__).resolve().parents[1] / "gnn_qot_estimation_b200" / "csrc"


def _cap(fname, name):
    m = re.search(rf"constexpr\s+int\s+{name}\s*=\s*(\d+)\s*;", (CSRC / fname).read_text())
    assert m, f"{name} not found in {fname}"
    return int(m.group(1))


TG = _cap("lightpath_stream.cu", "kTG")                  # graphs per tile
T_NODES = _cap("lightpath_stream.cu", "kTNodes")         # x window of a tile
T_EDGES = _cap("lightpath_stream.cu", "kTEdges")         # destination window of a tile
T_MAX_E = _cap("lightpath_stream.cu", "kTMaxE")          # edges of a fast-path graph
GROUP_TILES = _cap("lightpath_stream.cu", "kGroupTiles")  # tiles per readout group of the in-kernel head
MAX_N = _cap("lightpath_common.cuh", "kMaxN")            # nodes of a fast-path graph
SUB_MSG = _cap("lightpath_common.cuh", "kSubMsg")        # messages of a fast-path row: sources + the self loop
HUB = SUB_MSG - 1                                        # the largest LUT in-degree the fast path keeps
F, LUT_COL = 5, 1


# ------------------------------------------------------------------------------------------------------------------
# graphs
# ------------------------------------------------------------------------------------------------------------------
@dataclass
class Graph:
    x: np.ndarray                 # [n, 5] float32, the LUT flag in column LUT_COL
    src: np.ndarray               # [E] int64, graph-local ids
    dst: np.ndarray               # [E] int64, graph-local ids
    tag: str = ""
    ext: dict = field(default_factory=dict)   # edge -> "prev" | "neg" | "N" | "big": its source lies outside the graph

    @property
    def n(self):
        return int(self.x.shape[0])

    @property
    def E(self):
        return int(self.src.shape[0])

    def lut(self):
        return np.nonzero(self.x[:, LUT_COL] == 1.0)[0]

    def indeg(self):
        """In-edges of the (first) LUT node: what the fast path counts against kSubMsg - 1."""
        return int((self.dst == self.lut()[0]).sum())

    def kept(self):
        """Messages the LUT row keeps from its in-edges: self loops and sources outside [0, N) are dropped."""
        il = self.lut()[0]
        ins = np.nonzero(self.dst == il)[0]
        return sum(1 for e in ins if self.src[e] != il and self.ext.get(int(e)) not in ("neg", "N", "big"))


def _rand_x(rng, n, luts):
    x = rng.random((n, F), dtype=np.float32) + np.float32(0.05)
    x[:, LUT_COL] = 0.0
    x[list(luts), LUT_COL] = 1.0
    return x


def _directed_edges(rng, n, E, il, deg, loops, dups, at):
    src = rng.integers(0, n, E)
    if il is None or deg is None:
        return src, rng.integers(0, n, E)
    others = np.array([v for v in range(n) if v != il])
    dst = others[rng.integers(0, len(others), E)]
    pos = np.sort(rng.choice(E, deg, replace=False)) if at is None else np.asarray(sorted(set(at)))
    if at is not None and len(pos) < deg:
        rest = np.setdiff1d(np.arange(E), pos)
        pos = np.sort(np.concatenate([pos, rng.choice(rest, deg - len(pos), replace=False)]))
    distinct = deg - loops - dups
    s = rng.choice(others, distinct, replace=False)
    s = np.concatenate([s, np.full(loops, il), s[rng.integers(0, max(distinct, 1), dups)]])
    rng.shuffle(s)
    src[pos], dst[pos] = s, il
    return src, dst


def _sym_edges(rng, n, E, il, deg, loops):
    """The from_networkx layout of an undirected graph: both directions of every pair, no duplicate pair, edges
    sorted by (source, destination).  The LUT node has `deg` in-edges (`loops` of them its self loop)."""
    assert loops in (0, 1)
    others = [v for v in range(n) if v != il]
    nb = (deg or 0) - loops
    edges = []
    if il is not None:
        for v in rng.choice(others, nb, replace=False):
            edges += [(il, int(v)), (int(v), il)]
        edges += [(il, il)] * loops
    rest = E - len(edges)
    assert rest >= 0
    if rest % 2:
        edges.append((others[0], others[0]))   # a self loop off the LUT row fixes the parity
    pairs = [(u, v) for i, u in enumerate(others) for v in others[i + 1:]]
    for k in rng.choice(len(pairs), rest // 2, replace=False):
        u, v = pairs[k]
        edges += [(u, v), (v, u)]
    edges.sort()
    e = np.array(edges, dtype=np.int64).reshape(-1, 2)
    return e[:, 0], e[:, 1]


def make_graph(rng, n, E, lut=0, deg=None, loops=0, dups=0, at=None, sym=False, luts=None, tag=""):
    """A graph of n nodes and E edges.  lut: position of its LUT node (negative: from the end; None: no LUT node);
    luts: several LUT nodes.  deg: exact in-degree of the LUT row, `loops` of them self loops, `dups` repeating an
    earlier source (directed builder only); at: edge positions the row's in-edges take (the rest random).
    sym: the verified from_networkx layout (PackedGraphStore.verify_layout)."""
    if luts is None:
        luts = [] if lut is None else [lut % n]
    il = luts[0] if luts else None
    x = _rand_x(rng, n, luts)
    if sym:
        assert dups == 0 and at is None
        src, dst = _sym_edges(rng, n, E, il, deg, loops)
    else:
        src, dst = _directed_edges(rng, n, E, il, deg, loops, dups, at)
    return Graph(x, src.astype(np.int64), dst.astype(np.int64), tag or f"n={n},E={E},deg={deg}")


def filler(rng, n):
    """A graph without LUT node and without edges: no readout row, it only takes space in its tile."""
    return Graph(_rand_x(rng, n, []), np.zeros(0, np.int64), np.zeros(0, np.int64), f"filler{n}")


def small_graphs(rng, k, sym=False, nlo=8, nhi=24):
    """k ordinary fast-path graphs: n ~ U{nlo..nhi}, a LUT row of 3..7 in-edges, about 2n edges."""
    out = []
    for _ in range(k):
        n = int(rng.integers(nlo, nhi + 1))
        deg = int(rng.integers(3, min(8, n)))
        E = 2 * deg + 2 * int(rng.integers(1, min(n, (n - 1) * (n - 2) // 2) + 1))
        out.append(make_graph(rng, n, E, lut=int(rng.integers(0, n)), deg=deg, sym=sym))
    return out


# ------------------------------------------------------------------------------------------------------------------
# batches
# ------------------------------------------------------------------------------------------------------------------
def assemble(graphs, lut_extra=None):
    """Host Batch of the graphs in the reference layout; `ext` sources resolved against this batch.
    lut_extra {graph: k}: lut_ptr claims k more rows for that graph than its x holds (a stale index array)."""
    from gnn_qot_estimation_b200 import Batch
    ns = np.array([g.n for g in graphs], np.int64)
    es = np.array([g.E for g in graphs], np.int64)
    ptr = np.concatenate([[0], np.cumsum(ns)])
    eptr = np.concatenate([[0], np.cumsum(es)])
    N = int(ptr[-1])
    srcs, dsts = [], []
    for i, g in enumerate(graphs):
        s = g.src + ptr[i]
        for e, kind in g.ext.items():
            assert kind != "prev" or ptr[i] > 0
            s[e] = {"prev": ptr[i] - 1, "neg": -1, "N": N, "big": 1 << 40}[kind]
        srcs.append(s)
        dsts.append(g.dst + ptr[i])
    counts = np.array([len(g.lut()) for g in graphs], np.int64)
    for gi, k in (lut_extra or {}).items():
        counts[gi] += k
    lut_ptr = np.concatenate([[0], np.cumsum(counts)])
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64))
    return Batch(x=torch.from_numpy(np.concatenate([g.x for g in graphs])),
                 edge_index=torch.stack([t(np.concatenate(srcs)), t(np.concatenate(dsts))]),
                 batch=t(np.repeat(np.arange(len(graphs)), ns)), ptr=t(ptr), edge_ptr=t(eptr), lut_ptr=t(lut_ptr),
                 num_graphs=len(graphs), lut_col=LUT_COL)


def store_of(graphs):
    """The graphs as a host PackedGraphStore (no `ext` sources): what verify_layout judges."""
    from gnn_qot_estimation_b200.batch import PackedGraphStore
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64))
    return PackedGraphStore(t(np.concatenate([[0], np.cumsum([g.n for g in graphs])])),
                            t(np.concatenate([[0], np.cumsum([g.E for g in graphs])])),
                            t(np.concatenate([g.src for g in graphs])), t(np.concatenate([g.dst for g in graphs])),
                            node_feat=torch.from_numpy(np.concatenate([g.x for g in graphs])), lut_col=LUT_COL)


def to_device(hb, dev, node_off=0, edge_off=0, sym=False):
    """The batch on `dev`, x and edge_index as views `node_off` nodes / `edge_off` int64 words into larger
    allocations that end where the views end (x then starts 20 * node_off bytes after a 512-byte boundary)."""
    from gnn_qot_estimation_b200 import Batch
    N, E = hb.x.shape[0], hb.edge_index.shape[1]
    xs = torch.full(((node_off + N) * F,), float("nan"), device=dev)
    x = xs[node_off * F:].view(N, F)
    x.copy_(hb.x)
    es = torch.full((edge_off + 2 * E,), -1, dtype=torch.int64, device=dev)
    ei = es[edge_off:].view(2, E)
    ei.copy_(hb.edge_index)
    return Batch(x=x, edge_index=ei, batch=hb.batch.to(dev), ptr=hb.ptr.to(dev), edge_ptr=hb.edge_ptr.to(dev),
                 lut_ptr=hb.lut_ptr.to(dev), num_graphs=hb.num_graphs, lut_col=LUT_COL, sym_by_src=sym)


def oracle_batch(hb):
    """What the reference is given: the edges whose source lies outside [0, N) (the kernel drops them) removed."""
    from gnn_qot_estimation_b200 import Batch
    N = hb.x.shape[0]
    s = hb.edge_index[0]
    keep = (s >= 0) & (s < N)
    return Batch(x=hb.x.double(), edge_index=hb.edge_index[:, keep], batch=hb.batch, ptr=hb.ptr,
                 num_graphs=hb.num_graphs, lut_col=LUT_COL)


def x_lead(node_off, nb0):
    """Bytes between the 16-byte aligned start of a tile's x copy and node nb0 of a batch slice at node_off."""
    return (node_off + nb0) * F * 4 % 16


def kernel_paths(hb, verified=False):
    """What lp_stream_kernel does with each graph of the batch, restated from lightpath_stream.cu (the window
    sizing of st_producer, the `fits` / hub / source checks of st_consume_tile): 'fast', 'generic', 'none'
    (no LUT node: no row) or 'flagged' (lut_ptr disagrees with x: status bit 1, the generic path fills the rows)."""
    ptr, eptr, lptr = hb.ptr.numpy(), hb.edge_ptr.numpy(), hb.lut_ptr.numpy()
    src, dst = hb.edge_index[0].numpy(), hb.edge_index[1].numpy()
    flag = hb.x[:, LUT_COL].numpy() == 1.0
    B, N = hb.num_graphs, hb.x.shape[0]
    out = []
    for g in range(B):
        t0 = g // TG * TG
        t1 = min(t0 + TG, B)
        xn, en = ptr[t1] - ptr[t0], eptr[t1] - eptr[t0]
        staged = 0 < xn <= T_NODES and en <= T_EDGES
        n0, n1, e0, e1 = ptr[g], ptr[g + 1], eptr[g], eptr[g + 1]
        rows = lptr[g + 1] - lptr[g]
        fits = staged and n1 - n0 <= MAX_N and e1 - e0 <= T_MAX_E and rows <= MAX_N
        lut = np.nonzero(flag[n0:n1])[0] + n0
        cnt = len(lut)
        if cnt != rows:
            out.append("flagged")
        elif cnt == 0:
            out.append("none")
        elif not fits or cnt > 1:
            out.append("generic")
        else:
            il = lut[0]
            ins = np.nonzero(dst[e0:e1] == il)[0] + e0
            if len(ins) > SUB_MSG - 1:
                out.append("generic")
                continue
            if verified:      # the out-run of il: edges [#{dst < il}, + deg) of the graph, destinations as sources
                start = e0 + int((dst[e0:e1] < il).sum())
                s = dst[start:start + len(ins)]
                foreign = bool(((s < n0) | (s >= n1)).any())
            else:
                s = src[ins]
                foreign = bool(((s >= 0) & (s < N) & ((s < n0) | (s >= n1))).any())
            out.append("generic" if foreign else "fast")
    return out


# ------------------------------------------------------------------------------------------------------------------
# cases: each on one side of one boundary; `subjects` = (batch, graph) pairs whose path is the point of the case
# ------------------------------------------------------------------------------------------------------------------
@dataclass
class Case:
    name: str
    batches: list                 # list of graph lists, one launch over all
    subjects: list = field(default_factory=list)
    node_off: int = 0
    edge_off: int = 0
    lut_extra: dict = field(default_factory=dict)   # batch -> {graph: k}
    status: tuple = ()            # batches whose status word must be 1
    force_sym: bool = False       # verified mark set although verify_layout would refuse the layout

    def host(self):
        return [assemble(gs, self.lut_extra.get(i)) for i, gs in enumerate(self.batches)]


def _seed(name, sym):
    return sum(map(ord, name)) * 7919 + (1 if sym else 0)


def _tile_split(total, k=TG):
    base, rem = divmod(total, k)
    return [base + (i < rem) for i in range(k)]


def case_tile_nodes(d, sym):
    """A tile of 16 graphs spanning kTNodes + d nodes and few edges, between two ordinary tiles."""
    rng = np.random.default_rng(_seed("tile_nodes", sym) + d)
    tile = [make_graph(rng, n, 12, lut=i % n, deg=5, sym=sym) for i, n in enumerate(_tile_split(T_NODES + d))]
    gs = small_graphs(rng, TG, sym) + tile + small_graphs(rng, 5, sym)
    return Case(f"tile_nodes_{T_NODES + d}", [gs], [(0, TG + i) for i in range(TG)])


def case_tile_edges(d, sym):
    """A tile of 16 graphs spanning kTEdges + d edges and few nodes."""
    rng = np.random.default_rng(_seed("tile_edges", sym) + d)
    tile = [make_graph(rng, 20, E, lut=-1 - i % 3, deg=6, sym=sym) for i, E in enumerate(_tile_split(T_EDGES + d))]
    gs = small_graphs(rng, 3, sym) + small_graphs(rng, TG - 3, sym) + tile
    return Case(f"tile_edges_{T_EDGES + d}", [gs], [(0, TG + i) for i in range(TG)])


def case_graph_n(n, sym):
    """Graphs of n nodes (kMaxN / kMaxN + 1) at slots 5 and 16 (the next tile's first) among small graphs."""
    rng = np.random.default_rng(_seed("graph_n", sym) + n)
    gs = small_graphs(rng, 17, sym)
    for slot, lut in ((5, 0), (16, -1)):
        gs[slot] = make_graph(rng, n, 40, lut=lut, deg=6, sym=sym, tag=f"n={n}")
    return Case(f"graph_n_{n}", [gs], [(0, 5), (0, 16)])


def case_graph_e(E, sym):
    """Graphs of E edges (kTMaxE - 1 .. kTMaxE + 1) and 48 nodes; the LUT row's in-edges at both ends of the
    8 lanes' contiguous runs of c = ((E + 7) >> 3) | 1 edges (directed builder)."""
    rng = np.random.default_rng(_seed("graph_e", sym) + E)
    c = ((E + 7) >> 3) | 1
    at = None if sym else [p for p in (0, c - 1, c, 2 * c - 1, 7 * c - 1, 7 * c, E - 1) if p < E]
    gs = small_graphs(rng, 20, sym)
    gs[2] = make_graph(rng, 48, E, lut=7, deg=10, loops=1, at=at, sym=sym, tag=f"E={E}")
    gs[19] = make_graph(rng, 48, E, lut=-1, deg=HUB, at=at, sym=sym, tag=f"E={E},deg={HUB}")
    return Case(f"graph_e_{E}", [gs], [(0, 2), (0, 19)])


def case_hub(sym):
    """LUT rows with in-degree kSubMsg - 2 .. kSubMsg, with and without self loops / duplicate edges, and rows
    keeping 7, 8 and 9 messages (8 per round of the online softmax), the LUT node first, last and inside."""
    rng = np.random.default_rng(_seed("hub", sym))
    gs, subj = [], []
    flavours = [(0, 0), (1, 0)] + ([] if sym else [(2, 0), (0, 2), (1, 3)])
    for deg in (HUB - 1, HUB, HUB + 1):
        for loops, dups in flavours:
            for lut in (0, -1):
                gs.append(make_graph(rng, 30, 64, lut=lut, deg=deg, loops=loops, dups=dups, sym=sym,
                                     tag=f"indeg={deg},loops={loops},dups={dups},lut={lut}"))
    for kept in (7, 8, 9):
        for loops in (0, 1):
            gs.append(make_graph(rng, 24, 50, lut=11, deg=kept + loops, loops=loops, sym=sym,
                                 tag=f"kept={kept},loops={loops}"))
    order = rng.permutation(len(gs))
    gs = [gs[i] for i in order]
    subj = [(0, i) for i in range(len(gs))]
    return Case("hub", [gs], subj)


def case_lut_ends(sym):
    """The LUT node at position 0 and n - 1 of graphs of 2, 9, 33 and kMaxN nodes."""
    rng = np.random.default_rng(_seed("lut_ends", sym))
    gs = []
    for n in (2, 9, 33, MAX_N):
        for lut in (0, -1):
            deg = 1 if n == 2 else 5
            gs.append(make_graph(rng, n, 2 if n == 2 else 3 * n, lut=lut, deg=deg, sym=sym, tag=f"n={n},lut={lut}"))
    return Case("lut_ends", [gs], [(0, i) for i in range(len(gs))])


def case_tensor_end(node_off, sym):
    """19 graphs (the last tile holds 3) as a view node_off nodes into a larger allocation: the last tile's x window
    ends at the end of x with x_lead(node_off, nb0) = 4 * ((node_off + nb0) % 4), its destination window at the end
    of edge_index (odd node_off: the view starts 8 bytes off a 16-byte boundary).  The last node is the last graph's
    LUT node and the last edge one of its in-edges, so the bytes a short copy would miss are read.  The graphs are
    the same for every offset (so the window's end takes every residue too); only the features are drawn anew."""
    rng = np.random.default_rng(_seed("tensor_end", sym))
    gs = small_graphs(rng, 18, sym)
    if sym:
        last = make_graph(rng, 21, 40, lut=-1, deg=12, loops=1, sym=True, tag="last")
    else:
        last = make_graph(rng, 21, 40, lut=-1, deg=12, at=[0, 39], tag="last")
    rng = np.random.default_rng(_seed("tensor_end", sym) + 1 + node_off)
    for g in gs + [last]:
        g.x = _rand_x(rng, g.n, g.lut())
    return Case(f"tensor_end_off{node_off}", [gs + [last]], [(0, 16), (0, 17), (0, 18)], node_off=node_off,
                edge_off=node_off % 2)


def case_sources():
    """Sources outside the graph: a node of the previous graph (generic path), and -1, N, 2^40 (outside [0, N):
    dropped, the fast path stays)."""
    rng = np.random.default_rng(_seed("sources", False))
    gs = small_graphs(rng, 20)
    for gi, kinds in ((3, ("prev",)), (6, ("neg", "N", "big")), (9, ("neg", "prev")), (19, ("big",))):
        g = make_graph(rng, 20, 50, lut=4, deg=9, tag=f"sources={kinds}")
        ins = np.nonzero(g.dst == 4)[0]
        g.ext = {int(e): k for e, k in zip(ins, kinds)}
        gs[gi] = g
    return Case("sources", [gs], [(0, 6), (0, 19)])


def case_sym_foreign_dst():
    """Verified layout except in one graph: an edge of the LUT node's out-run leads into the previous graph.  The
    kSym scan reads the row's sources from that run, finds a node outside the graph and hands it to the generic
    path; without the mark the source row is read and the graph is ordinary."""
    rng = np.random.default_rng(_seed("sym_foreign_dst", True))
    gs = small_graphs(rng, 20, True)
    gs[7] = make_graph(rng, 12, 30, lut=0, deg=4, sym=True)   # the node the stray edge reaches is not its LUT node
    g = make_graph(rng, 20, 60, lut=12, deg=6, sym=True, tag="foreign out-run")
    run = np.nonzero((g.src == 12) & (g.dst < 12))[0]
    g.dst = g.dst.copy()
    g.dst[run[0]] = -3                # graph-local -3: the previous graph's third node from the end
    gs[8] = g
    return Case("sym_foreign_dst", [gs], [(0, 8)], force_sym=True)


def case_all_generic(sym):
    """Two staged tiles in which every graph takes the generic path, each for a reason of its own."""
    rng = np.random.default_rng(_seed("all_generic", sym))
    gs = []
    for t in range(2):
        for i in range(TG):
            r = (i + t) % 6
            if r == 0:
                gs.append(make_graph(rng, 24, 48, lut=i % 24, deg=HUB + 1 + i % 5, sym=sym, tag="hub"))
            elif r == 1:
                gs.append(make_graph(rng, 20, 40, luts=[3, 17], sym=sym, deg=4, tag="two LUT nodes"))
            elif r == 2:
                gs.append(make_graph(rng, MAX_N + 1, 30, lut=-1, deg=5, sym=sym, tag="n>kMaxN"))
            elif r == 3:
                gs.append(make_graph(rng, 30, T_MAX_E + 1, lut=0, deg=5, sym=sym, tag="E>kTMaxE"))
            elif r == 4 and not sym and i > 0:
                g = make_graph(rng, 16, 40, lut=2, deg=6, tag="foreign source")
                g.ext = {int(np.nonzero(g.dst == 2)[0][0]): "prev"}
                gs.append(g)
            else:
                gs.append(make_graph(rng, 20, 46, lut=-1, deg=HUB + 2, loops=1, sym=sym, tag="hub with loop"))
    return Case("all_generic", [gs], [])


def case_generic_every_tile(sym):
    """Three batches of 1024 graphs (192 tiles: every SM works at once), a hub graph in every tile at a slot that
    moves with the tile, two LUT nodes in every third tile: the generic path's one scratch per CTA is contended
    inside tiles, between the tiles of one CTA and across CTAs."""
    rng = np.random.default_rng(_seed("generic_every_tile", sym))
    batches = []
    for _ in range(3):
        gs = small_graphs(rng, 1024, sym)
        for t in range(1024 // TG):
            gs[t * TG + t % TG] = make_graph(rng, 20, 48, lut=t % 20, deg=HUB + 1 + t % 4, sym=sym, tag="hub")
            if t % 3 == 0:
                s = t * TG + (t + 7) % TG
                gs[s] = make_graph(rng, 12, 30, luts=[1, 10], deg=3, sym=sym, tag="two LUT nodes")
        batches.append(gs)
    return Case("generic_every_tile", batches, [])


def case_tails(sym):
    """Batches of 1..17, 127, 128 and 129 graphs in one launch: partial tiles, the last graph's n_lut write, and
    readout groups of kGroupTiles tiles that are partly filled and span batch boundaries."""
    rng = np.random.default_rng(_seed("tails", sym))
    sizes = list(range(1, 18)) + [127, 128, 129]
    return Case("tails", [small_graphs(rng, b, sym, 6, 40) for b in sizes], [])


def case_lut_mismatch():
    """lut_ptr claims one row more than x holds LUT nodes for a staged graph with one LUT node, one without LUT
    node and one over the node cap (status bit 1; each graph's LUT nodes fill its first rows, the rest NaN), next
    to fast and generic graphs that are fine, in the second batch of the launch."""
    rng = np.random.default_rng(_seed("lut_mismatch", False))
    gs = small_graphs(rng, 20)
    gs[5] = make_graph(rng, MAX_N + 1, 40, lut=3, deg=5, tag="n>kMaxN")
    gs[6] = make_graph(rng, 20, 40, lut=3, deg=HUB + 1, tag="hub")
    gs[11] = make_graph(rng, 14, 30, lut=None, tag="no LUT node")
    gs[17] = make_graph(rng, MAX_N + 1, 40, lut=9, deg=5, tag="n>kMaxN")
    return Case("lut_mismatch", [small_graphs(rng, 9), gs], [], lut_extra={1: {4: 1, 11: 1, 17: 1}}, status=(1,))


SYM_CASES = {
    **{f"tile_nodes_{T_NODES + d}": (lambda s, d=d: case_tile_nodes(d, s)) for d in (0, 1)},
    **{f"tile_edges_{T_EDGES + d}": (lambda s, d=d: case_tile_edges(d, s)) for d in (0, 1)},
    **{f"graph_n_{n}": (lambda s, n=n: case_graph_n(n, s)) for n in (MAX_N, MAX_N + 1)},
    **{f"graph_e_{E}": (lambda s, E=E: case_graph_e(E, s)) for E in (T_MAX_E - 1, T_MAX_E, T_MAX_E + 1)},
    "hub": case_hub,
    "lut_ends": case_lut_ends,
    **{f"tensor_end_off{k}": (lambda s, k=k: case_tensor_end(k, s)) for k in range(4)},
    "all_generic": case_all_generic,
    "generic_every_tile": case_generic_every_tile,
    "tails": case_tails,
}
DIRECTED_CASES = {"sources": case_sources, "lut_mismatch": case_lut_mismatch, "sym_foreign_dst": case_sym_foreign_dst}


@functools.lru_cache(maxsize=None)
def build_case(name, sym):
    """The case `name` with the verified layout (sym) or the directed builder with self loops and duplicates."""
    if name in SYM_CASES:
        return SYM_CASES[name](sym)
    assert not sym or name == "sym_foreign_dst"
    return DIRECTED_CASES[name]()


# (case, verified) pairs the GPU test runs; sym_foreign_dst: the verified mark is forced onto a layout that breaks it
RUNS = [(c, v) for c in SYM_CASES for v in (False, True)] + [("sources", False), ("lut_mismatch", False),
                                                            ("sym_foreign_dst", False), ("sym_foreign_dst", True)]


# ------------------------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------------------------
def _state_dict(weights):
    """'ckpt0' / 'ckpt1': the shipped checkpoints; 'randK': random weights, attention vectors scaled by 8 (a
    peaked softmax: large jumps of the running maximum between 8-message rounds), BatchNorm with nontrivial
    running statistics and affine parameters."""
    if weights.startswith("ckpt"):
        return load_golden(f"ckpt_lightpath_model_{weights[4:]}.pt")["model_state_dict"]
    from gnn_qot_estimation_b200 import LightpathGNN
    seed = int(weights[4:])
    torch.manual_seed(1000 + seed)
    sd = {k: v.clone() for k, v in LightpathGNN(5, 32, 3, is_lut_index=LUT_COL, dropout_p=0.0).state_dict().items()}
    g = torch.Generator().manual_seed(seed)
    sd["conv1.att_src"] *= 8.0
    sd["conv1.att_dst"] *= 8.0
    sd["conv1.bias"] = 0.1 * torch.randn(sd["conv1.bias"].shape, generator=g)
    sd["norm1.module.running_mean"] = 0.3 * torch.randn(128, generator=g)
    sd["norm1.module.running_var"] = 0.2 + torch.rand(128, generator=g)
    sd["norm1.module.weight"] = 1.0 + 0.5 * torch.randn(128, generator=g)
    sd["norm1.module.bias"] = 0.2 * torch.randn(128, generator=g)
    return sd


_MODELS = {}


def _models(weights, dev):
    if weights not in _MODELS:
        from gnn_qot_estimation_b200 import LightpathGNN
        from oracle import LightpathGNNOracle
        sd = _state_dict(weights)
        m = LightpathGNN(5, 32, 3, is_lut_index=LUT_COL, dropout_p=0.0)
        m.load_state_dict(sd, strict=True)
        o = LightpathGNNOracle(5, 32, 3, is_lut_index=LUT_COL, dropout_p=0.0).double()
        o.load_state_dict(sd, strict=True)
        _MODELS[weights] = (m.to(dev).eval(), o.eval())
    return _MODELS[weights]


def _launch(m, dbs, split_head):
    plan = m.stream_plan(dbs, split_head=split_head)
    plan.out.fill_(float("nan"))
    plan.lut_batch.fill_(-7)
    plan.lut_node.fill_(-7)
    m.forward_stream(plan)
    torch.cuda.synchronize()
    return plan


def path_refs(m, graphs, split_head, dev):
    """Each graph alone in a staged tile (fillers of one node after it) and in a tile the producer does not stage
    (a filler of kTNodes + 1 nodes after it): its fast-path and its generic-path row (or its generic row twice, if a
    cap of its own sends it there), in order."""
    rng = np.random.default_rng(5)
    tiny = filler(rng, 1)
    big = filler(rng, T_NODES + 1)
    fast = [h for g in graphs for h in [g] + [tiny] * (TG - 1)]
    gen = [h for g in graphs for h in [g, big] + [tiny] * (TG - 2)]
    outs = []
    for gs in (fast, gen):
        hb = assemble(gs)
        plan = _launch(m, [to_device(hb, dev)], split_head)
        assert int(plan.status[0]) == 0
        outs.append(plan.out[:len(graphs)].cpu())
    return outs


def check_case(case, verified, split_head, weights, dev):
    m, o = _models(weights, dev)
    hbs = case.host()
    if verified and not case.force_sym:
        assert all(store_of(gs).verify_layout() for gs in case.batches), case.name
    dbs = [to_device(hb, dev, case.node_off, case.edge_off, verified) for hb in hbs]
    plan = _launch(m, dbs, split_head)
    assert plan.flags == (1 if verified else 0) | (2 if split_head else 0)
    for b, (hb, db) in enumerate(zip(hbs, dbs)):
        where = f"{case.name}: batch {b}"
        r = plan.result(b)
        lptr = hb.lut_ptr.numpy()
        paths = kernel_paths(hb, verified)
        assert int(r.status) == (1 if b in case.status else 0), where
        assert int(r.n_lut) == int(lptr[-1]), where
        # true rows (oracle order) and kernel rows of every graph lut_ptr describes correctly
        flag = hb.x[:, LUT_COL].numpy() == 1.0
        nodes = np.nonzero(flag)[0]
        gof = hb.batch.numpy()[nodes]
        krow, trow = [], []
        for g, p in enumerate(paths):
            t = np.nonzero(gof == g)[0]
            k = min(len(t), lptr[g + 1] - lptr[g])
            krow += list(range(lptr[g], lptr[g] + k))      # rows of the graph's LUT nodes, as far as lut_ptr has rows
            trow += list(t[:k])
            if p == "flagged":            # lut_ptr disagrees with x: the rows past its LUT nodes are NaN, lut_node -1
                rest = slice(lptr[g] + k, lptr[g + 1])
                assert torch.isnan(r.out[rest]).all(), (where, g)
                assert (r.lut_node[rest] == -1).all() and (r.lut_batch[rest] == g).all(), (where, g)
        krow, trow = torch.tensor(krow, dtype=torch.long), torch.tensor(trow, dtype=torch.long)
        out = r.out.cpu()[krow]
        assert torch.equal(r.lut_batch.cpu()[krow], torch.from_numpy(gof[trow.numpy()])), where
        assert torch.equal(r.lut_node.cpu()[krow].long(), torch.from_numpy(nodes[trow.numpy()])), where
        with torch.no_grad():
            eo, _ = o(oracle_batch(hb))
        eo = eo[trow]
        assert rel_err(out, eo) <= RTOL, (where, rel_err(out, eo))
        torch.testing.assert_close(out.double(), eo, rtol=RTOL, atol=ABS_FLOOR, msg=lambda s: f"{where}: {s}")
        # the one-launch-per-batch module path: the same rows; bit for bit when it uses the same readout head
        from gnn_qot_estimation_b200 import Batch
        view = Batch(x=db.x, edge_index=db.edge_index, ptr=db.ptr, edge_ptr=db.edge_ptr, lut_ptr=db.lut_ptr,
                     num_graphs=db.num_graphs, lut_col=LUT_COL, sym_by_src=verified)
        mr = m.forward_device(view)
        torch.cuda.synchronize()
        assert int(mr.status) == int(r.status), where
        assert int(mr.n_lut) == int(r.n_lut), where
        assert torch.equal(mr.lut_batch.cpu()[krow], r.lut_batch.cpu()[krow]), where
        assert torch.equal(mr.lut_node.cpu()[krow], r.lut_node.cpu()[krow]), where
        if split_head:
            torch.testing.assert_close(mr.out.cpu()[krow], out, rtol=RTOL, atol=ABS_FLOOR)
        else:
            assert torch.equal(mr.out.cpu()[krow], out), where
    # the path each subject took, bit for bit
    subj = [(b, g) for b, g in case.subjects if "prev" not in case.batches[b][g].ext.values()]
    if subj:
        graphs = [case.batches[b][g] for b, g in subj]
        fast, gen = path_refs(m, graphs, split_head, dev)
        ref_paths = kernel_paths(assemble([h for g in graphs for h in [g] + [filler(np.random.default_rng(5), 1)] *
                                           (TG - 1)]))
        told = 0
        for i, (b, g) in enumerate(subj):
            p = kernel_paths(hbs[b], verified)[g]
            row = int(hbs[b].lut_ptr[g])
            got = plan.result(b).out[row].cpu()
            tag = f"{case.name}: graph {g} ({case.batches[b][g].tag}) should take the {p} path"
            if ref_paths[TG * i] == "fast":      # its own caps allow the fast path
                # the in-kernel head (tcgen05, TF32 x3) and the generic path's FP32 head never agree to the bit; the
                # split build runs one head for both, so only the attention sums tell the paths apart there
                told += not torch.equal(fast[i], gen[i])
                assert split_head or not torch.equal(fast[i], gen[i]), f"{tag}: fast and generic rows coincide"
            assert torch.equal(got, fast[i] if p == "fast" else gen[i]), f"{tag}: {got.tolist()} vs fast " \
                f"{fast[i].tolist()} / generic {gen[i].tolist()}"
        if "fast" in ref_paths[::TG]:
            assert told, f"{case.name}: no subject's fast and generic rows differ, the paths are not told apart"


@pytest.mark.parametrize("split_head", [False, True])
@pytest.mark.parametrize("name,verified", RUNS)
def test_stream_caps(cuda, name, verified, split_head):
    check_case(build_case(name, verified), verified, split_head, "ckpt1", cuda)


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("split_head", [False, True])
@pytest.mark.parametrize("name", ["hub", "graph_e_%d" % T_MAX_E, "tensor_end_off1", "all_generic", "tails",
                                  "sources"])
def test_stream_caps_random_weights(cuda, name, split_head, seed):
    check_case(build_case(name, False), False, split_head, f"rand{seed}", cuda)


@pytest.mark.parametrize("split_head", [False, True])
@pytest.mark.parametrize("sizes", [[40, 40, 40, 40, 7], [33, 16, 70, 1, 48]])
def test_stream_sub_range(cuda, sizes, split_head):
    """forward_stream(plan, i, k) from every batch index of a 5-batch plan (uniform and searched tile counts)
    rewrites exactly batches [i, i + k), bit for bit as the full launch."""
    m, _ = _models("ckpt0", cuda)
    rng = np.random.default_rng(sum(sizes))
    dbs = [to_device(assemble(small_graphs(rng, s)), cuda) for s in sizes]
    plan = _launch(m, dbs, split_head)
    full = (plan.out.clone(), plan.lut_batch.clone(), plan.lut_node.clone())
    for i in range(5):
        for k in sorted({1, 5 - i}):
            plan.out.fill_(float("nan"))
            plan.lut_batch.fill_(-7)
            plan.lut_node.fill_(-7)
            m.forward_stream(plan, i, k)
            torch.cuda.synchronize()
            a, b = plan.off[i], plan.off[i + k]
            for buf, ref, blank in zip((plan.out, plan.lut_batch, plan.lut_node), full, (float("nan"), -7, -7)):
                assert torch.equal(buf[a:b], ref[a:b]), (i, k)
                rest = torch.cat([buf[:a], buf[b:]])
                assert (rest.isnan() if blank != -7 else rest == -7).all(), (i, k)
