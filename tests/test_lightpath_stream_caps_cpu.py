"""The case builders of test_lightpath_stream_caps_gpu.py sit on the boundaries they name (no GPU needed): tile
node and edge spans, per-graph n and E, LUT in-degree and kept messages, the x_lead residue and the tail bytes of a
window that ends at the end of x, the layout verify_layout accepts.  The caps come from the CUDA sources, so a
changed constant moves the cases with it; a later edit to a builder that moves a case off its boundary fails here."""
import numpy as np
import pytest

from test_lightpath_stream_caps_gpu import (F, GROUP_TILES, HUB, MAX_N, RUNS, SUB_MSG, T_EDGES, T_MAX_E, T_NODES, TG,
                                            build_case, kernel_paths, store_of, x_lead)


def _case(name, sym=False):
    c = build_case(name, sym)
    return c, c.host()


def test_caps_read_from_the_sources():
    assert TG == 16 and GROUP_TILES * TG == 128          # readout group = the 128 rows of one MMA
    assert 0 < MAX_N and 0 < T_MAX_E and SUB_MSG > 8      # 8 messages per softmax round: a row can cross one
    assert TG * MAX_N > T_NODES and TG * T_MAX_E > T_EDGES   # a tile of graphs within their own caps can overflow


@pytest.mark.parametrize("name,verified", RUNS)
def test_case_layout_and_paths(name, verified):
    """Every batch is well formed; the symmetric builder passes verify_layout, the directed one does not; every
    subject takes the path its boundary implies."""
    c, hbs = _case(name, verified)
    for gs, hb in zip(c.batches, hbs):
        ptr, eptr = hb.ptr.numpy(), hb.edge_ptr.numpy()
        assert ptr[-1] == hb.x.shape[0] and eptr[-1] == hb.edge_index.shape[1]
        ei = hb.edge_index.numpy()
        ext = sum(len(g.ext) for g in gs)
        g_of_e = np.repeat(np.arange(len(gs)), np.diff(eptr))
        inside = (ei >= ptr[g_of_e]) & (ei < ptr[g_of_e + 1])
        assert inside[1].sum() + (name == "sym_foreign_dst") == ei.shape[1]    # destinations inside their graph
        assert ei.shape[1] - inside[0].sum() == ext                              # sources: only the declared ones
        if verified and not c.force_sym:
            assert store_of(gs).verify_layout()
        elif name not in ("sources", "lut_mismatch", "sym_foreign_dst"):
            assert not store_of(gs).verify_layout()                              # duplicates / unpaired edges
    for b, g in c.subjects:
        hb = hbs[b]
        p = kernel_paths(hb, verified)[g]
        assert p in ("fast", "generic")
        assert c.batches[b][g].n <= MAX_N + 1


def _tile_span(hb, t):
    ptr, eptr = hb.ptr.numpy(), hb.edge_ptr.numpy()
    t1 = min(TG * (t + 1), hb.num_graphs)
    return ptr[t1] - ptr[TG * t], eptr[t1] - eptr[TG * t]


@pytest.mark.parametrize("sym", [False, True])
@pytest.mark.parametrize("d", [0, 1])
def test_tile_boundaries(sym, d):
    c, (hb,) = _case(f"tile_nodes_{T_NODES + d}", sym)
    xn, en = _tile_span(hb, 1)
    assert xn == T_NODES + d and en <= T_EDGES // 4
    assert all(g.n <= MAX_N and g.E <= T_MAX_E for g in c.batches[0][TG:2 * TG])
    assert set(kernel_paths(hb, sym)[TG:2 * TG]) == {"generic" if d else "fast"}
    c, (hb,) = _case(f"tile_edges_{T_EDGES + d}", sym)
    xn, en = _tile_span(hb, 1)
    assert en == T_EDGES + d and xn <= T_NODES // 2
    assert all(g.n <= MAX_N and g.E <= T_MAX_E for g in c.batches[0][TG:2 * TG])
    assert set(kernel_paths(hb, sym)[TG:2 * TG]) == {"generic" if d else "fast"}


@pytest.mark.parametrize("sym", [False, True])
def test_graph_boundaries(sym):
    for n in (MAX_N, MAX_N + 1):
        c, (hb,) = _case(f"graph_n_{n}", sym)
        for _, g in c.subjects:
            assert c.batches[0][g].n == n and kernel_paths(hb, sym)[g] == ("fast" if n == MAX_N else "generic")
        assert [g for _, g in c.subjects] == [5, TG]                               # inside a tile and first of the next
    for E in (T_MAX_E - 1, T_MAX_E, T_MAX_E + 1):
        c, (hb,) = _case(f"graph_e_{E}", sym)
        for _, gi in c.subjects:
            g = c.batches[0][gi]
            assert g.E == E and g.n <= MAX_N
            assert kernel_paths(hb, sym)[gi] == ("fast" if E <= T_MAX_E else "generic")
        assert max(c.batches[0][gi].indeg() for _, gi in c.subjects) == HUB
    # E = kTMaxE: 8 lanes x c edges exactly, c odd; the LUT row's in-edges at both ends of lane runs
    c = ((T_MAX_E + 7) >> 3) | 1
    assert 8 * c == T_MAX_E and c % 2 == 1
    if not sym:
        g = build_case(f"graph_e_{T_MAX_E}", False).batches[0][2]
        ins = set(np.nonzero(g.dst == g.lut()[0])[0].tolist())
        assert {0, c - 1, c, 7 * c - 1, 7 * c, T_MAX_E - 1} <= ins


@pytest.mark.parametrize("sym", [False, True])
def test_hub_rows(sym):
    c, (hb,) = _case("hub", sym)
    gs = c.batches[0]
    paths = kernel_paths(hb, sym)
    degs = {g.indeg() for g in gs}
    assert {SUB_MSG - 2, SUB_MSG - 1, SUB_MSG} <= degs
    assert {7, 8, 9} <= {g.kept() for g in gs}
    for i, g in enumerate(gs):
        assert paths[i] == ("fast" if g.indeg() <= SUB_MSG - 1 else "generic"), g.tag
    loops = lambda g: int(((g.src == g.lut()[0]) & (g.dst == g.lut()[0])).sum())
    dups = lambda g: g.indeg() - loops(g) - len(set(g.src[g.dst == g.lut()[0]].tolist()) - {g.lut()[0]})
    for deg in (SUB_MSG - 1, SUB_MSG):                   # each side of the cap with self loops, and with duplicates
        assert any(g.indeg() == deg and loops(g) for g in gs)
        assert sym or any(g.indeg() == deg and dups(g) for g in gs)
    assert {0, 1} <= {int(g.lut()[0] == g.n - 1) for g in gs}     # the LUT node first and last


def test_lut_ends():
    c, (hb,) = _case("lut_ends")
    pos = {(g.n, int(g.lut()[0])) for g in c.batches[0]}
    for n in (2, 9, 33, MAX_N):
        assert {(n, 0), (n, n - 1)} <= pos
    assert set(kernel_paths(hb)) == {"fast"}


@pytest.mark.parametrize("sym", [False, True])
def test_tensor_end_residues(sym):
    """The last tile's window ends at the end of x and edge_index; over node offsets 0..3 every x_lead residue
    occurs, and three of four windows end off a 16-byte boundary (the hand-copied tail)."""
    leads, tails = set(), []
    for k in range(4):
        c, (hb,) = _case(f"tensor_end_off{k}", sym)
        N, E, B = hb.x.shape[0], hb.edge_index.shape[1], hb.num_graphs
        t = (B - 1) // TG
        nb0, eb0 = int(hb.ptr[TG * t]), int(hb.edge_ptr[TG * t])
        assert 0 < B - TG * t < TG                                  # a partial last tile
        xn, en = _tile_span(hb, t)
        assert nb0 + xn == N and eb0 + en == E and xn <= T_NODES and en <= T_EDGES
        leads.add(x_lead(c.node_off, nb0))
        tails.append((c.node_off + N) * F * 4 % 16)                 # bytes past the last 16-byte boundary of x
        assert c.edge_off == k % 2
        last = c.batches[0][-1]
        assert last.lut()[0] == last.n - 1                          # the bytes a short copy would miss are read
        assert last.dst[-1] == last.n - 1                           # so is the last edge's destination
        assert kernel_paths(hb, sym)[-1] == "fast"
    assert leads == {0, 4, 8, 12}
    assert sorted(tails) == [0, 4, 8, 12]


def test_sources():
    c, (hb,) = _case("sources")
    p = kernel_paths(hb)
    kinds = {gi: set(c.batches[0][gi].ext.values()) for gi in range(hb.num_graphs) if c.batches[0][gi].ext}
    assert kinds == {3: {"prev"}, 6: {"neg", "N", "big"}, 9: {"neg", "prev"}, 19: {"big"}}
    assert [p[g] for g in (3, 6, 9, 19)] == ["generic", "fast", "generic", "fast"]
    N = hb.x.shape[0]
    src = hb.edge_index[0].numpy()
    assert {-1, N, 1 << 40} <= set(src.tolist())


def test_sym_foreign_dst():
    c, (hb,) = _case("sym_foreign_dst")
    assert kernel_paths(hb, True)[8] == "generic" and kernel_paths(hb, False)[8] == "fast"
    g7 = c.batches[0][7]
    assert g7.lut()[0] != g7.n - 3                                  # the stray edge does not reach a readout row


@pytest.mark.parametrize("sym", [False, True])
def test_generic_cases(sym):
    c, (hb,) = _case("all_generic", sym)
    assert hb.num_graphs == 2 * TG
    assert set(kernel_paths(hb, sym)) == {"generic"}
    for t in range(2):
        xn, en = _tile_span(hb, t)
        assert xn <= T_NODES and en <= T_EDGES                      # staged: every graph is generic on its own account
    c, hbs = _case("generic_every_tile", sym)
    assert sum(hb.num_graphs for hb in hbs) // TG >= 148            # more tiles than SMs
    for hb in hbs:
        p = kernel_paths(hb, sym)
        assert all("generic" in p[t:t + TG] for t in range(0, hb.num_graphs, TG))


def test_tails_and_mismatch():
    c, hbs = _case("tails")
    assert [hb.num_graphs for hb in hbs] == list(range(1, 18)) + [127, 128, 129]
    c, hbs = _case("lut_mismatch")
    p = kernel_paths(hbs[1])
    assert [p[g] for g in (4, 11, 17)] == ["flagged"] * 3 and p[5] == p[6] == "generic" and p.count("fast") == 15
    assert [len(c.batches[1][g].lut()) for g in (4, 11, 17)] == [1, 0, 1]
    assert set(kernel_paths(hbs[0])) == {"fast"}
