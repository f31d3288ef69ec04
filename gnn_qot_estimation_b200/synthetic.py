"""Seeded synthetic graph generators for the BASELINE.json configurations.

The reference's dataset (HHI ``.nc`` -> networkx pickles) is not shipped
(SURVEY.md 0.5), so every measurable workload is synthetic, in the exact tensor
layout the reference datasets emit (topological_training/dataset.py:75-123,
lightpath_training/dataset.py:86-123): edges in ``from_networkx`` order (both
directions of every undirected link, grouped by source node ascending).

Generators are vectorised torch code and run on any device (GPU for the 1M-graph
inference workload, CPU for tests).
"""
from __future__ import annotations

from typing import List, Tuple

import torch

from .batch import PackedGraphStore

# NSFNET T1 backbone: 14 nodes, 21 undirected links (BASELINE cfg 1/3).
NSFNET_LINKS: List[Tuple[int, int]] = [
    (0, 1), (0, 2), (0, 7), (1, 2), (1, 3), (2, 5), (3, 4), (3, 10), (4, 5), (4, 6),
    (5, 9), (5, 13), (6, 7), (7, 8), (8, 9), (8, 11), (8, 12), (10, 11), (10, 12),
    (11, 13), (12, 13),
]


def directed_from_undirected(num_nodes: int, links: List[Tuple[int, int]]):
    """Directed edge list in ``from_networkx`` order: for each source node ascending,
    its neighbours in adjacency-insertion order (SURVEY.md A.6).  Also returns, for
    each directed edge, the index of the undirected link it mirrors."""
    adj = [[] for _ in range(num_nodes)]
    for li, (u, v) in enumerate(links):
        adj[u].append((v, li))
        if u != v:
            adj[v].append((u, li))
    src, dst, lid = [], [], []
    for u in range(num_nodes):
        for v, li in adj[u]:
            src.append(u)
            dst.append(v)
            lid.append(li)
    return src, dst, lid


def nsfnet_store(num_graphs: int, seed: int = 0, device="cpu") -> PackedGraphStore:
    """cfg 1/3: `num_graphs` copies of NSFNET (14 nodes, 42 directed edges), edge_attr
    ~ U[0,1) per undirected link mirrored on both directions, y ~ U[0,1) [G,3];
    no node features (node_ids + embeddings)."""
    gen = torch.Generator(device="cpu").manual_seed(seed)
    src, dst, lid = directed_from_undirected(14, NSFNET_LINKS)
    n_e = len(src)
    link_attr = torch.rand(num_graphs, len(NSFNET_LINKS), 4, generator=gen)
    edge_feat = link_attr[:, torch.tensor(lid)].reshape(num_graphs * n_e, 4).contiguous()
    y = torch.rand(num_graphs, 3, generator=gen)
    node_ptr = torch.arange(num_graphs + 1, dtype=torch.int64) * 14
    edge_ptr = torch.arange(num_graphs + 1, dtype=torch.int64) * n_e
    es = torch.tensor(src, dtype=torch.int32).repeat(num_graphs)
    ed = torch.tensor(dst, dtype=torch.int32).repeat(num_graphs)
    return PackedGraphStore(node_ptr, edge_ptr, es, ed, None, edge_feat, y).to(device)


def lightpath_store(num_graphs: int, seed: int = 1, device="cpu", n_min: int = 8, n_max: int = 56,
                    lut_per_graph: int = 1) -> PackedGraphStore:
    """cfg 2/4: per graph n ~ U{n_min..n_max} lightpath nodes, ~2n random undirected
    interference links (duplicates collapsed like nx.Graph does; mean directed degree
    ~3.8), exactly ``lut_per_graph`` nodes with is_lut == 1.0 (column 1), the other four
    features ~ U[0,1); y ~ U[0,1) [G,3].  Feature order
    [freq, is_lut, mod_order, num_spans, path_len] (lightpath_training/dataset.py:45-48)."""
    dev = torch.device(device)
    gen = torch.Generator(device=dev).manual_seed(seed)
    G = num_graphs
    n = torch.randint(n_min, n_max + 1, (G,), generator=gen, device=dev, dtype=torch.int64)
    node_ptr = torch.zeros(G + 1, dtype=torch.int64, device=dev)
    node_ptr[1:] = torch.cumsum(n, 0)
    N = int(node_ptr[-1])
    m = 2 * n                                                  # undirected samples per graph
    mptr = torch.zeros(G + 1, dtype=torch.int64, device=dev)
    mptr[1:] = torch.cumsum(m, 0)
    M = int(mptr[-1])
    gid = torch.repeat_interleave(torch.arange(G, device=dev), m)
    ng = n[gid]
    u = (torch.rand(M, generator=gen, device=dev) * ng).long()
    u = torch.minimum(u, ng - 1)
    step = 1 + torch.minimum((torch.rand(M, generator=gen, device=dev) * (ng - 1)).long(), ng - 2)
    v = (u + step) % ng                                        # v != u
    lo, hi = torch.minimum(u, v), torch.maximum(u, v)
    key = (gid * 64 + lo) * 64 + hi                            # n_max <= 63
    key = torch.unique(key)                                    # nx.Graph keeps one edge per pair
    g_u = key // 4096
    lo, hi = (key // 64) % 64, key % 64
    # both directions, grouped by (graph, source) ascending, then by target
    dsrc = torch.cat([lo, hi])
    ddst = torch.cat([hi, lo])
    dg = torch.cat([g_u, g_u])
    order = torch.argsort((dg * 64 + dsrc) * 64 + ddst)
    dsrc, ddst, dg = dsrc[order], ddst[order], dg[order]
    edge_ptr = torch.zeros(G + 1, dtype=torch.int64, device=dev)
    edge_ptr[1:] = torch.cumsum(torch.bincount(dg, minlength=G), 0)
    x = torch.rand(N, 5, generator=gen, device=dev)
    x[:, 1] = 0.0
    for k in range(lut_per_graph):
        pos = torch.minimum((torch.rand(G, generator=gen, device=dev) * n).long(), n - 1)
        x[node_ptr[:-1] + pos, 1] = 1.0
    y = torch.rand(G, 3, generator=gen, device=dev)
    return PackedGraphStore(node_ptr, edge_ptr, dsrc.to(torch.int32), ddst.to(torch.int32), x, None, y, lut_col=1)


def random_topology_store(num_nodes: int = 10000, num_links: int = 40000, seed: int = 2,
                          device="cpu") -> PackedGraphStore:
    """cfg 5: ONE graph with `num_nodes` nodes and `num_links` random undirected links
    (both directions -> 2*num_links directed edges, grouped by source), edge_attr
    ~ U[0,1) per link mirrored.  No node features (embedding table of num_nodes rows)."""
    gen = torch.Generator(device="cpu").manual_seed(seed)
    u = torch.randint(0, num_nodes, (num_links,), generator=gen)
    v = (u + 1 + torch.randint(0, num_nodes - 1, (num_links,), generator=gen)) % num_nodes
    attr = torch.rand(num_links, 4, generator=gen)
    src = torch.cat([u, v])
    dst = torch.cat([v, u])
    ea = torch.cat([attr, attr])
    order = torch.argsort(src * num_nodes + dst, stable=True)
    src, dst, ea = src[order], dst[order], ea[order].contiguous()
    node_ptr = torch.tensor([0, num_nodes], dtype=torch.int64)
    edge_ptr = torch.tensor([0, src.numel()], dtype=torch.int64)
    y = torch.rand(1, 3, generator=gen)
    return PackedGraphStore(node_ptr, edge_ptr, src.to(torch.int32), dst.to(torch.int32), None, ea, y).to(device)


# --------------------------------------------------------------------------------------------- #
# raw "network status" samples: the input of to_graph.py (the HHI .nc dataset is not shipped)
# --------------------------------------------------------------------------------------------- #
LP_FEAT = ["conn_id", "src_id", "dst_id", "mod_order", "path_len", "num_spans", "freq", "osnr", "snr", "ber"]
METRICS = ["osnr", "snr", "ber", "class"]


def network_status_samples(num_samples: int, num_links: int = 40, num_freqs: int = 64, seed: int = 0,
                           spacing: float = 0.0375, max_lightpaths: int = 48, super_channel_p: float = 0.1,
                           num_nodes: int = 75):
    """Seeded stand-in for ``dataset["data"]`` of to_graph.py:124-129: a float32 array
    ``[sample, lp_feat, link, freq]`` that is zero on free channels and carries the lightpath's
    feature vector on every (link, frequency) channel it occupies, plus ``target [sample, 4]``,
    the frequency grid ``freqs [num_freqs]`` (float64, 192.2 + k*spacing) and the name lists.
    Every sample holds 8..max_lightpaths lightpaths routed over 1..6 random links with one
    frequency slot each (a few take two adjacent slots: super-channels, which to_graph.py turns
    into self loops); the last lightpath placed is the LUT (osnr = snr = ber = -1).  Endpoints are drawn
    from 1..num_nodes (small values give many lightpaths per node pair: nx.Graph keeps one edge, last
    attributes win, to_graph.py:175-178)."""
    import numpy as np
    rng = np.random.default_rng(seed)
    F = len(LP_FEAT)
    fi = {k: i for i, k in enumerate(LP_FEAT)}
    freqs = 192.2 + spacing * np.arange(num_freqs, dtype=np.float64)
    data = np.zeros((num_samples, F, num_links, num_freqs), dtype=np.float32)
    target = np.zeros((num_samples, len(METRICS)), dtype=np.float64)
    for s in range(num_samples):
        n_lp = int(rng.integers(8, max_lightpaths + 1))
        free = np.ones((num_links, num_freqs), dtype=bool)
        conn_ids = rng.permutation(np.arange(1, 4 * max_lightpaths))[:n_lp]
        placed = 0
        for k in range(n_lp):
            width = 2 if rng.random() < super_channel_p else 1
            links = rng.choice(num_links, size=min(int(rng.integers(1, 7)), num_links), replace=False)
            ok_q = [q for q in range(num_freqs - width + 1) if all(free[l, q:q + width].all() for l in links)]
            if not ok_q:
                continue
            q0 = int(rng.choice(ok_q))
            vec = np.zeros(F, dtype=np.float32)
            vec[fi["conn_id"]] = conn_ids[k]
            vec[fi["src_id"]], vec[fi["dst_id"]] = rng.choice(np.arange(1, num_nodes + 1), 2, replace=False)
            vec[fi["mod_order"]] = rng.choice([4, 8, 16, 32, 64])
            vec[fi["path_len"]] = int(rng.integers(24214, 7834746))
            vec[fi["num_spans"]] = int(rng.integers(1, 107))
            vec[fi["osnr"]], vec[fi["snr"]], vec[fi["ber"]] = rng.uniform(13, 33), rng.uniform(9, 29), rng.uniform(1e-11, 1e-2)
            for l in links:
                for q in range(q0, q0 + width):
                    v = vec.copy()
                    v[fi["freq"]] = freqs[q]
                    data[s, :, l, q] = v
                    free[l, q] = False
            placed += 1
            last = (links, q0, width)
        links, q0, width = last                       # the LUT: metrics unknown (-1), to be predicted
        for l in links:
            for q in range(q0, q0 + width):
                data[s, fi["osnr"], l, q] = data[s, fi["snr"], l, q] = data[s, fi["ber"], l, q] = -1.0
        target[s] = [rng.uniform(12.47, 33.49), rng.uniform(8.96, 29.98), rng.uniform(1.7e-12, 1.98e-2), rng.integers(0, 3)]
    return {"data": data, "target": target, "freqs": freqs, "lp_feat": list(LP_FEAT), "metric": list(METRICS)}


def lightpath_candidates(samples, per_sample: int, seed: int = 0):
    """Seeded candidate lightpaths for the network-status ``samples`` (the dict ``network_status_samples`` returns):
    ``per_sample`` candidates per sample, each on 1..6 distinct random links with one slot (or two adjacent slots,
    probability 0.1) that is free on every link of its path; ``feat = (float32(freqs[q0]), mod_order, num_spans,
    path_len)`` as ``network_status_samples`` writes a lightpath's first channel.  A sample too full to place a
    candidate after 64 draws gets fewer.  Returns ``to_graph.LightpathCandidates`` of CPU tensors (``.to(device)``)."""
    import numpy as np
    from .to_graph import LightpathCandidates
    rng = np.random.default_rng(seed)
    data, freqs = samples["data"], samples["freqs"]
    S, _, L, Q = data.shape
    occupied = np.any(data != 0, axis=1)                       # [S, L, Q]
    smp, lptr, links, q0s, widths, feats = [], [0], [], [], [], []
    for s in range(S):
        for _ in range(per_sample):
            for _try in range(64):
                width = 2 if rng.random() < 0.1 else 1
                path = rng.choice(L, size=min(int(rng.integers(1, 7)), L), replace=False)
                free = ~occupied[s, path].any(axis=0)          # [Q]
                ok = free[:Q - width + 1].copy()
                for u in range(1, width):
                    ok &= free[u:Q - width + 1 + u]
                cand = np.flatnonzero(ok)
                if cand.size:
                    break
            else:
                continue
            q0 = int(rng.choice(cand))
            smp.append(s)
            links.extend(int(l) for l in path)
            lptr.append(len(links))
            q0s.append(q0)
            widths.append(width)
            feats.append([np.float32(freqs[q0]), rng.choice([4, 8, 16, 32, 64]), int(rng.integers(1, 107)),
                          int(rng.integers(24214, 7834746))])
    return LightpathCandidates(torch.tensor(smp, dtype=torch.int64), torch.tensor(lptr, dtype=torch.int64),
                               torch.tensor(links, dtype=torch.int32), torch.tensor(q0s, dtype=torch.int32),
                               torch.tensor(widths, dtype=torch.int32),
                               torch.tensor(np.array(feats, dtype=np.float32).reshape(-1, 4)))


def lightpath_changes(samples, state, per_sample: int, seed: int = 0):
    """Seeded changes to the lightpaths of ``samples`` (the dict ``network_status_samples`` returns), whose network
    state ``state`` is (``to_graph.lightpath_network_state``; its node numbering gives ``node``).  ``per_sample``
    changes per sample, a mix of
      - retunes (0.35): the lightpath on its own links at another slot of its own width; half of them take the nearest
        slot, which overlaps its own slots for a super-channel;
      - reroutes (0.30): onto 1..6 distinct random links, its own width, new num_spans and path_len;
      - teardowns (0.20): an empty path (q0, width and feat are the lightpath's own, and unused);
      - insertions (0.15): node -1, as ``lightpath_candidates`` draws them.
    A move keeps the lightpath's mod_order and sets ``freq = float32(freqs[q0])``; its channels are free or its own on
    every link of its path.  A sample without lightpaths gets insertions only; a draw that finds no room after 64 tries
    is dropped.  Returns ``to_graph.LightpathChanges`` of CPU tensors (``.to(device)``)."""
    import numpy as np
    from .to_graph import LightpathChanges
    rng = np.random.default_rng(seed)
    data, freqs = samples["data"], samples["freqs"]
    fi = {k: i for i, k in enumerate(samples["lp_feat"])}
    S, _, L, Q = data.shape
    occupied = np.any(data != 0, axis=1)                       # [S, L, Q]
    conn_ids = state.conn_ids.cpu().numpy()
    ptr = state.batch.ptr.cpu().numpy()
    nodes, smp, lptr, links, q0s, widths, feats = [], [], [0], [], [], [], []

    def slots_ok(free, path, width):
        """[Q - width + 1] bool: start slots whose width slots are free on every link of path."""
        f = free[path].all(axis=0)
        ok = f[:Q - width + 1].copy()
        for u in range(1, width):
            ok &= f[u:Q - width + 1 + u]
        return np.flatnonzero(ok)

    def emit(node, s, path, q0, width, feat):
        nodes.append(node)
        smp.append(s)
        links.extend(int(l) for l in path)
        lptr.append(len(links))
        q0s.append(int(q0))
        widths.append(int(width))
        feats.append(feat)

    for s in range(S):
        conn = np.trunc(data[s, fi["conn_id"]])
        n0, n1 = int(ptr[s]), int(ptr[s + 1])
        for _ in range(per_sample):
            r = rng.random() if n1 > n0 else 1.0
            if r >= 0.85:                                          # insertion
                for _try in range(64):
                    width = 2 if rng.random() < 0.1 else 1
                    path = rng.choice(L, size=min(int(rng.integers(1, 7)), L), replace=False)
                    cand = slots_ok(~occupied[s], path, width)
                    if cand.size:
                        q0 = int(rng.choice(cand))
                        emit(-1, s, path, q0, width, [np.float32(freqs[q0]), rng.choice([4, 8, 16, 32, 64]),
                                                      int(rng.integers(1, 107)), int(rng.integers(24214, 7834746))])
                        break
                continue
            j = int(rng.integers(n0, n1))
            mine = occupied[s] & (conn == conn_ids[j])
            ls, qs = np.nonzero(mine)                              # row-major: (ls[0], qs[0]) is the first channel
            own_links = np.unique(ls)
            q_own, w = int(qs.min()), int(qs.max() - qs.min() + 1)
            mod, spans, plen = (data[s, fi[k], ls[0], qs[0]] for k in ("mod_order", "num_spans", "path_len"))
            free = ~occupied[s] | mine
            if r < 0.35:                                           # retune on its own links
                cand = slots_ok(free, own_links, w)
                other = cand[cand != q_own]
                if other.size == 0:
                    q0 = q_own
                elif rng.random() < 0.5:
                    d = np.abs(other - q_own)
                    q0 = int(rng.choice(other[d == d.min()]))
                else:
                    q0 = int(rng.choice(other))
                emit(j, s, own_links, q0, w, [np.float32(freqs[q0]), mod, spans, plen])
            elif r < 0.65:                                         # reroute
                for _try in range(64):
                    path = rng.choice(L, size=min(int(rng.integers(1, 7)), L), replace=False)
                    cand = slots_ok(free, path, w)
                    if cand.size:
                        q0 = int(rng.choice(cand))
                        emit(j, s, path, q0, w, [np.float32(freqs[q0]), mod, int(rng.integers(1, 107)),
                                                 int(rng.integers(24214, 7834746))])
                        break
            else:                                                  # teardown
                emit(j, s, [], q_own, w, [np.float32(freqs[q_own]), mod, spans, plen])
    return LightpathChanges(torch.tensor(nodes, dtype=torch.int64), torch.tensor(smp, dtype=torch.int64),
                            torch.tensor(lptr, dtype=torch.int64), torch.tensor(links, dtype=torch.int32),
                            torch.tensor(q0s, dtype=torch.int32), torch.tensor(widths, dtype=torch.int32),
                            torch.tensor(np.array(feats, dtype=np.float32).reshape(-1, 4)))


def lightpath_change_sets(samples, state, per_sample: int, seed: int = 0):
    """Seeded sets of simultaneous changes to the lightpaths of ``samples`` (as ``lightpath_changes``), for
    ``LightpathGNN.forward_change_sets``.  ``per_sample`` sets per sample, a mix of
      - restoration (0.25): a random link that carries lightpaths fails; each lightpath crossing it (at most
        ``ops.SET_MAX_CHANGES``) is rerouted onto 1..6 links that avoid it, its own width, at slots free once all of
        them are cleared and not taken by an earlier reroute of the set, or torn down when there is no room;
      - batch insertion (0.25): 2..8 new lightpaths; after the first, half of them share a link with an earlier one of
        the set at the slot right next to it, so that the two interfere;
      - defragmentation (0.25): 2..8 retunes of distinct lightpaths on their own links, starting with a slot swap of two
        lightpaths of equal width whenever the sample has a pair that can swap;
      - single changes (0.25): one change drawn as ``lightpath_changes`` draws it.
    Every placement is free once the set's moved and torn-down lightpaths are cleared, and the placements of a set are
    disjoint.  A sample without lightpaths gets batch insertions; a draw that finds no room is dropped, so a set may
    come out smaller (never empty).  Returns ``(to_graph.LightpathChanges, set_ptr [G+1] int64)`` of CPU tensors."""
    import numpy as np
    from .to_graph import LightpathChanges
    rng = np.random.default_rng(seed)
    data, freqs = samples["data"], samples["freqs"]
    fi = {k: i for i, k in enumerate(samples["lp_feat"])}
    S, _, L, Q = data.shape
    occupied = np.any(data != 0, axis=1)
    conn_ids = state.conn_ids.cpu().numpy()
    ptr = state.batch.ptr.cpu().numpy()
    rows, set_ptr = [], [0]

    def starts(free, path, width):
        f = free[np.asarray(path)].all(axis=0)
        ok = f[:Q - width + 1].copy()
        for u in range(1, width):
            ok &= f[u:Q - width + 1 + u]
        return np.flatnonzero(ok)

    def own(s, j):
        """(channels [L, Q] bool, own links, q0, width, (mod, spans, plen)) of node j of sample s."""
        mine = occupied[s] & (np.trunc(data[s, fi["conn_id"]]) == conn_ids[j])
        ls, qs = np.nonzero(mine)
        rest = tuple(data[s, fi[k], ls[0], qs[0]] for k in ("mod_order", "num_spans", "path_len"))
        return mine, np.unique(ls), int(qs.min()), int(qs.max() - qs.min() + 1), rest

    def take(free, path, q0, width):
        free[np.ix_(np.asarray(path), range(q0, q0 + width))] = False

    def rand_path():
        return rng.choice(L, size=min(int(rng.integers(1, 7)), L), replace=False)

    def new_feat(q0):
        return [np.float32(freqs[q0]), rng.choice([4, 8, 16, 32, 64]), int(rng.integers(1, 107)),
                int(rng.integers(24214, 7834746))]

    def restoration(s, n0, n1):
        carried = np.flatnonzero(occupied[s].any(axis=1))
        l_fail = int(rng.choice(carried))
        hit = [j for j in range(n0, n1) if own(s, j)[0][l_fail].any()][:64]
        info = {j: own(s, j) for j in hit}
        free = ~occupied[s]
        for j in hit:
            free |= info[j][0]
        out = []
        for j in hit:
            _, _, _, w, (mod, _, _) = info[j]
            for _try in range(16):
                path = rand_path()
                if l_fail in path:
                    continue
                cand = starts(free, path, w)
                if cand.size:
                    q0 = int(rng.choice(cand))
                    take(free, path, q0, w)
                    out.append((j, s, path, q0, w, [np.float32(freqs[q0]), mod, int(rng.integers(1, 107)),
                                                     int(rng.integers(24214, 7834746))]))
                    break
            else:
                out.append((j, s, [], info[j][2], w, [np.float32(freqs[info[j][2]]), mod, 0, 0]))
        return out

    def batch_insertion(s):
        free = ~occupied[s]
        out = []
        for i in range(int(rng.integers(2, 9))):
            w = 2 if rng.random() < 0.1 else 1
            placed = False
            if out and rng.random() < 0.5:                 # next to an earlier one of the set, on one of its links
                _, _, p, q, pw, _ = out[int(rng.integers(len(out)))]
                l = int(rng.choice(p))
                for q0 in (q + pw, q - w):
                    if 0 <= q0 and q0 + w <= Q and free[l, q0:q0 + w].all():
                        path = np.array([l] + [x for x in rand_path() if x != l][:2])
                        if free[np.ix_(path, range(q0, q0 + w))].all():
                            take(free, path, q0, w)
                            out.append((-1, s, path, q0, w, new_feat(q0)))
                            placed = True
                            break
            for _try in range(0 if placed else 16):
                path = rand_path()
                cand = starts(free, path, w)
                if cand.size:
                    q0 = int(rng.choice(cand))
                    take(free, path, q0, w)
                    out.append((-1, s, path, q0, w, new_feat(q0)))
                    break
        return out

    def defragmentation(s, n0, n1):
        info = {j: own(s, j) for j in range(n0, n1)}
        order = [int(j) for j in rng.permutation(np.arange(n0, n1))]
        want = int(rng.integers(2, 9))
        out, moved = [], []
        free = ~occupied[s]
        for a in order:                                    # a swap: a onto b's slots on a's links, b onto a's
            ma, la, qa, wa, ra = info[a]
            for b in order:
                mb, lb, qb, wb, rb = info[b]
                if b == a or wb != wa or qb == qa:
                    continue
                others = occupied[s] & ~ma & ~mb
                if others[np.ix_(la, range(qb, qb + wa))].any() or others[np.ix_(lb, range(qa, qa + wa))].any():
                    continue
                if set(la.tolist()) & set(lb.tolist()) and abs(qb - qa) < wa:
                    continue                               # the two new placements would share a channel
                free |= ma | mb
                take(free, la, qb, wa)
                take(free, lb, qa, wb)
                out += [(a, s, la, qb, wa, [np.float32(freqs[qb]), *ra]),
                        (b, s, lb, qa, wb, [np.float32(freqs[qa]), *rb])]
                moved += [a, b]
                break
            if moved:
                break
        for j in order:
            if len(out) >= want:
                break
            if j in moved:
                continue
            m, ls, q_own, w, r = info[j]
            f = free | m
            cand = starts(f, ls, w)
            cand = cand[cand != q_own]
            if cand.size:
                q0 = int(rng.choice(cand))
                free |= m
                take(free, ls, q0, w)
                out.append((j, s, ls, q0, w, [np.float32(freqs[q0]), *r]))
                moved.append(j)
        return out

    single = lightpath_changes(samples, state, per_sample, seed=int(rng.integers(1 << 31)))
    by_sample = {}
    for k in range(single.sample.shape[0]):
        a, b = int(single.link_ptr[k]), int(single.link_ptr[k + 1])
        by_sample.setdefault(int(single.sample[k]), []).append(
            (int(single.node[k]), int(single.sample[k]), single.links[a:b].tolist(), int(single.q0[k]),
             int(single.width[k]), single.feat[k].tolist()))
    for s in range(S):
        n0, n1 = int(ptr[s]), int(ptr[s + 1])
        singles = by_sample.get(s, [])
        for _ in range(per_sample):
            r = rng.random() if n1 > n0 else 0.3
            if r < 0.25:
                got = restoration(s, n0, n1)
            elif r < 0.5:
                got = batch_insertion(s)
            elif r < 0.75:
                got = defragmentation(s, n0, n1)
            else:
                got = [singles.pop(0)] if singles else []
            if got:
                rows.extend(got)
                set_ptr.append(len(rows))
    lptr = np.cumsum([0] + [len(r[2]) for r in rows])
    return (LightpathChanges(torch.tensor([r[0] for r in rows], dtype=torch.int64),
                             torch.tensor([r[1] for r in rows], dtype=torch.int64),
                             torch.tensor(lptr, dtype=torch.int64),
                             torch.tensor([int(l) for r in rows for l in r[2]], dtype=torch.int32),
                             torch.tensor([r[3] for r in rows], dtype=torch.int32),
                             torch.tensor([r[4] for r in rows], dtype=torch.int32),
                             torch.tensor(np.array([r[5] for r in rows], dtype=np.float32).reshape(-1, 4))),
            torch.tensor(set_ptr, dtype=torch.int64))


def lightpath_demands(samples, per_sample: int, options=(1, 4), seed: int = 0, bound_range=(0.1, 0.6)):
    """Seeded lightpath demands for the network-status ``samples`` (the dict ``network_status_samples`` returns), for
    ``LightpathGNN.forward_placements``.  ``per_sample`` demands per sample, each in a random sample with
    ``options[0]..options[1]`` options.  An option is a route of 1..6 distinct random links (free slots or not), a
    width of 1..3 slots, ``feat = (mod_order, num_spans, path_len)`` drawn as ``lightpath_candidates`` draws them and
    ``own_bound``; after the first, an option repeats an earlier route of the demand with another modulation format
    and width with probability 0.3.  ``own_bound`` is per demand: -inf on every option (probability 0.2: every free
    placement is feasible), +inf (0.2: none is) or, per option, uniform in ``bound_range`` (0.6: the spread of the
    reference model's column-0 predictions, so that a few placements are feasible).  Returns
    ``to_graph.LightpathDemands`` of CPU tensors (``.to(device)``)."""
    import numpy as np
    from .to_graph import LightpathDemands
    rng = np.random.default_rng(seed)
    S, _, L, _ = samples["data"].shape
    lo, hi = int(options[0]), int(options[1])
    if not 1 <= lo <= hi:
        raise ValueError("options must be (lo, hi) with 1 <= lo <= hi")
    smp, optr, lptr, links, widths, feats, bounds = [], [0], [0], [], [], [], []
    for _ in range(S * per_sample):
        smp.append(int(rng.integers(0, S)))
        kind = rng.random()
        routes = []
        for k in range(int(rng.integers(lo, hi + 1))):
            if routes and rng.random() < 0.3:
                path = routes[int(rng.integers(0, len(routes)))]
            else:
                path = [int(l) for l in rng.choice(L, size=min(int(rng.integers(1, 7)), L), replace=False)]
                routes.append(path)
            links.extend(path)
            lptr.append(len(links))
            widths.append(int(rng.integers(1, 4)))
            feats.append([rng.choice([4, 8, 16, 32, 64]), int(rng.integers(1, 107)), int(rng.integers(24214, 7834746))])
            bounds.append(-np.inf if kind < 0.2 else np.inf if kind < 0.4 else rng.uniform(*bound_range))
        optr.append(len(widths))
    return LightpathDemands(torch.tensor(smp, dtype=torch.int64), torch.tensor(optr, dtype=torch.int64),
                            torch.tensor(lptr, dtype=torch.int64), torch.tensor(links, dtype=torch.int32),
                            torch.tensor(widths, dtype=torch.int32),
                            torch.tensor(np.array(feats, dtype=np.float32).reshape(-1, 3)),
                            torch.tensor(np.array(bounds, dtype=np.float32)))


def lightpath_traffic(samples, per_sample: int, load: float, options=(1, 4), seed: int = 0, bound_range=(0.1, 0.6),
                      release_existing: float = 0.0):
    """Seeded dynamic traffic for the network-status ``samples``, for ``LightpathGNN.forward_traffic``: returns
    ``(demands, releases)``, ``to_graph.LightpathDemands`` and ``to_graph.LightpathReleases`` of CPU tensors.

    Per sample, ``per_sample`` demands arrive as a Poisson process of rate ``load`` (in Erlang, with unit-mean
    exponential holding times) and each holds its lightpath for its holding time.  Options are drawn as
    ``lightpath_demands`` draws them.  The demands of all samples are ordered by arrival time, so samples interleave.
    Each demand's departure is a release by demand whose ``before`` is the number of demands that arrived before the
    departure (one ``searchsorted`` over all arrivals); departures after the last arrival get ``before = D``.
    ``release_existing``: the fraction of each sample's lightpaths (the conn_ids on its channels) released by conn_id
    at uniform random times over the sample's arrival window."""
    import numpy as np
    from .to_graph import LightpathReleases
    if load <= 0:
        raise ValueError("load must be positive (Erlang)")
    rng = np.random.default_rng(seed)
    S = samples["data"].shape[0]
    base = lightpath_demands(samples, per_sample, options, seed=int(rng.integers(1 << 31)), bound_range=bound_range)
    optr = base.opt_ptr.numpy()
    # arrival times per sample, then one global order by time
    smp, t_arr, t_dep, opts = [], [], [], []
    for s in range(S):
        t = np.cumsum(rng.exponential(1.0 / load, per_sample))
        smp += [s] * per_sample
        t_arr.append(t)
        t_dep.append(t + rng.exponential(1.0, per_sample))
    t_arr, t_dep = np.concatenate(t_arr), np.concatenate(t_dep)
    order = np.argsort(t_arr, kind="stable")
    smp = np.asarray(smp, dtype=np.int64)[order]
    t_arr, t_dep = t_arr[order], t_dep[order]
    D = smp.shape[0]
    # demand k takes the options of base demand k (whose sample is redrawn here)
    sub = [list(range(int(optr[k]), int(optr[k + 1]))) for k in range(D)]
    lptr = base.link_ptr.numpy()
    o_idx = [p for k in range(D) for p in sub[k]]
    l_idx = [e for p in o_idx for e in range(int(lptr[p]), int(lptr[p + 1]))]
    from .to_graph import LightpathDemands
    t = lambda v: torch.tensor(np.asarray(v, dtype=np.int64))
    demands = LightpathDemands(t(smp), t(np.cumsum([0] + [len(x) for x in sub])),
                               t(np.cumsum([0] + [int(lptr[p + 1] - lptr[p]) for p in o_idx])),
                               base.links[t(l_idx)], base.width[t(o_idx)], base.feat[t(o_idx)],
                               base.own_bound[t(o_idx)])
    # departures of the demands: before = arrivals strictly earlier than the departure
    r_s, r_b, r_d, r_c, r_t = [], [], [], [], []
    before = np.searchsorted(t_arr, t_dep, side="left")
    for k in range(D):
        r_s.append(int(smp[k])); r_b.append(int(before[k])); r_d.append(k); r_c.append(-1); r_t.append(t_dep[k])
    # a share of the initial lightpaths released by conn_id at uniform times over the sample's arrivals
    if release_existing > 0:
        fi = {n: i for i, n in enumerate(samples["lp_feat"])}
        for s in range(S):
            d = samples["data"][s]
            conns = np.unique(np.trunc(d[fi["conn_id"]][np.any(d != 0, axis=0)]).astype(np.int64))
            pick = conns[rng.random(conns.shape[0]) < release_existing]
            mine = t_arr[smp == s]
            end = float(mine[-1]) if mine.size else 1.0
            for c in pick:
                tr = rng.uniform(0.0, end)
                r_s.append(s); r_b.append(int(np.searchsorted(t_arr, tr, side="left"))); r_d.append(-1)
                r_c.append(int(c)); r_t.append(tr)
    ro = np.argsort(np.asarray(r_t), kind="stable")            # releases in time order (the index is cosmetic)
    pick = lambda v: torch.tensor(np.asarray(v, dtype=np.int64)[ro] if len(v) else np.zeros(0, dtype=np.int64))
    return demands, LightpathReleases(pick(r_s), pick(r_b), pick(r_d), pick(r_c))


def lightpath_restoration_options(samples, state, options=(1, 4), seed: int = 0, bound_range=(0.1, 0.6)):
    """Seeded restoration options for every lightpath of ``state`` (built from the network-status ``samples``), for
    ``LightpathGNN.forward_restoration``: ``to_graph.LightpathDemands`` of CPU tensors with one demand per node of
    ``state.batch`` (``sample[v]`` = v's sample) and ``options[0]..options[1]`` options each.  Option 0 is the
    lightpath's current route (the links it occupies, ascending) and width (its slots on its first link) with its own
    (mod_order, num_spans, path_len), so a failure of one of its links always filters it out; the others are drawn as
    ``lightpath_demands`` draws them, as is ``own_bound`` (one kind per lightpath: -inf, +inf or uniform in
    ``bound_range`` per option).  One host copy of the state's channel map."""
    import numpy as np
    from .to_graph import LightpathDemands
    rng = np.random.default_rng(seed)
    lo, hi = int(options[0]), int(options[1])
    if not 1 <= lo <= hi:
        raise ValueError("options must be (lo, hi) with 1 <= lo <= hi")
    data = samples["data"]
    L = data.shape[2]
    fi = {k: i for i, k in enumerate(samples["lp_feat"])}
    chan = state.chan_node.cpu().numpy()
    node_ptr = state.batch.ptr.cpu().numpy()
    smp, optr, lptr, links, widths, feats, bounds = [], [0], [0], [], [], [], []
    for s in range(state.S):
        n0, n1 = int(node_ptr[s]), int(node_ptr[s + 1])
        c = chan[s]
        for v in range(n0, n1):
            ll, qq = np.nonzero(c == v)
            route = sorted(set(ll.tolist()))
            width = int((ll == route[0]).sum()) if route else 1
            l0, q0 = (int(ll[0]), int(qq[0])) if route else (0, 0)
            smp.append(s)
            kind = rng.random()
            routes = [route] if route else []
            for k in range(int(rng.integers(lo, hi + 1))):
                if k == 0 and route:
                    path, w = route, width
                    f = [float(data[s, fi[n], l0, q0]) for n in ("mod_order", "num_spans", "path_len")]
                else:
                    if routes and rng.random() < 0.3:
                        path = routes[int(rng.integers(0, len(routes)))]
                    else:
                        path = [int(l) for l in rng.choice(L, size=min(int(rng.integers(1, 7)), L), replace=False)]
                        routes.append(path)
                    w = int(rng.integers(1, 4))
                    f = [rng.choice([4, 8, 16, 32, 64]), int(rng.integers(1, 107)), int(rng.integers(24214, 7834746))]
                links.extend(path)
                lptr.append(len(links))
                widths.append(w)
                feats.append(f)
                bounds.append(-np.inf if kind < 0.2 else np.inf if kind < 0.4 else rng.uniform(*bound_range))
            optr.append(len(widths))
    return LightpathDemands(torch.tensor(smp, dtype=torch.int64), torch.tensor(optr, dtype=torch.int64),
                            torch.tensor(lptr, dtype=torch.int64), torch.tensor(links, dtype=torch.int32),
                            torch.tensor(widths, dtype=torch.int32),
                            torch.tensor(np.array(feats, dtype=np.float32).reshape(-1, 3)),
                            torch.tensor(np.array(bounds, dtype=np.float32)))
