"""Dense network-status samples at the capacity of the lightpath network-state kernels (TEST INFRASTRUCTURE, like
tg_cases.py): seeded numpy builders of ``[S, F, L, Q]`` samples in the format of ``synthetic.network_status_samples``
that place an exact number of lightpaths, up to QOT_TG_MAX_NODES = 256 per sample and QOT_TG_MAX_CHANNELS = 6144
occupied channels, plus hand-built symmetric, source-sorted graph stores at the fast-path bounds of every-node mode
(kEnMaxN = 128 nodes, kEnMaxE = 512 edges).

  hub          L = 128, Q = 32, threshold 0.05: lightpath 1 on every link at slot 10, single-link lightpaths at slots 9
               and 11 (0.0375 from the hub, 0.075 from each other) until there are 256; only slot 11 of link 127 stays
               free next to the hub.  n = 256, E = 510, the hub's in-degree is 255.
  clique       L = 8, Q = 256, threshold 10.0 (wider than the grid: every pair sharing a link interferes), 256
               lightpaths on 1..3 random links.  Rows of well over 64 messages, in-rows over 128.
  full_sparse  L = 40, Q = 80, threshold 0.05: samples of 256, 255, 1 and 48 lightpaths in one state, so the node
               offsets of the samples differ.
  full_grid    L = 64, Q = 96: 256 lightpaths of 8 links x 3 slots occupying every one of the 6144 channels
               (``extra``: that many more channels of lightpath 0 on an added slot column, over capacity)."""
import numpy as np

MAX_NODES = 256                # QOT_TG_MAX_NODES
MAX_CHANNELS = 6144            # QOT_TG_MAX_CHANNELS
EN_MAX_N, EN_MAX_E = 128, 512  # every-node fast path (csrc/lightpath_every_node.cu kEnMaxN / kEnMaxE)
HUB_THRESHOLD = 0.05
CLIQUE_THRESHOLD = 10.0


class SampleBuilder:
    """One sample [F, L, Q] on the grid 192.2 + spacing * q; lightpaths get distinct random conn_ids and random
    features (``synthetic.network_status_samples``'s distributions), one vector per channel with its own freq."""

    def __init__(self, L, Q, rng, spacing=0.0375):
        from gnn_qot_estimation_b200 import synthetic
        self.lp_feat = list(synthetic.LP_FEAT)
        self.metric = list(synthetic.METRICS)
        self.fi = {k: i for i, k in enumerate(self.lp_feat)}
        self.L, self.Q, self.rng = L, Q, rng
        self.freqs = 192.2 + spacing * np.arange(Q, dtype=np.float64)
        self.data = np.zeros((len(self.lp_feat), L, Q), dtype=np.float32)
        self.conn_pool = rng.permutation(np.arange(1, 4 * MAX_NODES + 8))
        self.count = 0
        self.last = None

    def vector(self):
        fi, rng = self.fi, self.rng
        v = np.zeros(len(self.lp_feat), dtype=np.float32)
        v[fi["conn_id"]] = self.conn_pool[self.count]
        v[fi["src_id"]], v[fi["dst_id"]] = rng.choice(np.arange(1, 76), 2, replace=False)
        v[fi["mod_order"]] = rng.choice([4, 8, 16, 32, 64])
        v[fi["path_len"]] = int(rng.integers(24214, 7834746))
        v[fi["num_spans"]] = int(rng.integers(1, 107))
        v[fi["osnr"]], v[fi["snr"]], v[fi["ber"]] = rng.uniform(13, 33), rng.uniform(9, 29), rng.uniform(1e-11, 1e-2)
        return v

    def put(self, vec, l, q):
        assert not self.data[:, l, q].any(), f"channel ({l}, {q}) is taken"
        v = vec.copy()
        v[self.fi["freq"]] = self.freqs[q]
        self.data[:, l, q] = v

    def place(self, links, q0, width=1):
        """A new lightpath on links x [q0, q0 + width); returns its conn_id."""
        vec = self.vector()
        for l in links:
            for q in range(q0, q0 + width):
                self.put(vec, l, q)
        self.count += 1
        self.last = (list(links), q0, width)
        return int(vec[self.fi["conn_id"]])

    def free(self):
        return ~np.any(self.data != 0, axis=0)

    def place_random(self, n_links, width=1):
        """A new lightpath on ``n_links`` random links at a random slot range free on all of them; False if none."""
        links = self.rng.choice(self.L, size=n_links, replace=False)
        free = self.free()
        ok = [q for q in range(self.Q - width + 1) if free[np.ix_(links, range(q, q + width))].all()]
        if not ok:
            return False
        self.place(sorted(int(l) for l in links), int(self.rng.choice(ok)), width)
        return True

    def finish(self, expect, overflow=False):
        """The sample, after asserting it holds exactly ``expect`` lightpaths and (unless ``overflow``) at most
        MAX_CHANNELS occupied channels.  The last lightpath placed is the LUT (osnr = snr = ber = -1)."""
        fi = self.fi
        occ = np.any(self.data != 0, axis=0)
        conns = np.unique(np.trunc(self.data[fi["conn_id"]][occ]))
        assert conns.size == self.count == expect, (conns.size, self.count, expect)
        assert overflow or int(occ.sum()) <= MAX_CHANNELS, int(occ.sum())
        if self.last is not None:
            links, q0, width = self.last
            for l in links:
                self.data[[fi["osnr"], fi["snr"], fi["ber"]], l, q0:q0 + width] = -1.0
        return self.data


def _pack(samples, freqs, lp_feat, metric, rng):
    data = np.stack(samples)
    target = np.stack([[rng.uniform(12.47, 33.49), rng.uniform(8.96, 29.98), rng.uniform(1.7e-12, 1.98e-2),
                        rng.integers(0, 3)] for _ in samples])
    return {"data": data, "target": target, "freqs": freqs, "lp_feat": lp_feat, "metric": metric}


def hub(seed=0):
    """One hub sample (threshold HUB_THRESHOLD).  Node order follows the row-major scan: link l holds the single at
    slot 9, then (link 0 only) the hub at slot 10, then the single at slot 11."""
    rng = np.random.default_rng(seed)
    b = SampleBuilder(128, 32, rng)
    for l in range(128):
        b.place([l], 9)
        if l == 0:
            b.place(list(range(128)), 10)
        if l < 127:
            b.place([l], 11)
    return _pack([b.finish(256)], b.freqs, b.lp_feat, b.metric, rng)


def clique(seed=0, n=256):
    """One clique sample (threshold CLIQUE_THRESHOLD): ``n`` lightpaths on 1..3 random links, one slot each (a few
    super-channels of two slots), grid spacing 0.0125 so that every frequency stays inside to_graph's range."""
    rng = np.random.default_rng(seed)
    b = SampleBuilder(8, 256, rng, spacing=0.0125)
    while b.count < n:
        assert b.place_random(int(rng.integers(1, 4)), 2 if rng.random() < 0.1 else 1)
    return _pack([b.finish(n)], b.freqs, b.lp_feat, b.metric, rng)


def full_sparse(seed=0, counts=(256, 255, 1, 48)):
    """Samples of exactly ``counts`` lightpaths each (threshold HUB_THRESHOLD) on 1..3 random links, 10% of them
    super-channels (self loops)."""
    rng = np.random.default_rng(seed)
    out = []
    for cnt in counts:
        b = SampleBuilder(40, 80, rng)
        while b.count < cnt:
            assert b.place_random(int(rng.integers(1, 4)), 2 if rng.random() < 0.1 else 1)
        out.append(b.finish(cnt))
    return _pack(out, b.freqs, b.lp_feat, b.metric, rng)


def full_grid(seed=0, extra=0):
    """Every channel of L = 64, Q = 96 occupied by 256 lightpaths of 8 links x 3 slots (threshold HUB_THRESHOLD:
    neighbouring slot groups interfere, every lightpath has a self loop).  ``extra`` > 0 adds a slot column and
    lightpath 0 on its first ``extra`` links: 6144 + extra occupied channels, still 256 lightpaths."""
    rng = np.random.default_rng(seed)
    b = SampleBuilder(64, 96 + (1 if extra else 0), rng)
    first = None
    for k in range(256):
        b.place(list(range(8 * (k // 32), 8 * (k // 32) + 8)), 3 * (k % 32), 3)
        if k == 0:
            first = b.data[:, 0, 0].copy()
    for l in range(extra):
        b.put(first, l, 96)
    data = b.finish(256, overflow=extra > 0)
    assert int(np.any(data != 0, axis=0).sum()) == MAX_CHANNELS + extra
    return _pack([data], b.freqs, b.lp_feat, b.metric, rng)


def count_sample(n, seed=0):
    """One sample of exactly ``n`` single-slot lightpaths on 1..3 random links of L = 40, Q = 80 (n may exceed
    MAX_NODES: a capacity probe)."""
    rng = np.random.default_rng(seed)
    b = SampleBuilder(40, 80, rng)
    while b.count < n:
        assert b.place_random(int(rng.integers(1, 4)))
    return _pack([b.finish(n)], b.freqs, b.lp_feat, b.metric, rng)


# --------------------------------------------------------------------------------------------- boundary stores
BOUNDARY_SHAPES = [(128, 512), (129, 512), (128, 514), (120, 500)]   # (nodes, directed edges incl. self loops)


def boundary_graph(n, E, rng, hub_degree=100, loops=2):
    """(x [n, 5] float32 with the flag column zero, edges [2, E] int64 sorted by (source, destination)): an undirected
    graph, both directions of every pair, ``loops`` self loops, node 0 adjacent to ``hub_degree`` others, random
    pairs up to exactly E directed edges."""
    assert (E - loops) % 2 == 0 and hub_degree < n
    pairs = {(0, int(j)) for j in rng.choice(np.arange(1, n), hub_degree, replace=False)}
    while len(pairs) < (E - loops) // 2:
        a, b = (int(v) for v in rng.choice(n, 2, replace=False))
        pairs.add((min(a, b), max(a, b)))
    d = {(a, b) for a, b in pairs} | {(b, a) for a, b in pairs}
    d |= {(int(v), int(v)) for v in rng.choice(np.arange(1, n), loops, replace=False)}
    ei = np.array(sorted(d), dtype=np.int64).T
    assert ei.shape[1] == E
    x = rng.random((n, 5), dtype=np.float32)
    x[:, 1] = 0.0
    return x, ei


def boundary_store(seed=0, shapes=BOUNDARY_SHAPES):
    """A PackedGraphStore (CPU) of one boundary graph per shape, in order; its layout passes verify_layout()."""
    import torch
    from gnn_qot_estimation_b200.batch import PackedGraphStore
    rng = np.random.default_rng(seed)
    xs, srcs, dsts, nptr, eptr = [], [], [], [0], [0]
    for n, E in shapes:
        x, ei = boundary_graph(n, E, rng)
        xs.append(x)
        srcs.append(ei[0])
        dsts.append(ei[1])
        nptr.append(nptr[-1] + n)
        eptr.append(eptr[-1] + E)
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dt)
    return PackedGraphStore(torch.tensor(nptr), torch.tensor(eptr), t(np.concatenate(srcs), torch.int32),
                            t(np.concatenate(dsts), torch.int32), t(np.concatenate(xs), torch.float32), None,
                            torch.zeros(len(shapes), 3), lut_col=1)
