"""Model check of the persistent tower kernel's synchronisation protocol (csrc/az_net.cu, az_k_tower_yrow; DESIGN.md section 4,
"persistent layer loop") -- no GPU needed.

The kernel has no grid-wide barrier: CTA pairs exchange two 64-bit counters per pair ("my first row of layer l is stored",
"my last row of layer l is stored"), a CTA's producer follows its own epilogue warps through a store counter, the weights
are swapped when a layer's last MMA has retired, and T / X are reused in place.  This file restates those rules as a
happens-before graph over the events of one launch (load of an input row, consumption by the MMAs, epilogue of an output
row, publication of its stores, weight swap) for a given number of leaf boards, and checks for MANY board counts that
  * the graph is acyclic even with the tightest resource limits (ring of one input row, one accumulator): no deadlock;
  * every read of a row is ordered after the store that produced it (RAW), including the halo rows of neighbouring pairs;
  * every in-place overwrite of a row is ordered after every read of its previous contents (WAR), by rules of the protocol
    alone (no ring / accumulator edges assumed: the producer may run arbitrarily far ahead);
  * every unit of every layer is processed exactly once, in the same order by producer, MMA issuer and epilogue.
The functions unit_range / segment / neighbour search are transcriptions of the device code (yr::unit_range, tw::segment and
the q_lo / q_hi loops); the graph rules are the waits of the three warp roles.  A model, not the kernel: the GPU tests
(`test_persistent_tower_equals_per_layer_kernels` and every network-driven MCTS test, whose ticks run hundreds of different
leaf counts bit-exactly) are the check of the code itself."""
import pytest

H = 6          # board rows = units per 32-board group
NBOARD = 16    # boards per CTA (32 per pair and group)
NPAIRS = 74


def unit_range(n_boards, pair, npairs=NPAIRS):
    groups = (n_boards + 2 * NBOARD - 1) // (2 * NBOARD)
    U = 6 * groups
    return U * pair // npairs, U * (pair + 1) // npairs


def segments(u0, u1):
    """Processing order of a pair's segments: (g, j_lo, j_hi) -- tw::segment()."""
    nseg = (u1 - 1) // H - u0 // H + 1
    out = []
    for k in range(nseg):
        i = k
        if nseg >= 2 and u1 % H != 0:   # a range that ends on a group boundary has no reader above
            i = nseg - 1 if k == 0 else k - 1
        g = u0 // H + i
        j_lo = u0 - g * H if i == 0 else 0
        j_hi = min(u1 - g * H, H)
        out.append((g, j_lo, j_hi))
    return out


class Graph:
    def __init__(self):
        self.ids, self.succ = {}, []

    def node(self, key):
        if key not in self.ids:
            self.ids[key] = len(self.succ)
            self.succ.append([])
        return self.ids[key]

    def edge(self, a, b):
        self.succ[self.node(a)].append(self.node(b))

    def topo(self):
        n = len(self.succ)
        indeg = [0] * n
        for s in self.succ:
            for t in s:
                indeg[t] += 1
        order, stack = [], [i for i in range(n) if indeg[i] == 0]
        while stack:
            v = stack.pop()
            order.append(v)
            for t in self.succ[v]:
                indeg[t] -= 1
                if indeg[t] == 0:
                    stack.append(t)
        return order if len(order) == n else None

    def ancestors(self):
        """bitset of ancestors (incl. self) per node; requires acyclicity"""
        order = self.topo()
        assert order is not None
        anc = [1 << i for i in range(len(self.succ))]
        for v in order:
            a = anc[v]
            for t in self.succ[v]:
                anc[t] |= a
        return anc


def build(n_boards, num_layers, resources=True, drop=()):
    """Events: ('L', p, l, g, y) input row y of group g requested by the producer; ('C', p, l, g, y) its stages consumed by the MMAs;
    ('A', p, l, u) accumulator of output row u complete; ('E', p, l, u) epilogue of u (the TMA stores are issued: the WRITE);
    ('S', p, l, u) stores complete and published (stored[] += 1, and the pair's counters if u is its first / last row);
    ('W', p, l) the layer's weights requested; ('F', p, l) every MMA of the layer retired (wfree)."""
    G = Graph()
    pairs = [p for p in range(NPAIRS) if unit_range(n_boards, p)[0] < unit_range(n_boards, p)[1]]
    rng = {p: unit_range(n_boards, p) for p in pairs}
    lower = {p: max([q for q in pairs if q < p], default=None) for p in pairs}
    upper = {p: min([q for q in pairs if q > p], default=None) for p in pairs}
    reads = {}     # (l, row) -> list of 'C' events that read that output row of layer l-1 at layer l
    order_check = []
    for p in pairs:
        u0, u1 = rng[p]
        q_lo = lower[p] if u0 % H != 0 else None
        q_hi = upper[p] if u1 % H != 0 else None
        prev_load = prev_cons = prev_epi = prev_store = None
        for l in range(num_layers):
            segs = segments(u0, u1)
            units = [g * H + j for (g, j_lo, j_hi) in segs for j in range(j_lo, j_hi)]
            order_check.append((p, l, units))
            if l > 0 and "wfree" not in drop:
                G.edge(('F', p, l - 1), ('W', p, l))            # warp 1: wfree, then the weight loads
            for (g, j_lo, j_hi) in segs:
                y_lo, y_hi = max(0, j_lo - 1), min(H - 1, j_hi)
                lo_halo = q_lo is not None and g * H + j_lo == u0
                hi_halo = q_hi is not None and g * H + j_hi == u1
                first = True
                for y in range(y_lo, y_hi + 1):
                    L, C = ('L', p, l, g, y), ('C', p, l, g, y)
                    if prev_load is not None:
                        G.edge(prev_load, L)                     # producer program order
                    if l > 0 and first:
                        for j in range(j_lo, j_hi):              # stored[] >= units through this segment of layer l-1
                            if "own" not in drop:
                                G.edge(('S', p, l - 1, g * H + j), L)
                        if lo_halo and "lo" not in drop:
                            G.edge(('S', q_lo, l - 1, rng[q_lo][1] - 1), L)     # done_up[q_lo]
                    if l > 0 and hi_halo and y == j_hi and "hi" not in drop:
                        G.edge(('S', q_hi, l - 1, rng[q_hi][0]), L)             # done[q_hi]
                    first = False
                    G.edge(L, C)                                 # full barrier
                    G.edge(('W', p, l), C)                       # bfull
                    if prev_cons is not None:
                        G.edge(prev_cons, C)                     # MMA issue order
                        if resources:
                            G.edge(prev_cons, L)                 # tightest ring: one input row in flight
                    prev_load, prev_cons = L, C
                    if l > 0:
                        reads.setdefault((l, g * H + y), []).append(C)
                    for j in (y - 1, y, y + 1):                  # output rows fed by input row y
                        if j_lo <= j < j_hi:
                            G.edge(C, ('A', p, l, g * H + j))
                for j in range(j_lo, j_hi):
                    u = g * H + j
                    A, E, S = ('A', p, l, u), ('E', p, l, u), ('S', p, l, u)
                    G.edge(A, E)                                 # tfull
                    G.edge(E, S)
                    if prev_epi is not None:
                        G.edge(prev_epi, E)                      # epilogue program order
                        G.edge(prev_store, S)                    # wait_group 0 per unit: publications are in order
                        if resources:
                            G.edge(prev_epi, A)                  # tightest accumulator ring: one slot
                    prev_epi, prev_store = E, S
            G.edge(prev_cons, ('F', p, l))
    return G, pairs, rng, reads, order_check


def check(n_boards, num_layers=4, drop=()):
    # 1. no deadlock under the tightest resource limits
    G, pairs, rng, reads, order_check = build(n_boards, num_layers, resources=True, drop=drop)
    assert G.topo() is not None, "cyclic wait graph (deadlock) at %d boards" % n_boards
    # 2. every unit exactly once, all roles in the same order (the three device loops share tw::segment)
    for p, l, units in order_check:
        assert sorted(units) == list(range(*rng[p])), (p, l)
    # 3. hazards, from protocol edges only
    G, pairs, rng, reads, _ = build(n_boards, num_layers, resources=False, drop=drop)
    anc = G.ancestors()
    owner = {}
    for p in pairs:
        for u in range(*rng[p]):
            owner[u] = p
    def before(a, b):
        return (anc[G.ids[b]] >> G.ids[a]) & 1
    n_raw = n_war = 0
    for p in pairs:                                               # the resident weights are overwritten in place, too
        for l in range(1, num_layers):
            assert before(('F', p, l - 1), ('W', p, l)), ("weights", n_boards, p, l)
    for (l, row), consumers in reads.items():
        q = owner[row]
        for c in consumers:
            load = ('L',) + c[1:]
            assert before(('S', q, l - 1, row), load), ("RAW", n_boards, l, row, c)   # the row read at layer l was stored at layer l-1
            n_raw += 1
            if l + 1 < num_layers:                                                     # ... and is overwritten in place at layer l+1
                assert before(c, ('E', q, l + 1, row)), ("WAR", n_boards, l, row, c)
                n_war += 1
    return len(pairs), n_raw, n_war


def test_tower_protocol_small_and_odd_sizes():
    """Every board count up to 20 groups = 640 boards (one unit per pair, neighbours without work, ranges inside one group, ...)."""
    seen_pairs = set()
    for n in list(range(1, 32 * 20 + 1)) + [1, 31, 32, 33, 63, 64, 65, 395, 396, 397]:
        npairs, n_raw, n_war = check(n)
        seen_pairs.add(npairs)
        assert n_raw > 0
    assert 6 in seen_pairs and 74 in seen_pairs      # one group = six pairs with one unit each ... all 74 pairs busy


def test_tower_protocol_bench_sizes():
    """Leaf counts of the bench (2700-3000 per tick, 4096 at the first tick): ranges of 7 and 10-11 units = 2-3 segments."""
    for n in (2688, 2750, 2751, 2817, 3000, 3999, 4096, 4128):
        npairs, n_raw, n_war = check(n, num_layers=4)
        assert npairs == 74 and n_war > 0
    check(2750, num_layers=14)   # the real layer count once


def test_tower_protocol_sweep_of_tick_sizes():
    """The leaf count changes every tick (anything from a few hundred to 4096): every 29th size up to one group past 4096."""
    for n in range(641, 4129, 29):
        check(n, num_layers=3)


def test_boundary_rows_are_processed_early():
    """What the reordering is for: with >= 2 segments the row the pair above waits for (last row) is published after at most
    the first segment, and the row the pair below waits for (first row) right after the first row of the second segment."""
    for n in (2750, 4096):
        for p in range(NPAIRS):
            u0, u1 = unit_range(n, p)
            segs = segments(u0, u1)
            if len(segs) < 2:
                continue
            units = [g * H + j for (g, j_lo, j_hi) in segs for j in range(j_lo, j_hi)]
            n_first_seg = segs[0][2] - segs[0][1]
            if u1 % H != 0:      # a pair above reads the last row
                assert units.index(u1 - 1) == n_first_seg - 1
                assert units.index(u0) == n_first_seg
            else:                # only the pair below reads a row of this pair: its first row, produced first
                assert units.index(u0) == 0
            if u0 % H != 0:      # the layer goes on for at least one more unit (~4 us) after the row the pair below waits for
                assert units.index(u0) + 1 <= len(units) - 1


@pytest.mark.parametrize("drop", ["hi", "lo", "own", "wfree"])
def test_the_model_notices_a_missing_wait(drop):
    """Sensitivity of the check: without the wait on the upper neighbour's first row, on the lower neighbour's last row, on
    the CTA's own store counter, or on `wfree`, some read / overwrite is no longer ordered."""
    with pytest.raises(AssertionError):
        for n in (2750, 4096, 100):
            check(n, drop=(drop,))
