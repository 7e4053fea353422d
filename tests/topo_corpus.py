"""Generated topologies for the tests of the tree solver's host-built schedules and of the dense fallback
(tests/test_emu_topologies.py on the emulated device, tests/test_gpu_topologies.py on the B200).

What mapdn_create builds for a net (the PQ forest re-rooted at the tree centres, the height- and depth-level schedules
with their lane inheritance, the contiguous-children encoding of hubs, the narrow suffix / prefix of the multi-warp
groups, the bank-conflict relabelling, the static first iteration) depends on the topology and the lane count only. The
corpus is made to reach each of these branches: families of shapes, each net deterministic from its name and seed.

Structure is built on abstract node ids (0 = slack bus); ``_finish`` then gives every net the element mix of
``conftest.random_tree_net`` (taps, line charging, shunts, element scaling, a parallel twin, an out-of-service branch
that would close a loop), puts the slack at a random bus index, lists branches in both directions, and sets a slack angle
and, on every other net, a flat-start magnitude ``vm_init`` different from the slack's."""
from collections import namedtuple

import numpy as np

from mapdn_b200.network import NetDesc, ProfileDesc

Entry = namedtuple("Entry", "name seed net")


class _Tree:
    """Edges (parent, child) on abstract ids; node 0 is the slack bus."""

    def __init__(self):
        self.n, self.edges = 1, []

    def add(self, parent):
        v = self.n
        self.n += 1
        self.edges.append((parent, v))
        return v

    def chain(self, parent, m):
        for _ in range(m):
            parent = self.add(parent)
        return parent

    def recursive(self, parent, m, rng):
        """Random recursive tree of m buses below ``parent``: each new bus hangs off a uniformly drawn earlier one."""
        nodes = [self.add(parent)]
        for _ in range(m - 1):
            nodes.append(self.add(nodes[rng.integers(0, len(nodes))]))
        return nodes

    def leveled(self, parent, widths):
        """A tree whose depth levels below its root have exactly ``widths`` buses (widths non-decreasing, each at most
        twice the one before). Children are dealt round-robin, so every bus above the last level has a child: the height
        levels are the depth levels reversed, and the root (two subtrees of full depth) is the centre."""
        level = [self.add(parent)]
        assert widths[0] == 1
        for w in widths[1:]:
            assert len(level) <= w <= 2 * len(level)
            level = [self.add(level[k % len(level)]) for k in range(w)]


def _recursive_net(npq, rng):
    t = _Tree()
    t.recursive(0, npq, rng)
    return t


def _families():
    """(name, seed, builder(rng) -> (_Tree, extra branches)) of the radial and meshed families."""
    out = []

    def fam(name, seed):
        def deco(fn):
            out.append((name, seed, fn))
            return fn
        return deco

    for npq, seed in ((30, 1), (90, 2), (199, 3)):
        fam(f"recursive{npq + 1}", seed)(lambda rng, npq=npq: (_recursive_net(npq, rng), []))

    @fam("recursive_forest", 4)               # the slack is one of the candidate parents: many deep trees
    def _(rng):
        t, nodes = _Tree(), [0]
        for _ in range(120):
            nodes.append(t.add(nodes[rng.integers(0, len(nodes))]))
        return t, []

    for npq, seed in ((40, 5), (41, 6)):      # diameter 39 (two centres) and 40 (one centre)
        fam(f"chain{npq + 1}", seed)(lambda rng, npq=npq: (_chain_tree(npq), []))

    @fam("caterpillar", 7)                    # a spine of 40 with legs of 1-3 buses on every other spine bus
    def _(rng):
        t, p = _Tree(), 0
        for k in range(40):
            p = t.add(p)
            if rng.random() < 0.5:
                t.chain(p, int(rng.integers(1, 4)))
        return t, []

    @fam("broom", 8)                          # a handle of 30 and 24 bristles at its end
    def _(rng):
        t = _Tree()
        end = t.chain(0, 30)
        for _ in range(24):
            t.add(end)
        return t, []

    @fam("binary_full", 9)                    # depth levels 1, 2, 4, ..., 128: a level exactly G wide for every G
    def _(rng):
        t = _Tree()
        t.leveled(0, [2 ** k for k in range(8)])
        return t, []

    @fam("leveled_33", 10)                    # a level of 33 (= 32 + 1) after one of 17
    def _(rng):
        t = _Tree()
        t.leveled(0, [1, 2, 3, 5, 9, 17, 33])
        return t, []

    @fam("leveled_g_plus_1", 11)              # levels of 5, 9, 17, 33, 65, 129: G + 1 for every G
    def _(rng):
        t = _Tree()
        t.leveled(0, [1, 2, 3, 5, 9, 17, 33, 65, 129])
        return t, []

    @fam("ternary_full", 12)                  # three children everywhere: the contiguous extras on every level
    def _(rng):
        t, level = _Tree(), None
        level = [t.add(0)]
        for _ in range(4):
            level = [t.add(p) for p in level for _ in range(3)]
        return t, []

    for k, seed in ((3, 13), (4, 14), (31, 15), (33, 16), (64, 17), (257, 18)):
        fam(f"hub{k}", seed)(lambda rng, k=k: (_hub_tree(k, rng), []))

    @fam("forest2", 19)                       # two deep random trees
    def _(rng):
        t = _Tree()
        t.recursive(0, 30, rng)
        t.recursive(0, 22, rng)
        return t, []

    @fam("forest5", 20)                       # single buses and chains of up to 30
    def _(rng):
        t = _Tree()
        for m in (1, 30, 1, 12, 5):
            t.chain(0, m)
        return t, []

    @fam("forest40", 21)
    def _(rng):
        t = _Tree()
        lengths = [1] * 28 + [30] + list(rng.integers(2, 14, 11))
        for m in rng.permutation(lengths):
            t.chain(0, int(m))
        return t, []

    for n, n_loops, seed in ((20, 1, 22), (60, 3, 23), (130, 6, 24), (200, 4, 25), (257, 2, 26)):
        fam(f"meshed{n}", seed)(lambda rng, n=n, n_loops=n_loops: _meshed(n, n_loops, rng))
    return out


def _chain_tree(npq):
    t = _Tree()
    t.chain(0, npq)
    return t


def _hub_tree(k, rng):
    """slack - 2 buses - hub with k children; the first child continues into a tail of 20 buses, a few others into
    short chains."""
    t = _Tree()
    hub = t.chain(0, 3)
    kids = [t.add(hub) for _ in range(k)]
    t.chain(kids[0], 20)
    for c in kids[1:4]:
        t.chain(c, int(rng.integers(1, 4)))
    return t


def _meshed(n, n_loops, rng):
    """A random recursive tree of n buses plus n_loops loop-closing branches (two of them with R/X > 3 where there are
    that many, so that the flat-start Jacobian needs row swaps)."""
    t = _recursive_net(n - 1, rng)
    have = {tuple(sorted(e)) for e in t.edges}
    extra = []
    while len(extra) < n_loops:
        a, b = (int(v) for v in rng.choice(n, 2, replace=False))
        if tuple(sorted((a, b))) in have:
            continue
        have.add(tuple(sorted((a, b))))
        extra.append((a, b, len(extra) < 2))
    return t, extra


def _finish(name, seed, tree, extra, rng):
    """Electrical parameters and elements for a structure; see the module docstring."""
    n = tree.n
    perm = rng.permutation(n)                                     # abstract id -> bus index; the slack lands anywhere
    f = np.array([perm[a] for a, _ in tree.edges]); t = np.array([perm[b] for _, b in tree.edges])
    nt = len(f)
    r = rng.uniform(1e-3, 2e-2, nt)
    x = r * rng.uniform(0.3, 2.0, nt)
    b = rng.uniform(0, 2e-3, nt)
    g = rng.uniform(0, 1e-4, nt)
    tap = np.ones(nt)
    is_line = np.ones(nt, np.uint8)
    k = rng.choice(nt, max(1, nt // 6), replace=False)
    tap[k] = rng.uniform(0.95, 1.05, len(k))
    is_line[k] = 0
    status = np.ones(nt, np.uint8)
    # loop-closing branches; `steep` ones have R/X in [3, 6]
    for a, c, steep in extra:
        f = np.r_[f, perm[a]]; t = np.r_[t, perm[c]]
        rr = rng.uniform(5e-3, 3e-2)
        r = np.r_[r, rr]; x = np.r_[x, rr / (rng.uniform(3.0, 6.0) if steep else rng.uniform(0.5, 2.0))]
        b = np.r_[b, 0.0]; g = np.r_[g, 0.0]; tap = np.r_[tap, 1.0]; is_line = np.r_[is_line, 1]; status = np.r_[status, 1]
    # a parallel twin of the first branch, and an out-of-service branch that would close a loop
    adj = {tuple(sorted((int(u), int(v)))) for u, v in zip(f, t)}
    while True:
        u, v = (int(w) for w in rng.choice(n, 2, replace=False))
        if (min(u, v), max(u, v)) not in adj:
            break
    f = np.r_[f, f[0], u]; t = np.r_[t, t[0], v]
    r = np.r_[r, r[0] * 1.3, 0.01]; x = np.r_[x, x[0] * 0.9, 0.01]
    b = np.r_[b, 0.0, 0.0]; g = np.r_[g, 0.0, 0.0]; tap = np.r_[tap, tap[0], 1.0]
    is_line = np.r_[is_line, is_line[0], 1].astype(np.uint8)
    status = np.r_[status, 1, 0].astype(np.uint8)
    flip = rng.random(len(f)) < 0.5
    f, t = np.where(flip, t, f), np.where(flip, f, t)
    # loads: none on some buses, two or three on others; sgens on distinct buses, two on one bus where there is room
    n_loads = rng.choice([0, 1, 1, 1, 2, 3], n)
    load_bus = np.repeat(np.arange(n), n_loads).astype(np.int32)
    n_sgen = int(min(6, max(2, n // 25)))
    sgen_bus = rng.choice(n, n_sgen, replace=False).astype(np.int32)
    sgen_bus[-1] = sgen_bus[0]
    zone = rng.integers(0, 4, n).astype(np.int32)
    zone[sgen_bus] = np.maximum(zone[sgen_bus], 1)
    slack_vm = float(rng.uniform(1.0, 1.04))
    vm_init = slack_vm + float(rng.choice([-0.03, -0.015, 0.01])) if seed % 2 else None
    return NetDesc(base_mva=10.0, n_bus=n, slack_bus=int(perm[0]), slack_vm=slack_vm,
                   slack_va_deg=float(rng.uniform(-6.0, 6.0)), vm_init=vm_init,
                   br_from=f, br_to=t, br_r=r, br_x=x, br_b=b, br_g=g, br_tap=tap, br_status=status, br_is_line=is_line,
                   bus_gs=rng.uniform(0, 0.05, n), bus_bs=rng.uniform(-0.05, 0.05, n),
                   load_bus=load_bus, load_scaling=rng.uniform(0.8, 1.2, len(load_bus)),
                   sgen_bus=sgen_bus, sgen_zone=zone[sgen_bus], sgen_scaling=rng.uniform(0.9, 1.1, n_sgen),
                   bus_zone=zone, name=name)


def corpus():
    """Every net of the corpus, in a fixed order."""
    out = []
    for name, seed, build in _families():
        rng = np.random.default_rng(seed)
        tree, extra = build(rng)
        out.append(Entry(name, seed, _finish(name, seed, tree, extra, rng)))
    return out


def by_name():
    return {e.name: e.net for e in corpus()}


def hub_net(k, seed=27):
    """A hub with k children (beyond the 257 the schedule encoding takes for k = 258)."""
    rng = np.random.default_rng(seed)
    return _finish(f"hub{k}", seed, _hub_tree(k, rng), [], rng)


def meshed_net(n, n_loops=1, seed=28):
    rng = np.random.default_rng(seed)
    tree, extra = _meshed(n, n_loops, rng)
    return _finish(f"meshed{n}", seed, tree, extra, rng)


def is_meshed(net):
    on = net.br_status > 0
    return len({(min(a, b), max(a, b)) for a, b in zip(net.br_from[on], net.br_to[on])}) != net.n_bus - 1


# ---- injections ----

def _load_moment(net):
    """max over buses of sum over the branches on the path from the slack (breadth-first tree of the in-service
    branches) of |z| x (number of loads behind the branch): the voltage drop in p.u. per p.u. of load on every load."""
    adj = [[] for _ in range(net.n_bus)]
    for k in np.nonzero(net.br_status)[0]:
        z = abs(complex(net.br_r[k], net.br_x[k]))
        adj[net.br_from[k]].append((net.br_to[k], z)); adj[net.br_to[k]].append((net.br_from[k], z))
    par, zpar, order = {net.slack_bus: (-1)}, {net.slack_bus: 0.0}, [net.slack_bus]
    for u in order:
        for v, z in adj[u]:
            if v not in par:
                par[v], zpar[v] = u, z
                order.append(v)
    behind = np.bincount(net.load_bus, minlength=net.n_bus).astype(float)
    for v in reversed(order[1:]):
        behind[par[v]] += behind[v]
    drop = {net.slack_bus: 0.0}
    for v in order[1:]:
        drop[v] = drop[par[v]] + zpar[v] * behind[v]
    return max(drop.values())


def nominal_load_mw(net, drop=0.03):
    """Load per load element (MW) that drops the voltage by about ``drop`` p.u. at the far end."""
    return drop / max(_load_moment(net), 1e-9) * net.base_mva


def injections(net, seed, B=3):
    """(p_load, q_load, p_sgen, q_sgen) of B envs: env 1 is heavy (about three times the nominal load, several more
    Newton iterations), env 2 light with a large PV infeed."""
    rng = np.random.default_rng(seed)
    p0 = nominal_load_mw(net)
    lo = np.array([0.5, 2.6, 0.1, 0.8, 1.0][:B] + [0.5] * max(0, B - 5))
    hi = np.array([1.0, 3.0, 0.6, 1.4, 2.0][:B] + [1.0] * max(0, B - 5))
    pl = p0 * rng.uniform(lo[:, None], hi[:, None], (B, net.n_load))
    ql = pl * rng.uniform(0.2, 0.5, (B, net.n_load))
    total = p0 * net.n_load
    pv = total / net.n_sgen * rng.uniform(0.0, 0.5, (B, net.n_sgen))
    pv[2 % B] *= 2.0
    q = pv * rng.uniform(-0.3, 0.3, (B, net.n_sgen))
    return pl, ql, pv, q


def profile(net, seed=2):
    """A three-day profile store for any corpus net, after oracle/ref_scenarios.py:_general_case, scaled to the net's
    nominal load."""
    rng = np.random.default_rng(seed)
    p0 = nominal_load_mw(net)
    T = 3 * 480 + 1
    pv_max = p0 * net.n_load / net.n_sgen * 0.5
    return ProfileDesc(pv=rng.uniform(0.2, 1.0, (T, net.n_sgen)) * pv_max,
                       load_p=rng.uniform(0.3, 1.2, (T, net.n_load)) * p0,
                       load_q=rng.uniform(0.1, 0.4, (T, net.n_load)) * p0, steps_per_hour=20, n_days=3)
