"""CPU tier: the host-built symbolic structure of mapdn_create on generated topologies (tests/topo_corpus.py), run on the
emulated device (tests/emu) against the oracle.

Which branch of the schedule builder runs depends on the topology and the lane count G only: the PQ forest (one tree per
slack neighbour, re-rooted at its centre), the height-level forward and depth-level back schedules with their lane
inheritance and store flags, the contiguous-children encoding of hubs (more than two children), the narrow suffix /
prefix that only warp 0 of a G = 64 / 128 group runs, the bank-conflict relabelling (max_children <= 2, G >= 8,
npq >= 8), and the static first iteration (first_tab, seeded by vm_init). Meshed nets take the dense-LU fallback."""
import os
import re
import sys

import numpy as np
import pytest
import scipy.linalg

from conftest import ROOT
import topo_corpus as T

sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
from emu_env import EmuEnv                                          # noqa: E402
from oracle.pandapower_nr import PandapowerEquivalent, dSbus_dV     # noqa: E402
from test_emu_geometry import _episodes_against_oracles             # noqa: E402
from test_emu_kernel import _oracle_droop                           # noqa: E402

LANES = (0, 4, 8, 16, 32, 64, 128)
GS = (4, 8, 16, 32, 64, 128)
MAX_SMEM = 232448                                # sharedMemPerBlockOptin of the emulated B200 (tests/emu/cuda_runtime.h)
CORPUS = T.corpus()
NETS = {e.name: e for e in CORPUS}
RADIAL = [e.name for e in CORPUS if not T.is_meshed(e.net)]
# The dense factorisations are slow in the emulation (one barrier per pivot column and lane stride): meshed200 and the
# whole env on meshed nets run on the device only (tests/test_gpu_topologies.py); meshed257 (m = 512) runs here.
MESHED = [e.name for e in CORPUS if T.is_meshed(e.net) and e.name != "meshed200"]
WHOLE_ENV = ["forest40", "recursive_forest", "hub64", "hub257", "leveled_33", "chain42", "caterpillar"]

_SCHED = {}                                      # (net name, G) -> what MAPDN_DEBUG_SCHED printed when the handle was built
_SCHED_RE = re.compile(r"\[sched\] G=(\d+) levels=(\d+) esteps=(\d+) real=(\d+) reg0=(\d+) load0=(\d+) load1=(\d+) \| "
                       r"bsteps=(\d+) real=(\d+) regp=(\d+)")
_RELABEL_RE = re.compile(r"\[relabel\] [^:]*: ([\d.]+) -> ([\d.]+)")


@pytest.fixture(autouse=True)
def _no_overrides(monkeypatch):
    for k in ("MAPDN_EMU_SMS", "MAPDN_PLAN", "MAPDN_HELPERS", "MAPDN_EPB", "MAPDN_NO_RELABEL"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("MAPDN_DEBUG_SCHED", "1")


def _create(capfd, net, lanes, prof=None, args=None, batch=1):
    """EmuEnv plus what the schedule builder printed; the latter is also kept in _SCHED (runs with the relabelling on)."""
    capfd.readouterr()
    try:
        env = EmuEnv(net, prof, args or dict(voltage_barrier_type="l1"), batch=batch, lanes_per_env=lanes)
    finally:
        err = capfd.readouterr().err
    m = _SCHED_RE.search(err)
    keys = ("G", "levels", "esteps", "ereal", "reg0", "load0", "load1", "bsteps", "breal", "regp")
    s = dict(zip(keys, (int(v) for v in m.groups())))
    r = _RELABEL_RE.search(err)
    s["relabelled"] = r is not None and float(r.group(2)) < float(r.group(1))
    if not os.environ.get("MAPDN_NO_RELABEL"):
        _SCHED[(net.name, s["G"])] = s
    return env, s


# ---- the forest as the builder must see it, computed here from the branch list ----

def forest_levels(net):
    """(height-level widths, depth-level widths, largest number of children) of the PQ forest: in-service branches with
    parallel twins merged, the slack removed, one tree per slack neighbour re-rooted at its centre (the middle of a
    diameter found by two breadth-first searches over ascending bus indices, the far end of the second one walked back
    half-way, as mapdn_create does)."""
    n, s = net.n_bus, net.slack_bus
    on = net.br_status > 0
    pairs = {(min(a, b), max(a, b)) for a, b in zip(net.br_from[on], net.br_to[on])}
    adj = [[] for _ in range(n)]
    for a, b in sorted(pairs):
        adj[a].append(b); adj[b].append(a)
    for a in adj:
        a.sort()

    def bfs(src):
        dist, frm, q = {src: 0}, {src: -1}, [src]
        for u in q:
            for v in adj[u]:
                if v != s and v not in dist:
                    dist[v], frm[v] = dist[u] + 1, u
                    q.append(v)
        return q, dist, frm

    roots, seen = [], set()
    for s0 in adj[s]:
        if s0 in seen:
            continue
        comp, _, _ = bfs(s0)
        seen.update(comp)
        q, dist, frm = bfs(comp[-1])
        c = q[-1]
        for _ in range(dist[q[-1]] // 2):
            c = frm[c]
        roots.append(c)
    depth, parent, order = {r: 0 for r in roots}, {r: -1 for r in roots}, list(roots)
    for u in order:
        for v in adj[u]:
            if v != s and v not in depth:
                depth[v], parent[v] = depth[u] + 1, u
                order.append(v)
    height = dict.fromkeys(order, 0)
    nchild = dict.fromkeys(order, 0)
    for v in reversed(order):
        if parent[v] >= 0:
            height[parent[v]] = max(height[parent[v]], height[v] + 1)
            nchild[parent[v]] += 1
    n_lev = max(height.values()) + 1
    hw, dw = np.bincount(list(height.values()), minlength=n_lev), np.bincount(list(depth.values()), minlength=n_lev)
    return hw, dw, max(nchild.values())


def schedule_shape(net, G):
    """(n_esteps, n_bsteps, n_wide_e, n_narrow_b) of the schedules for G, from the level widths."""
    hw, dw, _ = forest_levels(net)
    steps = lambda w: -(-w // G)
    n_esteps, n_bsteps = int(sum(steps(w) for w in hw)), int(sum(steps(w) for w in dw[1:]))
    if G <= 32:
        return n_esteps, n_bsteps, n_esteps, 0
    wide = [k for k, w in enumerate(hw) if w > 32]
    first_narrow = wide[-1] + 1 if wide else 0            # forward steps of the levels from here on: warp 0 only
    n_wide_e = int(sum(steps(w) for w in hw[:first_narrow]))
    last = 0
    while last + 1 < len(dw) and dw[last + 1] <= 32:       # back steps of the depth levels 1..last: warp 0 only
        last += 1
    return n_esteps, n_bsteps, n_wide_e, int(sum(steps(w) for w in dw[1:last + 1]))


def least_footprint(net, G):
    """A lower bound of the shared memory any plan of the planner needs: one step of envs (32 / G of them for G <= 32,
    one otherwise), each with its npq + 2 node records of 144 B and the sgen p / q, plus Y[i,parent], Y[parent,i], Y[i,i]
    and the node descriptors of the static blob."""
    npq, unit = net.n_bus - 1, max(1, 32 // G)
    return unit * 16 * (9 * (npq + 2) + net.n_sgen) + 56 * npq


# ---- solve against the oracle ----

def _references(name):
    e = NETS[name]
    pf = PandapowerEquivalent(e.net)
    inp = T.injections(e.net, e.seed)
    return inp, [pf.runpp(*(x[k] for x in inp)) for k in range(3)]


def _check_against(out, refs, label):
    for k, r in enumerate(refs):
        assert out["converged"][k] == r.converged and out["iterations"][k] == r.iterations, (label, k)
        if r.converged:
            assert np.abs(out["vm"][k] - r.vm_pu).max() < 1e-9, (label, k)
            assert np.abs(out["va_deg"][k] - r.va_degree).max() < 1e-8, (label, k)
            assert np.abs(out["p_bus"][k] - r.p_mw).max() < 1e-8 and np.abs(out["q_bus"][k] - r.q_mvar).max() < 1e-8, (label, k)
            assert np.abs(out["pl"][k] - r.pl_mw).max() < 1e-9, (label, k)


@pytest.mark.parametrize("name", RADIAL)
def test_tree_solver_matches_oracle_at_every_lane_count(capfd, monkeypatch, name):
    """B = 3 (env 1 heavy) at every lane count against PandapowerEquivalent: the convergence flag and the iteration count
    are equal, the solution within 1e-9. The schedule the builder reports has the step counts the level widths give. A
    lane count may be refused as too large only where no plan can fit; where the relabelling applied, the run without
    it (MAPDN_NO_RELABEL=1) is bit-identical."""
    net = NETS[name].net
    inp, refs = _references(name)
    ran = 0
    for lanes in LANES:
        if lanes and least_footprint(net, lanes) > MAX_SMEM:
            with pytest.raises(RuntimeError, match=r"network too large for the shared-memory resident solver \((\d+) B needed"):
                _create(capfd, net, lanes)
            continue
        env, s = _create(capfd, net, lanes)
        G = s["G"]
        assert lanes in (0, G)
        assert (s["esteps"], s["bsteps"]) == schedule_shape(net, G)[:2] and s["levels"] == len(forest_levels(net)[0]), (G, s)
        out = env.solve(*inp)
        env.close()
        _check_against(out, refs, G)
        ran += 1
        if s["relabelled"]:
            monkeypatch.setenv("MAPDN_NO_RELABEL", "1")
            env, s0 = _create(capfd, net, lanes)
            monkeypatch.delenv("MAPDN_NO_RELABEL")
            assert not s0["relabelled"]
            plain = env.solve(*inp)
            env.close()
            for k in out:
                assert np.array_equal(out[k], plain[k]), (G, k)
    assert ran >= 5


def test_too_large_is_refused_with_the_footprint(capfd):
    """The planner refuses a lane count no plan fits, and says how much shared memory the smallest plan needs."""
    net = NETS["hub257"].net
    with pytest.raises(RuntimeError, match="too large") as ex:
        _create(capfd, net, 4)
    needed, avail = (int(v) for v in re.search(r"\((\d+) B needed, (\d+) B available\)", str(ex.value)).groups())
    assert avail == MAX_SMEM and needed >= least_footprint(net, 4) > MAX_SMEM


def _first_jacobian(net):
    """The oracle's Jacobian at the flat start (newtonpf's J, PQ buses only)."""
    pf = PandapowerEquivalent(net)
    dVm, dVa = dSbus_dV(pf.Ybus, pf.flat_start())
    pq = pf.pq
    a, m = dVa[pq][:, pq].toarray(), dVm[pq][:, pq].toarray()
    return np.block([[a.real, m.real], [a.imag, m.imag]])


@pytest.mark.parametrize("name", MESHED)
def test_dense_fallback_matches_oracle(capfd, name):
    """Meshed nets up to 256 PQ buses (m = 2 npq up to 512: 16 lane strides per row) on the dense-LU fallback, which
    always runs one warp per env. Partial pivoting must swap rows: the flat-start Jacobian of the oracle needs it."""
    net = NETS[name].net
    inp, refs = _references(name)
    _, piv = scipy.linalg.lu_factor(_first_jacobian(net))
    assert np.any(piv != np.arange(len(piv)))
    env, s = _create(capfd, net, 0)
    assert s["G"] == 32 and env.dims["lanes_per_env"] == 32
    out = env.solve(*inp)
    env.close()
    _check_against(out, refs, name)


def test_topology_limits(capfd):
    with pytest.raises(RuntimeError, match="more than 257 children"):
        _create(capfd, T.hub_net(258), 32)
    with pytest.raises(RuntimeError, match=r"meshed \(1 loop-closing branches\) and has more than 256 PQ buses"):
        _create(capfd, T.meshed_net(258), 0)


@pytest.mark.parametrize("name", WHOLE_ENV)
def test_whole_env_matches_oracle(capfd, name):
    """reset + 3 noisy steps (and a second episode) against VoltageControlOracle, then the droop baseline with
    q_max_manual below s_rated against the script: the epilogue tables (bus_of_node, the observation program, the line
    tables) depend on the topology too."""
    e = NETS[name]
    net, prof = e.net, T.profile(e.net)
    args = dict(voltage_barrier_type="bowl", action_scale=0.8, seed=e.seed, line_weight=0.3)
    env, _ = _create(capfd, net, 0, prof, args, batch=2)
    _episodes_against_oracles(env, net, prof, args, steps=3, seed=e.seed)
    pl, ql, pv, _ = T.injections(net, e.seed + 1, B=2)
    s_rated = prof.s_max
    pv = np.minimum(pv, 0.9 * s_rated)
    qmm = s_rated * np.linspace(0.15, 0.6, net.n_sgen)
    out = env.droop(pl, ql, pv, s_rated, q_max_manual=qmm)
    env.close()
    for k in range(2):
        vm, q, loss, it = _oracle_droop(net, pl[k], ql[k], pv[k], s_rated, q_max_manual=qmm)
        assert it < 100, k                    # stopped by the rule, not by the iteration limit
        assert out["iterations"][k] == it and np.abs(out["vm"][k] - vm).max() < 1e-8, k
        assert np.abs(out["q"][k] - q).max() < 1e-8 and abs(out["loss"][k] - loss) < 1e-8, k


def test_corpus_reaches_every_branch_of_the_schedule_builder(capfd):
    """For every G: a net whose forward schedule inherits lanes (reg0) and fetches second children (load1), a net with
    a level wider than G, a hub (extra children), nets with and without the relabelling (G >= 8: it never applies below);
    for G = 64 / 128 nets with a narrow suffix of the forward sweep and a narrow prefix of the back sweep after / before
    wide steps. Uses the schedules the solve tests built; builds the ones missing."""
    seen = {G: dict(reg0_load1=[], wider=[], extra=[], relabelled=[], plain=[], narrow_e=[], narrow_b=[]) for G in GS}
    for name in RADIAL:
        net = NETS[name].net
        hw, dw, max_children = forest_levels(net)
        for G in GS:
            if least_footprint(net, G) > MAX_SMEM:
                continue
            if (name, G) not in _SCHED:
                _create(capfd, net, G)[0].close()
            s, c = _SCHED[(name, G)], seen[G]
            n_esteps, n_bsteps, n_wide_e, n_narrow_b = schedule_shape(net, G)
            if s["reg0"] > 0 and s["load1"] > 0:
                c["reg0_load1"].append(name)
            if max(hw.max(), dw.max()) > G:
                c["wider"].append(name)
            if max_children > 2:
                c["extra"].append(name)
            (c["relabelled"] if s["relabelled"] else c["plain"]).append(name)
            if 0 < n_wide_e < n_esteps:
                c["narrow_e"].append(name)
            if 0 < n_narrow_b < n_bsteps:
                c["narrow_b"].append(name)
    for G, c in seen.items():
        need = ["reg0_load1", "wider", "extra", "plain"] + (["relabelled"] if G >= 8 else []) + \
               (["narrow_e", "narrow_b"] if G > 32 else [])
        assert all(c[k] for k in need), (G, {k: len(v) for k, v in c.items()})
