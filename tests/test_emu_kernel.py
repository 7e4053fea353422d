"""CPU tier: the kernel SOURCE (mapdn_b200/csrc/env_kernel.cuh + the C-ABI host code) compiled with g++ against
tests/emu/cuda_runtime.h - a SIMT emulation with one OS thread per CUDA thread, counting barriers for
__syncthreads / bar.sync / bar.arrive / bar.red, exchange arrays for __shfl / __ballot - and executed against the oracle
and against the reference-executed fixtures. It proves the kernel's LOGIC (schedules, lock-step groups, multi-warp
groups, helper warps, RNG, epilogue) without a GPU; the `-m gpu` tests prove the sm_100a build. The emulated library is
test infrastructure: the product never loads it, and the device build is byte-identical with or without the
MAPDN_HOST_EMU guards (same SASS)."""
import json
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, random_tree_net
from mapdn_b200 import cases
from mapdn_b200.network import NetDesc, ProfileDesc

sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
from emu_env import EmuEnv                                          # noqa: E402
from oracle import ref_scenarios as S                               # noqa: E402
from oracle.pandapower_nr import PandapowerEquivalent               # noqa: E402
from oracle.voltage_control_ref import INFO_KEYS, VoltageControlOracle   # noqa: E402

TOL = 1e-9


@pytest.mark.parametrize("lanes", [0, 4, 16, 32, 64, 128])
def test_emulated_solve_matches_oracle_with_identical_iteration_counts(lanes):
    net, p, q = cases.baran_wu_nominal()
    env = EmuEnv(net, None, dict(voltage_barrier_type="l1"), batch=5, lanes_per_env=lanes)
    scale = np.array([1.0, 0.3, 1.6, 0.8, 2.2])[:, None]
    rng = np.random.default_rng(lanes)
    ps, qs = rng.uniform(0, 0.4, (5, 6)), rng.uniform(-0.3, 0.3, (5, 6))
    out = env.solve(p[None] * scale, q[None] * scale, ps, qs)
    pf = PandapowerEquivalent(net)
    for k in range(5):
        r = pf.runpp(p * scale[k, 0], q * scale[k, 0], ps[k], qs[k])
        assert out["converged"][k] == 1 and out["iterations"][k] == r.iterations
        assert np.abs(out["vm"][k] - r.vm_pu).max() < TOL and np.abs(out["va_deg"][k] - r.va_degree).max() < 1e-8
        assert np.abs(out["p_bus"][k] - r.p_mw).max() < TOL and np.abs(out["pl"][k] - r.pl_mw).max() < TOL
    env.close()


def test_emulated_solve_general_net_and_meshed_fallback():
    net = random_tree_net(23, 4, seed=11)                      # taps, charging, shunts, scaling, open branch, slack != 0
    rng = np.random.default_rng(0)
    pl, ql = rng.uniform(0, 0.3, (3, net.n_load)), rng.uniform(0, 0.1, (3, net.n_load))
    ps, qs = rng.uniform(0.1, 0.5, (3, 4)), rng.uniform(-0.2, 0.2, (3, 4))
    env = EmuEnv(net, None, dict(voltage_barrier_type="l1"), batch=3)
    out = env.solve(pl, ql, ps, qs)
    pf = PandapowerEquivalent(net)
    for k in range(3):
        r = pf.runpp(pl[k], ql[k], ps[k], qs[k])
        assert out["iterations"][k] == r.iterations and np.abs(out["vm"][k] - r.vm_pu).max() < TOL
        assert np.abs(out["q_bus"][k] - r.q_mvar).max() < TOL
    env.close()
    # Saadat Ex. 6.7 (meshed): the dense-LU fallback, published solution
    z = np.array([0.02 + 0.04j, 0.01 + 0.03j, 0.0125 + 0.025j])
    mesh = NetDesc(base_mva=100.0, n_bus=3, slack_bus=0, slack_vm=1.05, br_from=np.array([0, 0, 1]), br_to=np.array([1, 2, 2]),
                   br_r=z.real, br_x=z.imag, load_bus=np.array([1, 2]), sgen_bus=np.array([2]), sgen_zone=np.array([1]),
                   bus_zone=np.array([0, 1, 1]), name="saadat_6_7")
    env = EmuEnv(mesh, None, dict(voltage_barrier_type="l1"), batch=1)
    out = env.solve(np.array([[256.6, 138.6]]), np.array([[110.2, 45.2]]), np.zeros((1, 1)), np.zeros((1, 1)))
    V = out["vm"][0] * np.exp(1j * np.deg2rad(out["va_deg"][0]))
    assert np.abs(V - np.array([1.05, 0.98 - 0.06j, 1.00 - 0.05j])).max() < 1e-9
    env.close()


@pytest.mark.parametrize("name,barrier,batch,lanes", [("case33", "bowl", 5, 0), ("case33", "l1", 3, 4), ("case33", "bump", 9, 32),
                                                      ("case141", "l1", 3, 0), ("case33", "l2", 2, 64),
                                                      ("case322", "courant_beltrami", 2, 0)])
def test_emulated_trajectory_matches_oracle(name, barrier, batch, lanes):
    """reset (sampled start, noise, reset action) + noisy steps: helper warps, named barriers, Philox, epilogue."""
    net, prof = cases.make_case(name), cases.make_profiles(name, n_days=4)
    scale = cases.SCENARIOS[name]["action_scale"]
    env = EmuEnv(net, prof, dict(voltage_barrier_type=barrier, action_scale=scale, seed=5), batch=batch, lanes_per_env=lanes,
                 env_id_offset=100)
    ors = [VoltageControlOracle(net, prof, env.args, env_id=100 + i) for i in range(batch)]
    obs, st = env.reset()
    for i, o in enumerate(ors):
        oo, os_ = o.reset()
        assert np.abs(np.array(oo) - obs[i]).max() < TOL and np.abs(os_ - st[i]).max() < 1e-8
    rng = np.random.default_rng(1)
    for t in range(3 if name != "case322" else 2):
        a = rng.uniform(-scale, scale, (batch, net.n_sgen))
        r, term, info = env.step(a)
        it = env.get_field("nr_iters")[:, 0]
        for i, o in enumerate(ors):
            ro, to, io = o.step(a[i])
            assert abs(ro - r[i]) < TOL and to == bool(term[i]) and it[i] == o.g.res.iterations
            assert np.abs(np.array([io[k] for k in INFO_KEYS]) - info[i]).max() < TOL
            assert np.abs(np.array(o.get_obs()) - env.obs[i]).max() < TOL
    env.close()


@pytest.mark.parametrize("name", ["case33_bowl", "general_line_weight", "case33_state_space", "case33_divergence", "case141_l1",
                                  "case33_reset_keep"])
def test_emulated_kernel_reproduces_the_reference_executed_fixtures(name):
    """The kernel source, on the CPU, against trajectories the reference's own env code produced
    (tests/golden/ref_env_*.npz, see tests/test_reference_golden.py)."""
    replay_reference_fixture(name)


def replay_reference_fixture(name, lead=0):
    """Replays a reference-executed fixture on the emulated kernel. ``lead`` extra envs precede the fixture's envs in the
    batch (``env_id_offset = -lead`` keeps their env ids, hence their random streams), which moves them to a later CTA
    or a later round of the persistent loop. Returns the handle's dims."""
    g = np.load(S.fixture_path(ROOT, name))
    ops = [tuple(op) for op in json.loads(str(g["ops"]))]
    sc = S.SCENARIOS[name]
    net, prof = sc["build"]()
    ids = [lead + i for i in sc["env_ids"]]
    B = max(ids) + 1
    env = EmuEnv(net, prof, sc["args"], batch=B, env_id_offset=-lead)
    t = n_reset = 0
    for k_op, op in enumerate(ops):
        if op[0] == "step":
            a = np.zeros((B, net.n_sgen))
            a[ids] = g["actions"][t]
            r, term, info = env.step(a, add_noise=op[1])
            live = np.nonzero(g["alive"][t])[0]
            sel = [ids[k] for k in live]
            if live.size:
                assert np.abs(r[sel] - g["reward"][t, live]).max() < TOL and np.array_equal(term[sel], g["term"][t, live])
                assert np.abs(info[sel] - g["info"][t, live]).max() < TOL
            t += 1
            if live.size == 0:
                continue
        else:
            if op[0] in ("manual", "reset_keep"):
                start = np.zeros((B, 3), np.int32)
                for k, e in enumerate(ids):
                    start[e] = S.manual_of(sc, op, k) if op[0] == "manual" else g["start"][n_reset - 1, k]
                env.reset(start, add_noise=(op[0] == "reset_keep"))
            else:
                env.reset()
            n_reset += 1
            live, sel = np.arange(len(ids)), ids
        assert np.abs(env.obs[sel] - g["obs"][k_op, live][..., -env.dims["obs_dim"]:]).max() < TOL
        assert np.abs(env.get_state()[sel] - g["state"][k_op, live]).max() < 1e-8
    env.close()
    return env.dims


def _check_solve(net, lanes_list, B, rng, pl_hi, pv_hi):
    pf = PandapowerEquivalent(net)
    pl = rng.uniform(0.0, pl_hi, (B, net.n_load)); ql = 0.35 * pl
    pv = rng.uniform(0.0, pv_hi, (B, net.n_sgen)); q = rng.uniform(-0.3 * pv_hi, 0.3 * pv_hi, (B, net.n_sgen))
    for lanes in lanes_list:
        env = EmuEnv(net, None, dict(voltage_barrier_type="l1"), batch=1, lanes_per_env=lanes)
        out = env.solve(pl, ql, pv, q)
        for e in range(B):
            r = pf.runpp(pl[e], ql[e], pv[e], q[e])
            assert r.converged and out["converged"][e] == 1 and out["iterations"][e] == r.iterations
            assert np.abs(out["vm"][e] - r.vm_pu).max() < TOL and np.abs(out["va_deg"][e] - r.va_degree).max() < 1e-8
            assert np.abs(out["p_bus"][e] - r.p_mw).max() < 1e-8 and np.abs(out["pl"][e] - r.pl_mw).max() < TOL
        env.close()


def test_emulated_degenerate_topologies_and_hubs():
    """2-bus net, a star (forest of single-bus trees: no back sweep), a chain of 40 buses, and a net with a six-child hub
    plus a second hub (the > 2 children path of the sweeps), several lane counts - the same cases as the GPU tier."""
    rng = np.random.default_rng(5)
    two = NetDesc(base_mva=1.0, n_bus=2, slack_bus=1, slack_vm=1.01, br_from=[0], br_to=[1], br_r=[0.01], br_x=[0.02],
                  load_bus=[0], sgen_bus=[0], sgen_zone=[1], bus_zone=[1, 0])
    n = 9
    star = NetDesc(base_mva=1.0, n_bus=n, slack_bus=4, slack_vm=1.0, br_from=[4] * (n - 1), br_to=[b for b in range(n) if b != 4],
                   br_r=rng.uniform(0.005, 0.02, n - 1), br_x=rng.uniform(0.005, 0.02, n - 1), load_bus=np.arange(n),
                   sgen_bus=[0, 8], sgen_zone=[1, 2], bus_zone=[1, 1, 1, 1, 0, 2, 2, 2, 2])
    n = 40
    chain = NetDesc(base_mva=1.0, n_bus=n, slack_bus=0, slack_vm=1.0, br_from=np.arange(n - 1), br_to=np.arange(1, n),
                    br_r=rng.uniform(0.001, 0.004, n - 1), br_x=rng.uniform(0.001, 0.004, n - 1), load_bus=np.arange(1, n),
                    sgen_bus=[n - 1, n // 2], sgen_zone=[1, 1], bus_zone=[0] + [1] * (n - 1))
    for net in (two, star, chain):
        _check_solve(net, (0, 4, 32), 4, rng, 0.05, 0.2)
    f, t = [0], [1]
    nxt = 2
    for k in range(6):
        f += [1, nxt, nxt + 1]; t += [nxt, nxt + 1, nxt + 2]; nxt += 3
    for k in range(4):
        f.append(4); t.append(nxt); nxt += 1
    n = nxt
    hub = NetDesc(base_mva=1.0, n_bus=n, slack_bus=0, slack_vm=1.0, br_from=f, br_to=t, br_r=rng.uniform(0.002, 0.01, n - 1),
                  br_x=rng.uniform(0.002, 0.01, n - 1), load_bus=np.arange(1, n), sgen_bus=[3, 10, n - 1], sgen_zone=[1, 1, 1],
                  bus_zone=[0] + [1] * (n - 1))
    _check_solve(hub, (4, 8, 32, 64), 5, rng, 0.06, 0.3)


def test_emulated_divergence_flag_and_ragged_batches():
    net, p, q = cases.baran_wu_nominal()
    env = EmuEnv(net, None, dict(voltage_barrier_type="l1"), batch=1)
    out = env.solve(np.stack([p, p * 40, p]), np.stack([q, q * 40, q]), np.zeros((3, 6)), np.zeros((3, 6)))
    assert out["converged"].tolist() == [1, 0, 1] and out["iterations"][1] == 10
    assert np.abs(out["vm"][0] - out["vm"][2]).max() == 0.0
    pf = PandapowerEquivalent(net)
    for nb in (1, 2, 3, 17, 33):
        inp = cases.synthetic_inputs("case33", nb, seed=nb)
        qs = inp["action"] * np.sqrt(inp["s_max"] ** 2 - inp["p_pv"] ** 2)
        out = env.solve(inp["p_load"], inp["q_load"], inp["p_pv"], qs)
        for e in range(nb):
            assert np.abs(out["vm"][e] - pf.runpp(inp["p_load"][e], inp["q_load"][e], inp["p_pv"][e], qs[e]).vm_pu).max() < TOL
    env.close()


def test_emulated_node_relabelling_changes_addresses_not_results(monkeypatch):
    """The bank-conflict-aware node ids only move records inside shared memory; the static first-iteration factors are
    accumulated in a labelling-independent order: bit-identical results with and without the relabelling."""
    net, prof = cases.make_case("case33"), cases.make_profiles("case33", n_days=4)
    args = dict(seed=6, voltage_barrier_type="bowl")
    monkeypatch.setenv("MAPDN_NO_RELABEL", "1")
    e0 = EmuEnv(net, prof, args, batch=6)
    monkeypatch.delenv("MAPDN_NO_RELABEL")
    e1 = EmuEnv(net, prof, args, batch=6)
    o0, s0 = e0.reset(); o1, s1 = e1.reset()
    assert np.array_equal(o0, o1) and np.array_equal(s0, s1)
    rng = np.random.default_rng(0)
    for _ in range(3):
        a = rng.uniform(-0.8, 0.8, (6, 6))
        r0, t0, i0 = e0.step(a); r1, t1, i1 = e1.step(a)
        assert np.array_equal(r0, r1) and np.array_equal(i0, i1) and np.array_equal(e0.obs, e1.obs)
        assert np.array_equal(e0.get_field("vm"), e1.get_field("vm"))
    e0.close(); e1.close()


def _oracle_droop(net, pl, ql, pv, s_rated, max_ite=100, gain=0.1):
    """Literal restatement of reference traditional_control/pf_droop_matpower_all.m:121-152,196-231 (one instant)."""
    pf = PandapowerEquivalent(net)

    def droop(p, s, v, qmm):
        q_max = min(np.sqrt(s * s - p * p), qmm)
        if v <= 0.95: return q_max
        if v > 1.05: return -q_max
        if 1.0 <= v <= 1.0: return 0.0
        if v < 1.0: return (q_max - 0) / (0.95 - 1.0) * (v - 1.0)
        return (0 - q_max) / (1.0 - 1.05) * (1.0 - v)
    q_last = np.zeros(net.n_sgen); v_last = 100 * np.ones(net.n_sgen)
    for i in range(max_ite):
        res = pf.runpp(pl, ql, pv, q_last)
        v = res.vm_pu[net.sgen_bus]
        if np.linalg.norm(v_last - v) < 1e-4:
            break
        v_last = v
        q_new = np.array([droop(pv[j], s_rated[j], v[j], s_rated[j]) for j in range(net.n_sgen)])
        q_last = (1 - gain) * q_last + gain * q_new
    return res.vm_pu, q_last, res.pl_mw.sum(), i + 1


def test_emulated_droop_baseline_matches_the_script():
    """MODE_DROOP (one launch: the relaxed loop of <= 100 power flows, per-env stopping rule) on the tree solver and on the
    dense fallback of a meshed net."""
    net = cases.case33()
    inp = cases.synthetic_inputs("case33", 5, seed=4)
    env = EmuEnv(net, None, None, batch=1)
    out = env.droop(inp["p_load"], inp["q_load"], inp["p_pv"], inp["s_max"])
    for e in range(5):
        vm, q, loss, it = _oracle_droop(net, inp["p_load"][e], inp["q_load"][e], inp["p_pv"][e], inp["s_max"])
        assert out["iterations"][e] == it and np.abs(out["vm"][e] - vm).max() < 1e-8
        assert np.abs(out["q"][e] - q).max() < 1e-8 and abs(out["loss"][e] - loss) < 1e-8
    env.close()
    z = np.array([0.02 + 0.04j, 0.01 + 0.03j, 0.0125 + 0.025j, 0.015 + 0.03j])
    mesh = NetDesc(base_mva=100.0, n_bus=4, slack_bus=0, slack_vm=1.03, br_from=np.array([0, 0, 1, 2]), br_to=np.array([1, 2, 2, 3]),
                   br_r=z.real, br_x=z.imag, load_bus=np.array([1, 2, 3]), sgen_bus=np.array([2, 3]), sgen_zone=np.array([1, 1]),
                   bus_zone=np.array([0, 1, 1, 1]), name="mesh4")
    env = EmuEnv(mesh, None, None, batch=1)
    rng = np.random.default_rng(2)
    pl = rng.uniform(80, 260, (4, 3)); ql = pl * rng.uniform(0.2, 0.5, (4, 3)); pv = rng.uniform(0, 60, (4, 2))
    out = env.droop(pl, ql, pv, np.array([80.0, 80.0]))
    for e in range(4):
        vm, q, loss, it = _oracle_droop(mesh, pl[e], ql[e], pv[e], np.array([80.0, 80.0]))
        assert out["iterations"][e] == it and it > 2 and np.abs(out["vm"][e] - vm).max() < 1e-8 and np.abs(out["q"][e] - q).max() < 1e-7
    env.close()


@pytest.mark.parametrize("scenario,batch", [("case33", 6), ("case141", 2)])
def test_emulated_host_paths_deliver_the_same_transition(scenario, batch):
    """mapdn_step (device buffers) == mapdn_step_host (staged copies) == mapdn_step_host_pinned (zero-copy, padding not
    rewritten) == mapdn_step_host_compact (rows without the padding, copied or written directly), fp64 and fp32."""
    net, prof = cases.make_case(scenario), cases.make_profiles(scenario, n_days=3)
    envs = [EmuEnv(net, prof, dict(seed=11), batch=batch) for _ in range(6)]
    for e in envs:
        e.reset()
    slices, row = envs[0].compact_layout()
    assert len(slices) == net.n_sgen and row % 4 == 0 and sum(n for _, n in slices) <= row < sum(n for _, n in slices) + 4
    rng = np.random.default_rng(5)
    for t in range(2):
        act = rng.uniform(-0.6, 0.6, (batch, net.n_sgen))
        r, tm, info = envs[0].step(act)
        ref = envs[0].obs
        outs = [envs[1].step_host(act, path="staged"), envs[2].step_host(act, path="pinned"),
                envs[3].step_host(act, path="compact", direct=bool(t & 1)), envs[4].step_host(act, path="compact", f32=True, direct=not (t & 1)),
                envs[5].step_host(act, path="pinned", f32=True)]
        for k, (r2, t2, i2, o2) in enumerate(outs):
            assert np.array_equal(r, r2) and np.array_equal(tm, t2) and np.array_equal(info, i2), k
        assert np.array_equal(outs[0][3], ref) and np.array_equal(outs[1][3], ref) and np.array_equal(outs[4][3], ref.astype(np.float32))
        for o, dt in ((outs[2][3], np.float64), (outs[3][3], np.float32)):
            for a, (off, n) in enumerate(slices):
                assert np.array_equal(o[:, off:off + n], ref[:, a, :n].astype(dt)) and not np.any(ref[:, a, n:])
            assert not np.any(o[:, sum(n for _, n in slices):])
    for e in envs:
        e.close()


def test_plain_c_caller_through_the_emulated_library():
    """examples/c_abi_demo.c (strict C99, host buffers, no CUDA header) linked against the EMULATED library: the whole
    boundary - C caller -> extern "C" entry points -> host code -> kernel source - runs on the CPU and prints what the
    NumPy binding of the same library computes for the same feeder. (Against the real library the demo fails loudly
    without a GPU: tests/test_c_abi_demo.py.)"""
    import shutil
    import subprocess
    from emu_env import build as build_emu
    from test_c_abi_demo import SRC, _demo_inputs
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    lib = build_emu()
    exe = os.path.join(os.path.dirname(lib), "c_abi_demo_emu")
    r = subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-O2", "-I", os.path.join(ROOT, "include"), SRC,
                        "-o", exe, lib, "-Wl,-rpath," + os.path.dirname(lib), "-lm"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.strip().splitlines()
    got = [ln.split() for ln in lines if ln.startswith("step ")]
    assert lines[0].startswith("dims n_agents 2 obs_dim ") and len(got) == 10
    net, prof = _demo_inputs()
    env = EmuEnv(net, prof, dict(voltage_barrier_type="bowl", seed=2024, action_scale=0.8), batch=8)
    env.reset()
    for k in range(10):
        a = np.array([[-0.8 + 1.6 * ((e * 7 + g * 3 + k) % 11) / 10.0 for g in range(2)] for e in range(8)])
        rew, term, _ = env.step(a)
        rs, os_ = float(got[k][2]), float(got[k][3])
        assert abs(rs - float(rew.sum())) < 1e-12 * max(1.0, abs(rs)) and abs(os_ - float(env.obs.sum())) < 1e-12 * max(1.0, abs(os_))
        assert int(got[k][4]) == int(term.sum())
    env.close()
