"""CPU tier: the launch geometries mapdn_create picks at full batch size, run on the emulated device (tests/emu) against
the oracle. The planner chooses from the batch size and the SM count: lanes per env, envs per CTA, the number of rounds of
the persistent loop per CTA, the number of helper warps, and one of four shared-memory plans, each with its own code:

    plan 0  everything in shared memory
    plan 1  the scaled loads staged in the dead Newton fields of the node records (stage_in_records)
    plan 2  the once-per-step tables (Y[i,slack], observation program, line tables) in global memory
    plan 3  both

At small batches on 148 SMs it always picks plan 0 in one round. With one emulated SM (MAPDN_EMU_SMS=1) it picks the
full-size geometry at a batch the emulation can run; MAPDN_PLAN / MAPDN_HELPERS / MAPDN_EPB force the other choices."""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT
from mapdn_b200 import cases

sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
from emu_env import EmuEnv                                          # noqa: E402
from oracle import ref_scenarios as S                               # noqa: E402
from oracle.voltage_control_ref import INFO_KEYS, VoltageControlOracle   # noqa: E402
from test_emu_kernel import replay_reference_fixture               # noqa: E402

TOL = 1e-9
SMEM_PER_SM, SMEM_RESERVED = 233472, 1024          # emulated B200 (tests/emu/cuda_runtime.h)

# (scenario, batch): (lanes per env, envs per CTA, dynamic shared memory in bytes, plan, rounds per CTA)
FULL_SIZE = {("case33", 4096): (8, 28, 161792, 0, 1),       # BASELINE.json config 1
             ("case141", 2048): (32, 7, 182560, 0, 2),      # config 2
             ("case322", 1024): (64, 4, 229328, 3, 2),      # configs 3 and 5, the per-GPU shards of config 4
             ("case322", 512): (64, 4, 229328, 3, 1)}
ONE_SM = {("case33", 28): (8, 28, 161792, 0, 1),
          ("case141", 14): (32, 7, 182560, 0, 2),
          ("case322", 8): (64, 4, 229328, 3, 2)}


@pytest.fixture(autouse=True)
def _no_overrides(monkeypatch):
    for k in ("MAPDN_EMU_SMS", "MAPDN_PLAN", "MAPDN_HELPERS", "MAPDN_EPB", "MAPDN_NO_RELABEL"):
        monkeypatch.delenv(k, raising=False)


def _scenario(name, **extra):
    net, prof = cases.make_case(name), cases.make_profiles(name, n_days=4)
    sc = cases.SCENARIOS[name]
    return net, prof, dict(voltage_barrier_type=sc["barrier"], action_scale=sc["action_scale"], seed=5, **extra)


def _geometry(env):
    d = env.dims
    return d["lanes_per_env"], d["envs_per_block"], d["smem_bytes"]


def rounds_per_cta(batch, epb, smem, n_sm):
    """Rounds of the persistent loop (launch_env_kernel) for a footprint that fits one CTA per SM."""
    assert 2 * (smem + SMEM_RESERVED) > SMEM_PER_SM
    needed = -(-batch // epb)
    return -(-needed // min(needed, n_sm))


def _forced_plans(monkeypatch, net, prof, args, batch, lanes=0):
    out = []
    for plan in range(4):
        monkeypatch.setenv("MAPDN_PLAN", str(plan))
        e = EmuEnv(net, prof, args, batch=batch, lanes_per_env=lanes)
        out.append(_geometry(e))
        e.close()
    monkeypatch.delenv("MAPDN_PLAN")
    assert len({g[2] for g in out}) == 4, out          # the planner drops a forced plan that does not fit
    return out


@pytest.mark.parametrize("table,sms", [(FULL_SIZE, None), (ONE_SM, "1")])
def test_planner_geometry_table(monkeypatch, table, sms):
    """The geometries below are what the other tests of this file (and tests/test_gpu_geometry.py) run as the production
    path; a change of the planner must update them. The plan is identified by the footprint of the forced plans."""
    if sms:
        monkeypatch.setenv("MAPDN_EMU_SMS", sms)
    for (name, batch), (lanes, epb, smem, plan, rounds) in table.items():
        net, prof, args = _scenario(name)
        e = EmuEnv(net, prof, args, batch=batch)
        got = _geometry(e)
        e.close()
        assert got == (lanes, epb, smem), (name, batch, got)
        assert _forced_plans(monkeypatch, net, prof, args, batch)[plan][2] == smem, (name, batch)
        assert rounds_per_cta(batch, epb, smem, 1 if sms else 148) == rounds, (name, batch)


def _check_against_oracles(env, oracles, a=None):
    """reset (a is None) or step outputs of every env against its oracle: reward, terminated, the 11 info values, NR
    iterations, obs, state."""
    if a is None:
        obs, st = env.obs, env.state
        for i, o in enumerate(oracles):
            oo, os_ = o.reset()
            assert np.abs(np.array(oo) - obs[i]).max() < TOL and np.abs(os_ - st[i]).max() < 1e-8, i
        return
    r, term, info = env.reward, env.term, env.info
    it = env.get_field("nr_iters")[:, 0]
    st = env.get_state()
    for i, o in enumerate(oracles):
        ro, to, io = o.step(a[i])
        assert abs(ro - r[i]) < TOL and to == bool(term[i]) and it[i] == o.g.res.iterations, i
        assert np.abs(np.array([io[k] for k in INFO_KEYS]) - info[i]).max() < TOL, i
        assert np.abs(np.array(o.get_obs()) - env.obs[i]).max() < TOL, i
        assert np.abs(o.get_state() - st[i]).max() < 1e-8, i


def _episodes_against_oracles(env, net, prof, args, steps=3, seed=1):
    """Sampled reset with noise and the reset action, noisy steps, and a second episode (the episode counter re-keys the
    random streams), every env of the batch against its own oracle."""
    B, scale = env.batch, args["action_scale"]
    oracles = [VoltageControlOracle(net, prof, env.args, env_id=i) for i in range(B)]
    rng = np.random.default_rng(seed)
    for n_steps in (steps, 1):
        env.reset()
        _check_against_oracles(env, oracles)
        for t in range(n_steps):
            a = rng.uniform(-scale, scale, (B, net.n_sgen))
            env.step(a)
            _check_against_oracles(env, oracles, a)


@pytest.mark.parametrize("name,batch,line_weight", [("case33", 28, None), ("case33", 57, None), ("case141", 14, None),
                                                    ("case322", 8, None), ("case322", 8, 0.4)])
def test_production_geometry_on_one_sm_matches_oracle(monkeypatch, name, batch, line_weight):
    """The full-size geometry of ONE_SM (case33 x 57: two rounds of 32 envs) against the oracle, every env of both
    rounds. line_weight puts the line tables (global memory under plan 3) into the reward."""
    monkeypatch.setenv("MAPDN_EMU_SMS", "1")
    net, prof, args = _scenario(name, **({} if line_weight is None else dict(line_weight=line_weight)))
    env = EmuEnv(net, prof, args, batch=batch)
    lanes, epb, smem = _geometry(env)
    if (name, batch) in ONE_SM:
        assert (lanes, epb, smem) == ONE_SM[(name, batch)][:3]
    assert rounds_per_cta(batch, epb, smem, 1) == 2 or (name, batch) == ("case33", 28)
    _episodes_against_oracles(env, net, prof, args)
    env.close()


def _run_all_paths(env, name, net, seed=0):
    """reset, two noisy steps, a compact host step, solve and droop: every output, for bitwise comparison."""
    B = env.batch
    out = [a.copy() for a in env.reset()]
    rng = np.random.default_rng(seed)
    for t in range(2):
        out += [a.copy() for a in env.step(rng.uniform(-0.6, 0.6, (B, net.n_sgen)))] + [env.obs.copy()]
    out += [env.get_field(f) for f in ("vm", "va_deg", "line_loss", "q_sgen", "nr_iters")] + [env.get_state().copy()]
    out += list(env.step_host(rng.uniform(-0.6, 0.6, (B, net.n_sgen)), path="compact"))
    inp = cases.synthetic_inputs(name, B, seed=seed + 1)
    qs = inp["action"] * np.sqrt(inp["s_max"] ** 2 - inp["p_pv"] ** 2)
    out += list(env.solve(inp["p_load"], inp["q_load"], inp["p_pv"], qs).values())
    out += list(env.droop(inp["p_load"], inp["q_load"], inp["p_pv"], inp["s_max"], max_ite=8).values())
    return out


@pytest.mark.parametrize("name,lanes,batch", [("case33", 4, 6), ("case33", 8, 6), ("case141", 32, 3), ("case141", 64, 3)])
def test_every_plan_forced_is_bit_identical(monkeypatch, name, lanes, batch):
    """The four shared-memory plans only move data: step, solve, droop and the compact host step are bit-identical to
    plan 0 (case33 is relabelled for bank conflicts, so plans 2 and 3 also run the relabelled node ids against the
    global-memory tables). Plan 3 is also checked against the oracle."""
    net, prof, args = _scenario(name)
    geoms = _forced_plans(monkeypatch, net, prof, args, batch, lanes)
    assert all(g[0] == lanes for g in geoms)
    ref = None
    for plan in (0, 1, 2, 3):
        monkeypatch.setenv("MAPDN_PLAN", str(plan))
        env = EmuEnv(net, prof, args, batch=batch, lanes_per_env=lanes)
        assert _geometry(env) == geoms[plan]
        out = _run_all_paths(env, name, net)
        env.close()
        if ref is None:
            ref = out
        else:
            assert len(out) == len(ref)
            for k, (x, y) in enumerate(zip(out, ref)):
                assert np.array_equal(x, y), (plan, k)
    env = EmuEnv(net, prof, args, batch=batch, lanes_per_env=lanes)      # MAPDN_PLAN=3 still set
    _episodes_against_oracles(env, net, prof, args, steps=2)
    env.close()


def test_helper_warp_counts_are_bit_identical(monkeypatch):
    """1-4 helper warps draw the next profile rows and the noise of a CTA round; two rounds per CTA (case141 on one SM)."""
    monkeypatch.setenv("MAPDN_EMU_SMS", "1")
    net, prof, args = _scenario("case141")
    ref = None
    for helpers in ("1", "2", "3", "4"):
        monkeypatch.setenv("MAPDN_HELPERS", helpers)
        env = EmuEnv(net, prof, args, batch=14)
        assert _geometry(env) == ONE_SM[("case141", 14)][:3]
        out = [a.copy() for a in env.reset()]
        rng = np.random.default_rng(2)
        for t in range(2):
            out += [a.copy() for a in env.step(rng.uniform(-0.6, 0.6, (14, net.n_sgen)))] + [env.obs.copy()]
        out += [env.get_field("p_load"), env.get_field("p_sgen")]
        env.close()
        if ref is None:
            ref = out
        for k, (x, y) in enumerate(zip(out, ref)):
            assert np.array_equal(x, y), (helpers, k)


def test_reset_retries_and_divergence_under_plan3_in_the_second_round(monkeypatch):
    """The reference-executed divergence fixture (reset re-draws, the -200 branch, the rolled-back state) with the
    fixture's envs in the second round of the only CTA (32 envs ahead of them) under plan 3."""
    monkeypatch.setenv("MAPDN_EMU_SMS", "1")
    monkeypatch.setenv("MAPDN_PLAN", "3")
    monkeypatch.setenv("MAPDN_EPB", "32")
    d = replay_reference_fixture("case33_divergence", lead=32)
    assert d["envs_per_block"] == 32 and rounds_per_cta(d["batch"], 32, d["smem_bytes"], 1) == 2
    sc = S.SCENARIOS["case33_divergence"]
    assert d["smem_bytes"] == _forced_plans(monkeypatch, *sc["build"](), sc["args"], d["batch"])[3][2]


def test_dense_fallback_with_more_rounds_than_resident_groups(monkeypatch):
    """Meshed nets bound the dense workspace to 2 CTAs per SM (one slice per resident env group): on one SM, one env per
    CTA and 3 envs, CTA 0 runs env 0 and then env 2 in the same slice."""
    from test_gpu_solve import _case33_meshed
    monkeypatch.setenv("MAPDN_EMU_SMS", "1")
    monkeypatch.setenv("MAPDN_EPB", "1")
    net, prof = _case33_meshed(), cases.make_profiles("case33", n_days=4)
    args = dict(voltage_barrier_type="bowl", action_scale=0.8, seed=6)
    env = EmuEnv(net, prof, args, batch=3)
    assert env.dims["lanes_per_env"] == 32 and env.dims["envs_per_block"] == 1
    _episodes_against_oracles(env, net, prof, args, steps=1)
    env.close()
