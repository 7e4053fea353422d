"""GPU tier: the launch geometries of the full-size batches on the B200 (148 SMs), against the oracle. At these sizes the
planner runs a persistent loop of two rounds per CTA, and case322 runs shared-memory plan 3 (cold tables in global memory,
loads staged in the node records); see tests/test_emu_geometry.py for the table and the plans. MAPDN_PLAN /
MAPDN_HELPERS / MAPDN_EPB force the planner's other choices, which must not change a bit of the results."""
import numpy as np
import pytest
import torch

from mapdn_b200 import cases
from test_emu_geometry import FULL_SIZE

pytestmark = pytest.mark.gpu
TOL = 1e-9
N_SM = 148


@pytest.fixture(autouse=True)
def _no_overrides(monkeypatch):
    for k in ("MAPDN_PLAN", "MAPDN_HELPERS", "MAPDN_EPB", "MAPDN_NO_RELABEL"):
        monkeypatch.delenv(k, raising=False)


def _make(net, prof, args, batch):
    from mapdn_b200.env import BatchedVoltageControl
    return BatchedVoltageControl(net, prof, args, batch=batch)


def _scenario(name, barrier=None, line_weight=None):
    sc = cases.SCENARIOS[name]
    args = dict(voltage_barrier_type=barrier or sc["barrier"], action_scale=sc["action_scale"], seed=13)
    if line_weight is not None:
        args["line_weight"] = line_weight
    return cases.make_case(name), cases.make_profiles(name), args


def _geometry(env):
    d = env.dims
    return d["lanes_per_env"], d["envs_per_block"], d["smem_bytes"]


def _launch_grid(batch, epb, max_blocks):
    """(CTAs, rounds per CTA) of launch_env_kernel."""
    needed = -(-batch // epb)
    grid = min(needed, max_blocks)
    rounds = -(-needed // grid)
    return -(-needed // rounds), rounds


def _sample_ids(batch, epb, grid):
    """First and last group of the first CTAs of both rounds, the last env of round 1, the middle, the last env."""
    r2 = grid * epb
    ids = {0, 1, epb - 1, epb, 2 * epb - 1, batch // 2, r2 - 1, r2, r2 + 1, r2 + epb - 1, r2 + epb, batch - 1}
    return sorted(i for i in ids if 0 <= i < batch)


def _check(env, oracles, ids, a=None):
    """Reset (a is None) or step outputs of the sampled envs against their oracles: vm, reward, terminated, the 11 info
    values, NR iterations, obs and state."""
    from oracle.voltage_control_ref import INFO_KEYS
    torch.cuda.synchronize()
    obs, st, vm = env.obs.cpu().numpy(), env.get_state().cpu().numpy(), env.get_field("vm").cpu().numpy()
    if a is None:
        for o, i in zip(oracles, ids):
            oo, os_ = o.reset()
            assert np.abs(np.array(oo) - obs[i]).max() < TOL and np.abs(os_ - st[i]).max() < 1e-8, i
            assert np.abs(o.g.res.vm_pu - vm[i]).max() < TOL, i
        return
    r, term, info = env.reward.cpu().numpy(), env.terminated.cpu().numpy(), env.info.cpu().numpy()
    it = env.get_field("nr_iters")[:, 0].cpu().numpy()
    for o, i in zip(oracles, ids):
        ro, to, io = o.step(a[i])
        assert abs(ro - r[i]) < TOL and to == bool(term[i]) and it[i] == o.g.res.iterations, i
        assert np.abs(np.array([io[k] for k in INFO_KEYS]) - info[i]).max() < TOL, i
        assert np.abs(o.g.res.vm_pu - vm[i]).max() < TOL, i
        assert np.abs(np.array(o.get_obs()) - obs[i]).max() < TOL, i
        assert np.abs(o.get_state() - st[i]).max() < 1e-8, i


def _episodes(env, net, prof, args, ids, steps=3):
    """Sampled reset with noise and the reset action, noisy steps, and a second episode."""
    from oracle.voltage_control_ref import VoltageControlOracle
    oracles = [VoltageControlOracle(net, prof, env.args, env_id=i) for i in ids]
    rng = np.random.default_rng(4)
    scale = args["action_scale"]
    for n_steps in (steps, 1):
        env.reset()
        _check(env, oracles, ids)
        for t in range(n_steps):
            a = rng.uniform(-scale, scale, (env.batch, net.n_sgen))
            env.step(torch.tensor(a, device=env.device))
            _check(env, oracles, ids, a)


@pytest.mark.parametrize("name,batch,barrier,line_weight", [("case141", 2048, "l1", None), ("case322", 1024, "bowl", None),
                                                            ("case322", 1024, "bowl", 0.4)])
def test_full_size_geometry_matches_oracle(name, batch, barrier, line_weight):
    """BASELINE.json config 2 (case141 x 2048, L1) and config 5 (case322 x 1024, bowl) at their default geometry: two
    rounds per CTA, plan 3 for case322; envs of both rounds against the oracle."""
    assert torch.cuda.get_device_properties(0).multi_processor_count == N_SM
    net, prof, args = _scenario(name, barrier, line_weight)
    env = _make(net, prof, args, batch)
    lanes, epb, smem, plan, rounds = FULL_SIZE[(name, batch)]
    assert _geometry(env) == (lanes, epb, smem)
    grid, r = _launch_grid(batch, epb, N_SM)          # one CTA per SM at these footprints
    assert r == rounds == 2
    _episodes(env, net, prof, args, _sample_ids(batch, epb, grid))
    env.close()


def _all_paths(env, name, net):
    """reset, two noisy steps, fields, a compact host step, solve and droop: every output on the host."""
    from mapdn_b200.baselines import droop_control
    B = env.batch
    rng = np.random.default_rng(6)
    out = [t.cpu().numpy().copy() for t in env.reset()]
    for _ in range(2):
        a = torch.tensor(rng.uniform(-0.6, 0.6, (B, net.n_sgen)), device=env.device)
        out += [t.cpu().numpy().copy() for t in env.step(a)] + [env.obs.cpu().numpy().copy()]
    out += [env.get_field(f).cpu().numpy() for f in ("vm", "va_deg", "line_loss", "q_sgen", "nr_iters")]
    out += [env.get_state().cpu().numpy().copy()]
    out += [x.copy() for x in env.step_host(rng.uniform(-0.6, 0.6, (B, net.n_sgen)), layout="compact")]
    inp = cases.synthetic_inputs(name, B, seed=2)
    t = {k: torch.tensor(v, device=env.device) for k, v in inp.items()}
    qs = t["action"] * torch.sqrt(t["s_max"] ** 2 - t["p_pv"] ** 2)
    out += [v.cpu().numpy() for v in env.solve(t["p_load"], t["q_load"], t["p_pv"], qs).values()]
    out += [v.cpu().numpy() for v in droop_control(env, t["p_load"], t["q_load"], t["p_pv"], t["s_max"]).values()]
    return out


def _assert_bit_identical(outs, labels):
    for lab, out in zip(labels[1:], outs[1:]):
        assert len(out) == len(outs[0])
        for k, (x, y) in enumerate(zip(out, outs[0])):
            assert np.array_equal(x, y), (lab, k)


def test_forced_plans_are_bit_identical_on_case322_x_1024(monkeypatch):
    """The four shared-memory plans at full size on the device: the pieces the emulation skips (L2 prefetch of the cold
    tables, __ldg, the TMA copy of a 229 kB footprint) must not change a bit of reset, step, solve, droop and the compact
    host step."""
    net, prof, args = _scenario("case322")
    outs, geoms = [], []
    for plan in range(4):
        monkeypatch.setenv("MAPDN_PLAN", str(plan))
        env = _make(net, prof, args, 1024)
        geoms.append(_geometry(env))
        outs.append(_all_paths(env, "case322", net))
        env.close()
    assert len({g[2] for g in geoms}) == 4, geoms       # the planner drops a forced plan that does not fit
    assert geoms[3] == FULL_SIZE[("case322", 1024)][:3]
    _assert_bit_identical(outs, [f"plan {p}" for p in range(4)])


def test_helper_warps_and_envs_per_cta_are_bit_identical_on_case141_x_2048(monkeypatch):
    net, prof, args = _scenario("case141")
    outs, labels, epbs = [], [], set()
    for var, values in (("MAPDN_HELPERS", ("1", "2", "3", "4")), ("MAPDN_EPB", ("3", "5", "8"))):
        for v in values:
            monkeypatch.setenv(var, v)
            env = _make(net, prof, args, 2048)
            if var == "MAPDN_EPB":
                epbs.add(env.dims["envs_per_block"])
            outs.append(_all_paths(env, "case141", net))
            labels.append(f"{var}={v}")
            env.close()
        monkeypatch.delenv(var)
    assert len(epbs) == 3, epbs
    _assert_bit_identical(outs, labels)


def test_dense_fallback_past_the_workspace_bound_matches_oracle():
    """A meshed net caps the CTAs at 2 per SM (one dense workspace slice per resident env group; fewer where the
    registers limit the occupancy): with more envs than that, later rounds reuse the slices. Envs at the round boundaries
    of both possible grids against the oracle."""
    from test_gpu_solve import _case33_meshed
    net, prof = _case33_meshed(), cases.make_profiles("case33", n_days=4)
    args = dict(voltage_barrier_type="bowl", action_scale=0.8, seed=6)
    B = 3000
    env = _make(net, prof, args, B)
    epb = env.dims["envs_per_block"]
    assert env.dims["lanes_per_env"] == 32
    ids = {B - 1}
    for per_sm in (1, 2):
        grid, rounds = _launch_grid(B, epb, per_sm * N_SM)
        assert rounds >= 2
        ids |= {i for r in range(rounds) for i in (r * grid * epb, r * grid * epb + epb - 1, (r + 1) * grid * epb - 1)}
    _episodes(env, net, prof, args, sorted(i for i in ids if i < B), steps=2)
    env.close()
