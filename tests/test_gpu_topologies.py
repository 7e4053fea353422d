"""GPU tier: the generated topologies of tests/topo_corpus.py on the B200 (see tests/test_emu_topologies.py for what they
reach in the schedule builder). Every solve runs a batch large enough for at least two rounds of the persistent loop per
CTA (the meshed nets: for later rounds reusing the dense workspace slices); the three injection rows of a net are tiled
over the batch and every env is compared with the oracle."""
import numpy as np
import pytest
import torch

import topo_corpus as T
from test_emu_topologies import LANES, MAX_SMEM, NETS, RADIAL, WHOLE_ENV, least_footprint

pytestmark = pytest.mark.gpu
N_SM, SMEM_PER_SM, SMEM_RESERVED = 148, 233472, 1024
MESHED = [n for n, e in NETS.items() if T.is_meshed(e.net)]


@pytest.fixture(autouse=True)
def _no_overrides(monkeypatch):
    for k in ("MAPDN_PLAN", "MAPDN_HELPERS", "MAPDN_EPB", "MAPDN_NO_RELABEL", "MAPDN_DEBUG_SCHED"):
        monkeypatch.delenv(k, raising=False)


def _two_round_batch(env, meshed):
    """A batch with more env groups than can be resident at once: the launch grid is capped at the CTAs per SM the
    occupancy allows (at most 32, 2048 threads and the shared memory; 2 for a meshed net) times the SMs."""
    d = env.dims
    epb, threads = d["envs_per_block"], d["envs_per_block"] * d["lanes_per_env"]
    per_sm = 2 if meshed else min(32, 2048 // threads, SMEM_PER_SM // (d["smem_bytes"] + SMEM_RESERVED))
    return 2 * epb * per_sm * N_SM + 1


def _solve_tiled(env, name, meshed):
    from oracle.pandapower_nr import PandapowerEquivalent
    e = NETS[name]
    inp = T.injections(e.net, e.seed)
    pf = PandapowerEquivalent(e.net)
    refs = [pf.runpp(*(x[k] for x in inp)) for k in range(3)]
    nb = _two_round_batch(env, meshed)
    rows = np.arange(nb) % 3
    out = env.solve(*(torch.tensor(x[rows], device=env.device) for x in inp))
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in out.items()}
    for k, r in enumerate(refs):
        sel = rows == k
        assert np.all(out["converged"][sel] == r.converged) and np.all(out["iterations"][sel] == r.iterations), k
        if r.converged:
            assert np.abs(out["vm"][sel] - r.vm_pu).max() < 1e-9, k
            assert np.abs(out["va_deg"][sel] - r.va_degree).max() < 1e-8, k
            assert np.abs(out["p_bus"][sel] - r.p_mw).max() < 1e-8 and np.abs(out["q_bus"][sel] - r.q_mvar).max() < 1e-8, k
            assert np.abs(out["pl"][sel] - r.pl_mw).max() < 1e-9, k


@pytest.mark.parametrize("name", RADIAL)
def test_tree_solver_matches_oracle_at_every_lane_count(name):
    from mapdn_b200._capi import MapdnError
    from mapdn_b200.env import BatchedVoltageControl
    net = NETS[name].net
    ran = 0
    for lanes in LANES:
        if lanes and least_footprint(net, lanes) > MAX_SMEM:
            with pytest.raises(MapdnError, match="too large"):
                BatchedVoltageControl(net, None, None, batch=1, lanes_per_env=lanes)
            continue
        env = BatchedVoltageControl(net, None, None, batch=1, lanes_per_env=lanes)
        assert lanes in (0, env.dims["lanes_per_env"])
        _solve_tiled(env, name, False)
        env.close()
        ran += 1
    assert ran >= 5


@pytest.mark.parametrize("name", MESHED)
def test_dense_fallback_matches_oracle(name):
    from mapdn_b200.env import BatchedVoltageControl
    env = BatchedVoltageControl(NETS[name].net, None, None, batch=1)
    assert env.dims["lanes_per_env"] == 32
    _solve_tiled(env, name, True)
    env.close()


@pytest.mark.parametrize("name", WHOLE_ENV + ["meshed130", "meshed257"])
def test_whole_env_matches_oracle(name):
    """reset + 3 noisy steps and a second episode on sampled envs of a batch of 64, then the droop baseline with
    q_max_manual below s_rated."""
    from mapdn_b200.baselines import droop_control
    from mapdn_b200.env import BatchedVoltageControl
    from test_emu_kernel import _oracle_droop
    from test_gpu_geometry import _episodes
    e = NETS[name]
    net, prof = e.net, T.profile(e.net)
    args = dict(voltage_barrier_type="bowl", action_scale=0.8, seed=e.seed, line_weight=0.3)
    env = BatchedVoltageControl(net, prof, args, batch=64)
    _episodes(env, net, prof, args, [0, 1, 31, 63], steps=3)
    pl, ql, pv, _ = T.injections(net, e.seed + 1, B=2)
    s_rated = prof.s_max
    pv = np.minimum(pv, 0.9 * s_rated)
    qmm = s_rated * np.linspace(0.15, 0.6, net.n_sgen)
    out = droop_control(env, pl, ql, pv, s_rated, q_max_manual=qmm)
    out = {k: v.cpu().numpy() for k, v in out.items()}
    env.close()
    for k in range(2):
        vm, q, loss, it = _oracle_droop(net, pl[k], ql[k], pv[k], s_rated, q_max_manual=qmm)
        assert it < 100 and out["iterations"][k] == it and np.abs(out["vm"][k] - vm).max() < 1e-8, k
        assert np.abs(out["q"][k] - q).max() < 1e-8 and abs(out["loss"][k] - loss) < 1e-8, k
