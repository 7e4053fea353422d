"""The batched runner holds the conversation the REFERENCE's learners (models/*.py, utilities/trainer.py) expect.

tests/golden/ref_learner_*.npz record the reference learners' side of that conversation, written by
scripts/make_reference_extra_golden.py from the reference's own code: every get_actions / value / init_hidden call with a
fingerprint of its inputs and its outputs, the batch shapes the reference's optimisation steps received, and, for the
reference's own Model.train_process / Model.evaluation, the transitions and statistics it produced. Here a
:class:`RecordedLearner` replays that side: each call checks that the runner passes what the reference learner was
given and answers what the reference learner answered."""
import json
import types

import numpy as np
import pytest
import torch

from conftest import ROOT

GOLDEN = ROOT + "/tests/golden"


class FakeBatchedEnv:
    """CPU stand-in with the surface of BatchedVoltageControl the runner touches."""

    def __init__(self, B, n_agents, obs_dim, episode_limit, seed=0):
        self.batch, self.n_agents, self.n_actions, self.obs_size = B, n_agents, 1, obs_dim
        self.device = torch.device("cpu")
        self.g = torch.Generator().manual_seed(seed)
        self.obs = torch.zeros(B, n_agents, obs_dim, dtype=torch.float64)
        self.t = torch.zeros(B, dtype=torch.int64)
        self.episode_limit = episode_limit
        self.actions_seen = []

    def reset(self, mask=None, want_state=True, **kw):
        m = torch.ones(self.batch, dtype=torch.bool) if mask is None else mask.bool()
        new = torch.rand(self.batch, self.n_agents, self.obs_size, generator=self.g, dtype=torch.float64)
        self.obs = torch.where(m[:, None, None], new, self.obs)
        self.t = torch.where(m, torch.ones_like(self.t), self.t)
        return self.obs, None

    def step(self, a):
        assert a.dtype == torch.float64 and tuple(a.shape) == (self.batch, self.n_agents)
        self.actions_seen.append(a.clone())
        self.obs = torch.rand(self.batch, self.n_agents, self.obs_size, generator=self.g, dtype=torch.float64)
        self.t += 1
        reward = -a.abs().mean(dim=1)
        done = (self.t >= self.episode_limit).to(torch.uint8)
        info = torch.arange(11, dtype=torch.float64)[None, :].repeat(self.batch, 1)
        return reward, done, info


class RecordedLearner:
    """The recorded reference learner: same interface as the reference's models (get_actions, value,
    policy_dicts[0].init_hidden, args, unpack_data)."""

    def __init__(self, path, tol=1e-5):
        g = np.load(path)
        self.g, self.tol, self.k = g, tol, 0
        self.calls = json.loads(str(g["calls"]))
        data = g["data"]
        self.a = {k: data[o:o + int(np.prod(shape))].reshape(shape) for k, (o, shape) in json.loads(str(g["index"])).items()}
        self.args = types.SimpleNamespace(**json.loads(str(g["args"])))
        self.policy_dicts = [types.SimpleNamespace(init_hidden=self.init_hidden)]

    def _take(self, kind):
        k = self.k
        assert k < len(self.calls) and self.calls[k]["kind"] == kind, (k, kind)
        self.k += 1
        return k, self.calls[k]

    def _check(self, k, name, t):
        fp = self.a[f"c{k}_{name}"]
        nd = len(fp) - 2
        x = t.detach().double()
        assert list(t.shape) == fp[:nd].astype(int).tolist(), (k, name)
        for got, want in ((float(x.sum()), fp[nd]), (float((x * x).sum()), fp[nd + 1])):
            assert abs(got - want) <= self.tol * (1.0 + abs(want)), (k, name, got, want)

    def _out(self, k, name):
        return torch.tensor(self.a[f"c{k}_{name}"], dtype=torch.float32)

    def init_hidden(self):
        k, _ = self._take("init_hidden")
        return self._out(k, "hid")

    def get_actions(self, state, status, exploration, actions_avail, target, last_hid):
        k, c = self._take("get_actions")
        assert c["status"] == status and c["exploration"] == bool(exploration) and target is False
        self._check(k, "state", state)
        self._check(k, "last_hid", last_hid)
        lp = self._out(k, "log_prob_a") if c["log_prob"] else None
        return self._out(k, "action"), self._out(k, "action_pol"), lp, None, self._out(k, "hid")

    def value(self, obs, act):
        k, _ = self._take("value")
        self._check(k, "obs", obs)
        self._check(k, "act", act)
        return self._out(k, "value")

    def unpack_data(self, batch):
        raise TypeError("the recorded learner only consumes device batches")

    def done(self):
        return self.k == len(self.calls)


def _run_on_device_batches(alg):
    """The runner collects through the (recorded) reference learner on the CPU stand-in env; at every lock-step the update
    hook draws a device batch (same seeded generator as the recording) and hands it through attach(). Every field of every
    batch has the shape, dtype, device, sum and sum of squares of the batch the reference's own value / policy / mixer
    optimisation steps consumed and learned from when the recording was made."""
    from mapdn_b200.marl_runner import BatchedMarlRunner, DeviceTransitionBuffer, TRANSITION_FIELDS, attach
    B, n, od, T = 5, 3, 7, 6
    learner = RecordedLearner(f"{GOLDEN}/ref_learner_device_batches_{alg}.npz")
    args = learner.args
    assert args.max_steps == T
    net = attach(learner)
    env = FakeBatchedEnv(B, n, od, episode_limit=4)
    buf = DeviceTransitionBuffer(32, B, n, od, act_dim=1, hid_dim=args.hid_size, device=env.device)
    gen = torch.Generator(device=env.device).manual_seed(17)          # BATCH_SEED of the recording script
    want_fields = json.loads(str(learner.g["update_fields"]))
    want_fp = learner.a["update_fingerprints"]
    lock_steps, n_batches = [], [0]

    def update(runner, stat):                      # where the reference's own optimisation steps ran on a device batch
        lock_steps.append(runner.steps // B)
        if len(runner.buffer) >= 2 * args.batch_size:
            u = n_batches[0]
            n_batches[0] += 1
            batch = runner.buffer.get_batch(args.batch_size, n_windows=2, generator=gen)
            got = net.unpack_data(batch)
            assert len(got) == len(TRANSITION_FIELDS) == len(want_fields[u])
            for f, t, (shape, dtype, device), (s1, s2) in zip(TRANSITION_FIELDS, got, want_fields[u], want_fp[u]):
                assert [list(t.shape), str(t.dtype), t.device.type] == [shape, dtype, device], (u, f)
                x = t.detach().double()
                assert abs(float(x.sum()) - s1) <= 1e-5 * (1.0 + abs(s1)), (u, f)
                assert abs(float((x * x).sum()) - s2) <= 1e-5 * (1.0 + abs(s2)), (u, f)
    runner = BatchedMarlRunner(env, net, buf, update_fn=update)
    stat = runner.train_process({})
    assert n_batches[0] == len(want_fields) > 0
    assert lock_steps == learner.a["update_lock_steps"].astype(int).tolist()
    return learner, args, env, buf, runner, stat


def test_reference_maddpg_learns_from_device_batches():
    """The batches MADDPG's own optimisation steps learned from (changed weights, finite losses) when the recording was
    made are the ones the runner delivers now (checked field by field in _run_on_device_batches); the learning itself
    ran in the recording, not here. Also the runner's side of Model.train_process / evaluation: action range, transition
    layout, done / last_step, hidden-state restarts, mean_train_* / mean_test_*."""
    learner, args, env, buf, runner, stat = _run_on_device_batches("maddpg")
    B, n, od, T = 5, 3, 7, 6
    assert runner.steps == T * B and buf.count == T
    # translate_action (utilities/util.py:123-132): every action the env saw lies inside [bias - scale, bias + scale]
    a = torch.stack(env.actions_seen)
    assert float(a.abs().max()) <= 0.8 + 1e-12
    # transition layout == what Model.unpack_data would have produced
    b = buf.latest(T)
    st, ac, lp, v, nv, rw, ns, dn, ls, av, lh, h = b.unpacked()
    assert st.shape == (T * B, n, od) and ac.shape == (T * B, n, 1) and v.shape == (T * B, n, 1) and rw.shape == (T * B, n)
    assert dn.shape == (T * B, 1) and ls.shape == (T * B, 1) and av.shape == (T * B, n, 1) and lh.shape == (T * B, n, args.hid_size)
    # done at the env's episode_limit (4 -> after 3 steps), last_step additionally at t = max_steps - 1 (model.py:225)
    dn, ls = dn.view(T, B), ls.view(T, B)
    assert bool((dn[2] == 1).all()) and bool((dn[[0, 1, 3, 4]] == 0).all())
    assert bool((ls[T - 1] == 1).all()) and bool((ls[2] == 1).all()) and float(ls.sum()) == float(dn.sum()) + B * (1 - int(dn[T - 1, 0]))
    # hidden state restarts at zero after a terminated episode
    assert float(lh.view(T, B, n, -1)[3].abs().max()) == 0.0 and float(lh.view(T, B, n, -1)[1].abs().max()) > 0.0
    # mean_train_* (model.py:243-261): info k is the constant k in the stand-in env
    assert abs(stat["mean_train_total_line_loss"] - 8.0) < 1e-12 and "mean_train_reward" in stat
    ev = runner.evaluation({}, num_eval_episodes=B)
    assert abs(ev["mean_test_destroy"] - 10.0) < 1e-12 and np.isfinite(ev["mean_test_reward"])
    assert learner.done()


@pytest.mark.parametrize("alg", ["iddpg", "maddpg", "matd3", "sqddpg", "facmaddpg", "mappo", "ippo", "coma"])
def test_reference_algorithms_run_unchanged_on_device_batches(alg):
    """Eight of the ten algorithms of the reference's registry (models/model_registry.py) collect experience through the
    batched runner, whose device batches their own get_loss / optimiser steps consumed when the recording was made:
    deterministic and Gaussian policies, twin critics (MATD3: value width 2), coalition sampling (SQDDPG: value width
    sample_size), a mixer (FACMADDPG), PPO / COMA advantage code. Not covered, for reasons upstream: IAC (`self.cuda_` is
    never set: models/iac.py:90 raises AttributeError with the reference's own env too) and MAAC (its value() returns a
    concatenation that is not [batch, n, k]-shaped, models/maac.py:47-66)."""
    learner, args, env, buf, runner, stat = _run_on_device_batches(alg)
    B, T = 5, 6
    assert runner.steps == T * B and np.isfinite(stat["mean_train_reward"])
    a = torch.stack(env.actions_seen)
    assert float(a.abs().max()) <= 0.8 + 1e-12                       # translate_action keeps the env's action range
    ev = runner.evaluation({}, num_eval_episodes=B)
    assert np.isfinite(ev["mean_test_reward"]) and learner.done()


class OracleBatchedEnv:
    """CPU stand-in with the surface of BatchedVoltageControl the runner touches, backed by the oracle restatement of the
    env (one VoltageControlOracle per env id) - what the CUDA engine is held to by the parity tests."""

    def __init__(self, net, prof, env_args, batch):
        from oracle.voltage_control_ref import INFO_KEYS, VoltageControlOracle
        self.keys = INFO_KEYS
        self.envs = [VoltageControlOracle(net, prof, env_args, env_id=i) for i in range(batch)]
        self.batch, self.n_agents, self.n_actions = batch, net.n_sgen, 1
        self.device = torch.device("cpu")
        self.obs = None

    def _snap(self):
        self.obs = torch.tensor(np.array([np.array(e.get_obs()) for e in self.envs]))
        self.obs_size = self.obs.shape[-1]

    def reset(self, mask=None, want_state=True, **kw):
        for i, e in enumerate(self.envs):
            if mask is None or bool(mask[i]):
                e.reset()
        self._snap()
        return self.obs, None

    def step(self, a):
        out = [e.step(a[i].numpy()) for i, e in enumerate(self.envs)]
        self._snap()
        return (torch.tensor([o[0] for o in out]), torch.tensor([int(o[1]) for o in out], dtype=torch.uint8),
                torch.tensor([[o[2][k] for k in self.keys] for o in out]))


@pytest.mark.parametrize("alg", ["maddpg", "mappo"])
def test_runner_collects_what_the_reference_train_process_collects(alg):
    """End to end against the reference's OWN loop: `Model.train_process` (models/model.py:197-263) drove the reference's
    own env (oracle/ref_harness.py) with the reference's own learner when the recording was made; the batched runner
    drives the oracle-backed stand-in with the recorded learner. The learner's inputs, every field of every transition
    (state, action, value, next_value, reward, next_state, done, last_step, last_hid, hid) and the mean_train_* /
    mean_test_* statistics agree."""
    from mapdn_b200 import cases
    from mapdn_b200.marl_runner import BatchedMarlRunner, DeviceTransitionBuffer, attach
    net, prof = cases.make_case("case33"), cases.make_profiles("case33", n_days=4)
    env_args = dict(voltage_barrier_type="bowl", action_scale=0.8, action_bias=0.0, seed=21)
    learner = RecordedLearner(f"{GOLDEN}/ref_learner_train_process_{alg}.npz", tol=1e-4)
    g, args = learner.g, learner.args
    T = args.max_steps
    assert T == 5
    env = OracleBatchedEnv(net, prof, env_args, batch=1)
    env.reset()                                                                # episode 1, like the reference's constructor
    buf = DeviceTransitionBuffer(T, 1, net.n_sgen, env.obs_size, act_dim=1, hid_dim=args.hid_size, device=env.device)
    runner = BatchedMarlRunner(env, attach(learner), buf)
    stat = runner.train_process({})
    st, ac, lp, v, nv, rw, ns, dn, ls, av, lh, h = buf.latest(T).unpacked()
    ref = {k[6:]: learner.a[k] for k in learner.a if k.startswith("trans_")}
    tol = 2e-5                                                                 # the learner computes in fp32
    for t in range(T):
        assert np.abs(ref["state"][t] - st[t].numpy()).max() < tol and np.abs(ref["next_state"][t] - ns[t].numpy()).max() < tol
        assert np.abs(ref["action"][t].reshape(-1) - ac[t].numpy().reshape(-1)).max() < tol
        assert np.abs(ref["value"][t].reshape(-1) - v[t].numpy().reshape(-1)).max() < 1e-4
        assert np.abs(ref["next_value"][t].reshape(-1) - nv[t].numpy().reshape(-1)).max() < 1e-4
        assert np.abs(ref["reward"][t] - rw[t].numpy()).max() < tol
        assert float(ref["done"][t]) == float(dn[t]) and float(ref["last_step"][t]) == float(ls[t])
        assert np.abs(ref["last_hid"][t].reshape(-1) - lh[t].numpy().reshape(-1)).max() < tol
        assert np.abs(ref["hid"][t].reshape(-1) - h[t].numpy().reshape(-1)).max() < tol
    stat_ref = json.loads(str(g["stat"]))
    assert stat_ref
    for k, v_ref in stat_ref.items():
        assert abs(stat[k] - v_ref) < 1e-5, k
    # Model.evaluation (models/model.py:265-302): greedy episodes, per-episode means averaged over the episodes
    ev_ref = json.loads(str(g["evaluation"]))
    ev = runner.evaluation({}, num_eval_episodes=args.num_eval_episodes)
    assert len(ev_ref) == 12 and args.num_eval_episodes == 2
    for k, v_ref in ev_ref.items():
        assert abs(ev[k] - v_ref) < 1e-5, k
    assert learner.done()
