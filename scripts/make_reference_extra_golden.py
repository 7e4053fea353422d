#!/usr/bin/env python
"""Writes the golden files that record what the REFERENCE's own code did for the tests that compare against it beyond the
env trajectories of scripts/make_reference_golden.py:

* ref_csv_case33.npz          - what the reference env's CSV readers (voltage_control_env.py:407-438) produce: a
  seeded sample of the table rows, the column sums and the derived statistics;
* ref_env_case33_cow.npz      - the first step of case33_bowl with pandas' copy-on-write row semantics (oracle/ref_harness.py);
* ref_decentralised_mode.json - how the reference's constructor fails for mode="decentralised";
* ref_learner_<test>_<alg>.npz - the reference learners' side of the batched runner's calls (get_actions / value /
  init_hidden: inputs and outputs), the transitions and statistics of the reference's own Model.train_process /
  Model.evaluation, and, for every batch the reference's optimisation code received, each field's shape, dtype,
  device and sum / sum of squares.

Needs a checkout of the reference (MAPDN_REFERENCE_ROOT) with its Python dependencies (torch, pyyaml):

    MAPDN_REFERENCE_ROOT=<reference checkout> python scripts/make_reference_extra_golden.py
"""
import importlib.util
import json
import os
import sys
import tempfile
import types
from collections import namedtuple

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from mapdn_b200 import cases                                           # noqa: E402
from mapdn_b200.marl_runner import BatchedMarlRunner, DeviceTransitionBuffer, attach   # noqa: E402
from oracle import ref_harness as H                                   # noqa: E402
from oracle import ref_scenarios as S                                 # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
REF = H.REFERENCE_ROOT


def _module(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def csv_golden():
    net, prof = cases.make_case("case33"), cases.make_profiles("case33", n_days=3)
    with tempfile.TemporaryDirectory() as d:
        H.write_reference_data(d, net, prof)
        env = H.ReferenceRun(d, net, dict(pv_scale=1.3, demand_scale=0.7, seed=0), env_id=0).env
        tables = dict(pv=env.pv_data.values, load_p=env.active_demand_data.values, load_q=env.reactive_demand_data.values)
        rows = np.sort(np.random.default_rng(0).choice(len(tables["pv"]), 24, replace=False))
        np.savez_compressed(os.path.join(GOLDEN, "ref_csv_case33.npz"), rows=rows, n_rows=len(tables["pv"]),
                            **{k: v[rows] for k, v in tables.items()},
                            **{f"{k}_colsum": v.sum(axis=0) for k, v in tables.items()}, pv_std=np.asarray(env.pv_std), s_max=np.asarray(env.s_max),
                            load_p_std=np.asarray(env.active_demand_std), steps_per_hour=60 // env.time_delta,
                            n_days=(env.pv_data.index[-1] - env.pv_data.index[0]).days)


def cow_golden():
    mod = _module(os.path.join(ROOT, "scripts", "make_reference_golden.py"), "make_reference_golden")
    sc = dict(S.SCENARIOS["case33_bowl"], ops=[("init",), ("step", True)], env_ids=[0])
    pinned, cow = mod.record(sc, view_rows=True), mod.record(sc, view_rows=False)
    np.savez_compressed(os.path.join(GOLDEN, "ref_env_case33_cow.npz"),
                        **{f"pinned_{k}": v for k, v in pinned.items()}, **{f"cow_{k}": v for k, v in cow.items()})


def decentralised_golden():
    net, prof = cases.make_case("case33"), cases.make_profiles("case33", n_days=3)
    with tempfile.TemporaryDirectory() as d:
        H.write_reference_data(d, net, prof)
        try:
            H.ReferenceRun(d, net, dict(mode="decentralised", seed=0), env_id=0)
            rec = dict(raises=None)
        except Exception as e:  # noqa: BLE001
            rec = dict(raises=type(e).__name__, message=str(e))
    with open(os.path.join(GOLDEN, "ref_decentralised_mode.json"), "w") as f:
        json.dump(dict(mode="decentralised", constructor=rec), f, indent=1)
        f.write("\n")


# ---------------------------------------------------------------------------------------------------- learners
class Recorder:
    """Logs the calls the batched runner (or the reference's own loop) makes on a reference model."""

    def __init__(self, net):
        self.calls, self.arrays, self.on = [], {}, True
        ga, va, ih = net.get_actions, net.value, net.policy_dicts[0].init_hidden

        def put(k, name, t):
            if t is not None:
                self.arrays[f"c{k}_{name}"] = t.detach().cpu().numpy()

        def fingerprint(k, name, t):            # inputs: shape, sum and sum of squares (fp64) keep the files small
            x = t.detach().cpu().double()
            self.arrays[f"c{k}_{name}"] = np.r_[np.array(t.shape, np.float64), float(x.sum()), float((x * x).sum())]

        def get_actions(state, status, exploration, actions_avail, target, last_hid, **kw):
            out = ga(state, status=status, exploration=exploration, actions_avail=actions_avail, target=target,
                     last_hid=last_hid, **kw)
            if self.on:
                k = len(self.calls)
                self.calls.append(dict(kind="get_actions", status=status, exploration=bool(exploration),
                                       log_prob=out[2] is not None))
                fingerprint(k, "state", state); fingerprint(k, "last_hid", last_hid)
                for name, t in zip(("action", "action_pol", "log_prob_a", "hid"), (out[0], out[1], out[2], out[4])):
                    put(k, name, t)
            return out

        def value(obs, act):
            out = va(obs, act)
            if self.on:
                k = len(self.calls)
                self.calls.append(dict(kind="value"))
                fingerprint(k, "obs", obs); fingerprint(k, "act", act); put(k, "value", out)
            return out

        def init_hidden():
            out = ih()
            if self.on:
                k = len(self.calls)
                self.calls.append(dict(kind="init_hidden"))
                put(k, "hid", out)
            return out
        net.get_actions, net.value, net.policy_dicts[0].init_hidden = get_actions, value, init_hidden

    def save(self, path, args, **extra):
        """One flat fp64 vector + a JSON index {name: [offset, shape]} (hundreds of tiny npz members would dominate the
        file)."""
        keep = ("max_steps", "action_scale", "action_bias", "hid_size", "num_eval_episodes", "batch_size")
        arrays = dict(self.arrays, **{k: v for k, v in extra.items() if v.dtype.kind != "U"})
        index, flat, off = {}, [], 0
        for k, v in arrays.items():
            index[k] = [off, list(v.shape)]
            flat.append(np.asarray(v, np.float64).ravel())
            off += v.size
        np.savez_compressed(path, calls=np.array(json.dumps(self.calls)), index=np.array(json.dumps(index)),
                            data=np.concatenate(flat), args=np.array(json.dumps({k: getattr(args, k) for k in keep})),
                            **{k: v for k, v in extra.items() if v.dtype.kind == "U"})


def _on_path():
    for k in ("agents", "critics", "models", "utilities"):
        for name in [m for m in sys.modules if m == k or m.startswith(k + ".")]:
            del sys.modules[name]
        pkg = types.ModuleType(k)
        pkg.__path__ = [os.path.join(REF, k)]
        sys.modules[k] = pkg
    sys.path.append(REF)


def _trainer(alg, n_agents, obs_dim, max_steps, **over):
    import yaml
    from models.model_registry import Model as REGISTRY
    from utilities.trainer import PGTrainer
    d = yaml.safe_load(open(os.path.join(REF, "args", "default.yaml")))
    d.update(yaml.safe_load(open(os.path.join(REF, "args", "alg_args", alg + ".yaml")))["alg_args"])
    d.update(agent_num=n_agents, obs_size=obs_dim, action_dim=1, cuda=False, max_steps=max_steps, action_scale=0.8,
             action_bias=0.0, batch_size=8, **over)
    args = namedtuple("Args", d.keys())(**d)
    return args, PGTrainer(args, REGISTRY[alg], env=None, logger=None)


BATCH_SEED = 17           # the generator of the update batches' draws (tests/test_marl_runner_cpu.py uses the same)


def batch_fingerprint(t):
    x = t.detach().cpu().double()
    return [float(x.sum()), float((x * x).sum())]


def learner_on_device_batches(alg, T_mod):
    """The runner collects through the reference learner on the CPU stand-in env and the reference's optimisation steps
    run on the device batches (what tests/test_marl_runner_cpu.py replays)."""
    torch.manual_seed(0)
    B, n, od, T = 5, 3, 7, 6
    args, trainer = _trainer(alg, n, od, max_steps=T, hid_size=8)         # a narrow learner keeps the recording small
    net = attach(trainer.behaviour_net)
    rec = Recorder(net)
    env = T_mod.FakeBatchedEnv(B, n, od, episode_limit=4)
    buf = DeviceTransitionBuffer(32, B, n, od, act_dim=1, hid_dim=args.hid_size, device=env.device)
    gen = torch.Generator(device=env.device).manual_seed(BATCH_SEED)
    fields, fingerprints, updates, lock_step = [], [], [], []

    def update(runner, stat):
        lock_step.append(runner.steps // B)
        if len(runner.buffer) >= 2 * args.batch_size:
            rec.on = False
            batch = runner.buffer.get_batch(args.batch_size, n_windows=2, generator=gen)
            # what the reference's get_loss receives, before its reward normalisation (Model.unpack_data)
            fields.append([[list(t.shape), str(t.dtype), t.device.type] for t in batch.unpacked()])
            fingerprints.append([batch_fingerprint(t) for t in batch.unpacked()])
            w0 = [p.detach().clone() for p in trainer.behaviour_net.policy_dicts.parameters()]
            trainer.value_transition_process(stat, batch)
            trainer.policy_transition_process(stat, batch)
            if args.mixer:
                trainer.mixer_transition_process(stat, batch)
            updates.append(any(not torch.equal(a, b) for a, b in zip(w0, trainer.behaviour_net.policy_dicts.parameters())))
            rec.on = True
    runner = BatchedMarlRunner(env, net, buf, update_fn=update)
    stat = runner.train_process({})
    assert updates and all(updates) and np.isfinite(stat["mean_train_value_loss"])
    runner.evaluation({}, num_eval_episodes=B)
    rec.save(os.path.join(GOLDEN, f"ref_learner_device_batches_{alg}.npz"), args,
             update_fields=np.array(json.dumps(fields)), update_fingerprints=np.array(fingerprints),
             update_lock_steps=np.array(lock_step))


def learner_train_process(alg, T_mod):
    """The reference's own Model.train_process / Model.evaluation on the reference env (oracle/ref_harness.py)."""
    net, prof = cases.make_case("case33"), cases.make_profiles("case33", n_days=4)
    env_args = dict(voltage_barrier_type="bowl", action_scale=0.8, action_bias=0.0, seed=21)
    with tempfile.TemporaryDirectory() as d:
        H.write_reference_data(d, net, prof)
        ref = H.ReferenceRun(d, net, env_args, env_id=0)
        T = 5
        torch.manual_seed(0)                    # the learner's initial weights
        args, trainer = _trainer(alg, net.n_sgen, ref.env.get_obs_size(), max_steps=T)
        args = args._replace(replay_warmup=10 ** 9, num_eval_episodes=2)
        trainer.args = trainer.behaviour_net.args = args
        rec = Recorder(trainer.behaviour_net)

        class Hooked:
            def __init__(self, run):
                self._r = run

            def reset(self):
                self._r.draws.begin_reset()
                return self._r.env.reset()

            def step(self, a):
                self._r.draws.begin_step()
                return self._r.env.step(a)

            def __getattr__(self, k):
                return getattr(self._r.env, k)

        trainer.env = Hooked(ref)
        torch.manual_seed(5)
        stat_ref, ev_ref = {}, {}
        with ref._ctx():
            trainer.behaviour_net.train_process(stat_ref, trainer)
        trans = trainer.replay_buffer.buffer
        assert len(trans) == T
        with ref._ctx():
            trainer.behaviour_net.evaluation(ev_ref, trainer)
    tr = {f"trans_{f}": np.array([np.asarray(getattr(t, f), np.float32) for t in trans])
          for f in ("state", "action", "value", "next_value", "reward", "next_state", "done", "last_step", "last_hid", "hid")}
    rec.save(os.path.join(GOLDEN, f"ref_learner_train_process_{alg}.npz"), args,
             stat=np.array(json.dumps({k: float(v) for k, v in stat_ref.items() if k.startswith("mean_train_")})),
             evaluation=np.array(json.dumps({k: float(v) for k, v in ev_ref.items()})), **tr)


def main():
    if not H.reference_available():
        raise SystemExit(f"no reference checkout at {REF} (set MAPDN_REFERENCE_ROOT)")
    csv_golden()
    cow_golden()
    decentralised_golden()
    T_mod = _module(os.path.join(ROOT, "tests", "test_marl_runner_cpu.py"), "test_marl_runner_cpu")
    _on_path()
    for alg in ("iddpg", "maddpg", "matd3", "sqddpg", "facmaddpg", "mappo", "ippo", "coma"):
        learner_on_device_batches(alg, T_mod)
    for alg in ("maddpg", "mappo"):
        learner_train_process(alg, T_mod)
    for f in sorted(os.listdir(GOLDEN)):
        if f.startswith(("ref_csv", "ref_env_case33_cow", "ref_decentralised", "ref_learner")):
            print(f"{f}: {os.path.getsize(os.path.join(GOLDEN, f)) / 1024:.1f} kB")


if __name__ == "__main__":
    main()
