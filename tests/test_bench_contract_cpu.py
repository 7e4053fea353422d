"""bench.py contract checks that need no GPU: the configurations are BASELINE.json's, the reference arm prints the
required JSON line, the core count comes from affinity / cgroup quota."""
import json
import os
import re
import subprocess
import sys

from conftest import ROOT


def _bench():
    sys.path.insert(0, ROOT)
    import bench
    return bench


def test_configs_are_the_baseline_json_configs():
    bench = _bench()
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    texts = base["configs"][1:]                       # configs[0] is the reference's 1-env CPU correctness run
    assert len(texts) == len(bench.CONFIGS) == 4
    for cid, txt in zip(sorted(bench.CONFIGS), texts):
        c = bench.CONFIGS[cid]
        assert c["scenario"] in txt and str(c["batch"]) in txt
        assert re.search(c["barrier"], txt, re.I)
        assert f"{c['n_gpus']}×B200" in txt or f"{c['n_gpus']}xB200" in txt
    assert bench.CONFIGS[bench.HEADLINE]["scenario"] == "case33" and bench.CONFIGS[bench.HEADLINE]["batch"] == 4096


def test_usable_cores_respects_affinity():
    bench = _bench()
    n, src = bench.usable_cores()
    assert 1 <= n <= len(os.sched_getaffinity(0)) and src in ("sched_getaffinity", "cgroup cpu quota")


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3",
                          "--cpu-sample", "4", "--cpu-cores", "2"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "env-steps/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("port", "pandapower") and cb["cores"] == 2 and cb["one_core"]["value"] > 0
    assert "case33 x 4096 envs per GPU" in line["config"]["workload"]
    # rank != 0 of a torchrun launch exits quietly
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_fixture_leg_of_the_parity_record():
    """bench.py's `parity.reference_fixture` leg replays a reference-executed fixture through the engine; here through an
    oracle-backed CPU stand-in of the engine's surface, to check the replay logic itself."""
    import numpy as np
    import torch
    from oracle.voltage_control_ref import INFO_KEYS, VoltageControlOracle
    bench = _bench()

    class Standin:
        def __init__(self, net, prof, args, B):
            self.o = [VoltageControlOracle(net, prof, args, env_id=i) for i in range(B)]
            self.device, self.obs = torch.device("cpu"), None

        def _snap(self):
            self.obs = torch.tensor(np.array([np.array(o.get_obs()) for o in self.o]))

        def reset(self, start=None, add_noise=True):
            for i, o in enumerate(self.o):
                o.reset(start=None if start is None else tuple(start[i].tolist()), add_noise=add_noise)
            self._snap()

        def step(self, a, add_noise=True):
            out = [o.step(a[i].numpy(), add_noise=add_noise) for i, o in enumerate(self.o)]
            self._snap()
            return (torch.tensor([x[0] for x in out]), torch.tensor([int(x[1]) for x in out], dtype=torch.uint8),
                    torch.tensor([[x[2][k] for k in INFO_KEYS] for x in out]))

        def get_state(self):
            return torch.tensor(np.array([o.get_state() for o in self.o]))

        def close(self):
            pass
    for name in ("case33_bowl", "case33_divergence"):
        rec = bench.reference_fixture_check(0, name=name, make_env=Standin)
        assert rec["n_steps"] >= 6 and rec["max_abs_dreward"] < 1e-11 and rec["max_abs_dinfo"] < 1e-11
        assert rec["max_abs_dobs"] < 1e-11 and rec["max_abs_dstate"] < 1e-9


def test_dump_outputs_writes_what_the_step_returned(tmp_path):
    """--dump-outputs: the last step's reward / terminated / info / obs as float64 .npy; past 64 MiB a fixed, seeded sample
    of env rows (the same rows in every array) with their global env ids."""
    import numpy as np
    import torch
    bench = _bench()

    class Standin:
        def __init__(self, B, obs_dim, offset=0):
            g = torch.Generator().manual_seed(B)
            self.count, self.offset = B, offset
            self.reward = torch.rand(B, dtype=torch.float64, generator=g)
            self.terminated = (torch.rand(B, generator=g) < 0.5).to(torch.uint8)
            self.info = torch.rand(B, 11, dtype=torch.float64, generator=g)
            self.obs = torch.rand(B, 6, obs_dim, dtype=torch.float64, generator=g)

    env = Standin(64, 5)
    bench.dump_outputs(env, str(tmp_path / "small"))
    names = sorted(p.name for p in (tmp_path / "small").iterdir())
    assert names == ["info.npy", "obs.npy", "reward.npy", "terminated.npy"]
    for k in ("reward", "terminated", "info", "obs"):
        a = np.load(tmp_path / "small" / f"{k}.npy")
        assert a.dtype == np.float64 and np.array_equal(a, getattr(env, k).numpy().astype(np.float64))

    big = Standin(4096, 400, offset=4096)                          # 4096 x (1 + 1 + 11 + 2400) fp64 = 75 MiB
    for d in ("a", "b"):
        bench.dump_outputs(big, str(tmp_path / d))
    total = sum(p.stat().st_size for p in (tmp_path / "a").iterdir())
    assert total <= 64 << 20
    ids = np.load(tmp_path / "a" / "env_ids.npy").astype(np.int64) - big.offset
    assert np.array_equal(ids, np.load(tmp_path / "b" / "env_ids.npy").astype(np.int64) - big.offset)
    assert np.all(np.diff(ids) > 0) and len(ids) > 3000
    assert np.array_equal(np.load(tmp_path / "a" / "obs.npy"), big.obs.numpy()[ids])
    assert np.array_equal(np.load(tmp_path / "a" / "reward.npy"), big.reward.numpy()[ids])
