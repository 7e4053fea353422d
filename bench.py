#!/usr/bin/env python
"""Benchmark of the MAPDN var_voltage_control env step (BASELINE.json metric: env-steps/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1]): case33 (33-bus feeder), 4096 env instances per GPU, Bowl
voltage barrier, noise on, synthetic load/PV profiles and random actions (the reference's data
files are not in the repo). One "step" = one fused launch advancing every env by one transition:
action clip -> fp64 Newton-Raphson power flow -> reward/info -> next profile row + noise -> obs.

Prints ONE JSON line (rank 0). `value` = env-steps/s with actions already resident in HBM, timed
with CUDA events around each step (L2 flushed between steps, outside the event pairs), max over
ranks. `e2e` = the same through the host-buffer API (H2D of actions, D2H of reward / done / info /
obs inside the timed region). The same line carries

* `configs`: the other BASELINE.json configurations that belong to this GPU count, each with its own
  `ms_per_step`, `value`, `roofline`, `e2e`, Newton-iteration and divergence statistics: case141 x 2048 (L1) at
  N = 1, case322 x 1024 (L2) sharded over 2 GPUs at N = 2, case322 x 8192 (Bowl) sharded over 8 GPUs at N = 8; at
  N = 1 also one GPU's shard of the two sharded configs (512 / 1024 envs of case322), labelled `shard_of`;
* `newton_iters_mean`, `nonconverged_frac` of the benchmarked batch, and `parity`: max |dV| / |dreward| / |dobs|
  between the CUDA path and the oracle on >= 64 envs of a batch of the benchmarked shape, computed in this run, plus
  `parity.reference_fixture`: the same device replaying a trajectory that the reference's own env code produced
  (tests/golden/ref_env_case33_bowl.npz);
* `cpu_baseline`: the CPU arm timed on this box's usable cores (affinity + cgroup quota), with a 1-core rate.

`--impl reference` times the reference's CPU implementation of the path on the host cores: real pandapower
(`import pandapower`, also looked up under baseline/_ref) when it is importable, else the oracle port
(oracle/: pandapower-2.7.0-equivalent NR + env logic, NumPy/SciPy).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env-steps/sec (batched power-flow solves)"
# BASELINE.json configs[1..4]: (scenario, global batch, barrier, GPUs the batch is sharded over)
CONFIGS = {
    1: dict(scenario="case33", batch=4096, barrier="bowl", n_gpus=1),
    2: dict(scenario="case141", batch=2048, barrier="l1", n_gpus=1),
    3: dict(scenario="case322", batch=1024, barrier="l2", n_gpus=2),
    4: dict(scenario="case322", batch=8192, barrier="bowl", n_gpus=8),
}
HEADLINE = 1


def workload_string(sc, per_gpu, barrier):
    return (f"{sc} x {per_gpu} envs per GPU, {barrier} barrier, noise on, fused step "
            "(runpp-equivalent NR + reward + next row + obs)")


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference path on the host cores (pandapower when importable, else the oracle port)
# ------------------------------------------------------------------------------------------------
def usable_cores():
    """Cores this process may really use: scheduler affinity, capped by the cgroup CPU quota (a GPU lease is usually a
    slice of the box - os.cpu_count() reports the whole machine)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    src = "sched_getaffinity"
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                quota, period = txt[0], float(txt[1])
            else:
                quota, period = txt[0], float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota not in ("max", "-1"):
                q = int(math.ceil(float(quota) / period))
                if 0 < q < n:
                    n, src = q, "cgroup cpu quota"
            break
        except Exception:
            continue
    return max(1, n), src


def pandapower_available():
    ref = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(ref) and ref not in sys.path:
        sys.path.append(ref)
    try:
        import pandapower  # noqa: F401
        return True
    except Exception:
        return False


_W = {}


def _cpu_init(scenario, barrier, seed, use_pp):
    import multiprocessing as mp
    from mapdn_b200 import cases
    from oracle.voltage_control_ref import VoltageControlOracle
    wid = mp.current_process()._identity[0] if mp.current_process()._identity else 0
    net, prof = cases.make_case(scenario), cases.make_profiles(scenario)
    env = VoltageControlOracle(net, prof, dict(voltage_barrier_type=barrier, seed=seed,
                                               action_scale=cases.SCENARIOS[scenario]["action_scale"]), env_id=wid)
    if use_pp:                                  # the real pandapower.runpp behind the same env logic
        from oracle.pp_bridge import PandapowerBackend
        env.pf = PandapowerBackend(net)
    env.reset()
    _W["env"], _W["rng"] = env, np.random.default_rng(wid)


def _cpu_work(n_steps):
    env, rng = _W["env"], _W["rng"]
    t0 = time.perf_counter()
    for _ in range(n_steps):
        a = rng.uniform(env.low, env.high, env.n_agents)
        _, term, _ = env.step(a)            # reference hot path: step() ...
        env.get_obs()                       # ... followed by get_obs() (models/model.py:216-219)
        if term:
            env.reset()
    return time.perf_counter() - t0


class CpuArm:
    def __init__(self, scenario, barrier, seed=0, cores=None):
        import multiprocessing as mp
        self.cores, self.cores_source = usable_cores()
        if cores:
            self.cores, self.cores_source = int(cores), "--cpu-cores"
        self.use_pp = pandapower_available()
        self.kind = "pandapower" if self.use_pp else "port"
        os.environ.setdefault("OMP_NUM_THREADS", "1")
        os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
        os.environ.setdefault("MKL_NUM_THREADS", "1")
        self.pool = mp.get_context("spawn").Pool(self.cores, initializer=_cpu_init,
                                                 initargs=(scenario, barrier, seed, self.use_pp))
        self.pool.map(_cpu_work, [1] * self.cores)      # spin-up

    def describe(self):
        if self.use_pp:
            return "pandapower.runpp (imported) behind the reference env logic, one process per core"
        return ("oracle/ NumPy+SciPy restatement of pandapower 2.7.0 runpp + reference env logic (pandapower is not "
                "importable in this image), one process per core")

    def run(self, env_steps):
        per = max(1, env_steps // self.cores)
        t0 = time.perf_counter()
        self.pool.map(_cpu_work, [per] * self.cores)
        dt = time.perf_counter() - t0
        return per * self.cores, dt

    def run_one_core(self, env_steps):
        """The same work on ONE process while the others idle."""
        return env_steps, self.pool.apply(_cpu_work, (env_steps,))

    def close(self):
        self.pool.close()
        self.pool.join()


def run_reference(args):
    from mapdn_b200 import cases
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg = CONFIGS[HEADLINE]
    sc, barrier, B = args.scenario or cfg["scenario"], args.barrier or cfg["barrier"], args.batch or cfg["batch"]
    arm = CpuArm(sc, barrier, cores=args.cpu_cores)
    # env-steps per "step" of this arm: a bounded sample of the batch, sized from the rate seen in the first
    # warm-up pass so that warm-up + K timed steps take about two minutes whatever K is (at least one env-step per core)
    sample = args.cpu_sample or 2 * arm.cores
    n0, dt0 = arm.run(sample)
    if not args.cpu_sample:
        budget_steps = (n0 / dt0) * 100.0 / max(1, args.steps + args.warmup)
        sample = int(min(B, max(arm.cores, budget_steps // arm.cores * arm.cores)))
    for _ in range(max(0, args.warmup - 1)):
        arm.run(sample)
    done, t = 0, 0.0
    for _ in range(args.steps):
        n, dt = arm.run(sample)
        done += n
        t += dt
    n1, dt1 = arm.run_one_core(max(8, min(400, int(3.0 * n0 / dt0 / arm.cores))))
    arm.close()
    val = done / t
    net = cases.make_case(sc)
    line = dict(impl="reference", metric=METRIC, value=val, unit="env-steps/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=t / args.steps * 1e3, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f64", data="synthetic",
                config=dict(workload=workload_string(sc, B, barrier), n_bus=net.n_bus, n_agents=net.n_sgen,
                            sampled_env_steps_per_step=sample),
                cpu_baseline=dict(value=val, unit="env-steps/s", cores=arm.cores, cores_source=arm.cores_source,
                                  kind=arm.kind, one_core=dict(value=n1 / dt1, unit="env-steps/s", env_steps=n1),
                                  sample=f"{done} env-steps of {sc} ({sample} per step x {args.steps} steps): "
                                         + arm.describe()),
                e2e=dict(value=val, unit="env-steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons DURING the timed region: NVML polled every ~2 ms from a thread (the timed region of
    the default run is only tens of ms long); `nvidia-smi -lms 50` is the fallback when NVML is not usable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    REASON_BITS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20),
                   ("hw_thermal_slowdown", 0x40))            # nvmlClocksEventReason* bit masks

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nvml, self.samples = index, [], None, None, []
        self._stop = threading.Event()

    def _nvml_open(self):
        import pynvml
        import torch
        pynvml.nvmlInit()
        h = None
        try:
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)); int(reasons(h))      # probe once
        return pynvml, h, reasons, mx

    def _poll(self):
        pynvml, h, reasons, _ = self.nvml
        while not self._stop.is_set():
            try:
                self.samples.append((time.perf_counter(), float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)),
                                     int(reasons(h))))
            except Exception:
                break
            time.sleep(0.0005)

    def start(self):
        self.t_start = time.perf_counter()
        try:
            self.nvml = self._nvml_open()
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE, text=True,
                                         stderr=subprocess.DEVNULL)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append((time.perf_counter(), ln.strip()))

    def stop(self, t0, t1, t_load0=None):
        """Samples inside the timed region [t0, t1]; when the region is too short for three samples (20 steps last ~2.5 ms)
        the window is widened to the loaded period that contains it (warm-up steps + timed steps, from t_load0)."""
        if self.nvml is not None:
            self._stop.set()
            self.th.join(timeout=1.0)
            timed = [r for r in self.samples if t0 <= r[0] <= t1]
            rows, window = timed, "timed region"
            if len(rows) < 3 and t_load0 is not None:
                rows, window = [r for r in self.samples if t_load0 <= r[0] <= t1], "warm-up + timed region (GPU under the same load)"
            rows = rows or self.samples[-3:]
            if rows:
                bits = 0
                for r in rows:
                    bits |= r[2]
                return dict(sm_mhz=float(np.median([r[1] for r in rows])), sm_max_mhz=self.nvml[3],
                            reasons=sorted(nm for nm, b in self.REASON_BITS if bits & b), samples=len(rows),
                            samples_in_timed_region=len(timed), window=window, source="nvml")
            return None
        if self.proc is None:
            return None
        time.sleep(0.12)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.06] or [r for _, r in self.rows[-3:]]
        sm, mx, reasons = [], [], set()
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except Exception:
                continue
            for nm, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return None
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm),
                    source="nvidia-smi")


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class Timer:
    """max-over-ranks helpers"""

    def __init__(self, world, dev):
        self.world, self.dev = world, dev

    def sync_all(self):
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(self, x):
        import torch
        import torch.distributed as dist
        t = torch.tensor([x], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(env, out_dir):
    """Writes what the last timed ``env.step`` handed its caller (reward, terminated, info, and the observations the step
    left in ``env.obs``) as ``out_dir/<name>.npy``, float64 (terminated as 0/1). When the arrays exceed 64 MiB in all, a
    fixed sample of env rows (seed 0, sorted) is written instead, with their ids in ``env_ids.npy``."""
    out = dict(reward=env.reward, terminated=env.terminated, info=env.info, obs=env.obs)
    out = {k: v.cpu().numpy().astype(np.float64) for k, v in out.items()}
    B = env.count
    if sum(a.nbytes for a in out.values()) > DUMP_LIMIT_BYTES:
        row = sum(a.nbytes for a in out.values()) // B + 8          # + its env id
        keep = max(1, (DUMP_LIMIT_BYTES - (64 << 10)) // row)       # 64 KiB for the .npy headers
        ids = np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
        out = {k: a[ids] for k, a in out.items()}
        out["env_ids"] = (ids + env.offset).astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


def measure(sc, barrier, global_batch, K, W, Ke, tm, local, rank, flush, lanes=0, clocks=None, obs_dtypes=("f64",),
            min_warm=0, dump_dir=None):
    """Device-timed and end-to-end throughput of one configuration, sharded over the ranks of this job."""
    import torch
    from mapdn_b200 import cases
    from mapdn_b200.distributed import ShardedVoltageControl

    dev = torch.device("cuda", local)
    net, prof = cases.make_case(sc), cases.make_profiles(sc)
    env_args = dict(voltage_barrier_type=barrier, action_scale=cases.SCENARIOS[sc]["action_scale"], seed=0)
    env = ShardedVoltageControl(net, prof, env_args, global_batch=global_batch, device=local, lanes_per_env=lanes)
    B = env.count
    n_sets = 8
    g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
    lo, hi = env.action_space.low, env.action_space.high
    acts = lo + (hi - lo) * torch.rand(n_sets, B, env.n_agents, dtype=torch.float64, device=dev, generator=g)
    ep_len = env.episode_limit - 1
    state = dict(t=0)

    def one_step(i):
        if state["t"] == ep_len:            # every env terminated at episode_limit: start a new episode
            env.reset()
            state["t"] = 0
        env.step(acts[i % n_sets])
        state["t"] += 1

    env.reset()
    if clocks is not None:
        clocks.start()
        time.sleep(0.05)
    tm.sync_all()
    t_load0 = time.perf_counter()
    W = max(W, min_warm)              # every rank alike; the clock record needs some loaded time before the timed steps
    for i in range(W):
        one_step(i)
        if flush is not None:
            flush.zero_()
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    tm.sync_all()
    launches0 = env.launch_count
    w0 = time.perf_counter()
    for i in range(K):
        ev0[i].record()
        one_step(W + i)
        ev1[i].record()
        if flush is not None:
            flush.zero_()
    returns = env.gather_episode_returns()           # the path's only collective (SURVEY §8e)
    tm.sync_all()
    w1 = time.perf_counter()
    launches = env.launch_count - launches0
    clk = clocks.stop(w0, w1, t_load0) if clocks is not None else None
    dev_ms = tm.max_over_ranks(sum(a.elapsed_time(b) for a, b in zip(ev0, ev1)))
    if dump_dir is not None:
        dump_outputs(env, dump_dir)
    assert returns.shape[0] == global_batch and bool(torch.isfinite(returns).all())
    # side metrics of the last timed step (SURVEY §8d): Newton iterations per solve, diverged fraction
    iters = env.get_field("nr_iters")[:, 0]
    side = torch.stack([iters.mean(), (env.info[:, 10] > 0).double().mean()])
    if tm.world > 1:
        import torch.distributed as dist
        dist.all_reduce(side, op=dist.ReduceOp.SUM)
        side /= tm.world
    ms = dev_ms / K
    out = dict(scenario=sc, barrier=barrier, global_batch=global_batch, envs_per_gpu=B, n_gpus=tm.world,
               ms_per_step=ms, value=global_batch * K / (dev_ms * 1e-3), unit="env-steps/s", steps=K,
               lanes_per_env=env.dims["lanes_per_env"], envs_per_block=env.dims["envs_per_block"],
               smem_bytes_per_block=env.dims["smem_bytes"], n_bus=net.n_bus, n_agents=net.n_sgen, obs_dim=env.obs_size,
               newton_iters_mean=float(side[0].item()), nonconverged_frac=float(side[1].item()),
               gpu_launches=int(launches), wall_ms_per_step=(w1 - w0) / K * 1e3, warmup_steps_done=W)
    alg = env.dims["algorithmic_bytes_per_env_step"] * B            # per launch (this GPU's shard)
    out["_alg_bytes_per_launch"] = alg
    out["_clocks"] = clk

    # ---- end to end through the host-buffer API (numpy in / numpy out) ----
    rng = np.random.default_rng(rank)
    host_acts = [rng.uniform(lo, hi, (B, env.n_agents)) for _ in range(4)]
    for tag in obs_dtypes:
        odt = np.float32 if tag in ("f32", "compact_f32") else np.float64
        staged = {"staged": True, "compact_zc_f64": False}.get(tag)      # None: the layout's default path
        layout = "compact" if tag.startswith("compact") else "padded"
        env.reset(); state["t"] = 0
        for i in range(3):
            env.step_host(host_acts[i % 4], obs_dtype=odt, staged=staged, layout=layout)
        tm.sync_all()
        e0 = time.perf_counter()
        for i in range(Ke):
            if state["t"] == ep_len:
                env.reset(); state["t"] = 0
            env.step_host(host_acts[i % 4], obs_dtype=odt, staged=staged, layout=layout)
            state["t"] += 1
        tm.sync_all()
        dt = tm.max_over_ranks(time.perf_counter() - e0)
        if layout == "compact":
            obs_bytes = env.obs_row_len * (4 if odt is np.float32 else 8)
        elif staged:
            obs_bytes = env.n_agents * env.obs_size * 8
        else:
            obs_bytes = env.host_obs_bytes_per_env // (2 if tag == "f32" else 1)
        out[{"f64": "e2e", "f32": "e2e_obs_f32", "staged": "e2e_staged", "compact_f64": "e2e_compact",
             "compact_f32": "e2e_compact_f32", "compact_zc_f64": "e2e_compact_zero_copy"}[tag]] = dict(
            value=global_batch * Ke / dt, unit="env-steps/s", h2d_bytes_per_step=B * env.n_agents * 8,
            d2h_bytes_per_step=B * (8 + 1 + 11 * 8 + obs_bytes), steps=Ke, obs_dtype="f32" if odt is np.float32 else "f64",
            path="compact rows [B, sum of the agents' true lengths] (no zero padding): kernel -> device rows -> ONE "
                 "copy-engine D2H; actions / reward / terminated / info zero-copy" if layout == "compact" and staged is None else
                 "compact rows [B, sum of the agents' true lengths] (no zero padding), zero-copy like the padded path"
                 if layout == "compact" else
                 "staged copies: H2D actions, kernel, 4 x D2H (full padded obs rows)" if staged else
                 "zero-copy: the kernel reads actions from / writes results to pinned host memory; obs padding "
                 "(constant zeros) not rewritten")
    env.close()
    return out


def roofline_of(m, peak, peak_src, traffic=None, ncu=None):
    ms = m["ms_per_step"]
    achieved = m["_alg_bytes_per_launch"] / (ms * 1e-3) / 1e9
    return dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak, traffic=traffic,
                peak_source=f"{peak_src} (MEASURED_PEAKS.json hbm_gbs)" if peak_src == "measured" else "fallback 6.65 TB/s",
                kernel=f"env_kernel<{m['lanes_per_env']},STEP>", algorithmic_bytes_per_launch=m["_alg_bytes_per_launch"],
                ncu=ncu,
                binding_bound="dependent-instruction latency of the slowest env of the launch (5 Newton iterations), fp64 issue "
                              "inside a sweep step, shared-memory pipe (DESIGN.md §4); compulsory HBM traffic is a few kB per "
                              "env-step, far below the HBM roof")


def parity_check(sc, barrier, B, local, n_check=64, n_steps=3):
    """max |dV|, |dreward|, |dobs| between the CUDA path and the oracle on `n_check` envs of a batch of the benchmarked
    shape (same launch geometry), over a reset and `n_steps` steps."""
    import torch
    from mapdn_b200 import cases
    from mapdn_b200.env import BatchedVoltageControl
    from oracle.voltage_control_ref import VoltageControlOracle
    net, prof = cases.make_case(sc), cases.make_profiles(sc)
    env_args = dict(voltage_barrier_type=barrier, action_scale=cases.SCENARIOS[sc]["action_scale"], seed=0)
    env = BatchedVoltageControl(net, prof, env_args, batch=B, device=local)
    ids = np.unique(np.linspace(0, B - 1, n_check).round().astype(int))
    obs, _ = env.reset()
    obs = obs.cpu().numpy()
    ors = [VoltageControlOracle(net, prof, env.args, env_id=int(i)) for i in ids]
    dv = dr = do = 0.0
    for o, i in zip(ors, ids):
        oo, _ = o.reset()
        do = max(do, float(np.abs(np.array(oo) - obs[i]).max()))
    rng = np.random.default_rng(7)
    lo, hi = env.action_space.low, env.action_space.high
    for _ in range(n_steps):
        a = rng.uniform(lo, hi, (B, env.n_agents))
        r, term, _ = env.step(torch.tensor(a, device=env.device))
        r, vm, ob = r.cpu().numpy(), env.get_field("vm").cpu().numpy(), env.obs.cpu().numpy()
        for o, i in zip(ors, ids):
            ro, _, _ = o.step(a[i])
            dr = max(dr, abs(ro - r[i]))
            dv = max(dv, float(np.abs(o.g.res.vm_pu - vm[i]).max()))
            do = max(do, float(np.abs(np.array(o.get_obs()) - ob[i]).max()))
    env.close()
    out = dict(max_abs_dv=dv, max_abs_dreward=float(dr), max_abs_dobs=do, n_envs_checked=int(len(ids)),
               n_steps=n_steps, batch=B, oracle="oracle/ (env logic pinned by reference-executed fixtures, power flow by "
                                                "literature results; not pinned against pandapower itself)",
               tolerance=dict(dv=1e-6, dreward=1e-5))
    try:        # the same device against trajectories the reference's own env code produced (never fatal for the bench)
        out["reference_fixture"] = reference_fixture_check(local)
    except Exception as e:      # noqa: BLE001
        out["reference_fixture"] = dict(error=repr(e)[:300])
    return out


def reference_fixture_check(local, name="case33_bowl", make_env=None):
    """Replays a trajectory that the REFERENCE's own env code produced (tests/golden/ref_env_<name>.npz, written by
    scripts/make_reference_golden.py; oracle/ref_harness.py says what is real and what is substituted) through the CUDA
    engine on this device and returns the largest deviations. `make_env` is a test hook (CPU stand-in)."""
    import torch
    from oracle import ref_scenarios as S
    g = np.load(S.fixture_path(ROOT, name))
    ops = [tuple(op) for op in json.loads(str(g["ops"]))]
    sc = S.SCENARIOS[name]
    net, prof = sc["build"]()
    ids = sc["env_ids"]
    B = max(ids) + 1
    if make_env is None:
        from mapdn_b200.env import BatchedVoltageControl
        env = BatchedVoltageControl(net, prof, sc["args"], batch=B, device=local)
    else:
        env = make_env(net, prof, sc["args"], B)
    d_obs = d_state = d_reward = d_info = 0.0
    t = n_steps = n_reset = 0
    for k_op, op in enumerate(ops):
        if op[0] == "step":
            a = np.zeros((B, net.n_sgen))
            a[ids] = g["actions"][t]
            r, _, info = env.step(torch.tensor(a, device=env.device), add_noise=bool(op[1]))
            live = np.nonzero(g["alive"][t])[0]
            sel = [ids[k] for k in live]
            if live.size:
                d_reward = max(d_reward, float(np.abs(r[sel].cpu().numpy() - g["reward"][t, live]).max()))
                d_info = max(d_info, float(np.abs(info[sel].cpu().numpy() - g["info"][t, live]).max()))
                n_steps += 1
            t += 1
            if live.size == 0:
                continue
        else:
            if op[0] in ("manual", "reset_keep"):
                start = np.zeros((B, 3), np.int32)
                for k, e in enumerate(ids):
                    start[e] = S.manual_of(sc, op, k) if op[0] == "manual" else g["start"][n_reset - 1, k]
                env.reset(torch.tensor(start, device=env.device), add_noise=(op[0] == "reset_keep"))
            else:
                env.reset()
            n_reset += 1
            live, sel = np.arange(len(ids)), list(ids)
        obs = env.obs[sel].cpu().numpy()
        d_obs = max(d_obs, float(np.abs(obs - g["obs"][k_op, live][..., -obs.shape[-1]:]).max()))
        d_state = max(d_state, float(np.abs(env.get_state()[sel].cpu().numpy() - g["state"][k_op, live]).max()))
    env.close()
    return dict(fixture=f"tests/golden/ref_env_{name}.npz", produced_by="the reference's own VoltageControl code "
                "(voltage_control_env.py, unmodified) behind a substitute pandapower: oracle/ref_harness.py",
                n_envs=len(ids), n_operations=len(ops), n_steps=n_steps, max_abs_dreward=d_reward, max_abs_dinfo=d_info,
                max_abs_dobs=d_obs, max_abs_dstate=d_state)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from mapdn_b200 import cases

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    from mapdn_b200.distributed import bind_to_gpu_numa_node
    numa = bind_to_gpu_numa_node(local) if world > 1 else "single rank: not bound"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    tm = Timer(world, dev)
    head = CONFIGS[HEADLINE]
    sc = args.scenario or head["scenario"]
    barrier = args.barrier or cases.SCENARIOS[sc]["barrier"]
    B = args.batch or {"case33": 4096, "case141": 2048, "case322": 1024}[sc]
    custom = bool(args.scenario or args.batch or args.barrier or args.lanes)
    K, W = args.steps, args.warmup
    flush = None if args.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    Ke = max(3, min(K, args.e2e_steps))

    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_check(sc, barrier, B, local)
    clocks = ClockSampler(local) if rank == 0 else None
    m = measure(sc, barrier, B * world, K, W, Ke, tm, local, rank, flush, lanes=args.lanes, clocks=clocks,
                obs_dtypes=("f64", "f32", "staged", "compact_f64", "compact_f32", "compact_zc_f64"), min_warm=50,
                dump_dir=args.dump_outputs if rank == 0 else None)

    # ---- the other BASELINE.json configurations of this GPU count ----
    subs = []
    if not custom and not args.no_sub:
        Ks, Ws = max(10, min(K, 50)), 5
        plan = []
        for cid, c in CONFIGS.items():
            if cid == HEADLINE:
                continue
            if c["n_gpus"] == world:
                plan.append((cid, c, c["batch"], None))
            elif world == 1 and c["n_gpus"] > 1:
                plan.append((cid, c, c["batch"] // c["n_gpus"], dict(config=cid, shard=f"1 of {c['n_gpus']}")))
        for cid, c, gb, shard in plan:
            r = measure(c["scenario"], c["barrier"], gb, Ks, Ws, max(3, min(Ks, 10)), tm, local, rank, flush)
            r["baseline_config"] = cid
            if shard:
                r["shard_of"] = shard
            subs.append(r)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peaks, peak_src = None, "fallback"
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peak, peak_src = float(peaks["hbm_gbs"]), "measured"
    except Exception:
        peak = 6650.0
    traffic = {}
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    net = cases.make_case(sc)
    roofline = roofline_of(m, peak, peak_src, traffic.get(f"{sc}_B{B}"), (traffic.get("ncu") or {}).get(f"{sc}_B{B}"))
    for r in subs:
        r["roofline"] = roofline_of(r, peak, peak_src, traffic.get(f"{r['scenario']}_B{r['envs_per_gpu']}"))
        r["config"] = dict(workload=workload_string(r["scenario"], r["envs_per_gpu"], r["barrier"]))
        r.pop("_alg_bytes_per_launch"); r.pop("_clocks")

    # ---- CPU baseline: the reference path on the host cores, bounded sample ----
    cpu = None
    if world == 1 and not args.no_cpu:
        arm = CpuArm(sc, barrier, cores=args.cpu_cores)
        n0, dt0 = arm.run(2 * arm.cores)
        n, dt = arm.run(args.cpu_sample or int(min(200 * arm.cores, max(arm.cores, 15.0 * n0 / dt0))))
        n1, dt1 = arm.run_one_core(max(8, min(400, int(3.0 * n / dt / arm.cores))))
        arm.close()
        cpu = dict(value=n / dt, unit="env-steps/s", cores=arm.cores, cores_source=arm.cores_source, kind=arm.kind,
                   one_core=dict(value=n1 / dt1, unit="env-steps/s", env_steps=n1),
                   sample=f"{n} env-steps of {sc} ({barrier} barrier, noise on) in {dt:.1f} s: " + arm.describe())

    line = dict(metric=METRIC, value=m["value"], unit="env-steps/s", n_gpus=world, steps=K, warmup=W,
                ms_per_step=m["ms_per_step"], higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64",
                data="synthetic",
                config=dict(workload=workload_string(sc, B, barrier),
                            n_bus=net.n_bus, n_agents=net.n_sgen, obs_dim=m["obs_dim"], global_batch=B * world,
                            lanes_per_env=m["lanes_per_env"], envs_per_block=m["envs_per_block"],
                            parallelism=f"envs sharded over {world} GPU(s)", numa=numa,
                            warmup_steps_done=m["warmup_steps_done"],
                            l2="flushed between steps (256 MiB memset, outside the event pairs)" if flush is not None
                            else "not flushed", timing="sum of per-step CUDA-event pairs, max over ranks"),
                clocks=m["_clocks"], gpu_launches=m["gpu_launches"],
                e2e=m["e2e"], e2e_obs_f32=dict(m["e2e_obs_f32"], note="same call with observations delivered in fp32 "
                                                                      "(opt-in API)"),
                e2e_staged=dict(m["e2e_staged"], note="round-1 host path, kept for comparison"),
                e2e_compact=dict(m["e2e_compact"], note="opt-in host layout without the reference's zero padding "
                                                        "(step_host(layout='compact'), mapdn_step_host_compact)"),
                e2e_compact_f32=dict(m["e2e_compact_f32"], note="compact rows in fp32"),
                e2e_compact_zero_copy=dict(m["e2e_compact_zero_copy"], note="compact rows written by the kernel itself "
                                           "(step_host(layout='compact', staged=False))"),
                roofline=roofline, cpu_baseline=cpu, wall_ms_per_step=m["wall_ms_per_step"],
                newton_iters_mean=m["newton_iters_mean"], nonconverged_frac=m["nonconverged_frac"],
                side_metrics_note="Newton iterations / diverged fraction of the last timed step, mean over the batch",
                parity=parity, configs=subs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scenario", default=None, choices=["case33", "case141", "case322"],
                    help="ad-hoc run of one scenario (default: the BASELINE.json headline + its sub-configs)")
    ap.add_argument("--batch", type=int, default=0, help="envs per GPU (default: BASELINE.json config)")
    ap.add_argument("--barrier", default=None, choices=["l1", "l2", "bowl", "bump", "courant_beltrami"])
    ap.add_argument("--lanes", type=int, default=0)
    ap.add_argument("--no-flush", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the other BASELINE.json configurations")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--cpu-cores", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=50)
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step returned (rank 0's envs) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    if args.warmup < 3:
        args.warmup = 3
    return run_reference(args) if args.impl == "reference" else run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
