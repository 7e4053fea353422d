"""Race check of the kernel source on the CPU: the emulated library (tests/emu) built with -fsanitize=thread. Every CUDA
thread is an OS thread and every barrier (__syncwarp, __syncthreads, bar.sync / arrive / red) a mutex-protected counting
barrier, so ThreadSanitizer's happens-before analysis covers shared AND global memory (compute-sanitizer's racecheck only
sees shared memory) and is stricter than the hardware (no implicit warp-synchronous ordering).
    python scripts/emu_tsan.py            # builds /tmp/mapdn_emu_tsan/libemu_tsan.so, runs reset / step / solve / droop
Besides small single-round batches it runs the full-size launch geometries on one emulated SM (case141 and case322: two
rounds per CTA; case322: plan 3, cold tables in global memory and loads staged in the node records) and plan 3 forced at 4
and 8 lanes per env.
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = "/tmp/mapdn_emu_tsan"
LIB = os.path.join(OUT, "libemu_tsan.so")
CHILD = r'''
import sys, numpy as np
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/tests/emu")
import emu_env
emu_env.LIB = %(lib)r; emu_env.build = lambda force=False: emu_env.LIB
from emu_env import EmuEnv
from mapdn_b200 import cases
name, lanes, B = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
net, prof = cases.make_case(name), cases.make_profiles(name, n_days=3)
scale = cases.SCENARIOS[name]["action_scale"]
env = EmuEnv(net, prof, dict(seed=3, voltage_barrier_type="bowl", action_scale=scale), batch=B, lanes_per_env=lanes)
env.reset()
rng = np.random.default_rng(0)
for t in range(2):
    env.step(rng.uniform(-scale, scale, (B, net.n_sgen)))
env.step_host(rng.uniform(-scale, scale, (B, net.n_sgen)), path="compact")
inp = cases.synthetic_inputs(name, 3, seed=1)
env.solve(inp["p_load"], inp["q_load"], inp["p_pv"], np.zeros_like(inp["p_pv"]))
env.droop(inp["p_load"], inp["q_load"], inp["p_pv"], inp["s_max"], max_ite=6)
d = env.dims
print("ran", d["lanes_per_env"], d["envs_per_block"], d["smem_bytes"])
'''


def main():
    os.makedirs(OUT, exist_ok=True)
    subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fPIC", "-shared", "-pthread", "-fsanitize=thread", "-DMAPDN_HOST_EMU",
                    "-DMAPDN_EMU_DEFINE_GLOBALS", "-I", os.path.join(ROOT, "tests", "emu"), "-x", "c++",
                    os.path.join(ROOT, "mapdn_b200", "csrc", "mapdn_b200.cu"), "-o", LIB], check=True, stderr=subprocess.DEVNULL)
    tsan = subprocess.run(["g++", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    child = os.path.join(OUT, "child.py")
    open(child, "w").write(CHILD % dict(root=ROOT, lib=LIB))
    env = dict(os.environ, LD_PRELOAD=os.path.realpath(tsan), TSAN_OPTIONS="halt_on_error=0 report_signal_unsafe=0 exitcode=0")
    total = failed = 0
    one_sm, plan3 = dict(MAPDN_EMU_SMS="1"), dict(MAPDN_PLAN="3")
    for cfg, over in ((("case33", "8", "9"), {}), (("case33", "4", "5"), {}), (("case33", "64", "2"), {}),
                      (("case141", "32", "3"), {}), (("case322", "64", "2"), {}),
                      (("case33", "0", "28"), one_sm), (("case141", "0", "14"), one_sm), (("case322", "0", "8"), one_sm),
                      (("case33", "4", "5"), plan3), (("case33", "8", "9"), plan3)):
        res = subprocess.run([sys.executable, child, *cfg], env=dict(env, **over), capture_output=True, text=True)
        n = res.stderr.count("WARNING: ThreadSanitizer")
        total += n
        ran = [ln.split()[1:] for ln in res.stdout.splitlines() if ln.startswith("ran ")]
        failed += not ran
        geom = f"lanes/env={ran[0][0]} envs/CTA={ran[0][1]} smem={ran[0][2]} B" if ran else "B"
        print(f"{cfg[0]} {geom}={cfg[2]}{''.join(f' {k}={v}' for k, v in over.items())} (reset, 2 steps, compact host step, "
              f"solve, droop): {'completed' if ran else 'FAILED'}, ThreadSanitizer reports: {n}")
        if n:
            sys.stderr.write(res.stderr[:6000])
    return 1 if total or failed else 0


if __name__ == "__main__":
    sys.exit(main())
