"""TEST INFRASTRUCTURE ONLY. NumPy binding of ``tests/emu/_build/libmapdn_b200_emu.so`` - the product's C-ABI library
compiled with g++ against ``tests/emu/cuda_runtime.h`` (a CPU SIMT emulation: one OS thread per CUDA thread), so that the
CPU test tier executes the kernel SOURCE (``mapdn_b200/csrc/env_kernel.cuh``) against the oracle. "Device pointers" are
NumPy buffers. The product never loads this library (``mapdn_b200/_capi.py`` only knows ``libmapdn_b200.so``)."""
import ctypes as C
import os
import subprocess

import numpy as np

from mapdn_b200 import _capi

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "mapdn_b200", "csrc")
LIB = os.path.join(HERE, "_build", "libmapdn_b200_emu.so")
DEPS = [os.path.join(CSRC, f) for f in ("mapdn_b200.cu", "env_kernel.cuh", "kernel_params.h", "philox.cuh")] + [
    os.path.join(HERE, "cuda_runtime.h"), os.path.join(ROOT, "include", "mapdn_b200.h")]


def build(force=False):
    if not force and os.path.exists(LIB) and all(os.path.getmtime(d) <= os.path.getmtime(LIB) for d in DEPS):
        return LIB
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    cmd = ["g++", "-std=c++17", "-O1", "-g", "-fPIC", "-shared", "-pthread", "-DMAPDN_HOST_EMU", "-DMAPDN_EMU_DEFINE_GLOBALS",
           "-I", HERE, "-x", "c++", os.path.join(CSRC, "mapdn_b200.cu"), "-o", LIB]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("g++ failed building the emulated library:\n" + res.stderr[-4000:])
    return LIB


_L = None


def lib():
    global _L
    if _L is None:
        L = C.CDLL(build())
        vp = C.c_void_p
        L.mapdn_last_error.restype = C.c_char_p
        L.mapdn_create.argtypes = [C.POINTER(_capi.NetDescC), C.POINTER(_capi.ProfileDescC), C.POINTER(_capi.CfgC), C.c_int32,
                                   C.POINTER(vp)]
        L.mapdn_destroy.argtypes = [vp]
        L.mapdn_get_dims.argtypes = [vp, C.POINTER(_capi.DimsC)]
        L.mapdn_reset.argtypes = [vp, vp, vp, C.c_int32, vp, vp, vp, vp]
        L.mapdn_step.argtypes = [vp, vp, C.c_int32, vp, vp, vp, vp, vp]
        L.mapdn_get_obs.argtypes = [vp, vp, vp]
        L.mapdn_get_state.argtypes = [vp, vp, vp]
        L.mapdn_get_field.argtypes = [vp, C.c_int32, vp, vp]
        L.mapdn_solve.argtypes = [vp, C.c_int32] + [vp] * 11 + [vp]
        L.mapdn_droop.argtypes = [vp, C.c_int32] + [vp] * 5 + [C.c_double, C.c_double, C.c_int32] + [vp] * 5
        L.mapdn_step_host.argtypes = [vp, vp, C.c_int32, vp, vp, vp, vp, vp]
        L.mapdn_step_host_f32obs.argtypes = [vp, vp, C.c_int32, vp, vp, vp, vp, vp]
        L.mapdn_step_host_pinned.argtypes = [vp, vp, C.c_int32, vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp]
        L.mapdn_step_host_compact.argtypes = [vp, vp, C.c_int32, vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp]
        L.mapdn_obs_compact_layout.argtypes = [vp, vp, vp, vp]
        L.mapdn_wait.argtypes = [vp, vp]
        _L = L
    return _L


def _ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


class EmuEnv:
    """The slice of ``BatchedVoltageControl`` the emulator tests need, on NumPy arrays."""

    def __init__(self, net, prof, env_args=None, batch=1, lanes_per_env=0, env_id_offset=0):
        from mapdn_b200.env import DEFAULT_ENV_ARGS
        args = dict(DEFAULT_ENV_ARGS)
        args.update(env_args or {})
        self.args, self.net, self.batch = args, net, batch
        L = lib()
        cfg = _capi.CfgC(batch=batch, barrier=_capi.BARRIERS[args["voltage_barrier_type"]],
                         voltage_weight=float(args["voltage_weight"]),
                         q_weight=float(args["q_weight"] if args["q_weight"] is not None else 0.0),
                         line_weight=float(args["line_weight"] or 0.0), use_line_weight=int(args["line_weight"] is not None),
                         v_upper=float(args["v_upper"]), v_lower=float(args["v_lower"]), episode_limit=int(args["episode_limit"]),
                         action_low=float(-args["action_scale"] + args["action_bias"]),
                         action_high=float(args["action_scale"] + args["action_bias"]),
                         reset_action=int(bool(args["reset_action"])), seed=int(args["seed"]), env_id_offset=env_id_offset,
                         tol=0.0, max_iter=0, lanes_per_env=lanes_per_env,
                         state_space_mask=sum(_capi.STATE_SPACE_BITS[k] for k in set(args["state_space"])))
        nd, self._k1 = _capi.make_net_desc(net)
        pd_, self._k2 = (None, None) if prof is None else _capi.make_profile_desc(prof)
        h = C.c_void_p()
        self._chk(L.mapdn_create(C.byref(nd), None if pd_ is None else C.byref(pd_), C.byref(cfg), 0, C.byref(h)))
        self._h = h
        d = _capi.DimsC()
        self._chk(L.mapdn_get_dims(h, C.byref(d)))
        self.dims = {k: getattr(d, k) for k, _ in d._fields_}
        B = batch
        self.obs = np.zeros((B, d.n_agents, d.obs_dim))
        self.state = np.zeros((B, d.state_dim))
        self.reward, self.term, self.info = np.zeros(B), np.zeros(B, np.uint8), np.zeros((B, 11))
        self.reset_ok = np.ones(B, np.uint8)

    @staticmethod
    def _chk(st):
        if st != 0:
            raise RuntimeError(f"mapdn status {st}: {lib().mapdn_last_error().decode()}")

    def close(self):
        if self._h:
            lib().mapdn_destroy(self._h)
            self._h = None

    def solve(self, p_load, q_load, p_sgen, q_sgen):
        nb, d = p_sgen.shape[0], self.dims
        ins = [np.ascontiguousarray(a, np.float64) for a in (p_load, q_load, p_sgen, q_sgen)]
        out = dict(vm=np.zeros((nb, d["n_bus"])), va_deg=np.zeros((nb, d["n_bus"])), p_bus=np.zeros((nb, d["n_bus"])),
                   q_bus=np.zeros((nb, d["n_bus"])), pl=np.zeros((nb, d["n_line"])), iterations=np.zeros(nb, np.int32),
                   converged=np.zeros(nb, np.uint8))
        self._chk(lib().mapdn_solve(self._h, nb, *[_ptr(a) for a in ins], *[_ptr(out[k]) for k in
                                    ("vm", "va_deg", "p_bus", "q_bus", "pl", "iterations", "converged")], None))
        return out

    def reset(self, start=None, add_noise=True):
        st = None if start is None else np.ascontiguousarray(start, np.int32)
        self._chk(lib().mapdn_reset(self._h, _ptr(st), None, int(add_noise), _ptr(self.obs), _ptr(self.state),
                                    _ptr(self.reset_ok), None))
        return self.obs, self.state

    def step(self, actions, add_noise=True):
        a = np.ascontiguousarray(actions, np.float64)
        self._chk(lib().mapdn_step(self._h, _ptr(a), int(add_noise), _ptr(self.reward), _ptr(self.term), _ptr(self.info),
                                   _ptr(self.obs), None))
        return self.reward, self.term, self.info

    def get_state(self):
        self._chk(lib().mapdn_get_state(self._h, _ptr(self.state), None))
        return self.state

    def get_field(self, name):
        d = self.dims
        width = dict(vm=d["n_bus"], va_deg=d["n_bus"], p_bus=d["n_bus"], q_bus=d["n_bus"], p_sgen=d["n_sgen"],
                     q_sgen=d["n_sgen"], line_loss=d["n_line"], p_load=d["n_load"], q_load=d["n_load"],
                     sum_rewards=1, steps=1, start_row=1, nr_iters=1)[name]
        out = np.zeros((self.batch, width))
        self._chk(lib().mapdn_get_field(self._h, _capi.FIELDS[name], _ptr(out), None))
        return out

    # ---- host-buffer entry points (under the emulation every buffer is "pinned host memory") ----
    def compact_layout(self):
        n = self.dims["n_agents"]
        off, ln, row = (C.c_int32 * n)(), (C.c_int32 * n)(), C.c_int32(0)
        self._chk(lib().mapdn_obs_compact_layout(self._h, off, ln, C.byref(row)))
        return [(int(off[a]), int(ln[a])) for a in range(n)], int(row.value)

    def step_host(self, actions, add_noise=True, f32=False, path="pinned", direct=False):
        """path: "pinned" (zero-copy, padding skipped), "staged" (H2D + 4 x D2H), "compact" (rows without padding)."""
        a = np.ascontiguousarray(actions, np.float64)
        d, B = self.dims, self.batch
        dt = np.float32 if f32 else np.float64
        if path == "compact":
            obs = np.zeros((B, self.compact_layout()[1]), dt)
            self._chk(lib().mapdn_step_host_compact(self._h, _ptr(a), int(add_noise), _ptr(self.reward), _ptr(self.term),
                                                    _ptr(self.info), _ptr(obs), int(f32), int(direct), 1, None))
        elif path == "pinned":
            obs = np.zeros((B, d["n_agents"], d["obs_dim"]), dt)      # the padding is never written: it must start as zeros
            self._chk(lib().mapdn_step_host_pinned(self._h, _ptr(a), int(add_noise), _ptr(self.reward), _ptr(self.term),
                                                   _ptr(self.info), _ptr(obs), int(f32), 1, 1, None))
        else:
            obs = np.full((B, d["n_agents"], d["obs_dim"]), np.nan, dt)
            fn = lib().mapdn_step_host_f32obs if f32 else lib().mapdn_step_host
            self._chk(fn(self._h, _ptr(a), int(add_noise), _ptr(self.reward), _ptr(self.term), _ptr(self.info), _ptr(obs), None))
        return self.reward.copy(), self.term.copy(), self.info.copy(), obs

    def droop(self, p_load, q_load, p_pv, s_rated, gain=0.1, tol=1e-4, max_ite=100, q_max_manual=None):
        B, d = p_pv.shape[0], self.dims
        qmm = s_rated if q_max_manual is None else q_max_manual
        ins = [np.ascontiguousarray(x, np.float64) for x in (p_load, q_load, p_pv, s_rated, qmm)]
        vm, q, loss, it = np.zeros((B, d["n_bus"])), np.zeros((B, d["n_sgen"])), np.zeros(B), np.zeros(B, np.int32)
        self._chk(lib().mapdn_droop(self._h, B, *[_ptr(x) for x in ins], float(gain), float(tol), int(max_ite), _ptr(vm), _ptr(q),
                                    _ptr(loss), _ptr(it), None))
        return dict(vm=vm, q=q, loss=loss, iterations=it)
