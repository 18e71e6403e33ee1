"""ctypes binding of the engine kernel source (csrc/mj_*.cuh) compiled as test harnesses:

* tests/host_emulation/libemul*.so (emul.cpp): compiled for the host with one lane (`Emu`);
* tests/host_emulation/libdevemul_*.so (devemul.cu): compiled for sm_100a with 32 lanes and the product's engine flags, a
  batch of states per launch (`DevEmu`, needs a GPU to run; compiles without one).

Both stop a substep after one of its phases (`run(stage)`, phases.hpp) and read the workspace back through the same
readers.  TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(os.path.dirname(_HERE)), "earl_benchmark_b200", "csrc")
_LIB = None


class TaskSpec(C.Structure):
    _fields_ = [("frame_skip", C.c_int32), ("hand_site", C.c_int32), ("ree_site", C.c_int32), ("lee_site", C.c_int32),
                ("obj_geom", C.c_int32), ("obj_site", C.c_int32), ("max_newton", C.c_int32), ("obj_qpos_count", C.c_int32),
                ("mocap_low", C.c_float * 3), ("mocap_high", C.c_float * 3), ("action_scale", C.c_float),
                ("success_radius", C.c_float), ("obj_init_pos", C.c_float * 3), ("hand_init_pos", C.c_float * 3),
                ("grasp_site", C.c_int32), ("lpad_site", C.c_int32), ("rpad_site", C.c_int32), ("corner_site", C.c_int32 * 4)]


_LIBS = {}
# compile-time capacity sets of the engine: "small" the door / peg primary set (default build), "xl" the door / peg
# extra-large set of the redo pass, "kitchen" (23 dofs, 118 geoms) and "kitchen_xl" the kitchen's primary and redo sets
CAPSETS = {"small": [], "xl": ["-DMJ_CAPSET_XL"], "kitchen": ["-DMJ_CAPSET_KITCHEN"],
           "kitchen_xl": ["-DMJ_CAPSET_KITCHEN", "-DMJ_CAPSET_KITCHEN_XL"]}
STAGES = {"forward_parts": 0, "collide": 1, "constraints": 2, "solve": 3, "substeps": 4}


def _sources(main):
    return [os.path.join(_HERE, main), os.path.join(_HERE, "phases.hpp")] + \
        [os.path.join(_CSRC, f) for f in os.listdir(_CSRC) if f.startswith("mj_")]


def _stale(so, main):
    return not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in _sources(main))


def lib(capset="small"):
    """The one-lane host build of capacity set `capset` (CAPSETS)."""
    global _LIB
    if capset != "small":
        if capset not in _LIBS:
            _LIBS[capset] = _load(os.path.join(_HERE, f"libemul_{capset}.so"), CAPSETS[capset])
        return _LIBS[capset]
    if _LIB is None:
        _LIB = _load(os.path.join(_HERE, "libemul.so"), [])
    return _LIB


def _phase_readers(L):
    DP = np.ctypeslib.ndpointer(np.float64, flags="C")
    IP = np.ctypeslib.ndpointer(np.int32, flags="C")
    L.ph_caps.argtypes = [IP]
    L.ph_state.argtypes = [C.c_void_p, C.c_int, DP, DP, DP]
    L.ph_info.argtypes = [C.c_void_p, C.c_int, IP]
    L.ph_forward.argtypes = [C.c_void_p, C.c_int, DP, DP, DP, DP]
    L.ph_hits.argtypes = [C.c_void_p, C.c_int, IP]
    L.ph_contacts.argtypes = [C.c_void_p, C.c_int, DP, DP, DP, IP]
    L.ph_rows.argtypes = [C.c_void_p, C.c_int, IP, DP, DP, DP, DP, DP, IP, DP, DP]
    L.ph_solve.argtypes = [C.c_void_p, C.c_int, DP, DP, DP, DP]
    caps = np.zeros(7, np.int32)
    L.ph_caps(caps)
    L.caps = dict(zip(("MAXV", "LDM", "MAXEFC", "MAXCON", "MAXHIT", "MAXCAND", "MAXB"), (int(c) for c in caps)))


def _load(so, defines):
    if True:
        if _stale(so, "emul.cpp"):
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            subprocess.check_call([cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-ffp-contract=off"] + defines +
                                  ["-o", so, os.path.join(_HERE, "emul.cpp")])
        L = C.CDLL(so)
        L.emu_create.restype = C.c_void_p
        L.emu_create.argtypes = [C.c_char_p, C.c_longlong, C.POINTER(TaskSpec), C.c_char_p, C.c_int]
        L.emu_destroy.argtypes = [C.c_void_p]
        DP = np.ctypeslib.ndpointer(np.float64, flags="C")
        FP = np.ctypeslib.ndpointer(np.float32, flags="C")
        IP = np.ctypeslib.ndpointer(np.int32, flags="C")
        L.emu_set_state.argtypes = [C.c_void_p, DP, DP, DP, DP, DP, DP]
        L.emu_get_state.argtypes = [C.c_void_p, DP, DP, DP, DP]
        L.emu_substeps.argtypes = [C.c_void_p, C.c_int]
        L.emu_env_step.argtypes = [C.c_void_p, FP, FP]
        L.emu_forward_parts.argtypes = [C.c_void_p, DP, DP, DP]
        L.emu_info.argtypes = [C.c_void_p, C.c_int]
        L.emu_run.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.emu_spd_solve.argtypes = [C.c_int, FP, FP]
        _phase_readers(L)
        return L


def build_device(capsets=tuple(CAPSETS), out_dir=None):
    """nvcc-compile devemul.cu for each capacity set in `capsets` (in parallel): next to this file when the .so is missing
    or older than its sources, or always into `out_dir` when given; returns the paths.  Flags: the product's engine flags
    (earl_benchmark_b200.build.NVCC_FLAGS, FMA contraction on)."""
    from earl_benchmark_b200 import build as B
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    out, procs = [], []
    for c in capsets:
        so = os.path.join(out_dir or _HERE, f"libdevemul_{c}.so")
        out.append(so)
        if out_dir or _stale(so, "devemul.cu"):
            tmp = f"{so}.{os.getpid()}.tmp"
            cmd = [nvcc] + B.NVCC_FLAGS + CAPSETS[c] + ["-shared", "-o", tmp, os.path.join(_HERE, "devemul.cu")]
            procs.append((cmd, tmp, so, subprocess.Popen(cmd)))
    for cmd, tmp, so, p in procs:
        if p.wait() != 0:
            raise subprocess.CalledProcessError(p.returncode, cmd)
        os.replace(tmp, so)
    return out


_DEV_LIBS = {}


def dev_lib(capset="small"):
    """The 32-lane device build of capacity set `capset`."""
    if capset not in _DEV_LIBS:
        L = C.CDLL(build_device([capset])[0])
        DP = np.ctypeslib.ndpointer(np.float64, flags="C")
        FP = np.ctypeslib.ndpointer(np.float32, flags="C")
        IP = np.ctypeslib.ndpointer(np.int32, flags="C")
        E = [C.c_char_p, C.c_int]
        L.dev_create.restype = C.c_void_p
        L.dev_create.argtypes = [C.c_char_p, C.c_longlong, C.POINTER(TaskSpec), C.c_int] + E
        L.dev_destroy.argtypes = [C.c_void_p]
        L.dev_set_states.argtypes = [C.c_void_p, C.c_int, DP, DP, DP, DP, DP, DP] + E
        L.dev_run.argtypes = [C.c_void_p, C.c_int, C.c_int] + E
        L.dev_spd_solve.argtypes = [C.c_int, IP, FP, FP, IP] + E
        L.dev_append.argtypes = [C.c_int, C.c_int, C.c_int, IP, IP, IP, IP] + E
        L.dev_support.argtypes = [C.c_int, FP, C.c_int, DP, DP] + E
        _phase_readers(L)
        _DEV_LIBS[capset] = L
    return _DEV_LIBS[capset]


def _check(L, fn, *args):
    err = C.create_string_buffer(256)
    if getattr(L, fn)(*args, err, 256) != 0:
        raise RuntimeError(f"{fn}: {err.value.decode()}")


class _Phases:
    """Readers of the workspace a substep's phases leave behind (phases.hpp), for state `i` of the last run."""

    def _r(self, fn, i, *args):
        rc = getattr(self.L, fn)(self.h, int(i), *args)
        if rc < 0:
            raise IndexError(f"{fn}: state {i} out of range")
        return rc

    def info(self, i=0):
        out = np.zeros(7, np.int32)
        self._r("ph_info", i, out)
        return dict(zip(("nefc", "ncon", "nhit", "iter", "bad", "ncand", "broad_valid"), (int(x) for x in out)))

    def state(self, i=0):
        q, v, w = np.zeros(self.nq), np.zeros(self.nv), np.zeros(self.nv)
        self._r("ph_state", i, q, v, w)
        return q, v, w

    def forward(self, i=0):
        """xpos [nbody, 3], xmat [nbody, 9], M [nv, nv], bias [nv]"""
        x, R, M, b = np.zeros((self.nb, 3)), np.zeros((self.nb, 9)), np.zeros((self.nv, self.nv)), np.zeros(self.nv)
        self._r("ph_forward", i, x, R, M, b)
        return x, R, M, b

    def hits(self, i=0):
        """geom pairs [nhit, 2] of the broad phase's hit list, in list order"""
        p = np.zeros((self.L.caps["MAXHIT"], 2), np.int32)
        return p[:self._r("ph_hits", i, p)].copy()

    def contacts(self, i=0):
        """dist [ncon], pos [ncon, 3], frame [ncon, 9], geoms [ncon, 2]"""
        k = self.L.caps["MAXCON"]
        d, p, f, g = np.zeros(k), np.zeros((k, 3)), np.zeros((k, 9)), np.zeros((k, 2), np.int32)
        n = self._r("ph_contacts", i, d, p, f, g)
        return d[:n].copy(), p[:n].copy(), f[:n].copy(), g[:n].copy()

    def rows(self, i=0):
        """constraint rows: type, J [nefc, nv], pos, R, D, aref; per contact its first row, dim, mu and fri"""
        ke, kc = self.L.caps["MAXEFC"], self.L.caps["MAXCON"]
        t, J = np.zeros(ke, np.int32), np.zeros((ke, self.nv))
        pos, R, D, aref = np.zeros(ke), np.zeros(ke), np.zeros(ke), np.zeros(ke)
        con, mu, fri = np.zeros((kc, 2), np.int32), np.zeros(kc), np.zeros((kc, 5))
        n = self._r("ph_rows", i, t, J, pos, R, D, aref, con, mu, fri)
        nc = self.info(i)["ncon"]
        return dict(type=t[:n].copy(), J=J[:n].copy(), pos=pos[:n].copy(), R=R[:n].copy(), D=D[:n].copy(), aref=aref[:n].copy(),
                    con_row=con[:nc, 0].copy(), con_dim=con[:nc, 1].copy(), mu=mu[:nc].copy(), fri=fri[:nc].copy())

    def solved(self, i=0):
        """acc, fcon (= J' force), smooth (qfrc_smooth) [nv]; force [nefc]"""
        a, fc, sm, f = np.zeros(self.nv), np.zeros(self.nv), np.zeros(self.nv), np.zeros(self.L.caps["MAXEFC"])
        self._r("ph_solve", i, a, fc, sm, f)
        return dict(acc=a, fcon=fc, smooth=sm, force=f[:self.info(i)["nefc"]].copy())


class Emu(_Phases):
    def __init__(self, model, task, capset="small"):
        blob = model.to_blob()
        err = C.create_string_buffer(256)
        self.L = lib(capset)
        self.h = self.L.emu_create(blob, len(blob), C.byref(task), err, 256)
        if not self.h:
            raise RuntimeError(err.value.decode())
        self.nq, self.nv, self.nb = int(model.nq), int(model.nv), int(model.nbody)

    def __del__(self):
        if getattr(self, "h", None):
            self.L.emu_destroy(self.h)

    def set_state(self, qpos, qvel, warm, mocap_pos, mocap_quat=(1, 0, 1, 0), ctrl=(0, 0)):
        f = lambda a: np.ascontiguousarray(a, np.float64)  # noqa: E731
        self.L.emu_set_state(self.h, f(qpos), f(qvel), f(warm), f(mocap_pos), f(mocap_quat), f(ctrl))

    def get_state(self):
        q, v, w, mp = np.zeros(self.nq), np.zeros(self.nv), np.zeros(self.nv), np.zeros(3)
        self.L.emu_get_state(self.h, q, v, w, mp)
        return q, v, w, mp

    def substeps(self, n=1):
        self.L.emu_substeps(self.h, int(n))

    def env_step(self, action):
        obs = np.zeros(7, np.float32)
        self.L.emu_env_step(self.h, np.ascontiguousarray(action, np.float32), obs)
        return obs

    def forward_parts(self):
        M, b, x = np.zeros((self.nv, self.nv)), np.zeros(self.nv), np.zeros((self.nb, 3))
        self.L.emu_forward_parts(self.h, M, b, x)
        return M, b, x

    def info(self, what=0):
        """info("nefc" | "ncon" | "iter" | "bad" | "npair" | "nhit"): one counter; info(0): all of them (_Phases.info)"""
        if not isinstance(what, str):
            return super().info(what)
        return self.L.emu_info(self.h, {"nefc": 0, "ncon": 1, "iter": 2, "bad": 3, "npair": 4, "nhit": 5}[what])

    def run(self, stage, nsub=1):
        """The phases of one substep up to `stage` (STAGES); "substeps": `nsub` whole substeps."""
        self.L.emu_run(self.h, STAGES[stage], int(nsub))


class DevEmu(_Phases):
    """The engine on the GPU, one warp per state, up to `batch` states per launch (devemul.cu)."""

    def __init__(self, model, task, capset="small", batch=512):
        blob = model.to_blob()
        err = C.create_string_buffer(256)
        self.L = dev_lib(capset)
        self.h = self.L.dev_create(blob, len(blob), C.byref(task), int(batch), err, 256)
        if not self.h:
            raise RuntimeError(err.value.decode())
        self.nq, self.nv, self.nb, self.nu = int(model.nq), int(model.nv), int(model.nbody), int(model.nu)
        self.n = 0

    def __del__(self):
        if getattr(self, "h", None):
            self.L.dev_destroy(self.h)

    def set_states(self, qpos, qvel, warm, mocap_pos, mocap_quat=None, ctrl=None):
        f = lambda a, w: np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float64), (len(qpos), w)))  # noqa: E731
        n = len(qpos)
        mq = (1, 0, 1, 0) if mocap_quat is None else mocap_quat
        ct = np.zeros(self.nu) if ctrl is None else ctrl
        _check(self.L, "dev_set_states", self.h, n, f(qpos, self.nq), f(qvel, self.nv), f(warm, self.nv), f(mocap_pos, 3), f(mq, 4),
               f(ct, self.nu))
        self.n = n

    def run(self, stage, nsub=1):
        _check(self.L, "dev_run", self.h, STAGES[stage], int(nsub))


def spd_solve_device(n, A, x, capset="small"):
    """spd_solve<32> on matrices A [count, MAXV, LDM] float32 and right-hand sides x [count, MAXV] (both overwritten);
    returns the ok flags [count]."""
    ok = np.zeros(len(n), np.int32)
    _check(dev_lib(capset), "dev_spd_solve", len(n), np.ascontiguousarray(n, np.int32), A, x, ok)
    return ok


def append_device(which, flags, capset="small"):
    """compact_append<32> ("hit") or cand_append<32> ("cand") over flags [count, nitems] from empty lists: returns both
    whole list arrays, hit [count, MAXHIT] and cand [count, MAXCAND] (unwritten entries 0xffff), and (count, bad) or
    (count, broad_valid) [count, 2]."""
    L = dev_lib(capset)
    flags = np.ascontiguousarray(flags, np.int32)
    hit, cand = np.zeros((len(flags), L.caps["MAXHIT"]), np.int32), np.zeros((len(flags), L.caps["MAXCAND"]), np.int32)
    info = np.zeros((len(flags), 2), np.int32)
    _check(L, "dev_append", 0 if which == "hit" else 1, len(flags), flags.shape[1], flags, hit, cand, info)
    return hit, cand, info


def support_device(hull, dirs, capset="small"):
    """support_geom<32> of a mesh with vertices hull [nvert, 3] (at the origin, world axes, no margin) in directions
    dirs [ndir, 3]: support points [ndir, 3]."""
    hull, dirs = np.ascontiguousarray(hull, np.float32), np.ascontiguousarray(dirs, np.float64)
    out = np.zeros_like(dirs)
    _check(dev_lib(capset), "dev_support", len(hull), hull, len(dirs), dirs, out)
    return out


def door_task(model, max_newton=0):
    t = TaskSpec()
    t.frame_skip, t.max_newton, t.obj_qpos_count = 5, max_newton, 1
    t.grasp_site = t.lpad_site = t.rpad_site = -1
    t.corner_site[:] = [-1] * 4
    t.hand_site, t.ree_site, t.lee_site = model.site_id("body:hand"), model.site_id("rightEndEffector"), model.site_id("leftEndEffector")
    t.obj_geom, t.obj_site = model.geom_id("handle"), -1
    t.mocap_low[:] = [-0.5, 0.40, 0.05]
    t.mocap_high[:] = [0.5, 1.0, 0.5]
    t.action_scale, t.success_radius = 0.01, 0.02
    return t


def peg_task(model, max_newton=0):
    t = TaskSpec()
    t.frame_skip, t.max_newton, t.obj_qpos_count = 5, max_newton, 3
    t.grasp_site = t.lpad_site = t.rpad_site = -1
    t.corner_site[:] = [-1] * 4
    t.hand_site, t.ree_site, t.lee_site = model.site_id("body:hand"), model.site_id("rightEndEffector"), model.site_id("leftEndEffector")
    t.obj_geom, t.obj_site = -1, model.site_id("pegHead")
    t.mocap_low[:] = [-0.5, 0.40, 0.05]
    t.mocap_high[:] = [0.5, 1.0, 0.5]
    t.action_scale, t.success_radius = 0.01, 0.05
    return t


def kitchen_task(model, max_newton=0):
    """Engine-level task spec for the kitchen model (the kitchen task layer is not in the kernel source yet: only
    `substeps` is meaningful, the Sawyer observation fields point at a valid site)."""
    t = TaskSpec()
    t.frame_skip, t.max_newton, t.obj_qpos_count = 40, max_newton, 0
    t.grasp_site = t.lpad_site = t.rpad_site = -1
    t.corner_site[:] = [-1] * 4
    t.hand_site = t.ree_site = t.lee_site = model.site_id("end_effector")
    t.obj_geom, t.obj_site = -1, model.site_id("slide_site")
    t.mocap_low[:] = [-0.7, -0.1, 1.8]
    t.mocap_high[:] = [0.4, 0.5, 2.6]
    t.action_scale, t.success_radius = 0.01, 0.3
    return t
