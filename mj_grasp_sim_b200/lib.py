"""ctypes binding of libmgs_b200.so (the C ABI declared in include/mgs_b200.h).

The product path has no CPU fallback: if the shared library is missing, or there is no CUDA
device, every entry point raises.  `build()` compiles the library in-tree with nvcc for sm_100a.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from . import shard
from .model_desc import MgsModelDesc, make_desc

_PKG = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_PKG, "libmgs_b200.so")
SO_PATH_F64 = os.path.join(_PKG, "libmgs_b200_f64.so")
CSRC = os.path.join(_PKG, "csrc")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-shared",
              "-Xcompiler", "-fPIC", "-t", "4"]


class MgsRolloutCfg(C.Structure):
    _fields_ = [("nstep_close", C.c_int), ("nstep_lift", C.c_int), ("shake_steps", C.c_int), ("repose_on_close", C.c_int),
                ("lift_dist", C.c_double), ("shake_dist", C.c_double)]


class MgsModelInfo(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("nq", "nv", "nu", "nmocap", "state_stride", "diag_stride", "ncon_max", "nefc_max",
                                       "smem_bytes_per_env", "warps_per_block", "blocks_per_sm", "num_sms", "real_bytes",
                                       "lanes_per_env")]


class MgsError(RuntimeError):
    pass


def _sources():
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))] + [
        os.path.join(os.path.dirname(_PKG), "include", f) for f in ("mgs_b200.h", "mgs_model_desc.h")]


def source_stamp() -> str:
    """sha256 prefix over the library's sources (csrc/ + include/): compiled into the .so as mgs_build_stamp() so that a test
    can tell a stale prebuilt library from one built from the checked-out tree."""
    import hashlib
    h = hashlib.sha256()
    for s in _sources():
        h.update(os.path.basename(s).encode())
        h.update(open(s, "rb").read())
    return h.hexdigest()[:16]


def _built_stamp(so: str) -> str:
    try:
        return open(so + ".stamp").read().strip()
    except OSError:
        return ""


def build(force: bool = False, f64: bool = False) -> str:
    """Compile csrc/mgs_b200.cu -> libmgs_b200.so (sm_100a).  Cross-compiles without a GPU."""
    so = SO_PATH_F64 if f64 else SO_PATH
    stamp = source_stamp()
    if not force and os.path.exists(so) and _built_stamp(so) == stamp:
        return so
    # four translation units = four variants of the rollout kernel (16 / 12 warps per CTA with one environment per warp, and one
    # environment per 256-thread CTA with its state in shared or in global memory; see csrc/mgs_kernel_ops.h)
    cmd = ["nvcc"] + NVCC_FLAGS + (["-DMGS_REAL_DOUBLE"] if f64 else []) + [f'-DMGS_BUILD_STAMP="{stamp}"', "-o", so,
                                                                             os.path.join(CSRC, "mgs_b200.cu"), os.path.join(CSRC, "mgs_kernel_w12.cu"),
                                                                             os.path.join(CSRC, "mgs_kernel_wide.cu"), os.path.join(CSRC, "mgs_kernel_wide_g.cu"),
                                                                             os.path.join(CSRC, "mgs_sampler.cu")]
    subprocess.check_call(cmd)
    with open(so + ".stamp", "w") as f:
        f.write(stamp)
    return so


def bind(L, prefix="mgs_"):
    """Attach argtypes/restypes for the ABI (also used by the lane-1 test harness, prefix 'l1_')."""
    vp, ip, fp, dp, u8p = C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_ubyte)
    g = lambda n: getattr(L, prefix + n)
    g("last_error").restype = C.c_char_p
    g("model_destroy").argtypes = [vp]
    g("model_destroy").restype = None
    g("model_info").argtypes = [vp, C.POINTER(MgsModelInfo)]
    g("step_host").argtypes = [vp, C.c_int, C.c_int, vp, vp, vp]
    g("last_aux").argtypes = [vp, C.c_int, fp]
    g("set_qvel_clip").argtypes = [vp, C.c_double]
    if prefix == "mgs_":
        L.mgs_model_create.argtypes = [C.POINTER(MgsModelDesc), C.c_int, C.POINTER(vp)]
        L.mgs_model_create_ex.argtypes = [C.POINTER(MgsModelDesc), C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
        L.mgs_model_create_any.argtypes = [C.POINTER(MgsModelDesc), C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
        L.mgs_model_state_in_global.argtypes = [vp]
        L.mgs_grasp_collision_mask.argtypes = [vp, C.c_int, fp, fp, C.c_int, ip, C.c_int, u8p]
        L.mgs_grasp_stability.argtypes = [vp, C.c_int, fp, fp, C.c_int, ip, C.c_int, dp, C.POINTER(MgsRolloutCfg), u8p, ip]
        L.mgs_rollout_device.argtypes = [vp, C.c_int, C.c_int, vp, vp, C.c_int, ip, C.c_int, dp, C.POINTER(MgsRolloutCfg), vp, vp, vp]
        L.mgs_step_device.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp]
        L.mgs_clutter_collision_mask.argtypes = [vp, C.c_int, dp, fp, fp, C.c_int, ip, C.c_int, u8p]
        L.mgs_clutter_stable_mask.argtypes = [vp, C.c_int, dp, fp, fp, C.c_int, ip, C.c_int, dp, C.POINTER(MgsRolloutCfg), u8p, ip]
        L.mgs_clutter_scenes_collision_mask.argtypes = [vp, C.c_int, C.c_int, dp, ip, fp, fp, C.c_int, ip, C.c_int, u8p]
        L.mgs_clutter_scenes_stable_mask.argtypes = [vp, C.c_int, C.c_int, dp, ip, fp, fp, C.c_int, ip, C.c_int, C.c_int, dp,
                                                     C.POINTER(MgsRolloutCfg), u8p, ip]
        L.mgs_clutter_scenes_device.argtypes = [vp, C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, vp, vp, C.c_int, ip, C.c_int, dp,
                                                C.POINTER(MgsRolloutCfg), vp, vp, vp]
        L.mgs_launch_count.restype = C.c_longlong
        L.mgs_overflow_count.argtypes = [vp]
        L.mgs_build_stamp.restype = C.c_char_p
        L.mgs_antipodal_hits.argtypes = [C.c_int, C.c_int, dp, dp, C.c_int, dp, C.c_double, dp, dp, ip]
    else:
        L.l1_model_create.argtypes = [C.POINTER(MgsModelDesc), C.POINTER(vp)]
        L.l1_rollout_host.argtypes = [vp, C.c_int, C.c_int, fp, fp, C.c_int, ip, C.c_int, dp, C.POINTER(MgsRolloutCfg), u8p, ip]
        L.l1_clutter_host.argtypes = [vp, C.c_int, C.c_int, dp, fp, fp, C.c_int, ip, C.c_int, dp, C.POINTER(MgsRolloutCfg), u8p, ip]
    return L


_LIBS = {}


def load(f64: bool = False):
    so = SO_PATH_F64 if f64 else os.environ.get("MGS_B200_SO", SO_PATH)  # env override: A/B builds while profiling
    if so not in _LIBS:
        if not os.path.exists(so):
            raise MgsError(f"{so} is missing: build it with mj_grasp_sim_b200.lib.build() (nvcc, sm_100a). "
                           "There is no CPU fallback for the rollout path.")
        _LIBS[so] = bind(C.CDLL(so))
    return _LIBS[so]


def _fp(a): return a.ctypes.data_as(C.POINTER(C.c_float))
def _ip(a): return a.ctypes.data_as(C.POINTER(C.c_int))
def _dp(a): return a.ctypes.data_as(C.POINTER(C.c_double))
def _u8(a): return a.ctypes.data_as(C.POINTER(C.c_ubyte))


class BatchSim:
    """A compiled model resident on one GPU + the batched entry points.

    `lib`/`prefix` exist so the test tier can drive the lane-1 host build of the same source
    through the same wrapper; product code always uses the defaults (the CUDA library).

    `global_fallback=True` (mgs_model_create_any): a model whose environment state does not fit one CTA's shared memory runs with
    that state in global memory (kernel variant wide_g) instead of raising; `state_in_global` tells which one was made.
    """

    def __init__(self, model, device: int = 0, f64: bool = False, lib=None, prefix: str = "mgs_", ncon_max: int = 0, nefc_max: int = 0,
                 ground_name: str = "geom:ground", global_fallback: bool = False):
        self.model = model
        self.device = device
        self.L = lib if lib is not None else load(f64)
        self.p = prefix
        self.desc, self._keep = make_desc(model, ground_name)
        h = C.c_void_p()
        if prefix == "mgs_":
            ncon_max = ncon_max or int(os.environ.get("MGS_NCON_MAX", "0"))
            nefc_max = nefc_max or int(os.environ.get("MGS_NEFC_MAX", "0"))
            create = self.L.mgs_model_create_any if global_fallback else self.L.mgs_model_create_ex
            rc = create(C.byref(self.desc), device, ncon_max, nefc_max, C.byref(h))
        else:
            rc = self.L.l1_model_create(C.byref(self.desc), C.byref(h))
        self._check(rc)
        self.h = h
        self.info = MgsModelInfo()
        self._check(self._f("model_info")(self.h, C.byref(self.info)))
        self.real = np.float32 if self.info.real_bytes == 4 else np.float64
        self._order = None  # launch order of the most recent multi-scene call (last_aux maps its results back), else None

    def _f(self, name): return getattr(self.L, self.p + name)

    @property
    def state_in_global(self) -> bool:
        """True when the environments' state lives in a global-memory slab (variant wide_g), False when in shared memory."""
        if self.p != "mgs_":
            return False
        rc = self.L.mgs_model_state_in_global(self.h)
        if rc < 0:
            self._check(rc)
        return bool(rc)

    def _check(self, rc):
        if rc != 0:
            raise MgsError(self._f("last_error")().decode())

    def close(self):
        if getattr(self, "h", None):
            self._f("model_destroy")(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- state records -------------------------------------------------------------------
    def pack_state(self, qpos, qvel, qacc_ws=None, ctrl=None, mocap_pos=None, mocap_quat=None):
        m = self.model
        qpos = np.atleast_2d(qpos)
        n = len(qpos)
        s = np.zeros((n, self.info.state_stride), dtype=self.real)
        nq, nv, nu = m.nq, m.nv, m.nu
        s[:, :nq] = qpos
        s[:, nq:nq + nv] = qvel
        if qacc_ws is not None:
            s[:, nq + nv:nq + 2 * nv] = qacc_ws
        if ctrl is not None:
            s[:, nq + 2 * nv:nq + 2 * nv + nu] = ctrl
        o = nq + 2 * nv + nu
        if self.info.nmocap:
            s[:, o:o + 3] = m.mocap_pos0[0] if mocap_pos is None else mocap_pos
            s[:, o + 3:o + 7] = m.mocap_quat0[0] if mocap_quat is None else mocap_quat
        return s

    def unpack_state(self, s):
        m = self.model
        nq, nv, nu = m.nq, m.nv, m.nu
        o = nq + 2 * nv + nu
        return dict(qpos=s[:, :nq], qvel=s[:, nq:nq + nv], qacc_warmstart=s[:, nq + nv:nq + 2 * nv], ctrl=s[:, nq + 2 * nv:o],
                    mocap_pos=s[:, o:o + 3], mocap_quat=s[:, o + 3:o + 7])

    def unpack_diag(self, d):
        m = self.model
        nv, nb = m.nv, m.nbody
        o = 8
        out = dict(ncon=d[:, 0].astype(int), nefc=d[:, 1].astype(int), niter=d[:, 2].astype(int), bad=d[:, 3].astype(int),
                   overflow=d[:, 4].astype(int), ne=d[:, 5].astype(int), nf=d[:, 6].astype(int), nl=d[:, 7].astype(int))
        out["qacc"] = d[:, o:o + nv]; out["qacc_smooth"] = d[:, o + nv:o + 2 * nv]; out["qfrc_smooth"] = d[:, o + 2 * nv:o + 3 * nv]
        o += 3 * nv
        out["M"] = d[:, o:o + nv * nv].reshape(-1, nv, nv); o += nv * nv
        out["xpos"] = d[:, o:o + 3 * nb].reshape(-1, nb, 3); o += 3 * nb
        out["xquat"] = d[:, o:o + 4 * nb].reshape(-1, nb, 4); o += 4 * nb
        nc, ne = self.info.ncon_max, self.info.nefc_max
        out["contact"] = d[:, o:o + 5 * nc].reshape(-1, nc, 5); o += 5 * nc
        out["efc"] = d[:, o:o + 4 * ne].reshape(-1, ne, 4)
        return out

    def step(self, state, nstep=1, want_diag=False):
        """mj_step x nstep on a batch of state records (nstep=0: mj_forward).  Host arrays in/out."""
        state = np.ascontiguousarray(state, dtype=self.real)
        n = len(state)
        out = np.empty_like(state)
        diag = np.zeros((n, self.info.diag_stride), dtype=self.real) if want_diag else None
        self._order = None
        self._check(self._f("step_host")(self.h, n, nstep, state.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p),
                                         diag.ctypes.data_as(C.c_void_p) if want_diag else None))
        return (out, self.unpack_diag(diag)) if want_diag else out

    # ---- the two reference loops ---------------------------------------------------------
    def _prep(self, pose7, joints, joint_qposadr):
        pose7 = np.ascontiguousarray(pose7, dtype=np.float32).reshape(-1, 7)
        joints = np.ascontiguousarray(joints, dtype=np.float32)
        joints = joints.reshape(len(pose7), joints.shape[-1] if joints.ndim > 1 else len(np.atleast_1d(joint_qposadr)))
        jadr = np.ascontiguousarray(joint_qposadr, dtype=np.int32)
        return pose7, joints, jadr

    def collision_mask(self, pose7, joints, joint_qposadr, base_qposadr):
        pose7, joints, jadr = self._prep(pose7, joints, joint_qposadr)
        n = len(pose7)
        out = np.zeros(n, dtype=np.uint8)
        self._order = None
        if self.p == "mgs_":
            rc = self.L.mgs_grasp_collision_mask(self.h, n, _fp(pose7), _fp(joints), joints.shape[1], _ip(jadr), int(base_qposadr), _u8(out))
        else:
            rc = self.L.l1_rollout_host(self.h, 1, n, _fp(pose7), _fp(joints), joints.shape[1], _ip(jadr), int(base_qposadr), None, None, _u8(out), None)
        self._check(rc)
        return out.astype(bool)

    def stability(self, pose7, joints, joint_qposadr, base_qposadr, close_ctrl, cfg: MgsRolloutCfg):
        pose7, joints, jadr = self._prep(pose7, joints, joint_qposadr)
        n = len(pose7)
        cc = np.ascontiguousarray(close_ctrl, dtype=np.float64)
        out = np.zeros(n, dtype=np.uint8)
        steps = np.zeros(n, dtype=np.int32)
        self._order = None
        if self.p == "mgs_":
            rc = self.L.mgs_grasp_stability(self.h, n, _fp(pose7), _fp(joints), joints.shape[1], _ip(jadr), int(base_qposadr), _dp(cc),
                                            C.byref(cfg), _u8(out), _ip(steps))
        else:
            rc = self.L.l1_rollout_host(self.h, 2, n, _fp(pose7), _fp(joints), joints.shape[1], _ip(jadr), int(base_qposadr), _dp(cc),
                                        C.byref(cfg), _u8(out), _ip(steps))
        self._check(rc)
        return out.astype(bool), steps

    # ---- clutter table ---------------------------------------------------------------------
    def clutter_collision_mask(self, scene, pose7, joints, joint_qposadr, base_qposadr):
        pose7, joints, jadr = self._prep(pose7, joints, joint_qposadr)
        sc = np.ascontiguousarray(scene, dtype=np.float64)
        n = len(pose7)
        out = np.zeros(n, dtype=np.uint8)
        self._order = None
        if n == 0:
            return out.astype(bool)
        if self.p == "mgs_":
            rc = self.L.mgs_clutter_collision_mask(self.h, n, _dp(sc), _fp(pose7), _fp(joints), joints.shape[1], _ip(jadr), int(base_qposadr), _u8(out))
        else:
            rc = self.L.l1_clutter_host(self.h, 3, n, _dp(sc), _fp(pose7), _fp(joints), joints.shape[1], _ip(jadr), int(base_qposadr), None, None, _u8(out), None)
        self._check(rc)
        return out.astype(bool)

    def clutter_stable_mask(self, scene, pose7, joints, joint_qposadr, base_qposadr, close_ctrl, cfg: MgsRolloutCfg):
        pose7, joints, jadr = self._prep(pose7, joints, joint_qposadr)
        sc = np.ascontiguousarray(scene, dtype=np.float64)
        cc = np.ascontiguousarray(close_ctrl, dtype=np.float64)
        n = len(pose7)
        out = np.zeros(n, dtype=np.uint8)
        steps = np.zeros(n, dtype=np.int32)
        self._order = None
        if n == 0:
            return out.astype(bool), steps
        if self.p == "mgs_":
            rc = self.L.mgs_clutter_stable_mask(self.h, n, _dp(sc), _fp(pose7), _fp(joints), joints.shape[1], _ip(jadr), int(base_qposadr), _dp(cc),
                                                C.byref(cfg), _u8(out), _ip(steps))
        else:
            rc = self.L.l1_clutter_host(self.h, 4, n, _dp(sc), _fp(pose7), _fp(joints), joints.shape[1], _ip(jadr), int(base_qposadr), _dp(cc),
                                        C.byref(cfg), _u8(out), _ip(steps))
        self._check(rc)
        return out.astype(bool), steps

    def _clutter_scenes(self, mode, scenes, scene_index, pose7, joints, joint_qposadr, base_qposadr, close_ctrl, cfg, enough_stable):
        pose7, joints, jadr = self._prep(pose7, joints, joint_qposadr)
        n = len(pose7)
        sc = np.ascontiguousarray(scenes, dtype=np.float64).reshape(-1, self.info.state_stride)
        si = np.ascontiguousarray(scene_index, dtype=np.int32).reshape(-1)
        if len(si) != n:
            raise ValueError(f"scene_index has {len(si)} entries for {n} candidates")
        out = np.zeros(n, dtype=np.uint8)
        steps = np.zeros(n, dtype=np.int32)
        self._order = None
        if n == 0:
            return out.astype(bool), steps
        # round-robin across scenes, each scene's candidates in their own order: the device early stop is exact for that order
        # and wastes only the candidates of a scene that are in flight when its count is reached
        order = shard.scene_round_robin(si)
        p7, jj, so = np.ascontiguousarray(pose7[order]), np.ascontiguousarray(joints[order]), np.ascontiguousarray(si[order])
        lab, st = np.zeros(n, dtype=np.uint8), np.zeros(n, dtype=np.int32)
        cc = np.ascontiguousarray(close_ctrl if close_ctrl is not None else np.zeros(max(1, self.model.nu)), dtype=np.float64)
        cfgp = C.byref(cfg) if cfg is not None else None
        es = int(enough_stable or 0)
        if self.p == "mgs_":
            if mode == 3:
                rc = self.L.mgs_clutter_scenes_collision_mask(self.h, n, len(sc), _dp(sc), _ip(so), _fp(p7), _fp(jj), jj.shape[1], _ip(jadr),
                                                              int(base_qposadr), _u8(lab))
            else:
                rc = self.L.mgs_clutter_scenes_stable_mask(self.h, n, len(sc), _dp(sc), _ip(so), _fp(p7), _fp(jj), jj.shape[1], _ip(jadr),
                                                           int(base_qposadr), es, _dp(cc), cfgp, _u8(lab), _ip(st))
        else:
            rc = self.L.l1_clutter_scenes_host(self.h, mode, n, len(sc), _dp(sc), _ip(so), es if mode == 4 else 0, _fp(p7), _fp(jj),
                                               jj.shape[1], _ip(jadr), int(base_qposadr), _dp(cc), cfgp, _u8(lab), _ip(st))
        self._check(rc)
        self._order = order
        out[order], steps[order] = lab, st
        return out.astype(bool), steps

    def clutter_scenes_collision_mask(self, scenes, scene_index, pose7, joints, joint_qposadr, base_qposadr):
        """clutter_collision_mask over several scenes of this model in one launch: `scenes` [nscene][state_stride] records, candidate i
        starts from scenes[scene_index[i]]."""
        return self._clutter_scenes(3, scenes, scene_index, pose7, joints, joint_qposadr, base_qposadr, None, None, 0)[0]

    def clutter_scenes_stable_mask(self, scenes, scene_index, pose7, joints, joint_qposadr, base_qposadr, close_ctrl, cfg: MgsRolloutCfg,
                                   enough_stable: int = 0):
        """clutter_stable_mask over several scenes in one launch -> (labels bool[n], steps int32[n]).  enough_stable > 0: a candidate
        whose scene already had that many non-overflowed successes when it was pulled is not simulated (label False, last_aux
        `skipped`); the per-scene prefix rule (shard.apply_enough_stable) is left to the caller."""
        return self._clutter_scenes(4, scenes, scene_index, pose7, joints, joint_qposadr, base_qposadr, close_ctrl, cfg, enough_stable)

    def last_aux(self, n: int):
        """Per-candidate auxiliary results of the most recent launch: dict(overflow bool[n], bad bool[n], skipped bool[n],
        pos_drift f32[n], rot_drift_deg f32[n]) - see mgs_last_aux in include/mgs_b200.h.  After a multi-scene call they are in
        the caller's candidate order."""
        a = np.zeros((n, 4), dtype=np.float32)
        if n:
            self._check(self._f("last_aux")(self.h, n, _fp(a)))
        if self._order is not None and len(self._order) == n:
            b = np.empty_like(a)
            b[self._order] = a
            a = b
        fl = a[:, 0].astype(np.int32)
        return dict(overflow=(fl & 1).astype(bool), bad=(fl & 2).astype(bool), skipped=(fl & 4).astype(bool), pos_drift=a[:, 1].copy(),
                    rot_drift_deg=a[:, 2].copy())

    def set_qvel_clip(self, clip: float):
        """step(): clamp qvel to +-clip before every step (scene generation); 0 = off."""
        self._check(self._f("set_qvel_clip")(self.h, float(clip)))

    def overflow_count(self) -> int:
        """Environments of the last launch that dropped contacts (capacity too small)."""
        rc = self.L.mgs_overflow_count(self.h)
        if rc < 0:
            self._check(rc)
        return rc

    def rollout_device(self, mode, n, d_pose7_ptr, d_joints_ptr, nj, joint_qposadr, base_qposadr, close_ctrl, cfg, d_labels_ptr,
                       d_steps_ptr, stream_ptr=0):
        """Device-pointer variant (torch tensors' .data_ptr()); asynchronous on `stream_ptr`."""
        jadr = np.ascontiguousarray(joint_qposadr, dtype=np.int32)
        cc = np.ascontiguousarray(close_ctrl if close_ctrl is not None else np.zeros(max(1, self.model.nu)), dtype=np.float64)
        self._order = None
        self._check(self.L.mgs_rollout_device(self.h, mode, n, d_pose7_ptr, d_joints_ptr, nj, _ip(jadr), int(base_qposadr), _dp(cc),
                                              C.byref(cfg) if cfg is not None else None, d_labels_ptr, d_steps_ptr, stream_ptr))


def antipodal_hits(p1, dirs, tri, eps, pick_u, device: int = 0):
    """mgs_antipodal_hits (include/mgs_b200.h): (signed distance along dirs of the chosen hit [n] (NaN: none), number of valid hits [n])."""
    L = load()
    p1, dirs, tri, pick_u = (np.ascontiguousarray(a, dtype=np.float64) for a in (p1, dirs, tri, pick_u))
    n = len(p1)
    t, nv = np.full(n, np.nan), np.zeros(n, dtype=np.int32)
    if n and L.mgs_antipodal_hits(device, n, _dp(p1), _dp(dirs), len(tri), _dp(tri), float(eps), _dp(pick_u), _dp(t), _ip(nv)) != 0:
        raise MgsError(L.mgs_last_error().decode())
    return t, nv
