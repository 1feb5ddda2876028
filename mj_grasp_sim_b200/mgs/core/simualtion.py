"""Sim handle (file name keeps the reference's spelling, /root/reference/mgs/core/simualtion.py).

The reference's MjSimulation wraps one MjModel + MjData and its callers poke `sim.data` directly
(`sim.data.qpos[idxs] = ...`, `sim.data.ctrl[:] = ...`, `sim.data.mocap_pos[0, :] = ...`, then `mujoco.mj_forward`
/ `mujoco.mj_step`).  Here `model` is the compiled flat model and the batched rollouts live on the GPU inside the
C-ABI library; for the imperative protocol the handle keeps ONE host-side state record (qpos | qvel |
qacc_warmstart | ctrl | mocap pose) and exposes it through `data` as writable numpy views, so the same statements
work.  `mj_forward()` / `mj_step(nstep)` run that single environment through the same sm_100a kernel
(`mgs_step_host`, a one-candidate launch): drop-in semantics, not the fast path - the batched entry points of the
environments are.

Methods of the reference class (simualtion.py:30-61): get_joint_idxs (with the unknown-name quirk: `mj_name2id`
returns -1 and `jnt_qposadr[-1]` is the LAST joint's address - hit by Robotiq's two misnamed joints), set_qpos,
get_state / set_state in MuJoCo's mjSTATE_INTEGRATION layout, idle (viewer loop: not available headless)."""
from __future__ import annotations

from typing import List

import numpy as np

from ...lib import BatchSim  # module-level name on purpose: the CPU test tier swaps it for the 1-lane host build


class _Contacts:
    def __init__(self, geom):
        self.geom = geom  # int [ncon, 2] geom ids, like mjData.contact.geom


class SimData:
    """The mjData fields the reference's grasp path touches, as views into the handle's state record."""

    def __init__(self, sim):
        object.__setattr__(self, "_sim", sim)

    def _sl(self, name):
        m = self._sim.model
        nq, nv, nu = m.nq, m.nv, m.nu
        o = {"qpos": (0, nq), "qvel": (nq, nq + nv), "qacc_warmstart": (nq + nv, nq + 2 * nv), "ctrl": (nq + 2 * nv, nq + 2 * nv + nu),
             "mocap_pos": (nq + 2 * nv + nu, nq + 2 * nv + nu + 3), "mocap_quat": (nq + 2 * nv + nu + 3, nq + 2 * nv + nu + 7)}[name]
        return slice(*o)

    def __getattr__(self, name):
        sim = object.__getattribute__(self, "_sim")
        if name in ("qpos", "qvel", "qacc_warmstart", "ctrl"):
            sim._touch()
            return sim._record[self._sl(name)]
        if name == "mocap_pos":
            sim._touch()
            return sim._record[self._sl(name)].reshape(1, 3)
        if name == "mocap_quat":
            sim._touch()
            return sim._record[self._sl(name)].reshape(1, 4)
        if name == "time":
            return sim._time
        if name == "ncon":
            return len(sim._contact_geoms())
        if name == "contact":
            return _Contacts(sim._contact_geoms())
        raise AttributeError(name)

    def __setattr__(self, name, value):
        # `sim.data.mocap_pos = np.copy(pose.pos)` (robotiq2f85.py:241-242, shadow.py:380-381) rebinds in MuJoCo's bindings = a copy
        if name in ("qpos", "qvel", "qacc_warmstart", "ctrl", "mocap_pos", "mocap_quat"):
            self._sim._touch()
            self._sim._record[self._sl(name)] = np.asarray(value, dtype=np.float64).reshape(-1)
        elif name == "time":
            self._sim._time = float(value)
        else:
            raise AttributeError(name)


class MjSimulation:
    model = None
    GROUND_GEOM = "geom:ground"
    _sim = None
    _device = None
    _caps = (0, 0)
    gripper = None
    # True: a model whose environment state does not fit one CTA's shared memory keeps that state in global memory (kernel variant
    # wide_g) instead of failing at creation (BatchSim(global_fallback=True)).  Set by ClutterTableEnv, whose fp64 Shadow-hand scenes
    # and escalation capacities need it.
    GLOBAL_STATE_FALLBACK = False

    def _sim_kwargs(self) -> dict:
        # passed only when set, so that a BatchSim stand-in without the argument keeps working for the other environments
        return {"global_fallback": True} if self.GLOBAL_STATE_FALLBACK else {}

    @property
    def compute_f64(self) -> bool:
        """Precision policy of the batched kernel for this environment (gripper.COMPUTE_F64; MGS_PRECISION overrides)."""
        import os
        force = os.environ.get("MGS_PRECISION", "").lower()
        if force in ("f32", "f64"):
            return force == "f64"
        return bool(getattr(self.gripper, "COMPUTE_F64", False))

    # ---- the batched simulator is created on first use (needs a CUDA device; there is no CPU fallback)
    @property
    def sim(self):
        if self._sim is None:
            dev = self._device
            if dev is None:
                import torch
                dev = torch.cuda.current_device() if torch.cuda.is_available() else 0
            self._sim = BatchSim(self.model, device=dev, ncon_max=self._caps[0], nefc_max=self._caps[1], ground_name=self.GROUND_GEOM,
                                 f64=self.compute_f64, **self._sim_kwargs())
        return self._sim

    # ---- single-environment state -------------------------------------------------------------
    def _init_state(self):
        from ... import scenes
        self._record = scenes.record_from_model(self.model)
        self._time = 0.0
        self._diag = None

    def _touch(self):
        self._diag = None  # derived quantities (contacts) are stale until the next forward

    @property
    def data(self) -> SimData:
        return SimData(self)

    def mj_resetData(self):
        self._init_state()

    def _run(self, nstep: int):
        out, diag = self.sim.step(self._record[None].astype(self.sim.real), nstep, want_diag=True)
        self._record = out[0].astype(np.float64)  # nstep = 0 (mj_forward) moves only qacc_warmstart, as mj_fwdConstraint does
        self._time += nstep * float(self.model.opt["timestep"])
        self._diag = diag

    def mj_forward(self):
        """mujoco.mj_forward(sim.model, sim.data) on the handle's environment."""
        self._run(0)

    def mj_step(self, nstep: int = 1):
        """mujoco.mj_step(sim.model, sim.data, nstep)."""
        self._run(int(nstep))
        # contacts of mjData after mj_step are those of the LAST forward pass inside the step, which is what the diag holds

    def _contact_geoms(self):
        if self._diag is None:
            self.mj_forward()
        d, ar = self._diag, self.model.arr
        n = int(d["ncon"][0])
        pair = d["contact"][0, :n, 4].astype(np.int64)
        g1 = np.asarray(ar["cgeom_geomid"])[np.asarray(ar["pair_geom1"])[pair]]
        g2 = np.asarray(ar["cgeom_geomid"])[np.asarray(ar["pair_geom2"])[pair]]
        return np.stack([g1, g2], axis=1).astype(np.int32).reshape(n, 2)

    # ---- reference methods ----------------------------------------------------------------------
    def idle(self):
        raise NotImplementedError("MjSimulation.idle opens the interactive MuJoCo viewer (simualtion.py:30-35); there is no viewer on the batched path")

    def get_joint_idxs(self, joint_list: List[str]) -> List[int]:
        out = []
        for j in joint_list:
            jid = self.model.names["joint"].get(j, -1)
            out.append(int(self.model.jnt_qposadr[jid]))
        return out

    def set_qpos(self, qpos: np.ndarray, idxs: List[int]):
        assert idxs is not None
        self.data.qpos[np.asarray(idxs, dtype=np.int64)] = qpos  # sequential scatter: a repeated address keeps the last value
        self.mj_forward()

    # mjSTATE_INTEGRATION = time | qpos | qvel | act | qacc_warmstart (history) | ctrl | qfrc_applied | xfrc_applied | eq_active |
    # mocap_pos | mocap_quat (+ userdata, plugin state: empty here)
    def _layout(self):
        m = self.model
        nq, nv, nu, nb, neq = m.nq, m.nv, m.nu, m.nbody, int(m.arr["neq"])
        nmocap = int(m.arr["nmocap"])
        o_qpos, o_qvel = 1, 1 + nq
        o_ws = o_qvel + nv  # act is empty
        o_ctrl = o_ws + nv
        o_applied = o_ctrl + nu
        o_xfrc = o_applied + nv
        o_eq = o_xfrc + 6 * nb
        o_mpos = o_eq + neq
        return dict(qpos=o_qpos, qvel=o_qvel, ws=o_ws, ctrl=o_ctrl, eq=o_eq, mpos=o_mpos, size=o_mpos + 7 * nmocap)

    def get_state(self) -> np.ndarray:
        m, L = self.model, self._layout()
        nq, nv, nu = m.nq, m.nv, m.nu
        st = np.zeros(L["size"])
        st[0] = self._time
        r = self._record
        st[L["qpos"]:L["qpos"] + nq] = r[:nq]
        st[L["qvel"]:L["qvel"] + nv] = r[nq:nq + nv]
        st[L["ws"]:L["ws"] + nv] = r[nq + nv:nq + 2 * nv]
        st[L["ctrl"]:L["ctrl"] + nu] = r[nq + 2 * nv:nq + 2 * nv + nu]
        st[L["eq"]:L["eq"] + int(m.arr["neq"])] = 1.0
        st[L["mpos"]:] = r[nq + 2 * nv + nu:]
        return st

    def _record_from_state(self, state) -> np.ndarray:
        m, L = self.model, self._layout()
        nq, nv, nu = m.nq, m.nv, m.nu
        state = np.asarray(state, dtype=np.float64)
        if state.shape != (L["size"],):
            raise ValueError(f"state has {state.shape} entries, mjSTATE_INTEGRATION of this model has {L['size']}")
        return np.concatenate([state[L["qpos"]:L["qpos"] + nq], state[L["qvel"]:L["qvel"] + nv], state[L["ws"]:L["ws"] + nv],
                               state[L["ctrl"]:L["ctrl"] + nu], state[L["mpos"]:]])

    def set_state(self, state):
        self._record = self._record_from_state(state)
        self._time = float(np.asarray(state)[0])
        self._touch()  # the reference follows with mj_forward (simualtion.py:58-61): derived quantities are recomputed on demand
