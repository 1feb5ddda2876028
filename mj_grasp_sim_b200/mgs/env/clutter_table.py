"""ClutterTableEnv - drop-in for the grasp-evaluation part of /root/reference/mgs/env/clutter_table.py.

Same constructor and the same evaluation methods:
  grasp_collision_mask(poses, joints) -> bool[N]                                        (reference :330-367)
  grasp_stable_mask(poses, joints, env_state, nstep_lift, lift_dist, enough_stable)     (reference :272-321)
plus get_state / set_state in MuJoCo's mjSTATE_INTEGRATION layout (core/simualtion.py:51-61), gen_clutter /
settle / is_stable (:157-222, run as single-environment launches of the same kernel) and to_dict / from_dict
(:369-399).  Rendering (MjScanEnv) is out of scope.  All candidates of a call run in one batched launch.
"""
from __future__ import annotations

from copy import deepcopy

import numpy as np

from ... import scenes
from ...compiler.mjcf import compile_mjcf
from ...lib import BatchSim, MgsRolloutCfg
from ...shard import apply_enough_stable, evaluate_sharded
from ..core.simualtion import MjSimulation
from .gravityless_object_grasping import EscalatingSim
from ..util.geo.transforms import SE3Pose

XML = scenes.CLUTTER_XML  # same options / body order as the reference template (:41-79), lights and camera element dropped


class ClutterTableEnv(MjSimulation):
    def __init__(self, gripper, objects, scene_randomization=True, device: int | None = None, ncon_max: int = 0, nefc_max: int = 0):
        self.gripper, self.objects = gripper, objects
        self.gripper_xml, self.gripper_assets = gripper.to_xml()
        self.object_names = [o.name for o in objects]
        self.object_ids = [o.object_id for o in objects]
        self.objs_xml_concat, self.objs_assets = "", {}
        for o in objects:
            x, a = o.to_xml()
            self.objs_xml_concat += x
            self.objs_assets.update(a)
        self.model_xml = XML.format(gripper=self.gripper_xml, objects=self.objs_xml_concat)
        self.env_defintion = {"model_xml": self.model_xml, "assets": {**self.gripper_assets, **self.objs_assets}}
        self.model = compile_mjcf(self.model_xml, self.env_defintion["assets"])
        self._device, self._caps, self._sim = device, (ncon_max, nefc_max), None
        self._esc = EscalatingSim(self._make_sim)
        self._init_state()

    GROUND_GEOM = "geom:table"
    # the fp64 Shadow hand over four or more objects, and the 256-contact escalation rung of every clutter scene, do not fit one
    # CTA's shared memory: those models keep their environment state in global memory
    GLOBAL_STATE_FALLBACK = True

    def _make_sim(self, caps):
        if caps is None:
            return self.sim
        return BatchSim(self.model, device=self.sim.device, ncon_max=caps[0], nefc_max=caps[1], ground_name=self.GROUND_GEOM,
                        f64=self.compute_f64, **self._sim_kwargs())

    @property
    def last_overflow(self):
        return self._esc.last_overflow

    # ---- scene generation (single-environment launches) -------------------------------------
    def _step(self, rec, nstep):
        out = self.sim.step(rec[None].astype(self.sim.real), nstep)
        self._time += nstep * float(self.model.opt["timestep"])
        self._diag = None
        return out[0].astype(np.float64)

    def set_gripper_pose(self, pos):
        """park the gripper (what gen_scene does through gripper.set_pose before generating the clutter)"""
        m = self.model
        b = self.gripper.get_freejoint_idxs(self)[0]
        mo = m.nq + 2 * m.nv + m.nu
        self._record[b:b + 3] = pos
        self._record[mo:mo + 3] = pos

    def gen_clutter(self, seed: int | None = None):
        info = dict(base_qposadr=self.gripper.get_freejoint_idxs(self)[0],
                    object_qposadr=[int(self.model.jnt_qposadr[self.model.names["joint"][f"{n}:joint"]]) for n in self.object_names])
        sd = int(np.random.randint(1 << 30)) if seed is None else seed
        self.sim.set_qvel_clip(50.0)  # the reference clamps qvel before EVERY step of the drop / settle phases (:215-221)
        try:
            self._record = scenes.gen_clutter(self.model, info, self._step, sd)
        finally:
            self.sim.set_qvel_clip(0.0)

    def gen_clutter_batch(self, seeds, require_stable: bool = True):
        """Beyond the reference (which generates one scene per process, gen_scene.py:28-45): generate len(seeds) scenes
        of this gripper/object set in one batch of launches.  Returns a list of `to_dict()`-style scene dictionaries
        (only the stable ones when `require_stable`)."""
        info = dict(base_qposadr=self.gripper.get_freejoint_idxs(self)[0],
                    object_qposadr=[int(self.model.jnt_qposadr[self.model.names["joint"][f"{n}:joint"]]) for n in self.object_names])
        step = lambda r, k: self.sim.step(r.astype(self.sim.real), k).astype(np.float64)
        self.sim.set_qvel_clip(50.0)
        try:
            recs = scenes.gen_clutter_batch(self.model, info, step, seeds)
        finally:
            self.sim.set_qvel_clip(0.0)
        ok, after = scenes.scenes_stable(self.model, info, step, recs.copy())
        out, keep_rec, keep_time = [], self._record, self._time
        for k in range(len(recs)):
            if require_stable and not ok[k]:
                continue
            self._record, self._time = recs[k], 11.7
            out.append(self.to_dict())
        self._record, self._time = keep_rec, keep_time
        return out

    def gen_clutter_scenes(self, seeds):
        """Scene k = what gen_clutter(seeds[k]) followed by to_dict() makes on this environment (state time included), for all
        seeds in one batch of launches; None where is_stable() would then be False."""
        info = dict(base_qposadr=self.gripper.get_freejoint_idxs(self)[0],
                    object_qposadr=[int(self.model.jnt_qposadr[self.model.names["joint"][f"{n}:joint"]]) for n in self.object_names])
        step = lambda r, k: self.sim.step(r.astype(self.sim.real), k).astype(np.float64)
        self.sim.set_qvel_clip(50.0)
        try:
            recs = scenes.gen_clutter_batch(self.model, info, step, seeds)
        finally:
            self.sim.set_qvel_clip(0.0)
        ok, _ = scenes.scenes_stable(self.model, info, step, recs.copy())
        t = self._time
        for _ in range(9 * len(self.object_names) + 90):  # gen_clutter advances the time in steps of 100 (_step)
            t += 100 * float(self.model.opt["timestep"])
        out, keep_rec, keep_time = [], self._record, self._time
        for k in range(len(recs)):
            self._record, self._time = recs[k], t
            out.append(self.to_dict() if ok[k] else None)
        self._record, self._time = keep_rec, keep_time
        return out

    def settle(self):
        self._record = self._step(self._record, 10000)

    def is_stable(self):
        adr = [int(self.model.jnt_qposadr[self.model.names["joint"][f"{n}:joint"]]) for n in self.object_names]
        stats = np.zeros(len(adr))
        for _ in range(10):
            start = np.array([self._record[a:a + 3] for a in adr])
            self._record = self._step(self._record, 100)
            stats += np.abs(np.array([self._record[a:a + 3] for a in adr]) - start).sum(axis=1)
        return bool(stats.max() < 5e-3) if len(adr) else True

    def get_object(self, object_name: str):
        for obj in self.objects:
            if obj.name == object_name:
                return obj
        return None

    def _disable_bodies(self, body_ids):
        """What the reference does by zeroing geom_contype / geom_conaffinity and setting body_gravcomp = 1 on the live
        mjModel (remove_obj, :146-155): on the compiled model the candidate-pair list loses every pair that involves a
        geom of those bodies, the masks are zeroed and gravity compensation is switched on; the device copy of the model is
        rebuilt on next use."""
        ar = self.model.arr
        body_ids = set(int(b) for b in body_ids)
        if not body_ids:
            return
        gone_c = np.array([int(b) in body_ids for b in ar["cgeom_bodyid"]])
        keep = ~(gone_c[ar["pair_geom1"]] | gone_c[ar["pair_geom2"]])
        for k in ("pair_geom1", "pair_geom2", "pair_condim", "pair_friction", "pair_solref", "pair_solimp", "pair_margin", "pair_gap"):
            ar[k] = ar[k][keep]
        ar["npair"] = int(keep.sum())
        for g in np.nonzero(np.isin(ar["geom_bodyid"], list(body_ids)))[0]:
            ar["geom_contype"][g] = 0
            ar["geom_conaffinity"][g] = 0
        for b in body_ids:
            ar["body_gravcomp"][b] = 1.0
        self._esc.close()
        if self._sim is not None:
            self._sim.close()
            self._sim = None

    def remove_obj(self, obj):
        """ClutterTableEnv.remove_obj (reference :146-155): the object stops colliding and floats where it is."""
        self._disable_bodies([self.model.names["body"][obj.name]])

    def get_obj_pose(self, object_name: str) -> SE3Pose:
        """object free-joint pose in the world (reference :323-328)"""
        a = int(self.model.jnt_qposadr[self.model.names["joint"][f"{object_name}:joint"]])
        return SE3Pose(np.copy(self._record[a:a + 3]), np.copy(self._record[a + 3:a + 7]), "wxyz")

    # ---- grasp evaluation ---------------------------------------------------------------------
    def _process(self, poses: SE3Pose, joints):
        names = self.gripper.get_actuator_joint_names()
        joints = np.asarray(joints)
        if len(poses) != len(joints):
            raise ValueError(f"Number of poses ({len(poses)}) must match number of joint configurations ({len(joints)}).")
        processed = poses @ self.gripper.base_to_contact_transform()
        pose7 = processed.to_vec(layout="pq", type="wxyz").astype(np.float32).reshape(-1, 7)
        return pose7, joints.astype(np.float32).reshape(len(pose7), len(names)), np.array(self.get_joint_idxs(names), dtype=np.int32)

    def grasp_collision_mask(self, poses: SE3Pose, joints: np.ndarray):
        pose7, j32, jadr = self._process(poses, joints)
        p = np.asarray(poses.pos).reshape(-1, 3)
        in_bound = (p[:, 0] < 0.25) & (p[:, 0] > -0.25) & (p[:, 1] < 0.25) & (p[:, 1] > -0.25) & (p[:, 2] < 1.0) & (p[:, 2] > 0.0)  # :344-354
        out = np.zeros(len(pose7), dtype=bool)
        idx = np.nonzero(in_bound)[0]
        base = self.gripper.get_freejoint_idxs(self)[0]
        if len(idx):
            p7, jj, rec = pose7[idx], j32[idx], self._record

            def run_range(lo, hi):
                sel = lambda k: (p7[lo:hi], jj[lo:hi]) if k is None else (p7[lo:hi][k], jj[lo:hi][k])
                return self._esc.run(lambda sim, k: sim.clutter_collision_mask(rec, *sel(k), jadr, base), hi - lo)[0]
            out[idx] = evaluate_sharded(len(idx), run_range)
        return out

    def grasp_stable_mask(self, poses: SE3Pose, joints: np.ndarray, env_state, nstep_lift: int = 3000, lift_dist: float = 0.3, enough_stable=None):
        pose7, j32, jadr = self._process(poses, joints)
        scene = self._record_from_state(env_state)
        base = self.gripper.get_freejoint_idxs(self)[0]
        cfg = MgsRolloutCfg(self.gripper.NSTEP_CLOSE, nstep_lift, 0, self.gripper.REPOSE_ON_CLOSE, lift_dist, 0.0)
        ctrl = self.gripper.close_ctrl()

        def run_range(lo, hi):
            sel = lambda k: (pose7[lo:hi], j32[lo:hi]) if k is None else (pose7[lo:hi][k], j32[lo:hi][k])
            return self._esc.run(lambda sim, k: sim.clutter_stable_mask(scene, *sel(k), jadr, base, ctrl, cfg), hi - lo)[0][0]
        # enough_stable as the reference's early stop (:293-296), in rounds of one GPU-filling chunk per rank
        info = self.sim.info
        return evaluate_sharded(len(pose7), run_range, enough_stable, chunk=info.warps_per_block * info.blocks_per_sm * info.num_sms)

    # ---- many scenes of this model in one launch ----------------------------------------------------
    def _scene_records(self, env_states):
        return np.stack([self._record_from_state(s) for s in env_states]) if len(env_states) else np.zeros((0, self.sim.info.state_stride))

    def grasp_collision_mask_scenes(self, poses: SE3Pose, joints: np.ndarray, scene_index, env_states):
        """grasp_collision_mask for candidates of several scenes of this model (same gripper, objects and masks) in one launch:
        candidate i is tested in the scene env_states[scene_index[i]] (mjSTATE_INTEGRATION vectors).  Equals grasp_collision_mask
        called per scene with that scene's state set."""
        pose7, j32, jadr = self._process(poses, joints)
        si = np.asarray(scene_index, dtype=np.int64).reshape(-1)
        if len(si) != len(pose7):
            raise ValueError(f"scene_index has {len(si)} entries for {len(pose7)} candidates")
        recs = self._scene_records(env_states)
        p = np.asarray(poses.pos).reshape(-1, 3)
        in_bound = (p[:, 0] < 0.25) & (p[:, 0] > -0.25) & (p[:, 1] < 0.25) & (p[:, 1] > -0.25) & (p[:, 2] < 1.0) & (p[:, 2] > 0.0)  # :344-354
        out = np.zeros(len(pose7), dtype=bool)
        idx = np.nonzero(in_bound)[0]
        base = self.gripper.get_freejoint_idxs(self)[0]
        if len(idx):
            p7, jj, s = pose7[idx], j32[idx], si[idx]
            sel = lambda k: (s, p7, jj) if k is None else (s[k], p7[k], jj[k])
            out[idx] = self._esc.run(lambda sim, k: sim.clutter_scenes_collision_mask(recs, *sel(k), jadr, base), len(idx))[0]
        return out

    def grasp_stable_mask_scenes(self, poses: SE3Pose, joints: np.ndarray, scene_index, env_states, nstep_lift: int = 3000, lift_dist: float = 0.3,
                                 enough_stable=None):
        """grasp_stable_mask for candidates of several scenes of this model in one launch; candidate i starts from
        env_states[scene_index[i]], and each scene's candidates are taken in their order here.  `enough_stable` applies per scene,
        as the early stop of the device (include/mgs_b200.h, mgs_clutter_scenes_*): the result equals grasp_stable_mask called once
        per scene with the same enough_stable.  Overflowed candidates are re-run up the capacity ladder without the early stop."""
        pose7, j32, jadr = self._process(poses, joints)
        si = np.asarray(scene_index, dtype=np.int64).reshape(-1)
        if len(si) != len(pose7):
            raise ValueError(f"scene_index has {len(si)} entries for {len(pose7)} candidates")
        recs = self._scene_records(env_states)
        base = self.gripper.get_freejoint_idxs(self)[0]
        cfg = MgsRolloutCfg(self.gripper.NSTEP_CLOSE, nstep_lift, 0, self.gripper.REPOSE_ON_CLOSE, lift_dist, 0.0)
        ctrl = self.gripper.close_ctrl()
        es = int(enough_stable) if enough_stable is not None else 0

        def call(sim, k):
            if k is None:
                return sim.clutter_scenes_stable_mask(recs, si, pose7, j32, jadr, base, ctrl, cfg, enough_stable=es)
            return sim.clutter_scenes_stable_mask(recs, si[k], pose7[k], j32[k], jadr, base, ctrl, cfg, enough_stable=0)
        lab = np.asarray(self._esc.run(call, len(pose7))[0][0], dtype=bool)
        if enough_stable is not None:
            for s in np.unique(si):
                rows = si == s
                lab[rows] = apply_enough_stable(lab[rows], enough_stable)
        return lab

    # ---- persistence (scene.npz payload) --------------------------------------------------------
    def to_dict(self):
        m = self.model
        state = {"geom_conaffinity": deepcopy(m.geom_conaffinity), "geom_contype": deepcopy(m.geom_contype),
                 "geom_rgba": np.ones((int(m.arr["ngeom"]), 4)), "body_gravcomp": deepcopy(m.body_gravcomp), "state": self.get_state()}
        return {"gripper": deepcopy(self.gripper), "objects": deepcopy(self.objects), "env_state": state}

    @classmethod
    def from_dict(cls, state_dict):
        env = cls(state_dict["gripper"], state_dict["objects"], scene_randomization=False)
        env.set_state(state_dict["env_state"]["state"])
        st = state_dict["env_state"]
        # restore edited masks (reference :394-397): bodies whose geoms were switched off (remove_obj) are switched off here too
        off = (np.asarray(st["geom_contype"]) == 0) & (np.asarray(st["geom_conaffinity"]) == 0) & \
              ((env.model.geom_contype != 0) | (env.model.geom_conaffinity != 0))
        other = (np.asarray(st["geom_contype"]) != env.model.geom_contype) | (np.asarray(st["geom_conaffinity"]) != env.model.geom_conaffinity)
        if (other & ~off).any():
            raise NotImplementedError("only masks that switch whole geoms off (remove_obj) can be restored")
        bodies = set(int(b) for b in env.model.geom_bodyid[off])
        for b in bodies:
            if not off[env.model.geom_bodyid == b].all():
                raise NotImplementedError("partially disabled bodies are not supported")
        env._disable_bodies(bodies)
        env.model.arr["body_gravcomp"][:] = np.asarray(st["body_gravcomp"], dtype=np.float64)
        return env
