"""gen_scene - clutter scene generation + per-scene grasp filtering (/root/reference/mgs/cli/gen_scene.py:28-208).

  gen_stable_scene  drop/settle the objects (ClutterTableEnv.gen_clutter), refuse unstable scenes (ValueError, :42-43)
  filter_grasps     per-object stable grasps -> world frame (o2w @ grasp, :58-60) -> batched collision mask ->
                    batched close+lift rollout with enough_stable = min(128, num_objects * 32) (:115-121)
  run               writes <MGS_OUTPUT_DIR>/<gripper name>/<hash>/scene.npz {scene_definition: pickled dict} and one
                    <object id>_<object name>.npz {pose, joints} per object (:178-205)
  filter_grasps_scenes / run_batch   the same for many scenes of one gripper and object set: scenes generated in one batch of
                    launches, one collision launch and one stable launch for all scenes (beyond the reference, which makes one
                    scene per process)

Per-object grasps come from <MGS_INPUT_DIR>/<gripper name>/<object id>/stable_grasps.npz as in the reference
(:15-25), or are passed in memory (`grasps={object_id: (pose[N,4,4], joints[N,nj])}`).

  python -m mj_grasp_sim_b200.mgs.cli.gen_scene gripper=PandaGripper objects=hull:0,hull:1,hull:2 [seed=0 | seeds=0,1,2,...]
"""
import os
from copy import deepcopy

import numpy as np

from ..env.selector import get_env, get_env_from_dict
from ..gripper.selector import get_gripper
from ..obj.selector import get_objects
from ..util.file import generate_unique_hash
from ..util.geo.transforms import SE3Pose
from ._common import parse_kv


def get_grasps(gripper_name, obj_id):
    g = np.load(os.path.join(os.getenv("MGS_INPUT_DIR"), gripper_name, obj_id, "stable_grasps.npz"))
    return g["pose"], g["joints"]


def _parked_env(gripper_name, object_ids, env_name):
    objs = get_objects(object_ids)
    gripper = get_gripper(gripper_name, default_pose=SE3Pose(np.array([5.0, 5.0, 1.0]), np.array([1.0, 0.0, 0.0, 0.0]), type="wxyz"))
    env = get_env(env_name, deepcopy(gripper), deepcopy(objs))
    env.set_gripper_pose(np.array([5.0, 5.0, 1.0]))
    return env


def gen_stable_scene(gripper_name, object_ids, env_name="clutter_table", seed=None):
    env = _parked_env(gripper_name, object_ids, env_name)
    env.gen_clutter(seed)
    scene_dict = env.to_dict()
    if not env.is_stable():
        raise ValueError("Scene unstable")
    return scene_dict


class GraspTable:
    """Column store of world-frame grasp candidates of one scene: pose[N,4,4], joints[N,nj] and, per row, the index of the
    object the grasp was generated for (`owner`, into `objects` = [(name, id), ...])."""

    def __init__(self, pose, joints, owner, objects):
        self.pose, self.joints, self.owner, self.objects = pose, joints, owner, objects

    @classmethod
    def from_scene(cls, env, source):
        """`source(object_id) -> (pose[N,4,4] in the object frame, joints[N,nj])`; rows are moved to the world frame with the
        object's settled pose (gen_scene.py:58-60).  Objects without candidates do not get an owner slot."""
        cols, objects = ([], [], []), []
        for name, oid in zip(env.object_names, env.object_ids):
            pose, joints = source(oid)
            if len(pose) == 0:
                continue
            cols[0].append((env.get_obj_pose(name) @ SE3Pose.from_mat(np.array(pose, copy=True))).to_mat())
            cols[1].append(np.asarray(joints))
            cols[2].append(np.full(len(pose), len(objects), dtype=np.int32))
            objects.append((name, oid))
        if not objects:
            raise ValueError("No collision free grasps")
        return cls(*(np.concatenate(c) for c in cols), objects)

    def __len__(self):
        return len(self.pose)

    def take(self, sel, move_owner=True):
        """rows `sel` (mask or index array).  move_owner=False leaves the owner column in its old order - only meaningful for
        a permutation, see `filter_grasps(reference_index_quirk=True)`."""
        return GraspTable(self.pose[sel], self.joints[sel], self.owner[sel] if move_owner else self.owner, self.objects)

    def se3(self):
        return SE3Pose.from_mat(np.array(self.pose, copy=True), type="wxyz")

    def per_object(self):
        for k in np.unique(self.owner):
            rows = self.owner == k
            name, oid = self.objects[k]
            yield k, {"object_id": oid, "object_name": name, "pose": self.pose[rows], "joints": self.joints[rows]}


def filter_grasps(gripper_name, scene_def, env_name="clutter_table", grasps=None, only_collision_free=False, save_collision_grasps=False,
                  enough_collision_free=128, rng=None, reference_index_quirk=False):
    """Per-scene filtering (gen_scene.py:48-172): collision mask over every object's candidates, then (unless
    `only_collision_free`) the close+lift rollout on a random permutation of the survivors with
    enough_stable = min(128, 32 * num_objects).  Returns (per-object survivors, per-object colliding candidates).

    Known reference defect, NOT reproduced by default: the reference permutes poses and joints but its statement for the
    object-index column is a comparison, not an assignment (gen_scene.py:113), so stable grasps are filed under the object
    whose row they landed on after the shuffle.  `reference_index_quirk=True` reproduces that attribution bit for bit."""
    env = get_env_from_dict(env_name, deepcopy(scene_def))
    table = GraspTable.from_scene(env, (lambda oid: grasps[oid]) if grasps is not None else (lambda oid: get_grasps(gripper_name, oid)))
    free = np.asarray(env.grasp_collision_mask(table.se3(), np.array(table.joints, copy=True)), dtype=bool)
    if int(free.sum()) < enough_collision_free:
        raise ValueError("Not enough collision free grasps!")
    keep, colliding = table.take(free), table.take(~free)
    if not only_collision_free:
        keep = keep.take((rng or np.random.default_rng()).permutation(len(keep)), move_owner=not reference_index_quirk)
        want = min(128, 32 * len(env.object_names))
        stable = np.asarray(env.grasp_stable_mask(keep.se3(), np.array(keep.joints, copy=True), deepcopy(scene_def["env_state"]["state"]),
                                                  enough_stable=want), dtype=bool)
        if int(stable.sum()) < want:
            raise ValueError("Not enough stable grasps!")
        keep = keep.take(stable)
    return _split(keep, colliding, save_collision_grasps)


def _split(keep, colliding, save_collision_grasps):
    valid, invalid = [], []
    rejected = dict(colliding.per_object()) if save_collision_grasps else {}
    for k, entry in keep.per_object():
        valid.append(entry)
        if k in rejected:  # only objects that kept at least one grasp get a "_collision" file (:150-160)
            invalid.append(rejected[k])
    return valid, invalid


_SHARED_MASKS = ("geom_contype", "geom_conaffinity", "body_gravcomp")


def _concat(tables, keys):
    """(rows of tables[k] for k in keys, back to back, as one GraspTable; scene index of every row)"""
    t = GraspTable(np.concatenate([tables[k].pose for k in keys]), np.concatenate([tables[k].joints for k in keys]), None, None)
    return t, np.concatenate([np.full(len(tables[k]), k, dtype=np.int64) for k in keys])


def filter_grasps_scenes(gripper_name, scene_defs, env_name="clutter_table", grasps=None, only_collision_free=False, save_collision_grasps=False,
                         enough_collision_free=128, rng=None, reference_index_quirk=False):
    """filter_grasps for many scenes of ONE model (same gripper, object ids, geom masks and gravcomp; ValueError otherwise): one
    collision launch and one stable launch serve all scenes.  Returns, per scene, the (valid, invalid) pair of filter_grasps or the
    ValueError it would have raised.  The result equals successive filter_grasps calls sharing one generator `rng`: each accepted
    scene draws its permutation in scene order, and scenes rejected for too few collision-free grasps draw nothing."""
    if not scene_defs:
        return []
    ref = scene_defs[0]
    model_key = lambda d: (type(d["gripper"]).__name__, [o.object_id for o in d["objects"]])
    for d in scene_defs[1:]:
        if model_key(d) != model_key(ref) or any(not np.array_equal(np.asarray(d["env_state"][k]), np.asarray(ref["env_state"][k]))
                                                 for k in _SHARED_MASKS):
            raise ValueError("the scenes of one call must share one model: gripper, object ids, geom masks and gravcomp")
    env = get_env_from_dict(env_name, deepcopy(ref))
    source = (lambda oid: grasps[oid]) if grasps is not None else (lambda oid: get_grasps(gripper_name, oid))
    states = [np.asarray(d["env_state"]["state"], dtype=np.float64) for d in scene_defs]
    out, tables = [None] * len(scene_defs), {}
    for k in range(len(scene_defs)):
        env.set_state(states[k])
        try:
            tables[k] = GraspTable.from_scene(env, source)
        except ValueError as e:
            out[k] = e
    if tables:
        allt, si = _concat(tables, list(tables))
        free = np.asarray(env.grasp_collision_mask_scenes(allt.se3(), np.array(allt.joints, copy=True), si, states), dtype=bool)
    rng = rng or np.random.default_rng()
    keep, colliding = {}, {}
    for k, t in tables.items():
        f = free[si == k]
        if int(f.sum()) < enough_collision_free:
            out[k] = ValueError("Not enough collision free grasps!")
            continue
        keep[k], colliding[k] = t.take(f), t.take(~f)
        if not only_collision_free:
            keep[k] = keep[k].take(rng.permutation(len(keep[k])), move_owner=not reference_index_quirk)
    if keep and not only_collision_free:
        want = min(128, 32 * len(env.object_names))
        allk, si = _concat(keep, list(keep))
        stable = np.asarray(env.grasp_stable_mask_scenes(allk.se3(), np.array(allk.joints, copy=True), si, states, enough_stable=want), dtype=bool)
        for k in list(keep):
            st = stable[si == k]
            if int(st.sum()) < want:
                out[k] = ValueError("Not enough stable grasps!")
                del keep[k]
            else:
                keep[k] = keep[k].take(st)
    for k in keep:
        out[k] = _split(keep[k], colliding[k], save_collision_grasps)
    return out


def _write(output_dir, scene_dict, valid, invalid):
    os.makedirs(output_dir, exist_ok=True)
    np.savez(os.path.join(output_dir, "scene"), scene_definition=scene_dict)
    for g in valid:
        np.savez(os.path.join(output_dir, g["object_id"] + "_" + g["object_name"]), pose=g["pose"], joints=g["joints"])
    for g in invalid:
        np.savez(os.path.join(output_dir, g["object_id"] + "_" + g["object_name"] + "_collision"), pose=g["pose"], joints=g["joints"])
    return output_dir


def run(gripper_name, object_ids, env_name="clutter_table", seed=None, grasps=None, output_dir=None, **kw):
    output_dir = output_dir or os.getenv("MGS_OUTPUT_DIR")
    assert output_dir is not None, "No ouput_dir defined!"
    output_dir = os.path.join(output_dir, gripper_name, generate_unique_hash(16))
    scene_dict = gen_stable_scene(gripper_name, object_ids, env_name, seed)
    valid, invalid = filter_grasps(gripper_name, scene_dict, env_name, grasps=grasps, **kw)
    return _write(output_dir, scene_dict, valid, invalid)


def run_batch(gripper_name, object_ids, seeds, env_name="clutter_table", grasps=None, output_dir=None, **kw):
    """`run` for every seed: scene k is the scene gen_stable_scene(seed=seeds[k]) makes, generated in one batch of launches, and
    filter_grasps_scenes filters all of them.  Every accepted scene is written as `run` writes it.  Returns, per seed, the output
    directory or the ValueError that `run` would have raised (unstable scene, too few collision-free or stable grasps)."""
    output_dir = output_dir or os.getenv("MGS_OUTPUT_DIR")
    assert output_dir is not None, "No ouput_dir defined!"
    defs = _parked_env(gripper_name, object_ids, env_name).gen_clutter_scenes(list(seeds))
    ok = [k for k, d in enumerate(defs) if d is not None]
    res = filter_grasps_scenes(gripper_name, [defs[k] for k in ok], env_name, grasps=grasps, **kw)
    out = [ValueError("Scene unstable") if d is None else None for d in defs]
    for k, r in zip(ok, res):
        out[k] = r if isinstance(r, Exception) else _write(os.path.join(output_dir, gripper_name, generate_unique_hash(16)), defs[k], *r)
    return out


if __name__ == "__main__":
    kv = parse_kv()
    try:
        if "seeds" in kv:
            for r in run_batch(kv.get("gripper", "PandaGripper"), kv.get("objects", "hull:0,hull:1,hull:2").split(","),
                               [int(x) for x in kv["seeds"].split(",")], kv.get("env", "clutter_table")):
                print(r)
        else:
            print(run(kv.get("gripper", "PandaGripper"), kv.get("objects", "hull:0,hull:1,hull:2").split(","), kv.get("env", "clutter_table"),
                      int(kv["seed"]) if "seed" in kv else None))
    except Exception as e:  # the reference's main swallows and prints (:175-208)
        print(e)
