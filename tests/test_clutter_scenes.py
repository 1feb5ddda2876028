"""Many clutter scenes of one model in one launch (mgs_clutter_scenes_*): the scene index per candidate, the device enough_stable early
stop, the round-robin launch order, scene sharding over ranks, and the ClutterTableEnv / gen_scene layers on top."""
import os
import subprocess
import sys

import numpy as np
import pytest

from hostsim import lane1_scenes
from mj_grasp_sim_b200 import lib as mlib
from mj_grasp_sim_b200 import scenes, shard

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCHED = (500, 300, 0, 0, 0.05, 0.0)    # the short schedule of tests/test_clutter.py
# lift shorter than the first contact test (step 100 of the lift): every candidate that does not blow up is a success, which makes
# the early stop's skipped set known in advance
ALL_SUCCEED = (500, 50, 0, 0, 0.05, 0.0)


def test_scene_round_robin():
    s = np.array([2, 0, 2, 1, 0, 2, 2, 5])
    order = shard.scene_round_robin(s)
    assert sorted(order.tolist()) == list(range(len(s)))
    assert s[order].tolist() == [0, 1, 2, 5, 0, 2, 2, 2]             # round-robin across scenes, scenes in increasing order
    for k in np.unique(s):                                              # each scene keeps its own order
        pos = [int(i) for i in order if s[i] == k]
        assert pos == sorted(pos)
    launched = np.arange(len(s)) * 10
    back = np.empty_like(launched)
    back[order] = launched
    assert np.array_equal(back[order], launched) and np.array_equal(np.argsort(order), np.nonzero(back[:, None] == launched[None])[1])
    assert len(shard.scene_round_robin([])) == 0


def test_plan_scenes_balances_whole_scenes():
    plan = shard.plan_scenes([5, 1, 4, 4], 2)
    assert sorted(sum(plan, [])) == [0, 1, 2, 3]
    load = [sum([5, 1, 4, 4][s] for s in p) for p in plan]
    assert max(load) - min(load) <= 2


@pytest.fixture(scope="module")
def three_scenes():
    """Panda + 3 objects (tests/test_clutter.py's model), three scenes from gen_clutter_batch, five candidates per scene, the
    candidates of the scenes interleaved in a fixed shuffled order."""
    m, info = scenes.build_clutter_scene("panda", [0, 1, 2])
    L = lane1_scenes.sim(m, f64=False)
    recs = scenes.gen_clutter_batch(m, info, lambda r, n: L.step(r.astype(np.float32), n).astype(np.float64), [0, 1, 2])
    pose7, joints, si = [], [], []
    for k in range(3):
        H, w = scenes.clutter_candidates(m, info, recs[k], 5, k)
        pose7.append(scenes.process_poses(H, "panda").astype(np.float32))
        joints.append(scenes.panda_width_to_joints(w).astype(np.float32))
        si.append(np.full(5, k))
    perm = np.random.default_rng(0).permutation(15)
    return m, info, recs, np.concatenate(pose7)[perm], np.concatenate(joints)[perm], np.concatenate(si)[perm]


def _args(info):
    return info["joint_qposadr"], info["base_qposadr"]


@pytest.mark.parametrize("f64", [False, True])
def test_multi_scene_equals_per_scene_lane1(three_scenes, f64):
    m, info, recs, pose7, joints, si = three_scenes
    L = lane1_scenes.sim(m, f64=f64)
    cfg = mlib.MgsRolloutCfg(*SCHED)
    free = L.clutter_scenes_collision_mask(recs, si, pose7, joints, *_args(info))
    lab, steps = L.clutter_scenes_stable_mask(recs, si, pose7, joints, *_args(info), info["close_ctrl"], cfg)
    aux = L.last_aux(len(si))
    assert not aux["skipped"].any() and not aux["bad"].any()
    for k in range(3):
        rows = si == k
        f1 = L.clutter_collision_mask(recs[k], pose7[rows], joints[rows], *_args(info))
        l1, s1 = L.clutter_stable_mask(recs[k], pose7[rows], joints[rows], *_args(info), info["close_ctrl"], cfg)
        assert np.array_equal(free[rows], f1)
        assert np.array_equal(lab[rows], l1) and np.array_equal(steps[rows], s1)


@pytest.mark.parametrize("enough", [1, 2, 4])
def test_device_early_stop_lane1(three_scenes, enough):
    """The host build runs candidates one after another, so the skipped set is exactly the candidates after each scene's
    enough-th success, and the prefix rule per scene of the full labels gives the final labels."""
    m, info, recs, pose7, joints, si = three_scenes
    L = lane1_scenes.sim(m, f64=False)
    cfg = mlib.MgsRolloutCfg(*ALL_SUCCEED)
    full, full_steps = L.clutter_scenes_stable_mask(recs, si, pose7, joints, *_args(info), info["close_ctrl"], cfg)
    over = L.last_aux(len(si))["overflow"]
    assert full.all() and 0 < over.sum() < 3  # one candidate drops contacts at this capacity: its success is not counted
    lab, steps = L.clutter_scenes_stable_mask(recs, si, pose7, joints, *_args(info), info["close_ctrl"], cfg, enough_stable=enough)
    skipped = L.last_aux(len(si))["skipped"]
    expect, count = np.zeros(len(si), dtype=bool), np.zeros(3, dtype=int)
    for i in range(len(si)):  # each scene's candidates in their order: skipped once the scene counts `enough` non-overflowed successes
        expect[i] = count[si[i]] >= enough
        count[si[i]] += int(not expect[i] and full[i] and not over[i])
    assert np.array_equal(skipped, expect) and expect.any()
    assert not lab[skipped].any() and not steps[skipped].any()
    assert np.array_equal(lab[~skipped], full[~skipped]) and np.array_equal(steps[~skipped], full_steps[~skipped])
    for k in range(3):
        rows = si == k
        assert np.array_equal(shard.apply_enough_stable(lab[rows], enough), shard.apply_enough_stable(full[rows], enough))


def test_scene_index_out_of_range_lane1(three_scenes):
    """The kernel's own range check (the lane-1 entry point does not validate): label 0, 0 steps, aux bit 1; the other candidates
    are unaffected."""
    m, info, recs, pose7, joints, si = three_scenes
    L = lane1_scenes.sim(m, f64=False)
    cfg = mlib.MgsRolloutCfg(*ALL_SUCCEED)
    bad_si = si.copy()
    bad_si[[0, 5]] = [3, -1]
    lab, steps = L.clutter_scenes_stable_mask(recs, bad_si, pose7, joints, *_args(info), info["close_ctrl"], cfg, enough_stable=100)
    aux = L.last_aux(len(si))
    out = np.zeros(len(si), dtype=bool)
    out[[0, 5]] = True
    assert np.array_equal(aux["bad"], out) and not lab[out].any() and not steps[out].any() and not aux["skipped"].any()
    assert lab[~out].all() and (steps[~out] > 0).all()
    free = L.clutter_scenes_collision_mask(recs, bad_si, pose7, joints, *_args(info))
    assert not free[out].any() and np.array_equal(L.last_aux(len(si))["bad"], out)


WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import numpy as np, torch.distributed as dist
from mj_grasp_sim_b200 import scenes, shard
from mj_grasp_sim_b200.lib import MgsRolloutCfg
from hostsim import lane1_scenes
dist.init_process_group("gloo")
rank = dist.get_rank()
m, info = scenes.build_clutter_scene("panda", [0, 1, 2])
L = lane1_scenes.sim(m)
recs = scenes.gen_clutter_batch(m, info, lambda r, n: L.step(r.astype(np.float32), n).astype(np.float64), [0, 1, 2])
si = np.array([0, 1, 2, 2, 0, 2, 1, 2])
H, w = scenes.clutter_candidates(m, info, recs[0], len(si), 0)
pose7, joints = scenes.process_poses(H, "panda").astype(np.float32), scenes.panda_width_to_joints(w).astype(np.float32)
cfg = MgsRolloutCfg(500, 50, 0, 0, 0.05, 0.0)
args = (info["joint_qposadr"], info["base_qposadr"], info["close_ctrl"], cfg)
def run_scenes(idx):
    lab, _ = L.clutter_scenes_stable_mask(recs, si[idx], pose7[idx], joints[idx], *args, enough_stable=2)
    return lab
got = shard.evaluate_scenes_sharded(si, 3, run_scenes)
ref, _ = L.clutter_scenes_stable_mask(recs, si, pose7, joints, *args, enough_stable=2)
assert np.array_equal(got, ref) and 0 < ref.sum() < len(si), (got, ref)  # scene 2's last two are skipped
if rank == 0:
    print("GLOO_OK", got.astype(int))
dist.destroy_process_group()
"""


def test_two_rank_scene_sharding(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                          "--master-port", "29547", str(script)], capture_output=True, text=True, env=env, timeout=300)
    assert "GLOO_OK" in out.stdout, out.stdout + out.stderr


# ------------------------------------------------------------------------------------------------------------------- GPU tier
def _gpu_sim(m, f64=False, variant=None, **kw):
    """BatchSim of the CUDA library; `variant` forces the kernel variant (MGS_KERNEL_VARIANT) for this model only."""
    old = os.environ.pop("MGS_KERNEL_VARIANT", None)
    if variant:
        os.environ["MGS_KERNEL_VARIANT"] = variant
    try:
        return mlib.BatchSim(m, ground_name="geom:table", f64=f64, global_fallback=True, **kw)
    finally:
        os.environ.pop("MGS_KERNEL_VARIANT", None)
        if old is not None:
            os.environ["MGS_KERNEL_VARIANT"] = old


def _panda_scenes(S, nper, seed0=0):
    m, info = scenes.build_clutter_scene("panda", [0, 1, 2])
    G = _gpu_sim(m)
    recs = scenes.gen_clutter_batch(m, info, lambda r, n: G.step(r.astype(G.real), n).astype(np.float64), list(range(seed0, seed0 + S)))
    G.close()
    pose7, joints, si = [], [], []
    for k in range(S):
        H, w = scenes.clutter_candidates(m, info, recs[k], nper, k)
        pose7.append(scenes.process_poses(H, "panda").astype(np.float32))
        joints.append(scenes.panda_width_to_joints(w).astype(np.float32))
        si.append(np.full(nper, k))
    perm = np.random.default_rng(1).permutation(S * nper)
    return m, info, recs, np.concatenate(pose7)[perm], np.concatenate(joints)[perm], np.concatenate(si)[perm]


def _assert_multi_equals_per_scene(G, recs, si, pose7, joints, info, sched):
    cfg = mlib.MgsRolloutCfg(*sched)
    free = G.clutter_scenes_collision_mask(recs, si, pose7, joints, *_args(info))
    lab, steps = G.clutter_scenes_stable_mask(recs, si, pose7, joints, *_args(info), info["close_ctrl"], cfg)
    aux = G.last_aux(len(si))
    assert not aux["skipped"].any()
    for k in range(len(recs)):
        rows = si == k
        f1 = G.clutter_collision_mask(recs[k], pose7[rows], joints[rows], *_args(info))
        l1, s1 = G.clutter_stable_mask(recs[k], pose7[rows], joints[rows], *_args(info), info["close_ctrl"], cfg)
        assert np.array_equal(free[rows], f1), k
        assert np.array_equal(lab[rows], l1) and np.array_equal(steps[rows], s1), k
        assert np.array_equal(aux["bad"][rows], G.last_aux(int(rows.sum()))["bad"]), k
    return lab, aux


@pytest.mark.gpu
@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("variant", [None, "wide", "wide_g"])
def test_gpu_multi_scene_equals_per_scene(variant, f64):
    m, info, recs, pose7, joints, si = _panda_scenes(3, 64)
    G = _gpu_sim(m, f64=f64, variant=variant)
    assert G.state_in_global == (variant == "wide_g") and (G.info.lanes_per_env == 256) == (variant is not None or f64)
    _, aux = _assert_multi_equals_per_scene(G, recs, si, pose7, joints, info, SCHED)
    assert not aux["bad"].any()
    # the plain entry point validates the index on the host
    with pytest.raises(mlib.MgsError):
        G.clutter_scenes_collision_mask(recs, np.where(si == 2, 3, si), pose7, joints, *_args(info))
    G.close()


@pytest.mark.gpu
@pytest.mark.parametrize("f64", [False, True])
def test_gpu_config5_two_scenes(f64):
    """Config 5 (Shadow hand + ten objects, nv = 94), two scenes: fp32 on its default variant at the bench's 80 contacts, fp64 on
    wide_g (its product path)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import clutter_shadow_bench as csb
    m, info = scenes.build_clutter_scene("shadow", list(range(10)))
    G = _gpu_sim(m, f64=f64, ncon_max=0 if f64 else csb.NCON_MAX)
    assert G.state_in_global == f64
    recs = scenes.gen_clutter_batch(m, info, lambda r, n: G.step(r.astype(G.real), n).astype(np.float64), [7, 8])
    pose7, joints, si = [], [], []
    for k in range(2):
        p, j = csb.make_inputs(scenes, m, info, recs[k], 48)
        pose7.append(p); joints.append(j); si.append(np.full(48, k))
    perm = np.random.default_rng(2).permutation(96)
    pose7, joints, si = np.concatenate(pose7)[perm], np.concatenate(joints)[perm], np.concatenate(si)[perm]
    lab, _ = _assert_multi_equals_per_scene(G, recs, si, pose7, joints, info, (300, 200, 0, 0, 0.02, 0.0))
    assert lab.any() and not lab.all()
    G.close()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [None, "wide"])
def test_gpu_skipping_is_deterministic(variant):
    """One scene, n = 3 x the resident environment slots, all copies of one candidate that succeeds, enough_stable = 1: every
    environment's second pull sees its own increment, so at most one candidate per slot is simulated."""
    m, info, recs, pose7, joints, si = _panda_scenes(1, 1)
    G = _gpu_sim(m, variant=variant)
    cfg = mlib.MgsRolloutCfg(*ALL_SUCCEED)
    one, _ = G.clutter_stable_mask(recs[0], pose7, joints, *_args(info), info["close_ctrl"], cfg)
    assert one.all() and not G.last_aux(1)["overflow"].any()
    slots = G.info.num_sms * G.info.blocks_per_sm * G.info.warps_per_block
    n = 3 * slots
    lab, steps = G.clutter_scenes_stable_mask(recs[:1], np.zeros(n, dtype=np.int32), np.repeat(pose7, n, 0), np.repeat(joints, n, 0),
                                              *_args(info), info["close_ctrl"], cfg, enough_stable=1)
    aux = G.last_aux(n)
    assert aux["skipped"].sum() >= n - slots
    assert np.array_equal(lab, ~aux["skipped"]) and not steps[aux["skipped"]].any()
    final = shard.apply_enough_stable(lab, 1)
    assert final[0] and not final[1:].any()
    G.close()


def _panda_env(ncon_max=0, nefc_max=0):
    from mj_grasp_sim_b200.mgs.env.clutter_table import ClutterTableEnv
    from mj_grasp_sim_b200.mgs.gripper.selector import get_gripper
    from mj_grasp_sim_b200.mgs.obj.hull import ObjectConvexHull
    from mj_grasp_sim_b200.mgs.util.geo.transforms import SE3Pose
    objs = []
    for i in range(3):
        pts, mass = scenes.random_hull_points(10 + i, 24)
        objs.append(ObjectConvexHull(SE3Pose(np.array([-8.0, -8.0 + 0.5 * i, 0.06]), np.array([1.0, 0, 0, 0]), "wxyz"), f"o{i}", [pts], mass))
    return ClutterTableEnv(get_gripper("PandaGripper"), objs, ncon_max=ncon_max, nefc_max=nefc_max)


@pytest.mark.gpu
def test_gpu_env_scenes_with_escalation_equal_per_scene():
    """ClutterTableEnv.grasp_*_mask_scenes at a forced small first-pass capacity (some candidates overflow and go up the capacity
    ladder) equal the single-scene methods called once per scene, with and without enough_stable; the workspace bounds test too."""
    from mj_grasp_sim_b200.mgs.util.geo.transforms import SE3Pose
    env = _panda_env(ncon_max=8, nefc_max=64)
    defs = [d for d in env.gen_clutter_scenes([3, 4, 5, 6]) if d is not None][:3]
    assert len(defs) >= 2
    states = [d["env_state"]["state"] for d in defs]
    m = env.model
    info = dict(object_qposadr=[int(m.jnt_qposadr[m.names["joint"][f"o{i}:joint"]]) for i in range(3)])
    H, w, si = [], [], []
    for k, st in enumerate(states):
        env.set_state(st)
        h, ww = scenes.clutter_candidates(m, info, env._record, 40, 10 + k)
        H.append(h); w.append(ww); si.append(np.full(40, k))
    H, w, si = np.concatenate(H), np.concatenate(w), np.concatenate(si)
    H[:3, 0, 3] += 1.0  # out of the workspace bounds
    joints = scenes.panda_width_to_joints(w)
    poses = SE3Pose.from_mat(H)
    env.gripper.NSTEP_CLOSE = 500
    free = env.grasp_collision_mask_scenes(poses, joints, si, states)
    assert not free[:3].any()
    results = {None: env.grasp_stable_mask_scenes(poses, joints, si, states, nstep_lift=50, lift_dist=0.05)}
    first = env.last_overflow
    results[5] = env.grasp_stable_mask_scenes(poses, joints, si, states, nstep_lift=50, lift_dist=0.05, enough_stable=5)
    assert results[None].sum() > results[5].sum() > 0
    for k, st in enumerate(states):
        rows = si == k
        env.set_state(st)
        sub = SE3Pose.from_mat(H[rows])
        assert np.array_equal(env.grasp_collision_mask(sub, joints[rows]), free[rows]), k
        for e, lab in results.items():
            assert np.array_equal(env.grasp_stable_mask(sub, joints[rows], st, nstep_lift=50, lift_dist=0.05, enough_stable=e), lab[rows]), (k, e)
    assert first["first_pass"] > 0 and first["after_escalation"] == 0, first


def _object_frame_grasps(scene):
    from mj_grasp_sim_b200.mgs.env.clutter_table import ClutterTableEnv
    env0 = ClutterTableEnv.from_dict(scene)
    grasps = {}
    for k, (name, oid) in enumerate(zip(env0.object_names, env0.object_ids)):
        a = int(env0.model.jnt_qposadr[env0.model.names["joint"][f"{name}:joint"]])
        H, w = scenes.clutter_candidates(env0.model, dict(object_qposadr=[a]), env0._record, 96, 30 + k)
        o2w = env0.get_obj_pose(name).to_mat().astype(np.float64).reshape(4, 4)
        grasps[oid] = (np.einsum("ij,njk->nik", np.linalg.inv(o2w), H), scenes.panda_width_to_joints(w))
    return grasps


def _files(d):
    out = {}
    for f in sorted(os.listdir(d)):
        z = np.load(os.path.join(d, f), allow_pickle=True)
        out[f] = {k: z[k] for k in z.files}
    return out


def _same_scene(a, b):
    assert type(a["gripper"]).__name__ == type(b["gripper"]).__name__
    assert [o.object_id for o in a["objects"]] == [o.object_id for o in b["objects"]]
    for k in ("geom_conaffinity", "geom_contype", "geom_rgba", "body_gravcomp", "state"):
        assert np.array_equal(np.asarray(a["env_state"][k]), np.asarray(b["env_state"][k])), k


@pytest.mark.gpu
def test_gpu_gen_scene_batch_equals_loop(tmp_path):
    from mj_grasp_sim_b200.mgs.cli import gen_scene
    ids = ["hull:20:24", "hull:21:24", "hull:22:24"]
    seeds = [5, 6, 7, 8]
    single = {}
    for s in seeds:
        try:
            single[s] = gen_scene.gen_stable_scene("PandaGripper", ids, seed=s)
        except ValueError as e:
            single[s] = e
    ok = [s for s in seeds if isinstance(single[s], dict)]
    assert len(ok) >= 2
    grasps = _object_frame_grasps(single[ok[0]])
    kw = dict(grasps=grasps, only_collision_free=True, save_collision_grasps=True, enough_collision_free=8)
    got = gen_scene.run_batch("PandaGripper", ids, seeds, output_dir=str(tmp_path / "batch"), **kw)
    written = 0
    for s, r in zip(seeds, got):
        if isinstance(single[s], ValueError):
            assert isinstance(r, ValueError) and str(r) == "Scene unstable"
            continue
        try:
            d = gen_scene.run("PandaGripper", ids, seed=s, output_dir=str(tmp_path / "loop"), **kw)
        except ValueError as e:  # e.g. too few collision-free grasps in this scene
            assert isinstance(r, ValueError) and str(r) == str(e)
            continue
        a, b = _files(r), _files(d)
        assert a.keys() == b.keys()
        _same_scene(a["scene.npz"]["scene_definition"].item(), b["scene.npz"]["scene_definition"].item())
        _same_scene(a["scene.npz"]["scene_definition"].item(), single[s])
        for f in a:
            if f != "scene.npz":
                assert all(np.array_equal(a[f][k], b[f][k]) for k in a[f]), f
        written += 1
    assert written >= 1
    # the stable pass: one generator shared by the loop and by the batch
    defs = [single[s] for s in ok]
    kw = dict(grasps=grasps, enough_collision_free=8)
    rng = np.random.default_rng(0)
    loop = []
    for d in defs:
        try:
            loop.append(gen_scene.filter_grasps("PandaGripper", d, rng=rng, **kw))
        except ValueError as e:
            loop.append(e)
    rng_b = np.random.default_rng(0)
    batch = gen_scene.filter_grasps_scenes("PandaGripper", defs, rng=rng_b, **kw)
    assert rng.bit_generator.state == rng_b.bit_generator.state  # the same draws, in the same order
    for x, y in zip(loop, batch):
        if isinstance(x, ValueError):
            assert isinstance(y, ValueError) and str(x) == str(y)
        else:
            for gx, gy in zip(x[0] + x[1], y[0] + y[1]):
                assert gx["object_id"] == gy["object_id"] and np.array_equal(gx["pose"], gy["pose"]) and np.array_equal(gx["joints"], gy["joints"])
            assert len(x[0]) == len(y[0]) and len(x[1]) == len(y[1])
    bad = dict(defs[0], objects=defs[0]["objects"][:2])
    with pytest.raises(ValueError):
        gen_scene.filter_grasps_scenes("PandaGripper", [defs[0], bad], **kw)
