"""Environment state in global memory (kernel variant wide_g, mgs_model_create_any): the environment-per-CTA kernel with its
per-environment slice in a global-memory slab, for models whose state does not fit one CTA's shared memory - the fp64 Shadow hand
over a cluttered table (the product path of ClutterTableEnv with the Shadow hand) and the 256-contact escalation rung of clutter
scenes.

CPU tier: the variant is in both builds without local memory, and the environments ask for it where they should.
GPU tier: the same code in the other address space gives the same results (to the last bits: see _compare); config 5 runs on the default product path (fp64);
clutter environments over capacity are re-run; the fp64 trajectory matches the oracle."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _with_env(var, value, make):
    """make() with os.environ[var] = value (None: unset), restored afterwards."""
    old = os.environ.get(var)
    if value is None:
        os.environ.pop(var, None)
    else:
        os.environ[var] = value
    try:
        return make()
    finally:
        if old is None:
            os.environ.pop(var, None)
        else:
            os.environ[var] = old


def _variant_sim(mlib, m, variant, **kw):
    """BatchSim on a forced kernel variant (the library reads MGS_KERNEL_VARIANT when the model is created)."""
    return _with_env("MGS_KERNEL_VARIANT", variant, lambda: mlib.BatchSim(m, **kw))


# ---------------------------------------------------------------------------------------------------------------- CPU tier
@pytest.mark.parametrize("f64", [False, True])
def test_both_builds_have_the_global_state_variant_without_local_memory(f64):
    from mj_grasp_sim_b200 import lib as mlib
    so = mlib.build(f64=f64)
    out = subprocess.run(["cuobjdump", "-res-usage", so], capture_output=True, text=True, check=True).stdout
    lines = out.splitlines()
    k = [i for i, ln in enumerate(lines) if "Function" in ln and "mgs_rollout_kernel_wide_g" in ln]
    assert len(k) == 1, "mgs_rollout_kernel_wide_g missing"
    assert "LOCAL:0" in lines[k[0] + 1], lines[k[0] + 1]


class _Info:
    def __init__(self, ncon_max):
        self.ncon_max, self.nefc_max, self.warps_per_block, self.blocks_per_sm, self.num_sms, self.real_bytes = ncon_max, 0, 1, 1, 148, 4


class _RecordingSim:
    """Stands in for BatchSim: records how the environment asked for each instance."""
    calls = []

    def __init__(self, model, device=0, ncon_max=0, nefc_max=0, ground_name="geom:ground", f64=False, **kw):
        _RecordingSim.calls.append(dict(ncon_max=ncon_max, **kw))
        self.device, self.info = device, _Info(ncon_max or 64)

    def close(self):
        pass


def _record(monkeypatch):
    from mj_grasp_sim_b200.mgs.core import simualtion as simmod
    from mj_grasp_sim_b200.mgs.env import clutter_table as ct
    from mj_grasp_sim_b200.mgs.env import gravityless_object_grasping as gog
    _RecordingSim.calls = []
    for mod in (simmod, ct, gog):
        monkeypatch.setattr(mod, "BatchSim", _RecordingSim)
    return _RecordingSim.calls


def test_clutter_env_asks_for_the_global_fallback_on_every_rung(monkeypatch):
    from mj_grasp_sim_b200.mgs.env.clutter_table import ClutterTableEnv
    from mj_grasp_sim_b200.mgs.gripper.selector import get_gripper
    from mj_grasp_sim_b200.mgs.obj.selector import get_objects
    calls = _record(monkeypatch)
    env = ClutterTableEnv(get_gripper("PandaGripper"), get_objects(["hull:50:16", "hull:51:16"]), device=0, ncon_max=16)
    env._esc.small, env._esc.mid, env._esc.big  # first pass (16 contacts), 32-contact rung, largest rung
    assert [c["ncon_max"] for c in calls] == [16, 32, 256]
    assert all(c.get("global_fallback") is True for c in calls), calls


def test_single_object_env_never_asks_for_it(monkeypatch):
    from mj_grasp_sim_b200.mgs.env.gravityless_object_grasping import GravitylessObjectGrasping
    from mj_grasp_sim_b200.mgs.gripper.selector import get_gripper
    from mj_grasp_sim_b200.mgs.obj.selector import get_object
    calls = _record(monkeypatch)
    env = GravitylessObjectGrasping(get_gripper("PandaGripper"), get_object("hull:0"), device=0, ncon_max=16)
    env._esc.small, env._esc.mid, env._esc.big
    assert [c["ncon_max"] for c in calls] == [16, 32, 256]
    assert not any(c.get("global_fallback") for c in calls), calls


# ---------------------------------------------------------------------------------------------------------------- GPU tier
@pytest.fixture(scope="module")
def libs():
    from mj_grasp_sim_b200 import lib as mlib
    from oracle import oracle as orc
    mlib.load()
    return mlib, orc


def _tools():
    p = os.path.join(ROOT, "tools")
    if p not in sys.path:
        sys.path.insert(0, p)
    import clutter_shadow_bench as csb
    return csb


def _place(m, info, pose7, joints, scene=None):
    """state records: the hand placed at pose7 / joints (over `scene` when given), closing"""
    n = len(pose7)
    st = np.tile(m.qpos0 if scene is None else scene[:m.nq], (n, 1))
    b = info["base_qposadr"]
    st[:, b:b + 7] = pose7
    for k, a in enumerate(info["joint_qposadr"]):
        st[:, a] = joints[:, k]
    return st


# wide and wide_g are one source compiled for two address spaces of the environment slice, but not to the same arithmetic: with the
# slice address taken from the constant bank instead of the shared window, the compiler contracts a few more multiply-adds into FMAs
# (PTX of the fp32 build: 917 fma.rn.f32 in wide_g against 912 in wide; fp64: 915 against 911 fma.rn.f64).  Results therefore
# agree to the last bits, not bitwise, and contact chaos amplifies last-bit differences over a rollout.  What stays exact is what
# does not integrate over time: the collision mask (one forward pass) and the model's capacities.
def _compare(W, G, run, step_states, nstep, tol, oracle_labels=None, min_agree=15 / 16):
    (fw, lw, sw), (fg, lg, sg) = run(W), run(G)
    assert np.array_equal(fw, fg)
    assert np.array_equal(run(G)[1], lg)  # each variant on its own is deterministic
    if oracle_labels is None:
        assert (lw == lg).mean() >= min_agree, (lw == lg).mean()
    else:
        assert (lg == oracle_labels).mean() >= min_agree and (lw == oracle_labels).mean() >= min_agree
    step_states = step_states[fw]  # collision-free placements: a start in penetration is violent and amplifies any last bit
    uw, ug = W.unpack_state(W.step(step_states, nstep)), G.unpack_state(G.step(step_states, nstep))
    err = np.abs(uw["qpos"] - ug["qpos"]).max() / max(1.0, np.abs(uw["qpos"]).max())
    assert err <= tol, err


@pytest.mark.gpu
@pytest.mark.parametrize("f64", [False, True])
def test_same_code_in_global_memory_single_object(libs, shadow_hull, f64):
    """Forced wide and wide_g on the Shadow hand: same collision mask, labels as close as the warp-variant comparison of the wide
    variant requires (15 of 16), 50-step states within that comparison's bounds."""
    mlib, _ = libs
    m, info, pose7, joints = shadow_hull
    n = 16
    pose7, joints = pose7[:n], joints[:n]
    W, G = _variant_sim(mlib, m, "wide", f64=f64), _variant_sim(mlib, m, "wide_g", f64=f64)
    assert not W.state_in_global and G.state_in_global and G.info.lanes_per_env == 256 and G.info.blocks_per_sm >= 1
    assert (W.info.ncon_max, W.info.nefc_max, W.info.smem_bytes_per_env) == (G.info.ncon_max, G.info.nefc_max, G.info.smem_bytes_per_env)
    sched = mlib.MgsRolloutCfg(300, 100, 20, 0, 0.02, 0.02)
    args = (pose7, joints, info["joint_qposadr"], info["base_qposadr"])
    run = lambda S: (S.collision_mask(*args),) + tuple(S.stability(*args, info["close_ctrl"], sched))
    st0 = _place(m, info, pose7, joints)
    st = W.pack_state(st0, np.zeros((n, m.nv)), ctrl=np.tile(info["close_ctrl"], (n, 1)), mocap_pos=pose7[:, :3], mocap_quat=pose7[:, 3:7])
    _compare(W, G, run, st, 50, 1e-8 if f64 else 5e-4)


@pytest.mark.gpu
def test_same_code_in_global_memory_config5(libs):
    """The same on config 5 (Shadow hand over ten objects, fp32, 80 contacts: the largest capacity that fits shared memory): same
    collision mask, labels of the short schedule within the config-5 bar against the oracle for both (0.85), first 10 steps within the
    fp32 trajectory bound (1e-4 relative)."""
    from mj_grasp_sim_b200 import scenes
    csb = _tools()
    mlib, orc = libs
    m, info = scenes.build_clutter_scene("shadow", list(range(10)))
    W = _variant_sim(mlib, m, "wide", ground_name="geom:table", ncon_max=csb.NCON_MAX)
    G = _variant_sim(mlib, m, "wide_g", ground_name="geom:table", ncon_max=csb.NCON_MAX)
    assert not W.state_in_global and G.state_in_global and W.info.real_bytes == G.info.real_bytes == 4
    rec = scenes.gen_clutter(m, info, lambda r, k: W.step(r[None].astype(np.float32), k)[0].astype(np.float64), 7)
    n = 64
    pose7, joints = csb.make_inputs(scenes, m, info, rec, n)
    sched = (300, 200, 0, 0, 0.02, 0.0)
    args = (rec, pose7, joints, info["joint_qposadr"], info["base_qposadr"])
    run = lambda S: (S.clutter_collision_mask(*args),) + tuple(S.clutter_stable_mask(*args, info["close_ctrl"], mlib.MgsRolloutCfg(*sched)))
    a = (pose7.astype(np.float64), info["base_qposadr"], joints.astype(np.float64), info["joint_qposadr"], info["close_ctrl"], orc.RolloutCfg(*sched),
         os.cpu_count() or 1)
    olab, _ = orc.batch(m, 3, *a, scene=rec, ground_name="geom:table")
    st = np.tile(rec, (n, 1))
    st[:, :m.nq] = _place(m, info, pose7, joints, rec)
    nq, nv, nu = m.nq, m.nv, m.nu
    st[:, nq + 2 * nv:nq + 2 * nv + nu] = info["close_ctrl"]
    st[:, nq + 2 * nv + nu:nq + 2 * nv + nu + 7] = pose7
    _compare(W, G, run, st.astype(np.float32), 10, 1e-4, oracle_labels=olab.astype(bool), min_agree=0.85)


def _config5_env(ncon_max=0):
    """ClutterTableEnv(ShadowHand, the ten hull objects of config 5) through the reference-facing constructor"""
    from mj_grasp_sim_b200 import scenes
    from mj_grasp_sim_b200.mgs.env.clutter_table import ClutterTableEnv
    from mj_grasp_sim_b200.mgs.gripper.selector import get_gripper
    from mj_grasp_sim_b200.mgs.obj.hull import ObjectConvexHull
    from mj_grasp_sim_b200.mgs.util.geo.transforms import SE3Pose
    objs = []
    for i in range(10):
        pts, mass = scenes.random_hull_points(i, 24)
        objs.append(ObjectConvexHull(SE3Pose(np.array([-8.0, -8.0 + 0.5 * i, 0.06]), np.array([1.0, 0, 0, 0]), "wxyz"), f"obj{i}", [pts], mass))
    env = ClutterTableEnv(get_gripper("ShadowHand"), objs, ncon_max=ncon_max)
    env.set_gripper_pose([0.0, 0.0, 1.5])
    return env


def _config5_candidates(env, n):
    """the config-5 candidates (tools/clutter_shadow_bench.make_inputs) as the env's inputs: SE3Pose [n] + joints [n, 22]"""
    from mj_grasp_sim_b200 import scenes
    from mj_grasp_sim_b200.mgs.util.geo.transforms import SE3Pose
    m = env.model
    adr = [int(m.jnt_qposadr[m.names["joint"][f"obj{i}:joint"]]) for i in range(10)]
    H, _ = scenes.clutter_candidates(m, dict(object_qposadr=adr), env._record, n, 2)
    Rt = np.array([[0.0, 0.0, 1.0], [-1.0, 0.0, 0.0], [0.0, -1.0, 0.0]])
    T = np.eye(4)
    T[:3, :3] = Rt
    T[:3, 3] = -Rt @ np.array([0.01, -0.06, 0.12])
    g = scenes.GRIPPERS["shadow"]
    jid = [m.names["joint"][j] for j in g["joints"]]
    joints = np.clip(np.asarray(g["open_pose"])[None] + np.random.default_rng(3).normal(scale=0.05, size=(n, 22)), m.jnt_range[jid, 0], m.jnt_range[jid, 1])
    return SE3Pose.from_mat(H @ T, type="wxyz"), joints.astype(np.float32), adr


@pytest.mark.gpu
def test_config5_on_the_default_product_path(libs, tmp_path, monkeypatch):
    """ClutterTableEnv with the Shadow hand over ten objects, no MGS_PRECISION: the fp64 model (388 KB per environment at 64 contacts)
    runs with its state in global memory - scene generation, collision mask and labels against the oracle, at least as close to it
    as the fp32 path on the same candidates (one flip of slack), nothing left over capacity, deterministic, and the scene dictionary
    round trip through eval_grasps."""
    import json
    from mj_grasp_sim_b200.mgs.cli import eval_grasps
    from mj_grasp_sim_b200.mgs.env.clutter_table import ClutterTableEnv
    monkeypatch.delenv("MGS_PRECISION", raising=False)
    monkeypatch.delenv("MGS_KERNEL_VARIANT", raising=False)
    mlib, orc = libs
    env = _config5_env()
    S = env.sim
    assert env.compute_f64 and S.info.real_bytes == 8 and S.state_in_global and S.info.lanes_per_env == 256
    env.gen_clutter(seed=7)
    m = env.model
    poses, joints, adr = _config5_candidates(env, 64)
    z = np.array([env._record[a + 2] for a in adr])
    assert (z > 0.0).all() and (z < 0.3).all(), z  # every object came to rest on the table
    state = env.get_state()
    env.gripper.NSTEP_CLOSE = 300
    free = env.grasp_collision_mask(poses, joints)
    lab = env.grasp_stable_mask(poses, joints, state, nstep_lift=200, lift_dist=0.02)
    assert env.last_overflow["after_escalation"] == 0, env.last_overflow
    assert np.array_equal(env.grasp_stable_mask(poses, joints, state, nstep_lift=200, lift_dist=0.02), lab)
    pose7, j32, jadr = env._process(poses, joints)
    base = env.gripper.get_freejoint_idxs(env)[0]
    sched = (300, 200, 0, 0, 0.02, 0.0)
    a = (pose7.astype(np.float64), base, j32.astype(np.float64), jadr, env.gripper.close_ctrl(), orc.RolloutCfg(*sched), os.cpu_count() or 1)
    ofree, _ = orc.batch(m, 2, *a, scene=env._record, ground_name="geom:table")
    olab, _ = orc.batch(m, 3, *a, scene=env._record, ground_name="geom:table")
    assert np.array_equal(free, ofree)
    F = mlib.BatchSim(m, ground_name="geom:table", ncon_max=80)  # the fp32 path on the same scene record and candidates
    flab, _ = F.clutter_stable_mask(env._record, pose7, j32, jadr, base, env.gripper.close_ctrl(), mlib.MgsRolloutCfg(*sched))
    agree, agree32 = (lab == olab).mean(), (flab == olab).mean()
    print(f"config 5, 64 candidates: fp64 global-state path {agree:.4f}, fp32 path {agree32:.4f} label agreement with the oracle")
    assert agree >= 0.85 and agree >= agree32 - 1.0 / len(lab), (agree, agree32)
    # scene dictionary round trip, then the reference's eval_grasps on it
    env2 = ClutterTableEnv.from_dict(env.to_dict())
    assert env2.sim.state_in_global and np.array_equal(env2.grasp_collision_mask(poses, joints), free)
    d = tmp_path / "ShadowHand" / "scene0"
    d.mkdir(parents=True)
    np.savez(d / "scene.npz", scene_definition=env.to_dict())
    np.savez(d / "inference_grasps.npz", pose=poses.to_mat()[:8].astype(np.float64).reshape(-1, 4, 4), joints=joints[:8])
    res = eval_grasps.run("ShadowHand", 0, input_dir=str(tmp_path))
    assert res["num_objects"] == 10 and 0.0 <= res["success_rate"] <= 1.0
    assert json.load(open(d / "grasp_evaluation.json")) == res


@pytest.mark.gpu
def test_clutter_environments_over_capacity_are_re_run(libs, monkeypatch):
    """Config 5 in fp32 with a 16-contact first pass: the environments over capacity climb the ladder - 32 contacts in shared
    memory, then 256 contacts, which only fits with the state in global memory - and none is left; the others keep the labels of a
    first-pass-only run bit for bit.  The settled pile alone holds more than 16 contacts, so that last check is repeated with a
    48-contact first pass on the same scene, where some environments stay within capacity."""
    monkeypatch.setenv("MGS_PRECISION", "f32")
    monkeypatch.delenv("MGS_KERNEL_VARIANT", raising=False)
    mlib, _ = libs
    env = _config5_env(ncon_max=16)
    env.gen_clutter(seed=7)
    poses, joints, _ = _config5_candidates(env, 64)
    state = env.get_state()
    env.gripper.NSTEP_CLOSE = 300
    lab = env.grasp_stable_mask(poses, joints, state, nstep_lift=200, lift_dist=0.02)
    ov = env.last_overflow
    assert ov["first_pass"] > 0 and ov["after_escalation"] == 0, ov
    esc = env._esc
    assert esc.small.info.ncon_max == 16 and not esc.small.state_in_global
    assert esc._mid and esc._mid.info.ncon_max == 32 and not esc._mid.state_in_global
    assert esc._big and esc._big.info.ncon_max == 256 and esc._big.state_in_global
    pose7, j32, jadr = env._process(poses, joints)
    base = env.gripper.get_freejoint_idxs(env)[0]
    cfg = mlib.MgsRolloutCfg(300, 200, 0, 0, 0.02, 0.0)
    first, _ = esc.small.clutter_stable_mask(env._record_from_state(state), pose7, j32, jadr, base, env.gripper.close_ctrl(), cfg)
    over = esc.small.last_aux(len(lab))["overflow"]
    assert over.sum() == ov["first_pass"]
    assert np.array_equal(lab[~over], first[~over])
    env48 = _config5_env(ncon_max=48)
    env48.set_state(state)
    env48.gripper.NSTEP_CLOSE = 300
    lab48 = env48.grasp_stable_mask(poses, joints, state, nstep_lift=200, lift_dist=0.02)
    assert env48.last_overflow["after_escalation"] == 0 and env48._esc._big.state_in_global
    first48, _ = env48._esc.small.clutter_stable_mask(env48._record_from_state(state), pose7, j32, jadr, base, env48.gripper.close_ctrl(), cfg)
    over48 = env48._esc.small.last_aux(len(lab))["overflow"]
    print(f"first pass over capacity: {int(over.sum())} of {len(lab)} at 16 contacts, {int(over48.sum())} at 48")
    assert (~over48).any() and np.array_equal(lab48[~over48], first48[~over48])


@pytest.mark.gpu
def test_config5_first_50_steps_fp64_in_global_memory(libs):
    """Trajectory on the product path of config 5 (fp64, state in global memory, 8 collision-free candidates): first 10 steps
    within 1e-7 relative of the oracle with the same contact counts (the fp64 bound of the single-object hands), step 50 within an
    event bound."""
    _tools()
    import clutter_first50
    rows = clutter_first50.run(8, 50, 10, f64=True)
    assert rows[0]["same_ncon"] == rows[0]["n"] == 8 and rows[0]["qpos_rel"] <= 1e-7, rows[0]
    # measured on B200: 3e-11 at step 10; by step 50 one of the 8 candidates has gone through a contact event the oracle took
    # differently (29 against 23 contacts) and sits at 2.1e-2 - above the fp32 test's 1e-2, hence the looser bound here
    assert rows[-1]["qpos_rel"] <= 5e-2, rows[-1]
