"""Config 5: qpos / qvel of the environment-per-CTA kernel vs the oracle over the first 50 steps after the hand is placed over the
settled 10-object scene and told to close (8 candidates).  fp32 (default): 80 contacts, state in shared memory; f64: the product
path of ClutterTableEnv with the Shadow hand - default capacity, state in global memory.
On a B200: python tools/clutter_first50.py [f32|f64]"""
import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tools"))
from mj_grasp_sim_b200 import scenes
from mj_grasp_sim_b200.lib import BatchSim
from oracle import oracle as orc
import clutter_shadow_bench as csb


def run(n=8, nstep=50, every=10, collision_free=True, f64=False):
    m, info = scenes.build_clutter_scene("shadow", list(range(10)))
    if f64:
        G = BatchSim(m, ground_name="geom:table", f64=True, global_fallback=True)
    else:
        G = BatchSim(m, ground_name="geom:table", ncon_max=csb.NCON_MAX)
    print(f"{'fp64' if f64 else 'fp32'}, {G.info.ncon_max} contacts, state in {'global' if G.state_in_global else 'shared'} memory", flush=True)
    step_fn = lambda r, k: G.step(r[None].astype(G.real), k)[0].astype(np.float64)
    rec = scenes.gen_clutter(m, info, step_fn, 7)
    pose7, joints = csb.make_inputs(scenes, m, info, rec, 16 * n)
    free = G.clutter_collision_mask(rec, pose7, joints, info["joint_qposadr"], info["base_qposadr"])
    if collision_free:  # the candidates the stability rollout is normally run on
        pose7, joints = pose7[free][:n], joints[free][:n]
    else:
        pose7, joints = pose7[:n], joints[:n]
    n = len(pose7)
    nq, nv, nu = m.nq, m.nv, m.nu
    st = np.tile(rec, (n, 1))
    b = info["base_qposadr"]
    st[:, b:b + 7] = pose7
    for k, a in enumerate(info["joint_qposadr"]):
        st[:, a] = joints[:, k]
    st[:, nq + 2 * nv:nq + 2 * nv + nu] = info["close_ctrl"]
    st[:, nq + 2 * nv + nu:nq + 2 * nv + nu + 7] = pose7
    S = orc.OracleSim(m, ground_name="geom:table")
    free = G.clutter_collision_mask(rec, pose7, joints, info["joint_qposadr"], info["base_qposadr"])
    print("collision-free at placement:", free.astype(int), flush=True)
    out = []
    cur = st.astype(G.real)
    ref = [st[i].copy() for i in range(n)]
    for t in range(every, nstep + 1, every):
        cur, d = G.step(cur, every, want_diag=True)
        qe = ve = 0.0
        same = 0
        per = []
        for i in range(n):
            S.set_record(ref[i]); S.step(every); ref[i] = S.get_record()
            e = np.abs(cur[i, :nq] - ref[i][:nq])
            per.append((float(e.max()), int(e.argmax()), int(d["ncon"][i]), int(S.ncon)))
            qe = max(qe, np.abs(cur[i, :nq] - ref[i][:nq]).max() / max(1.0, np.abs(ref[i][:nq]).max()))
            ve = max(ve, np.abs(cur[i, nq:nq + nv] - ref[i][nq:nq + nv]).max() / max(1.0, np.abs(ref[i][nq:nq + nv]).max()))
            same += int(d["ncon"][i] == S.ncon)
        out.append(dict(step=t, qpos_rel=float(qe), qvel_rel=float(ve), same_ncon=same, n=n))
        print(out[-1], "per candidate (max |dq|, coordinate, ncon kernel, ncon oracle):", [(round(a, 6), b, c, dd) for a, b, c, dd in per], flush=True)
    return out


if __name__ == "__main__":
    run(f64=len(sys.argv) > 1 and sys.argv[1] == "f64")
