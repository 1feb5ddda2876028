"""Config 5 label agreement at a larger n than the GPU test affords by default: the test's scene (seed 7) and schedule
(close 300 + lift 200), n candidates through the CUDA path (environment-per-CTA variant) and through the oracle.
  f32 (default): 80 contacts, state in shared memory (the bench line's configuration);
  f64: the product path of ClutterTableEnv with the Shadow hand - default capacity, state in global memory.
The variant can be forced (wide | wide_g; default: the library's choice).
On a B200: python tools/cfg5_labels.py [n] [f32|f64] [variant] -> one JSON line, also written to
$MGS_OUT_DIR/cfg5_labels[_f64].json (default: the current directory)"""
import json, os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tools"))
from mj_grasp_sim_b200 import scenes, lib as mlib
from oracle import oracle as orc
import clutter_shadow_bench as csb

n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
f64 = len(sys.argv) > 2 and sys.argv[2] == "f64"
if len(sys.argv) > 3:
    os.environ["MGS_KERNEL_VARIANT"] = sys.argv[3]
m, info = scenes.build_clutter_scene("shadow", list(range(10)))
G = mlib.BatchSim(m, ground_name="geom:table", ncon_max=0 if f64 else csb.NCON_MAX, f64=f64, global_fallback=True)
step_fn = lambda r, k: G.step(r[None].astype(G.real), k)[0].astype(np.float64)
rec = scenes.gen_clutter(m, info, step_fn, 7)
pose7, joints = csb.make_inputs(scenes, m, info, rec, n)
sched = (300, 200, 0, 0, 0.02, 0.0)
t = time.time()
free = G.clutter_collision_mask(rec, pose7, joints, info["joint_qposadr"], info["base_qposadr"])
lab, steps = G.clutter_stable_mask(rec, pose7, joints, info["joint_qposadr"], info["base_qposadr"], info["close_ctrl"], mlib.MgsRolloutCfg(*sched))
t_gpu = time.time() - t
over = G.last_aux(n)["overflow"].astype(bool)
a = (pose7.astype(np.float64), info["base_qposadr"], joints.astype(np.float64), info["joint_qposadr"], info["close_ctrl"], orc.RolloutCfg(*sched), os.cpu_count() or 1)
t = time.time()
ofree, _ = orc.batch(m, 2, *a, scene=rec, ground_name="geom:table")
olab, osteps = orc.batch(m, 3, *a, scene=rec, ground_name="geom:table")
t_or = time.time() - t
lab, olab = lab.astype(bool), olab.astype(bool)
row = dict(n=n, free_equal=bool(np.array_equal(free, ofree)), oracle_stable=float(olab.mean()), overflowed=int(over.sum()),
           agree_all=float((lab == olab).mean()), agree_not_overflowed=float((lab == olab)[~over].mean()),
           false_pos=int((lab & ~olab).sum()), false_neg=int((~lab & olab).sum()),
           steps_equal_where_labels_equal=float((steps[lab == olab] == osteps[lab == olab]).mean()), gpu_s=round(t_gpu, 1), oracle_s=round(t_or, 1),
           caps=[int(G.info.ncon_max), int(G.info.nefc_max)], precision="f64" if f64 else "f32", state_in_global=G.state_in_global,
           variant="wide_g" if G.state_in_global else ("wide" if G.info.lanes_per_env == 256 else "warp per environment"))
print(json.dumps(row), flush=True)
out_dir = os.environ.get("MGS_OUT_DIR", ".")
os.makedirs(out_dir, exist_ok=True)
json.dump(row, open(os.path.join(out_dir, "cfg5_labels%s.json" % ("_f64" if f64 else "")), "w"), indent=1)
