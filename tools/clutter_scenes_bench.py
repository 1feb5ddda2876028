"""Config 5 over many scenes: per-scene evaluation in enough_stable rounds against one multi-scene launch with the device early stop.

Workload (BASELINE.json configs[4]): the Shadow hand over ten hull objects, S scenes from gen_clutter_batch (seeds 7, 8, ...; untimed,
stepped by the fp32 kernel so every arm sees the same records), K top-down candidates per scene (clutter_shadow_bench.make_inputs),
the full schedule (close 3000 + lift 0.3 m over 3000 steps), enough_stable = 128 (gen_scene's rule for ten objects).  Three arms per
precision, alternated, `repeats` times each:
  A  today's way: one grasp_stable_mask-style evaluation per scene, in shard.evaluate_sharded rounds of one GPU-filling chunk
  B  one mgs_clutter_scenes_stable_mask launch over all scenes with the device early stop, then the prefix rule per scene
  C  the same launch without the early stop (every candidate simulated; comparable to bench.py's clutter_shadow env-steps/s)
Precisions: f32 = fp32 with the state in shared memory at 80 contacts (the clutter_shadow configuration), f64 = fp64 on wide_g (the
product path of ClutterTableEnv with the Shadow hand).  All arms go through the host entry points (inputs staged, results copied
back), timed with a host clock around calls that end in a stream synchronise.  No escalation: overflowed candidates are reported.
A and B must give the same labels; the tool exits with an error otherwise (after writing the JSON).

On a B200: python tools/clutter_scenes_bench.py [S=4] [K=444] [repeats=2] [precisions=f32,f64] -> $MGS_OUT_DIR/clutter_scenes_bench.json
(default: the current directory).  The scene-sharded path (shard.evaluate_scenes_sharded) is not timed here."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tools"))
from mj_grasp_sim_b200 import scenes, shard, lib as mlib  # noqa: E402
import clutter_shadow_bench as csb  # noqa: E402

OUT = os.environ.get("MGS_OUT_DIR", ".")
ENOUGH = 128


def smi(q):
    try:
        return subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=10).stdout.strip()
    except Exception as ex:
        return f"unavailable ({ex})"


def workload(S, K):
    m, info = scenes.build_clutter_scene("shadow", list(range(10)))
    gen = mlib.BatchSim(m, ground_name="geom:table", ncon_max=csb.NCON_MAX)
    t = time.perf_counter()
    recs = scenes.gen_clutter_batch(m, info, lambda r, k: gen.step(r.astype(np.float32), k).astype(np.float64), [7 + s for s in range(S)])
    t_gen = time.perf_counter() - t
    gen.close()
    pose7, joints = zip(*(csb.make_inputs(scenes, m, info, recs[s], K) for s in range(S)))
    return m, info, recs, np.concatenate(pose7), np.concatenate(joints), np.repeat(np.arange(S), K), t_gen


def make_sim(m, precision):
    if precision == "f32":
        return mlib.BatchSim(m, ground_name="geom:table", ncon_max=csb.NCON_MAX)
    os.environ["MGS_KERNEL_VARIANT"] = "wide_g"
    try:
        return mlib.BatchSim(m, ground_name="geom:table", f64=True, global_fallback=True)
    finally:
        os.environ.pop("MGS_KERNEL_VARIANT", None)


def run_arms(sim, info, recs, pose7, joints, si, repeats):
    S = len(recs)
    cfg = mlib.MgsRolloutCfg(*csb.SCHED)
    args = (info["joint_qposadr"], info["base_qposadr"])
    chunk = sim.info.warps_per_block * sim.info.blocks_per_sm * sim.info.num_sms

    def arm_a():
        labels, steps, sim_n, over = np.zeros(len(si), dtype=bool), 0, 0, 0
        for s in range(S):
            rows = np.nonzero(si == s)[0]

            def run_range(lo, hi):
                nonlocal steps, sim_n, over
                lab, st = sim.clutter_stable_mask(recs[s], pose7[rows[lo:hi]], joints[rows[lo:hi]], *args, info["close_ctrl"], cfg)
                steps += int(st.sum()); sim_n += hi - lo; over += int(sim.last_aux(hi - lo)["overflow"].sum())
                return lab
            labels[rows] = shard.evaluate_sharded(len(rows), run_range, ENOUGH, chunk=chunk)
        return labels, steps, sim_n, 0, over

    def arm_scenes(enough):
        lab, st = sim.clutter_scenes_stable_mask(recs, si, pose7, joints, *args, info["close_ctrl"], cfg, enough_stable=enough)
        aux = sim.last_aux(len(si))
        if enough:
            for s in range(S):
                lab[si == s] = shard.apply_enough_stable(lab[si == s], enough)
        return lab, int(st.sum()), int(len(si) - aux["skipped"].sum()), int(aux["skipped"].sum()), int(aux["overflow"].sum())

    arms = {"A_per_scene_rounds": arm_a, "B_scenes_device_stop": lambda: arm_scenes(ENOUGH), "C_scenes_no_stop": lambda: arm_scenes(0)}
    res = {k: dict(wall_s=[], env_steps=[], simulated=[], skipped=[], overflowed=[]) for k in arms}
    labels = {}
    sim.clutter_stable_mask(recs[0], pose7[:chunk], joints[:chunk], *args, info["close_ctrl"], mlib.MgsRolloutCfg(50, 50, 0, 0, 0.01, 0.0))
    for r in range(repeats):
        for k, fn in arms.items():
            t = time.perf_counter()
            lab, steps, simulated, skipped, over = fn()
            w = time.perf_counter() - t
            for key, v in zip(("wall_s", "env_steps", "simulated", "skipped", "overflowed"), (w, steps, simulated, skipped, over)):
                res[k][key].append(v)
            labels.setdefault(k, lab)
            print(r, k, f"{w:.1f} s, {steps} env-steps, {simulated} simulated, {skipped} skipped", flush=True)
    out = {}
    for k, v in res.items():
        w = float(np.median(v["wall_s"]))
        out[k] = dict(wall_s=[round(x, 2) for x in v["wall_s"]], median_wall_s=round(w, 2), env_steps=v["env_steps"][0],
                      env_steps_per_s=[round(s / x) for s, x in zip(v["env_steps"], v["wall_s"])], candidates_labelled_per_s=round(len(si) / w, 1),
                      candidates_simulated=v["simulated"][0], skipped=v["skipped"][0], overflowed=v["overflowed"][0],
                      stable_after_prefix_rule=int(labels[k].sum()) if k != "C_scenes_no_stop" else None,
                      stable_raw=int(labels[k].sum()) if k == "C_scenes_no_stop" else None)
    same = bool(np.array_equal(labels["A_per_scene_rounds"], labels["B_scenes_device_stop"]))
    a, b = out["A_per_scene_rounds"]["median_wall_s"], out["B_scenes_device_stop"]["median_wall_s"]
    return dict(arms=out, labels_A_equal_B=same, B_over_A_wall=round(b / a, 3), chunk=chunk, state_in_global=sim.state_in_global,
                ncon_max=sim.info.ncon_max, bytes_per_env=sim.info.smem_bytes_per_env), same


def main():
    S = int(sys.argv[1]) if len(sys.argv) > 1 else 4
    K = int(sys.argv[2]) if len(sys.argv) > 2 else 444
    repeats = int(sys.argv[3]) if len(sys.argv) > 3 else 2
    precisions = sys.argv[4].split(",") if len(sys.argv) > 4 else ["f32", "f64"]
    os.makedirs(OUT, exist_ok=True)
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu == 0:
        raise SystemExit("no CUDA device: this tool measures on the GPU")
    card = dict(name=smi("name"), power_limit=smi("power.limit"), sm_clock=smi("clocks.sm"), sm_clock_max=smi("clocks.max.sm"))
    m, info, recs, pose7, joints, si, t_gen = workload(S, K)
    result = dict(what=f"config 5 (Shadow hand + 10 objects), {S} scenes x {K} candidates, full schedule close 3000 + lift 3000, "
                       f"enough_stable = {ENOUGH}; arms alternated, host entry points, wall time", card=card,
                  scenes=S, candidates_per_scene=K, scene_generation_s_untimed=round(t_gen, 1), precisions={})
    ok = True
    for p in precisions:
        sim = make_sim(m, p)
        result["precisions"][p], same = run_arms(sim, info, recs, pose7, joints, si, repeats)
        ok = ok and same
        sim.close()
    card["sm_clock_after"] = smi("clocks.sm")
    result["gpus_visible"] = ngpu
    result["scene_sharded_n2"] = "not measured"
    print(json.dumps(result), flush=True)
    json.dump(result, open(os.path.join(OUT, "clutter_scenes_bench.json"), "w"), indent=1)
    if not ok:
        raise SystemExit("arms A and B gave different labels")


if __name__ == "__main__":
    main()
