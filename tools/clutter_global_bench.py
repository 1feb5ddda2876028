"""Config 5 with the environment state in global memory (kernel variant wide_g) against the shared-memory kernel, in one GPU process.

Scene and candidates of bench.py --workload clutter_shadow (tools/clutter_shadow_bench.py): the Shadow hand over ten hull objects
settled by the fp32 kernel (seed 7, the same record for every arm), 296 candidates per step (two per SM), the full schedule
(close 3000 + lift 0.3 m over 3000 steps), L2 flushed (256 MiB fill) before every timed step.  Three arms, alternated, three
timed steps each after one warm-up step per arm:
  f32_wide    fp32, 80 contacts, state in shared memory        (the bench line's configuration)
  f32_wide_g  fp32, 80 contacts, state in global memory        (what the address space alone costs)
  f64_wide_g  fp64, default 64 contacts, state in global memory (the product path of ClutterTableEnv with the Shadow hand)
Per arm: env-steps/s over device time (CUDA events), environments over capacity, and the labels of the first K candidates
against the oracle on the same schedule.  Before that, a short A/B of the L1/shared carveout of wide_g (MGS_CARVEOUT), and after
it tools/cfg5_labels.py at fp64, n = 256.  Card name, power limit and SM clocks are recorded in the same process.

On a B200: python tools/clutter_global_bench.py -> $MGS_OUT_DIR/clutter_global_bench.json (+ cfg5_labels_f64.json; default: the
current directory)"""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402
from mj_grasp_sim_b200 import scenes, lib as mlib  # noqa: E402
from oracle import oracle as orc  # noqa: E402
import clutter_shadow_bench as csb  # noqa: E402

OUT = os.environ.get("MGS_OUT_DIR", ".")
REPEATS, K_ORACLE = 3, 16
ARMS = {"f32_wide": dict(f64=False, variant="wide", ncon=csb.NCON_MAX),
        "f32_wide_g": dict(f64=False, variant="wide_g", ncon=csb.NCON_MAX),
        "f64_wide_g": dict(f64=True, variant=None, ncon=0)}


def smi(q):
    try:
        return subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=10).stdout.strip()
    except Exception as ex:
        return f"unavailable ({ex})"


def make_sim(m, arm):
    old = os.environ.pop("MGS_KERNEL_VARIANT", None)
    if arm["variant"]:
        os.environ["MGS_KERNEL_VARIANT"] = arm["variant"]
    try:
        return mlib.BatchSim(m, ground_name="geom:table", ncon_max=arm["ncon"], f64=arm["f64"], global_fallback=True)
    finally:
        os.environ.pop("MGS_KERNEL_VARIANT", None)
        if old is not None:
            os.environ["MGS_KERNEL_VARIANT"] = old


def main():
    os.makedirs(OUT, exist_ok=True)
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(dev)
    flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)  # 256 MiB > 126 MB of L2
    card = dict(name=smi("name"), power_limit=smi("power.limit"), sm_clock=smi("clocks.sm"), sm_clock_max=smi("clocks.max.sm"))
    m, info = scenes.build_clutter_scene("shadow", list(range(10)))
    sims = {k: make_sim(m, a) for k, a in ARMS.items()}
    gen = sims["f32_wide"]
    rec = scenes.gen_clutter(m, info, lambda r, k: gen.step(r[None].astype(np.float32), k)[0].astype(np.float64), 7)
    n = csb.N_PER_SM * gen.info.num_sms
    pose7, joints = csb.make_inputs(scenes, m, info, rec, n)
    jadr = np.ascontiguousarray(info["joint_qposadr"], dtype=np.int32)
    cc = np.ascontiguousarray(info["close_ctrl"], dtype=np.float64)
    d_pose, d_joint = torch.from_numpy(pose7).to(dev), torch.from_numpy(joints).to(dev)
    d_lab = torch.zeros(n, dtype=torch.uint8, device=dev)
    d_steps = torch.zeros(n, dtype=torch.int32, device=dev)
    d_scene = {k: torch.from_numpy(rec.astype(s.real)).to(dev) for k, s in sims.items()}
    L = {k: mlib.load(a["f64"]) for k, a in ARMS.items()}
    for lib in L.values():
        lib.mgs_clutter_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_int,
                                           C.POINTER(C.c_double), C.POINTER(mlib.MgsRolloutCfg), C.c_void_p, C.c_void_p, C.c_void_p]

    def timed(k, cfg, count):
        """one launch of `count` candidates of arm k on `stream` after an L2 flush: (device ms, env-steps, labels, overflowed)"""
        s = sims[k]
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            rc = L[k].mgs_clutter_device(s.h, 4, count, d_scene[k].data_ptr(), d_pose.data_ptr(), d_joint.data_ptr(), joints.shape[1],
                                         jadr.ctypes.data_as(C.POINTER(C.c_int)), int(info["base_qposadr"]), cc.ctypes.data_as(C.POINTER(C.c_double)),
                                         C.byref(cfg), d_lab.data_ptr(), d_steps.data_ptr(), stream.cuda_stream)
            s._check(rc)
            e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1), int(d_steps[:count].sum().item()), d_lab[:count].cpu().numpy().astype(bool), s.overflow_count()

    # carveout of wide_g (fp64 product path): max L1 (the library's choice) vs the driver default, alternated, short schedule, one wave
    short = mlib.MgsRolloutCfg(300, 200, 0, 0, 0.02, 0.0)
    carve = {"max_l1": [], "default": []}
    timed("f64_wide_g", short, gen.info.num_sms)
    for _ in range(REPEATS):
        for c in carve:
            if c == "default":
                os.environ["MGS_CARVEOUT"] = "default"
            ms, steps, _, _ = timed("f64_wide_g", short, gen.info.num_sms)
            os.environ.pop("MGS_CARVEOUT", None)
            carve[c].append(steps / ms * 1e3)
    print("carveout A/B (fp64 wide_g, env-steps/s):", {c: [round(v) for v in r] for c, r in carve.items()}, flush=True)

    full = mlib.MgsRolloutCfg(*csb.SCHED)
    res = {k: dict(rate=[], ms=[], overflowed=[], labels=None) for k in ARMS}
    for k in ARMS:
        timed(k, full, n)  # warm-up
    for r in range(REPEATS):
        for k in ARMS:
            ms, steps, lab, over = timed(k, full, n)
            res[k]["rate"].append(steps / ms * 1e3)
            res[k]["ms"].append(ms)
            res[k]["overflowed"].append(over)
            if res[k]["labels"] is None:
                res[k]["labels"] = lab
                res[k]["stable_fraction"] = float(lab.mean())
            else:
                res[k]["labels_repeat_identical"] = bool(np.array_equal(res[k]["labels"], lab))
            print(r, k, f"{steps / ms * 1e3:.0f} env-steps/s, {ms:.0f} ms, {over} over capacity", flush=True)
    card["sm_clock_after"] = smi("clocks.sm")
    t = time.time()
    a = (pose7[:K_ORACLE].astype(np.float64), info["base_qposadr"], joints[:K_ORACLE].astype(np.float64), info["joint_qposadr"], info["close_ctrl"],
         orc.RolloutCfg(*csb.SCHED), os.cpu_count() or 1)
    olab, _ = orc.batch(m, 3, *a, scene=rec, ground_name="geom:table")
    t_or = time.time() - t
    olab = olab.astype(bool)
    arms = {}
    for k, r in res.items():
        s = sims[k]
        arms[k] = dict(env_steps_per_s=[round(v) for v in r["rate"]], median_env_steps_per_s=round(float(np.median(r["rate"]))),
                       ms_per_step=[round(v, 1) for v in r["ms"]], envs_over_capacity=r["overflowed"], of_candidates=n,
                       stable_fraction=r["stable_fraction"], labels_repeat_identical=r.get("labels_repeat_identical"),
                       labels_equal_oracle_first_k=float((r["labels"][:K_ORACLE] == olab).mean()),
                       precision="f64" if ARMS[k]["f64"] else "f32", state_in_global=s.state_in_global, ncon_max=s.info.ncon_max,
                       nefc_max=s.info.nefc_max, bytes_per_env=s.info.smem_bytes_per_env, blocks_per_sm=s.info.blocks_per_sm)
    out = dict(what="config 5 (Shadow hand + 10 objects, nv = 94), full schedule close 3000 + lift 3000, %d candidates per step, "
                    "L2 flushed before every timed step; arms alternated, %d timed steps each after one warm-up" % (n, REPEATS),
               card=card, carveout_ab_fp64_wide_g_short_schedule={c: [round(v) for v in r] for c, r in carve.items()},
               arms=arms, oracle_sample=dict(k=K_ORACLE, stable_fraction=float(olab.mean()), seconds=round(t_or, 1), threads=os.cpu_count()),
               labels_f64_vs_f32_wide_equal=float((res["f64_wide_g"]["labels"] == res["f32_wide"]["labels"]).mean()),
               labels_f32_wide_g_vs_f32_wide_equal=float((res["f32_wide_g"]["labels"] == res["f32_wide"]["labels"]).mean()))
    print(json.dumps(out), flush=True)
    json.dump(out, open(os.path.join(OUT, "clutter_global_bench.json"), "w"), indent=1)
    for s in sims.values():
        s.close()
    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "cfg5_labels.py"), "256", "f64"], check=True)


if __name__ == "__main__":
    main()
