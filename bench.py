#!/usr/bin/env python
"""bench.py - grasp-evaluation rollout throughput on B200 (and the CPU arm beside it).

Workloads (config.workload).  Default = BASELINE.json configs[1] as SURVEY.md 8(d) states it: Robotiq 2F-85 on EIGHT synthetic
convex-hull objects (hull sizes n_v = 16 / 32 / 64, YCB geom recipe), 4096 antipodal-style grasp candidates per object, the
reference's stability rollout (close 3000 + lift 3000 + shake 2000 `mj_step` at dt = 1 ms; failed candidates stop early) - the
loop of /root/reference/mgs/env/gravityless_object_grasping.py:127-295.  A "step" is one full pass of the hot path over ONE
object's 4096 candidates; step k works on object k mod 8, so K >= 8 steps cover all of them.  The same JSON line carries, under
"also", Panda-on-convex (the gripper the north-star's target sentence names; same objects) and - at N = 1 - one line each
for the Allegro and LEAP hands (configs[3]).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--workload robotiq|panda|allegro|leap|mixed|clutter_shadow] [--dump-outputs DIR]

  value  = env-steps/s with inputs resident in HBM, timed with CUDA events on the launch stream
  e2e    = the same metric through the host-pointer C-ABI call (pinned H2D + kernel + D2H inside the call)
  --impl reference = the CPU arm: the fp64 oracle port (MuJoCo is not installable here) on all host threads, on a bounded
           sample of the SAME candidate sets.
  --dump-outputs DIR = after the run, DIR/<line>_labels.npy and DIR/<line>_steps.npy (float32, one value per candidate) hold what
           the last timed step of each line of the JSON result returned (<line> = the workload, or its name under "also"; the
           mixed batch returns labels only, in bucket order).  The inputs are seeded, so two builds can be compared file by file.

Multi-GPU (torchrun, one rank per GPU): robotiq / panda / hands are WEAK scaling - every rank runs the same object sequence, so
a loss of efficiency is the machine's, not a difference in work; `per_rank` holds every rank's kernel time.  `--workload mixed`
is BASELINE configs[2]: 65,536 candidates (8 objects x {vx300, panda} x 4096) as one STRONG-scaling job, bucketed by model,
chunks handed out dynamically (mj_grasp_sim_b200/mixed.py).  `--workload clutter_shadow` is configs[4] at one GPU-filling
batch per rank: the Shadow hand over a settled 10-object clutter scene (environment-per-CTA kernel variant).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_CAND = 4096
N_OBJECTS = 8
HULL_NV = (16, 32, 64)  # object k: seed k, n_v = HULL_NV[k % 3]
ROLLOUT = dict(nstep_close=3000, nstep_lift=3000, shake_steps=500, repose_on_close=0, lift_dist=0.1, shake_dist=0.02)
SCHED_TXT = "close3000+lift3000+shake2000"
# --workload: gripper, explicit per-environment capacities (contacts, constraint rows; 0 = the model's default), description
WORKLOADS = {
    "robotiq": dict(gripper="robotiq2f85", caps=(24, 110), objects=N_OBJECTS,
                    desc=f"configs[1]: robotiq 2f-85 gripper, 8 synthetic convex-hull objects (n_v 16/32/64, ycb recipe), 4096 antipodal candidates per object, one object per step, {SCHED_TXT}"),
    "panda": dict(gripper="panda", caps=(24, 100), objects=N_OBJECTS,
                  desc=f"panda gripper, 8 synthetic convex-hull objects (n_v 16/32/64, ycb recipe), 4096 antipodal candidates per object, one object per step, {SCHED_TXT}"),
    "allegro": dict(gripper="allegro", caps=(0, 0), objects=2, n=1024,
                    desc=f"configs[3]: allegro hand (16 dof, Newton), synthetic convex-hull objects, 1024 candidates per object, one object per step, {SCHED_TXT}"),
    "leap": dict(gripper="leap", caps=(0, 0), objects=2, n=1024,
                 desc=f"configs[3]: leap hand (16 dof, Newton), synthetic convex-hull objects, 1024 candidates per object, one object per step, {SCHED_TXT}"),
}
MIXED_DESC = (f"configs[2]: vx300 + panda mixed batch, 65536 candidates = 8 synthetic convex-hull objects (n_v 16/32/64) x 2 grippers x 4096, "
              f"bucketed by model, sharded over the ranks in GPU-filling chunks (dynamic hand-out), {SCHED_TXT}")
CLUTTER_DESC = ("configs[4]: shadow hand over one settled 10-object clutter scene (24-vertex hulls, gravity, table + walls), top-down candidates, "
                "clutter program close3000+lift1000 with the gripper-contact test every 100 steps")


def b_step(model):
    """Algorithmic HBM bytes per env-step (SURVEY 8(d)): fp32 state in and out once per step."""
    return 4 * (2 * model.nq + 4 * model.nv + model.nu + 7) + 1


def rollout_cfg(gripper):
    from mj_grasp_sim_b200 import scenes
    r = dict(ROLLOUT)
    r["repose_on_close"] = scenes.GRIPPERS[gripper]["repose"]
    return r


def make_object_workload(gripper, k, n=N_CAND):
    from mj_grasp_sim_b200 import scenes
    nv = int(os.environ.get("MGS_BENCH_HULL_NV", "0")) or HULL_NV[k % len(HULL_NV)]  # (MGS_BENCH_HULL_NV=32 MGS_BENCH_OBJECTS=1: round 1's workload)
    return scenes.workload(gripper, "hull", k, n, n_v=nv)


class ClockSampler:
    def __init__(self, index=0):
        self.index, self.rows, self.stop = index, [], False
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons, "samples": len(sm)}


def cpu_arm(model, info, pose7, joints, gripper, target_seconds, threads):
    """Time the oracle port on the first candidates of one set until `target_seconds` have passed;
    returns (env_steps, candidates, seconds)."""
    from oracle.oracle import RolloutCfg, batch
    r = rollout_cfg(gripper)
    cfg = RolloutCfg(r["nstep_close"], r["nstep_lift"], r["shake_steps"], r["repose_on_close"], r["lift_dist"], r["shake_dist"])
    chunk = max(threads * 2, 8)
    done, steps, t0 = 0, 0, time.perf_counter()
    while done < len(pose7):
        sl = slice(done, min(len(pose7), done + chunk))
        _, st = batch(model, 1, pose7[sl].astype(np.float64), info["base_qposadr"], joints[sl].astype(np.float64), info["joint_qposadr"],
                      info["close_ctrl"], cfg, threads)
        steps += int(st.sum())
        done = sl.stop
        if time.perf_counter() - t0 >= target_seconds:
            break
    return steps, done, time.perf_counter() - t0


def run_reference(args, rank, world):
    """CPU arm: the oracle port over all host threads; step k = a bounded sample (the FIRST candidates) of the same candidate set
    the GPU arm's step k evaluates (object k mod 8)."""
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    key = args.workload if args.workload in WORKLOADS else "panda"  # mixed / clutter: the CPU arm reports the Panda leg
    W = WORKLOADS[key]
    threads = os.cpu_count() or 1
    nobj = min(W["objects"], max(1, args.steps))
    sets = [make_object_workload(W["gripper"], k) for k in range(nobj)]
    for j in range(args.warmup):
        m, info, pose7, joints = sets[j % nobj]
        cpu_arm(m, info, pose7[:threads], joints[:threads], W["gripper"], 0.0, threads)
    per_step = max(4.0, min(30.0, 90.0 / max(1, args.steps)))
    steps, cands, t_total = 0, 0, 0.0
    for k in range(args.steps):
        m, info, pose7, joints = sets[k % nobj]
        s, n, dt = cpu_arm(m, info, pose7, joints, W["gripper"], per_step, threads)
        steps += s; cands += n; t_total += dt
    value = steps / t_total
    line = {"impl": "reference", "metric": "env_steps_per_s", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / max(1, args.steps), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": W["desc"] if args.workload in WORKLOADS else (MIXED_DESC if args.workload == "mixed" else CLUTTER_DESC),
                       "sample": f"first {cands // max(1, args.steps)} candidates (mean) of each step's 4096-candidate set, {cands} in total over {args.steps} bounded steps"},
            "grasps_per_s": cands / t_total,
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port", "grasps_per_s": cands / t_total,
                             "sample": f"oracle port (fp64 C restatement, MuJoCo not installable), {cands} candidates, ~{per_step:.0f}s per step"},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def dump_outputs(path, outputs):
    """outputs: {line: {array name: per-candidate array}} -> path/<line>_<array name>.npy in float32 (labels are 0 / 1, step
    counts stay below 2^24, so float32 holds both exactly)."""
    os.makedirs(path, exist_ok=True)
    for line, arrays in outputs.items():
        for name, a in arrays.items():
            np.save(os.path.join(path, f"{line}_{name}.npy"), np.asarray(a, dtype=np.float32))


def load_json(*path):
    try:
        return json.load(open(os.path.join(ROOT, *path)))
    except Exception:
        return {}


def run_ours(args, rank, world, local_rank):
    import torch
    from mj_grasp_sim_b200 import scenes
    from mj_grasp_sim_b200.lib import BatchSim, MgsRolloutCfg, load
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a CUDA device: the rollout path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = load()
    dev = torch.device("cuda", local_rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream = torch.cuda.current_stream()
    peaks = load_json("MEASURED_PEAKS.json")
    peak = float(peaks.get("hbm_gbs", 6650.0))
    # per workload: dram bytes of one rollout launch (tools/ncu_traffic.py) and warp-instructions per env-step of the steady hold
    # phase (tools/ncu_summary.py --json) - both derived by committed scripts from ncu captures, nothing typed in here
    traffic = load_json("profiles", "traffic_r2.json") or load_json("profiles", "traffic_r1.json")
    issue = load_json("profiles", "issue_slots_r2.json")
    outputs = {} if args.dump_outputs else None  # line -> arrays of its last timed step (--dump-outputs)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_ranks(x):
        """float per rank -> list over ranks (on every rank)"""
        if dist is None:
            return [float(x)]
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        out = torch.empty(world, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(out, t)
        return out.cpu().tolist()

    def per_rank_block(dev_s_list, e2e_s_list, steps_list):
        a = np.array(dev_s_list)
        return {"kernel_s": [round(x, 4) for x in dev_s_list], "kernel_s_min": float(a.min()), "kernel_s_mean": float(a.mean()), "kernel_s_max": float(a.max()),
                "e2e_s": [round(x, 4) for x in e2e_s_list], "env_steps": [int(x) for x in steps_list]}

    def roofline(key, bs, steps_per_launch, mean_launch_s):
        achieved = bs * steps_per_launch / mean_launch_s / 1e9
        tr = traffic.get(key, {})
        return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": tr.get("bytes_per_launch"), "traffic_gbs": tr.get("gbs"), "traffic_source": tr.get("source"),
                "algorithmic_bytes_per_launch": bs * steps_per_launch, "kernel": "mgs_rollout_kernel", "bytes_per_env_step": bs,
                "peak_source": "MEASURED_PEAKS.json (of measured)" if peaks else "fallback 6.65 TB/s (of fallback)",
                "note": "state stays in shared memory for the whole rollout; the kernel is issue/latency bound, not HBM bound (see issue_slots)"}

    def issue_block(key, value_per_gpu, mhz):
        it = issue.get(key)
        if not it:
            return None
        ipe = float(it["warp_instr_per_env_step"])
        peak_issue = 148 * 4 * (mhz or 1965.0) * 1e6
        return {"warp_instr_per_env_step": ipe, "source": it.get("source"), "achieved_ginst_s": ipe * value_per_gpu / 1e9,
                "peak_ginst_s": peak_issue / 1e9, "frac": ipe * value_per_gpu / peak_issue}

    # ------------------------------------------------------------------------------------------------ single-model workloads
    def measure(key, steps, warmup, with_cpu, line=None):
        """W warm-up + K timed passes on device-resident inputs (CUDA events), then K passes through the host-pointer C ABI.
        Step k works on object k mod n_objects.  Returns the JSON fields of that workload (rank 0) or None.  `line`: the name
        of its outputs (default: key)."""
        W = WORKLOADS[key]
        gripper = W["gripper"]
        N_CAND = W.get("n", 4096)
        ncon_max, nefc_max = W["caps"]
        if args.caps and key == args.workload:
            ncon_max, nefc_max = (int(x) for x in args.caps.split(","))
        f64 = gripper in scenes.F64_GRIPPERS and os.environ.get("MGS_PRECISION", "").lower() != "f32"  # precision policy of the product path
        cfg = MgsRolloutCfg(**rollout_cfg(gripper))
        nobj = min(int(os.environ.get("MGS_BENCH_OBJECTS", "0")) or W["objects"], max(steps, 1))
        sets = []
        for k in range(nobj):
            model, info, pose7, joints = make_object_workload(gripper, k, N_CAND)
            sim = BatchSim(model, device=local_rank, ncon_max=ncon_max, nefc_max=nefc_max, f64=f64)
            sets.append(dict(model=model, info=info, pose7=pose7, joints=joints, sim=sim, d_pose=torch.from_numpy(pose7).to(dev),
                             d_joint=torch.from_numpy(joints).to(dev)))
        d_lab = torch.zeros(N_CAND, dtype=torch.uint8, device=dev)
        d_steps = torch.zeros(N_CAND, dtype=torch.int32, device=dev)
        L = load(f64)

        def one_step(k):
            s = sets[k % nobj]
            s["sim"].rollout_device(2, N_CAND, s["d_pose"].data_ptr(), s["d_joint"].data_ptr(), s["joints"].shape[1], s["info"]["joint_qposadr"],
                                    s["info"]["base_qposadr"], s["info"]["close_ctrl"], cfg, d_lab.data_ptr(), d_steps.data_ptr(), stream.cuda_stream)

        for j in range(warmup):
            flush.fill_(1)
            one_step(j)
        barrier()
        launches0 = L.mgs_launch_count()
        kern_ms, total_steps, overflowed, stable = [], 0, 0, 0
        with ClockSampler(local_rank) as clk:
            barrier()
            t_begin = time.perf_counter()
            for k in range(steps):
                flush.fill_(1)  # L2 flush between timed iterations
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                one_step(k)
                e1.record(stream)
                e1.synchronize()
                kern_ms.append(e0.elapsed_time(e1))
                total_steps += int(d_steps.sum().item())
                stable += int(d_lab.sum().item())
                overflowed += sets[k % nobj]["sim"].overflow_count()
            barrier()
            t_wall = time.perf_counter() - t_begin
        if outputs is not None:
            outputs[line or key] = dict(labels=d_lab.cpu().numpy(), steps=d_steps.cpu().numpy())
        launches = sum(gather_ranks(L.mgs_launch_count() - launches0))
        dev_s = sum(kern_ms) / 1e3
        # end-to-end through the host-pointer C ABI (pinned staging, H2D + kernel + D2H inside the call)
        barrier()
        e2e_steps, t0 = 0, time.perf_counter()
        for k in range(steps):
            s = sets[k % nobj]
            lab, st = s["sim"].stability(s["pose7"], s["joints"], s["info"]["joint_qposadr"], s["info"]["base_qposadr"], s["info"]["close_ctrl"], cfg)
            e2e_steps += int(st.sum())
        barrier()
        e2e_s = time.perf_counter() - t0
        dev_l, e2e_l, st_l, e2e_st_l = gather_ranks(dev_s), gather_ranks(e2e_s), gather_ranks(total_steps), gather_ranks(e2e_steps)
        stable_l, over_l = gather_ranks(stable), gather_ranks(overflowed)
        if dist is not None:
            # the only data-path exchange: gather the success labels (uint8[N] per rank) on every rank
            gathered = torch.empty(world * N_CAND, dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(gathered, d_lab)
        out = None
        if rank == 0:
            model0, sim0 = sets[0]["model"], sets[0]["sim"]
            dev_max, e2e_max = max(dev_l), max(e2e_l)
            value = sum(st_l) / dev_max
            bs = b_step(model0)
            clocks = clk.summary()
            out = {"metric": "env_steps_per_s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": steps,
                   "warmup": warmup, "ms_per_step": 1e3 * dev_max / steps, "higher_is_better": True, "scaling": "weak",
                   "vs_baseline": None, "dtype": "f64" if f64 else "f32", "data": "synthetic",
                   "config": {"workload": W["desc"], "candidates_per_gpu_per_step": N_CAND, "objects": nobj, "hull_vertices": [HULL_NV[k % 3] for k in range(nobj)],
                              "per_rank_work": "identical (every rank runs the same object sequence)",
                              "l2": "flushed between timed iterations (256 MiB fill)",
                              "stable_fraction": sum(stable_l) / (world * N_CAND * steps),
                              "capacity": {"ncon_max": sim0.info.ncon_max, "nefc_max": sim0.info.nefc_max, "envs_overflowed": int(sum(over_l)),
                                           "of_candidates": world * N_CAND * steps,
                                           "policy": "first-pass capacities; an environment over capacity is flagged per candidate and the product path (mgs.env) re-runs it on larger ones - not done inside this timed region"},
                              "envs_per_sm": sim0.info.warps_per_block * sim0.info.blocks_per_sm, "smem_bytes_per_env": sim0.info.smem_bytes_per_env},
                   "grasps_per_s": world * N_CAND * steps / dev_max,
                   "e2e": {"value": sum(e2e_st_l) / e2e_max, "unit": "env-steps/s", "h2d_bytes_per_step": int(sets[0]["pose7"].nbytes + sets[0]["joints"].nbytes),
                           "d2h_bytes_per_step": int(N_CAND * 5), "grasps_per_s": world * N_CAND * steps / e2e_max},
                   "gpu_launches": int(launches),
                   "roofline": roofline(key, bs, total_steps / steps, float(np.mean(kern_ms)) / 1e3),
                   "per_rank": per_rank_block(dev_l, e2e_l, st_l),
                   "clocks": clocks, "wall_s": t_wall}
            ib = issue_block(key, value / world, clocks.get("sm_mhz"))
            if ib:
                out["issue_slots"] = ib
            if with_cpu:
                from oracle import oracle as orc
                orc.build()
                threads = os.cpu_count() or 1
                s = sets[0]
                st, n, dt = cpu_arm(s["model"], s["info"], s["pose7"], s["joints"], gripper, 12.0, threads)
                out["cpu_baseline"] = {"value": st / dt, "unit": "env-steps/s", "cores": threads, "kind": "port", "grasps_per_s": n / dt,
                                       "sample": f"oracle port (fp64 C restatement; MuJoCo not installable offline), first {n} of object 0's {N_CAND} candidates, {dt:.1f}s"}
        for s in sets:
            s["sim"].close()
        return out

    # ------------------------------------------------------------------------------------------------ cfg3: mixed batch
    def measure_mixed(steps, warmup):
        from mj_grasp_sim_b200.mixed import Bucket, run_mixed
        cfgs, sets = {}, []
        # bucket order: all Panda buckets, then all VX300 buckets - ranks pull from the queue in turn, and an alternating list would
        # hand every Panda bucket to one rank and every VX300 bucket to the other (measured at N = 2: 27.6 s vs 32.3 s of kernel time)
        for gripper, caps in (("panda", WORKLOADS["panda"]["caps"]), ("vx300", (24, 100))):
            for k in range(N_OBJECTS):
                model, info, pose7, joints = make_object_workload(gripper, k)
                sim = BatchSim(model, device=local_rank, ncon_max=caps[0], nefc_max=caps[1])
                cfgs[gripper] = MgsRolloutCfg(**rollout_cfg(gripper))
                sets.append(dict(name=f"{gripper}:hull{k}", gripper=gripper, model=model, info=info, pose7=pose7, joints=joints, sim=sim,
                                 d_pose=torch.from_numpy(pose7).to(dev), d_joint=torch.from_numpy(joints).to(dev),
                                 d_lab=torch.zeros(N_CAND, dtype=torch.uint8, device=dev), d_steps=torch.zeros(N_CAND, dtype=torch.int32, device=dev)))
        host = [False]

        def runner(s):
            def run(lo, hi):
                n = hi - lo
                if host[0]:  # end-to-end leg: host arrays through the host-pointer ABI
                    t0 = time.perf_counter()
                    lab, st = s["sim"].stability(s["pose7"][lo:hi], s["joints"][lo:hi], s["info"]["joint_qposadr"], s["info"]["base_qposadr"],
                                                 s["info"]["close_ctrl"], cfgs[s["gripper"]])
                    return lab, int(st.sum()), time.perf_counter() - t0
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                nj = s["joints"].shape[1]
                s["sim"].rollout_device(2, n, s["d_pose"].data_ptr() + lo * 28, s["d_joint"].data_ptr() + lo * nj * 4, nj, s["info"]["joint_qposadr"],
                                        s["info"]["base_qposadr"], s["info"]["close_ctrl"], cfgs[s["gripper"]], s["d_lab"].data_ptr() + lo,
                                        s["d_steps"].data_ptr() + lo * 4, stream.cuda_stream)
                e1.record(stream)
                e1.synchronize()
                return s["d_lab"][lo:hi].cpu().numpy(), int(s["d_steps"][lo:hi].sum().item()), e0.elapsed_time(e1) / 1e3
            return run
        buckets = [Bucket(s["name"], N_CAND, runner(s), 1.0) for s in sets]
        info0 = sets[0]["sim"].info
        # one hand-out = one wave of resident environments at the CTA size a whole-bucket launch would use (4096 Panda candidates
        # run as 2 waves of 14 environments per SM: chunk = 14 x 148 = 2072), so a chunk costs the same per candidate as a full launch
        slots = info0.warps_per_block * info0.blocks_per_sm * info0.num_sms
        waves = -(-N_CAND // slots)
        chunk = min(N_CAND, -(-N_CAND // (waves * info0.num_sms)) * info0.num_sms)
        # ... unless there are plenty of buckets per rank: inside ONE launch the second wave starts warp by warp as the first one drains,
        # two launches have a full stop between them (measured at N = 1: 8.44 M env-steps/s with whole buckets, 7.10 M with one-wave chunks)
        if len(sets) >= 4 * world:
            chunk = N_CAND
        for _ in range(warmup):
            flush.fill_(1)
            run_mixed(buckets[:2 * min(world, N_OBJECTS)], N_CAND, device=dev)  # warm-up: one launch of each model per rank
        barrier()
        launches0 = lib.mgs_launch_count()
        tot = dict(kernel_s=0.0, env_steps=0, chunks=0, candidates=0)
        stable, overflowed = 0, 0
        with ClockSampler(local_rank) as clk:
            barrier()
            t_begin = time.perf_counter()
            for _ in range(steps):
                flush.fill_(1)
                labels, st = run_mixed(buckets, chunk, device=dev)
                for k in tot:
                    tot[k] += st[k]
                stable += int(sum(l.sum() for l in labels))
            barrier()
            t_wall = time.perf_counter() - t_begin
        if outputs is not None:
            outputs["mixed"] = dict(labels=np.concatenate(labels))
        launches = sum(gather_ranks(lib.mgs_launch_count() - launches0))
        host[0] = True
        barrier()
        t0 = time.perf_counter()
        e2e_steps = 0
        for _ in range(steps):
            labels, st = run_mixed(buckets, chunk, device=dev)
            e2e_steps += st["env_steps"]
        barrier()
        e2e_s = time.perf_counter() - t0
        dev_l, st_l, ch_l = gather_ranks(tot["kernel_s"]), gather_ranks(tot["env_steps"]), gather_ranks(tot["chunks"])
        e2e_l, e2e_st_l = gather_ranks(e2e_s), gather_ranks(e2e_steps)
        out = None
        if rank == 0:
            n_total = N_CAND * len(sets)
            dev_max = max(dev_l)
            value = sum(st_l) / dev_max
            bs = b_step(sets[0]["model"])
            out = {"metric": "env_steps_per_s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": steps, "warmup": warmup,
                   "ms_per_step": 1e3 * dev_max / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                   "data": "synthetic",
                   "config": {"workload": MIXED_DESC, "candidates_total": n_total, "buckets": len(sets), "chunk": chunk,
                              "hand_out": "dynamic (atomic counter in the rendezvous store)" if world > 1 else "sequential",
                              "l2": "flushed between timed iterations (256 MiB fill)", "stable_fraction": stable / (n_total * steps)},
                   "grasps_per_s": n_total * steps / dev_max,
                   "e2e": {"value": sum(e2e_st_l) / max(e2e_l), "unit": "env-steps/s", "h2d_bytes_per_step": int(sum(s["pose7"].nbytes + s["joints"].nbytes for s in sets)),
                           "d2h_bytes_per_step": int(n_total * 5), "grasps_per_s": n_total * steps / max(e2e_l)},
                   "gpu_launches": int(launches),
                   "roofline": roofline("panda", bs, sum(st_l) / max(1, sum(ch_l)), sum(dev_l) / max(1, sum(ch_l))),
                   "per_rank": dict(per_rank_block(dev_l, e2e_l, st_l), chunks=[int(c) for c in ch_l]),
                   "clocks": clk.summary(), "wall_s": t_wall}
        for s in sets:
            s["sim"].close()
        return out

    # ------------------------------------------------------------------------------------------------ cfg5: shadow in clutter
    def measure_clutter(steps, warmup, with_cpu):
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import clutter_shadow_bench as csb
        return csb.measure(args, rank, world, local_rank, steps, warmup, with_cpu, dict(
            torch=torch, dist=dist, dev=dev, flush=flush, stream=stream, barrier=barrier, gather_ranks=gather_ranks, per_rank_block=per_rank_block,
            roofline=roofline, ClockSampler=ClockSampler, desc=CLUTTER_DESC, cpu_arm=None, outputs=outputs))

    with_cpu = world == 1 and not args.no_cpu
    if args.workload == "mixed":
        line = measure_mixed(args.steps, args.warmup)
    elif args.workload == "clutter_shadow":
        line = measure_clutter(args.steps, args.warmup, with_cpu)
    else:
        line = measure(args.workload, args.steps, args.warmup, with_cpu)
    also = {}
    if args.workload == "robotiq" and not args.no_also:
        # secondary workloads in the same line.  Panda on convex objects = the gripper the north-star's target sentence names;
        # the two 16-dof hands (configs[3]) only at N = 1 and with few steps: they are reported, not the headline
        side = [("panda_on_convex", "panda", min(args.steps, 8), 3, with_cpu)]
        if world == 1 and not args.no_hands:
            side += [("allegro", "allegro", 1, 2, False), ("leap", "leap", 1, 2, False)]
        for name, key, k, w, cpu in side:
            r = measure(key, k, w, cpu, line=name)
            if rank == 0:
                also[name] = {q: r[q] for q in ("value", "unit", "steps", "warmup", "ms_per_step", "grasps_per_s", "dtype", "e2e", "config", "roofline", "issue_slots",
                                                  "gpu_launches", "per_rank", "cpu_baseline") if q in r}
    if rank == 0:
        if also:
            line["also"] = also
            line["gpu_launches"] += sum(a["gpu_launches"] for a in also.values())
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="robotiq", choices=sorted(WORKLOADS) + ["mixed", "clutter_shadow"], help="robotiq = BASELINE.json configs[1] (default)")
    ap.add_argument("--no-also", action="store_true", help="skip the secondary measurements (Panda-on-convex, hands)")
    ap.add_argument("--no-hands", action="store_true", help="skip the Allegro / LEAP lines")
    ap.add_argument("--caps", default="", help="override the primary workload's per-environment capacities: ncon_max,nefc_max")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the labels and step counts of each line's last timed step to DIR/<line>_<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the CPU arm evaluates a time-bounded sample, not a fixed set)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
