"""bench.py --workload clutter_shadow: BASELINE.json configs[4] on one GPU-filling batch per rank.

Scene: the Shadow hand over TEN 24-vertex hull objects dropped and settled on the clutter table by the same kernel
(scenes.gen_clutter = ClutterTableEnv.gen_clutter, /root/reference/mgs/env/clutter_table.py:197-222; untimed set-up), nv = 94.
Step: ClutterTableEnv.grasp_stable_mask's loop body (clutter_table.py:288-317, reference defaults: close 3000 steps, lift 0.3 m
over 3000 steps with the gripper-contact test every 100 steps) for N top-down candidates.  The model runs the
environment-per-CTA kernel variant (one 256-thread CTA per environment, one environment per SM).
Weak scaling: every rank evaluates the same N candidates of the same scene (1 M candidates over 8 GPUs = 422 such batches per rank).
"""
import os
import time

import numpy as np

N_PER_SM = 2       # candidates per SM and step: two waves of the one resident environment
SCHED = (3000, 3000, 0, 0, 0.3, 0.0)
NCON_MAX = 80      # contacts per environment (370 rows): what fits next to the dense 94 x 94 Newton Hessian in one SM's shared memory


def b_step(model):
    return 4 * (2 * model.nq + 4 * model.nv + model.nu + 7) + 1


def make_inputs(scenes, m, info, rec, n):
    H, w = scenes.clutter_candidates(m, info, rec, n, 2)
    g = scenes.GRIPPERS["shadow"]
    Rt = np.array([[0.0, 0.0, 1.0], [-1.0, 0.0, 0.0], [0.0, -1.0, 0.0]])
    T = np.eye(4)
    T[:3, :3] = Rt
    T[:3, 3] = -Rt @ np.array([0.01, -0.06, 0.12])
    pose7 = scenes.process_poses(H @ T, "shadow")
    jid = [m.names["joint"][j] for j in g["joints"]]
    joints = np.clip(np.asarray(g["open_pose"])[None] + np.random.default_rng(3).normal(scale=0.05, size=(n, 22)), m.jnt_range[jid, 0], m.jnt_range[jid, 1])
    return pose7.astype(np.float32), joints.astype(np.float32)


def measure(args, rank, world, local_rank, steps, warmup, with_cpu, ctx):
    from mj_grasp_sim_b200 import scenes
    from mj_grasp_sim_b200.lib import BatchSim, MgsRolloutCfg, load
    torch, dev, flush, stream = ctx["torch"], ctx["dev"], ctx["flush"], ctx["stream"]
    f64 = os.environ.get("MGS_PRECISION", "").lower() == "f64"  # (the fp64 build of the nv = 94 scene does not fit one SM at this capacity)
    m, info = scenes.build_clutter_scene("shadow", list(range(10)))
    ncon = int(args.caps.split(",")[0]) if args.caps else NCON_MAX
    sim = BatchSim(m, device=local_rank, ground_name="geom:table", ncon_max=ncon, f64=f64)
    L = load(f64)
    t0 = time.perf_counter()
    step_fn = lambda r, k: sim.step(r[None].astype(sim.real), k)[0].astype(np.float64)
    rec = scenes.gen_clutter(m, info, step_fn, 7)
    t_scene = time.perf_counter() - t0
    n = N_PER_SM * sim.info.num_sms * sim.info.warps_per_block * sim.info.blocks_per_sm
    pose7, joints = make_inputs(scenes, m, info, rec, n)
    cfg = MgsRolloutCfg(*SCHED)
    d_scene = torch.from_numpy(rec.astype(sim.real)).to(dev)
    d_pose, d_joint = torch.from_numpy(pose7).to(dev), torch.from_numpy(joints).to(dev)
    d_lab = torch.zeros(n, dtype=torch.uint8, device=dev)
    d_steps = torch.zeros(n, dtype=torch.int32, device=dev)
    jadr = np.ascontiguousarray(info["joint_qposadr"], dtype=np.int32)
    cc = np.ascontiguousarray(info["close_ctrl"], dtype=np.float64)
    import ctypes as C
    L.mgs_clutter_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_int,
                                     C.POINTER(C.c_double), C.POINTER(MgsRolloutCfg), C.c_void_p, C.c_void_p, C.c_void_p]

    def one_step():
        rc = L.mgs_clutter_device(sim.h, 4, n, d_scene.data_ptr(), d_pose.data_ptr(), d_joint.data_ptr(), joints.shape[1], jadr.ctypes.data_as(C.POINTER(C.c_int)),
                                  int(info["base_qposadr"]), cc.ctypes.data_as(C.POINTER(C.c_double)), C.byref(cfg), d_lab.data_ptr(), d_steps.data_ptr(), stream.cuda_stream)
        sim._check(rc)

    for _ in range(warmup):
        flush.fill_(1)
        one_step()
    ctx["barrier"]()
    launches0 = L.mgs_launch_count()
    kern_ms, total_steps, overflowed, stable = [], 0, 0, 0
    with ctx["ClockSampler"](local_rank) as clk:
        ctx["barrier"]()
        t_begin = time.perf_counter()
        for _ in range(steps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            one_step()
            e1.record(stream)
            e1.synchronize()
            kern_ms.append(e0.elapsed_time(e1))
            total_steps += int(d_steps.sum().item())
            stable += int(d_lab.sum().item())
            overflowed += sim.overflow_count()
        ctx["barrier"]()
        t_wall = time.perf_counter() - t_begin
    if ctx["outputs"] is not None:
        ctx["outputs"]["clutter_shadow"] = dict(labels=d_lab.cpu().numpy(), steps=d_steps.cpu().numpy())
    launches = sum(ctx["gather_ranks"](L.mgs_launch_count() - launches0))
    dev_s = sum(kern_ms) / 1e3
    ctx["barrier"]()
    e2e_steps, t0 = 0, time.perf_counter()
    for _ in range(steps):
        lab, st = sim.clutter_stable_mask(rec, pose7, joints, info["joint_qposadr"], info["base_qposadr"], info["close_ctrl"], cfg)
        e2e_steps += int(st.sum())
    ctx["barrier"]()
    e2e_s = time.perf_counter() - t0
    g = ctx["gather_ranks"]
    dev_l, e2e_l, st_l, e2e_st_l, stable_l, over_l = g(dev_s), g(e2e_s), g(total_steps), g(e2e_steps), g(stable), g(overflowed)
    out = None
    if rank == 0:
        dev_max, e2e_max = max(dev_l), max(e2e_l)
        value = sum(st_l) / dev_max
        bs = b_step(m)
        out = {"metric": "env_steps_per_s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": steps, "warmup": warmup,
               "ms_per_step": 1e3 * dev_max / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64" if f64 else "f32",
               "data": "synthetic",
               "config": {"workload": ctx["desc"], "candidates_per_gpu_per_step": n, "nv": int(m.nv), "geom_pairs": int(len(m.pair_geom1)),
                          "kernel_variant": f"{sim.info.lanes_per_env} threads per environment, {sim.info.warps_per_block * sim.info.blocks_per_sm} environment(s) per SM",
                          "per_rank_work": "identical (every rank evaluates the same candidates of the same scene)",
                          "l2": "flushed between timed iterations (256 MiB fill)", "stable_fraction": sum(stable_l) / (world * n * steps),
                          "capacity": {"ncon_max": sim.info.ncon_max, "nefc_max": sim.info.nefc_max, "envs_overflowed": int(sum(over_l)), "of_candidates": world * n * steps},
                          "smem_bytes_per_env": sim.info.smem_bytes_per_env, "scene_generation_s_untimed": round(t_scene, 1)},
               "grasps_per_s": world * n * steps / dev_max,
               "e2e": {"value": sum(e2e_st_l) / e2e_max, "unit": "env-steps/s", "h2d_bytes_per_step": int(pose7.nbytes + joints.nbytes + rec.size * 4),
                       "d2h_bytes_per_step": int(n * 5), "grasps_per_s": world * n * steps / e2e_max},
               "gpu_launches": int(launches),
               "roofline": ctx["roofline"]("clutter_shadow", bs, total_steps / steps, float(np.mean(kern_ms)) / 1e3),
               "per_rank": ctx["per_rank_block"](dev_l, e2e_l, st_l), "clocks": clk.summary(), "wall_s": t_wall}
        if with_cpu:
            from oracle import oracle as orc
            orc.build()
            threads = os.cpu_count() or 1
            k = min(n, max(threads, 8))
            t0 = time.perf_counter()
            olab, osteps = orc.batch(m, 3, pose7[:k].astype(np.float64), info["base_qposadr"], joints[:k].astype(np.float64), info["joint_qposadr"], info["close_ctrl"],
                                     orc.RolloutCfg(*SCHED), threads, scene=rec, ground_name="geom:table")
            dt = time.perf_counter() - t0
            d_lab_h = d_lab.cpu().numpy().astype(bool)
            out["cpu_baseline"] = {"value": float(osteps.sum()) / dt, "unit": "env-steps/s", "cores": threads, "kind": "port", "grasps_per_s": k / dt,
                                   "sample": f"oracle port (fp64 C restatement), first {k} of the step's {n} candidates, {dt:.1f}s",
                                   "labels_equal_on_sample": float((d_lab_h[:k] == olab).mean())}
    sim.close()
    return out
