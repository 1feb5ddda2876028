// mgs_rollout.cuh - the fused per-candidate programs (reference L4 logic on the device).
//
//   MGS_MODE_COLLISION : grasp_collision_mask body   (gravityless_object_grasping.py:112-122)
//   MGS_MODE_STABILITY : grasp_stability_evaluation_from_joints body (:158-277): reset, place,
//                        close nstep_close steps, contact test, lift with the periodic contact
//                        test, shake back / right / left, label
//   MGS_MODE_STEP      : generic "load state, mj_step x nstep, store state" used by parity tests
// One warp runs one candidate start to finish; state never leaves shared memory in between.
#pragma once
#include "mgs_solver.cuh"

#define MGS_DIAG_HEADER 8
static inline int mgs_diag_stride(int nv, int nbody, int ncon_max, int nefc_max) {
  return MGS_DIAG_HEADER + 3 * nv + nv * nv + 7 * nbody + 5 * ncon_max + 4 * nefc_max;
}

MGS_DEV void mpr_cache_g_reset_w() {
#ifndef MGS_HOST
  if (IO.mpr_cache_g) {
    int *g = IO.mpr_cache_g + (size_t)MGS_ENV_SLOT * MD.npair * 4;
    #pragma unroll 1
    PFOR(i, 4 * MD.npair) g[i] = (i & 3) == 3 ? 0 : -1;
  }
#endif
}

MGS_DEVN void reset_w(Env &e) {
  #pragma unroll 1
  PFOR(i, MD.nq) { EF(qpos)[i] = LDG(MD.qpos0 + i); QPOS_LO_CLEAR(i); }
  #pragma unroll 1
  PFOR(i, MD.nv) { EF(qvel)[i] = 0; EF(qacc_ws)[i] = 0; }
  #pragma unroll 1
  PFOR(i, MD.nu) EF(ctrl)[i] = 0;
  #pragma unroll 1
  PFOR(i, MD.nmocap) {
    for (int k = 0; k < 3; k++) EF(mocap)[7 * i + k] = LDG(MD.mocap_pos0 + 3 * i + k);
    for (int k = 0; k < 4; k++) EF(mocap)[7 * i + 3 + k] = LDG(MD.mocap_quat0 + 4 * i + k);
  }
  EH.bad = 0; EH.overflow = 0; EH.ncon = 0; EH.nefc = 0;
  #pragma unroll 1
  PFOR(i, 4 * LY.ncache) IARR(EF(mpr_cache))[i] = (i & 3) == 3 ? 0 : -1;
  mpr_cache_g_reset_w();
  WSYNC();
}

// set_qpos(joints) + set_pose(base): simualtion.py:45-49, gripper/base.py:48-59
MGS_DEVN void place_w(Env &e, const float *pose7, const float *joints) {
  // `data.qpos[idxs] = qpos` is a sequential scatter: when two entries of idxs name the same address (Robotiq's two misnamed
  // joints both resolve to the object's x, robotiq2f85.py:275,279) the LAST one wins.  One lane writes them in order.
  if (joints) {
    #pragma unroll 1
    PFOR(one, 1) {
      #pragma unroll 1
      for (int k = 0; k < PRM.nj; k++) { EF(qpos)[PRM.joint_qposadr[k]] = (real)LDG(joints + k); QPOS_LO_CLEAR(PRM.joint_qposadr[k]); }
    }
    WSYNC();
  }
  #pragma unroll 1
  PFOR(k, 7) {
    real v = (real)LDG(pose7 + k);
    EF(qpos)[PRM.base_qposadr + k] = v;
    QPOS_LO_CLEAR(PRM.base_qposadr + k);
    EF(mocap)[k] = v;
  }
  WSYNC();
}

MGS_DEV real round32(real x) { return (real)(float)x; }

// linear mocap ramp of n steps from start to target (targets are never quite reached: t/n, t<n)
MGS_DEVN int ramp_w(Env &e, const real *start, const real *target, int n, int check_every, int *steps) {
  #pragma unroll 1
  for (int t = 0; t < n; t++) {
    real f = (real)t / (real)n;
    #pragma unroll 1
    PFOR(k, 3) EF(mocap)[k] = start[k] + (target[k] - start[k]) * f;
    WSYNC();
    if (step_w(e, 1, steps)) return 1;
    if (check_every > 0 && t > 0 && t % check_every == 0 && !contact_with_object_w(e, 0)) return 1;
  }
  return 0;
}

// qpos address of the grasped object's free joint: the object fragment comes last in the scene template, so it is the last joint
MGS_DEV int object_qposadr() {
  const int j = MD.njnt - 1;
  return (j >= 0 && LDG(MD.jnt_type + j) == JNT_FREE) ? LDG(MD.jnt_qposadr + j) : -1;
}

// object drift over the close phase (gravityless_object_grasping.py:175-200; get_object_transform casts to float32):
// |dp| and the rotation angle acos(2 <q0,q1>^2 - 1) in degrees
MGS_DEV void drift_w(const Env &e, const real *before, float *out) {
  const int a = object_qposadr();
  if (a < 0 || !out) return;
  float dp = 0, dot = 0;
  for (int k = 0; k < 3; k++) { const float d = (float)before[k] - (float)EF(qpos)[a + k]; dp += d * d; }
  for (int k = 3; k < 7; k++) dot += (float)before[k] * (float)EF(qpos)[a + k];
  dot = fminf(1.0f, fmaxf(-1.0f, dot));
  const float ang = acosf(fminf(1.0f, fmaxf(-1.0f, 2.0f * dot * dot - 1.0f)));
  if (MGS_LANE == 0) { out[0] = sqrtf(dp); out[1] = ang * 57.29577951308232f; }
}

MGS_DEVN int stability_program_w(Env &e, const float *pose7, const float *joints, int *steps, float *drift) {
  reset_w(e);
  place_w(e, pose7, joints);
  forward_w(e);
  MGS_STAGE_BARRIER(5);  // the integrate slot of a step (keeps the CTA stage-aligned)
  real obj0[7] = {0, 0, 0, 1, 0, 0, 0};
  {
    const int a = object_qposadr();
    if (a >= 0) for (int k = 0; k < 7; k++) obj0[k] = EF(qpos)[a + k];
  }
  // close_gripper_at (panda.py:225-241 and the five siblings): mocap <- pose, ctrl <- close signal
  if (PRM.repose_on_close) place_w(e, pose7, (const float *)0);
  #pragma unroll 1
  PFOR(k, 7) EF(mocap)[k] = (real)LDG(pose7 + k);
  #pragma unroll 1
  PFOR(u, MD.nu) EF(ctrl)[u] = PRM.close_ctrl[u];
  WSYNC();
  if (step_w(e, PRM.nstep_close, steps)) return 0;
  if (!contact_with_object_w(e, 0)) return 0;
  drift_w(e, obj0, drift);
  // lift (:205-226)
  real start[3], target[3];
  copy3(start, EF(mocap));
  copy3(target, start);
  target[2] = start[2] + PRM.lift_dist;
  WSYNC();
  if (ramp_w(e, start, target, PRM.nstep_lift, 100, steps)) return 0;
  if (!contact_with_object_w(e, 0)) return 0;
  // shake (:229-276); current_mocap_pose passes through SE3Pose => float32 pos/quat/rotation
  real p32[3], q32[4], Rm[9], tb[3], tr[3], tl[3];
  for (int k = 0; k < 3; k++) p32[k] = round32(EF(mocap)[k]);
  for (int k = 0; k < 4; k++) q32[k] = round32(EF(mocap)[3 + k]);
  normquat(q32);
  quat2mat(Rm, q32);
  for (int k = 0; k < 9; k++) Rm[k] = round32(Rm[k]);
  for (int k = 0; k < 3; k++) tb[k] = p32[k] - Rm[3 * k + 2] * PRM.shake_dist;  // back = R (0,0,-1)
  copy3(start, EF(mocap));
  WSYNC();
  if (ramp_w(e, start, tb, PRM.shake_steps, 0, steps)) return 0;
  if (!contact_with_object_w(e, 0)) return 0;
  for (int k = 0; k < 3; k++) tr[k] = tb[k] + Rm[3 * k + 1] * PRM.shake_dist;  // right = R (0,1,0)
  copy3(start, EF(mocap));
  WSYNC();
  if (ramp_w(e, start, tr, PRM.shake_steps, 0, steps)) return 0;
  if (!contact_with_object_w(e, 0)) return 0;
  // left: restarts from the START of the right move (reference quirk: ~2 cm mocap jump at t=0)
  for (int k = 0; k < 3; k++) tl[k] = start[k] - Rm[3 * k + 1] * (2 * PRM.shake_dist);
  if (ramp_w(e, start, tl, 2 * PRM.shake_steps, 0, steps)) return 0;
  if (!contact_with_object_w(e, 0)) return 0;
  return 1;
}

// load a scene record (qpos | qvel | qacc_warmstart | ctrl | mocap) from global memory
MGS_DEVN void load_record_w(Env &e, const real *in) {
  EH.bad = 0; EH.overflow = 0; EH.ncon = 0; EH.nefc = 0;
  #pragma unroll 1
  PFOR(i, 4 * LY.ncache) IARR(EF(mpr_cache))[i] = (i & 3) == 3 ? 0 : -1;
  mpr_cache_g_reset_w();
  #pragma unroll 1
  PFOR(i, MD.nq) { EF(qpos)[i] = in[i]; QPOS_LO_CLEAR(i); }
  #pragma unroll 1
  PFOR(i, MD.nv) { EF(qvel)[i] = in[MD.nq + i]; EF(qacc_ws)[i] = in[MD.nq + MD.nv + i]; }
  #pragma unroll 1
  PFOR(i, MD.nu) EF(ctrl)[i] = in[MD.nq + 2 * MD.nv + i];
  #pragma unroll 1
  PFOR(i, 7 * MD.nmocap) EF(mocap)[i] = in[MD.nq + 2 * MD.nv + MD.nu + i];
  WSYNC();
}

// ClutterTableEnv.grasp_stable_mask body (clutter_table.py:288-317): restore the scene, place, close, lift with
// the gripper-contact test at (t+1) % 100 == 0 (early break); label = lift survived
MGS_DEVN int clutter_stable_program_w(Env &e, const real *scene, const float *pose7, const float *joints, int *steps) {
  load_record_w(e, scene);
  place_w(e, pose7, joints);
  forward_w(e);
  MGS_STAGE_BARRIER(5);
  if (PRM.repose_on_close) place_w(e, pose7, (const float *)0);
  #pragma unroll 1
  PFOR(k, 7) EF(mocap)[k] = (real)LDG(pose7 + k);
  #pragma unroll 1
  PFOR(u, MD.nu) EF(ctrl)[u] = PRM.close_ctrl[u];
  WSYNC();
  if (step_w(e, PRM.nstep_close, steps)) return 0;
  real start[3], target[3];
  copy3(start, EF(mocap));
  copy3(target, start);
  target[2] = start[2] + PRM.lift_dist;
  WSYNC();
  #pragma unroll 1
  for (int t = 0; t < PRM.nstep_lift; t++) {
    const real f = (real)t / (real)PRM.nstep_lift;
    #pragma unroll 1
    PFOR(k, 3) EF(mocap)[k] = start[k] + (target[k] - start[k]) * f;
    WSYNC();
    if (step_w(e, 1, steps)) return 0;
    if ((t + 1) % 100 == 0 && !contact_with_object_w(e, 0)) return 0;
  }
  return 1;
}

MGS_DEVN void write_diag_w(const Env &e, real *o) {
  const int nv = MD.nv;
  #pragma unroll 1
  PFOR(k, 1) { o[0] = (real)EH.ncon; o[1] = (real)EH.nefc; o[2] = (real)EH.niter; o[3] = (real)EH.bad; o[4] = (real)EH.overflow; o[5] = (real)EH.ne; o[6] = (real)EH.nf; o[7] = (real)EH.nl; }
  real *p = o + MGS_DIAG_HEADER;
  #pragma unroll 1
  PFOR(d, nv) { p[d] = EF(qacc)[d]; p[nv + d] = EF(qacc_smooth)[d]; p[2 * nv + d] = EF(qfrc_smooth)[d]; }
  p += 3 * nv;
  #pragma unroll 1
  PFOR(i, nv * nv) {  // the diagnostics carry M dense
    const int r = i / nv, c = i - r * nv;
    p[i] = (LDG(MD.dof_treeadr + r) == LDG(MD.dof_treeadr + c)) ? EF(M)[LDG(MD.dof_rowoff + r) + c] : R_(0.0);
  }
  p += nv * nv;
  #pragma unroll 1
  PFOR(i, 3 * MD.nbody) p[i] = EF(xpos)[i];
  p += 3 * MD.nbody;
  #pragma unroll 1
  PFOR(i, 4 * MD.nbody) p[i] = EF(xquat)[i];
  p += 4 * MD.nbody;
  #pragma unroll 1
  PFOR(c, LY.ncon_max) {
    int ok = c < EH.ncon;
    p[5 * c] = ok ? EF(con_dist)[c] : 0;
    for (int k = 0; k < 3; k++) p[5 * c + 1 + k] = ok ? EF(con_pos)[3 * c + k] : 0;
    p[5 * c + 4] = ok ? (real)IARR(EF(con_pair))[c] : -1;
  }
  p += 5 * LY.ncon_max;
  #pragma unroll 1
  PFOR(i, LY.nefc_max) {
    int ok = i < EH.nefc;
    p[4 * i] = ok ? EF(efc_aref)[i] : 0; p[4 * i + 1] = ok ? EF(efc_D)[i] : 0;
    p[4 * i + 2] = ok ? EF(efc_force)[i] : 0; p[4 * i + 3] = ok ? EF(efc_jar)[i] : 0;
  }
}

// run one candidate / environment on this warp
MGS_DEVN void run_env_w(Env &e, int env) {
  int steps = 0;
  MGS_CLK_RESET();
  if (PRM.mode == MGS_MODE_STEP) {
    load_record_w(e, IO.state_in + (size_t)env * IO.state_stride);
    if (PRM.nstep > 0) step_w(e, PRM.nstep, &steps);
    else { forward_w(e); MGS_STAGE_BARRIER(5); }
    real *out = IO.state_out + (size_t)env * IO.state_stride;
    #pragma unroll 1
    PFOR(i, MD.nq) out[i] = EF(qpos)[i];
    #pragma unroll 1
    PFOR(i, MD.nv) { out[MD.nq + i] = EF(qvel)[i]; out[MD.nq + MD.nv + i] = EF(qacc_ws)[i]; }
    #pragma unroll 1
    PFOR(i, MD.nu) out[MD.nq + 2 * MD.nv + i] = EF(ctrl)[i];
    #pragma unroll 1
    PFOR(i, 7 * MD.nmocap) out[MD.nq + 2 * MD.nv + MD.nu + i] = EF(mocap)[i];
    if (IO.diag_out) write_diag_w(e, IO.diag_out + (size_t)env * IO.diag_stride);
    #pragma unroll 1
    PFOR(k, 1) {
      if (IO.labels) IO.labels[env] = (uint8_t)(EH.bad ? 0 : 1);
      if (IO.steps) IO.steps[env] = steps;
      if (IO.aux) { float *a = IO.aux + 4 * (size_t)env; a[0] = (float)((EH.overflow ? 1 : 0) | (EH.bad ? 2 : 0)); a[1] = a[2] = a[3] = 0; }
#ifndef MGS_HOST
      if (EH.overflow) atomicAdd(IO.work_counter + 1, 1u);
#endif
    }
    MGS_CLK_PRINT(env, steps);
    WSYNC();
    return;
  }
  const float *pose7 = IO.pose7 + (size_t)env * 7, *joints = IO.joints + (size_t)env * PRM.nj;
  float *aux = IO.aux ? IO.aux + 4 * (size_t)env : (float *)0;
  if (aux && MGS_LANE == 0) { aux[1] = nanf(""); aux[2] = nanf(""); aux[3] = 0; }
  int label, skipped = 0;
  const bool clutter = PRM.mode == MGS_MODE_CLUTTER_COLLISION || PRM.mode == MGS_MODE_CLUTTER_STABLE;
  if (PRM.mode == MGS_MODE_COLLISION) {
    reset_w(e);
    place_w(e, pose7, joints);
    forward_w(e);
    MGS_STAGE_BARRIER(5);
    label = (EH.ncon == 0);  // collision-free mask: no contact of any kind (check_contact, :306-307)
  } else if (clutter) {
    // Scene of this candidate, and the enough_stable skip.  One thread decides (the one that pulls candidates and counts successes,
    // so its next pull sees its own increment) and broadcasts: threads of the 256-thread variant that read the counter at different
    // moments could otherwise disagree.  The counter is read with a volatile load, never through the read-only path.
    const int s = IO.scene_index ? LDG(IO.scene_index + env) : 0;
    int gate = 0;  // 0 = simulate, 1 = scene index out of range, 2 = skipped
    if (IO.scene_index && (s < 0 || s >= IO.nscene)) gate = 1;  // no index array: scene 0, whatever nscene says
    else if (IO.scene_success && MGS_LANE == 0 && *(volatile unsigned int *)(IO.scene_success + s) >= (unsigned int)IO.enough_stable) gate = 2;
    gate = wbcasti(gate, 0);
    const real *scene = IO.state_in + (size_t)(gate ? 0 : s) * IO.state_stride;
    if (gate) {
      EH.bad = gate == 1;
      skipped = gate == 2;
      label = 0;
    } else if (PRM.mode == MGS_MODE_CLUTTER_COLLISION) {
      // ClutterTableEnv.grasp_collision_mask body (clutter_table.py:356-364); bounds test done by the host
      load_record_w(e, scene);
      place_w(e, pose7, joints);
      forward_w(e);
      MGS_STAGE_BARRIER(5);
      label = !contact_with_object_w(e, 1);
    } else {
      label = clutter_stable_program_w(e, scene, pose7, joints, &steps);
    }
  } else {
    label = stability_program_w(e, pose7, joints, &steps, aux ? aux + 1 : (float *)0);
  }
  #pragma unroll 1
  PFOR(k, 1) {
    IO.labels[env] = (uint8_t)label;
    if (IO.steps) IO.steps[env] = steps;
    if (aux) aux[0] = (float)((EH.overflow ? 1 : 0) | (EH.bad ? 2 : 0) | (skipped ? 4 : 0));
#ifndef MGS_HOST
    if (EH.overflow) atomicAdd(IO.work_counter + 1, 1u);
#endif
    // a success on the candidate's full contact set is final: count it for the early stop of its scene (the index is re-read here
    // rather than kept live over the rollout)
    if (clutter && IO.scene_success && label && !EH.overflow) {
      const int s = IO.scene_index ? LDG(IO.scene_index + env) : 0;
#ifdef MGS_HOST
      IO.scene_success[s]++;
#else
      atomicAdd(IO.scene_success + s, 1u);
#endif
    }
  }
  if (IO.state_out) {
    real *out = IO.state_out + (size_t)env * IO.state_stride;
    #pragma unroll 1
    PFOR(i, MD.nq) out[i] = EF(qpos)[i];
    #pragma unroll 1
    PFOR(i, MD.nv) { out[MD.nq + i] = EF(qvel)[i]; out[MD.nq + MD.nv + i] = EF(qacc_ws)[i]; }
    #pragma unroll 1
    PFOR(i, MD.nu) out[MD.nq + 2 * MD.nv + i] = EF(ctrl)[i];
    #pragma unroll 1
    PFOR(i, 7 * MD.nmocap) out[MD.nq + 2 * MD.nv + MD.nu + i] = EF(mocap)[i];
  }
  MGS_CLK_PRINT(env, steps);
  WSYNC();
}
