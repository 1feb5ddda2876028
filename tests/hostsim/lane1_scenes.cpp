// lane1_scenes.cpp - TEST HARNESS ONLY.  The lane-1 host build (lane1.cpp: the device source compiled with -DMGS_HOST as a 1-lane
// scalar program) plus the multi-scene clutter entry point, so that the CPU-only tier can check the scene index and the
// enough_stable early stop of run_env_w.  Never linked into the product library.
#include "lane1.cpp"

// scene_index is not checked here: the kernel's own range check is what the tests exercise
extern "C" int l1_clutter_scenes_host(L1Model *M, int mode, int n, int nscene, const double *scenes, const int *scene_index, int enough_stable,
                                      const float *pose7, const float *joints, int nj, const int *joint_qposadr, int base_qposadr,
                                      const double *close_ctrl, const MgsRolloutCfg *cfg, uint8_t *labels, int *steps) {
  RolloutParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.mode = mode; prm.n = n; prm.nj = nj; prm.base_qposadr = base_qposadr;
  for (int k = 0; k < nj; k++) prm.joint_qposadr[k] = joint_qposadr[k];
  if (cfg) {
    prm.nstep_close = cfg->nstep_close; prm.nstep_lift = cfg->nstep_lift; prm.shake_steps = cfg->shake_steps;
    prm.repose_on_close = cfg->repose_on_close; prm.lift_dist = (real)cfg->lift_dist; prm.shake_dist = (real)cfg->shake_dist;
  }
  if (close_ctrl) for (int u = 0; u < M->dm.nu; u++) prm.close_ctrl[u] = (real)close_ctrl[u];
  std::vector<real> rec((size_t)nscene * M->state_stride);
  for (size_t i = 0; i < rec.size(); i++) rec[i] = (real)scenes[i];
  std::vector<unsigned int> success(nscene > 0 ? nscene : 1, 0u);
  BatchIO io;
  memset(&io, 0, sizeof(io));
  io.pose7 = pose7; io.joints = joints; io.labels = labels; io.steps = steps;
  io.state_in = rec.data(); io.state_stride = M->state_stride;
  io.scene_index = scene_index; io.nscene = nscene;
  if (enough_stable > 0) { io.scene_success = success.data(); io.enough_stable = enough_stable; }
  run_all(M, prm, io);
  return 0;
}
