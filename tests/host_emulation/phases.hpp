// Engine phases of one substep stopped after a given stage, and readers of the workspace they leave behind.
// TEST INFRASTRUCTURE shared by the one-lane host build (emul.cpp) and the 32-lane device build (devemul.cu), so that
// both are stopped at the same point and read the same way.  The product library never links or loads this file.
#pragma once

#include "../../earl_benchmark_b200/csrc/mj_step.cuh"

namespace earl {
namespace mj {

// forward: kinematics + mass matrix + bias forces; collide: kinematics + mass matrix + collision (substep's order);
// constraints: + constraint rows and contact rows; solve: + bias forces, qfrc_smooth and the Newton solve (everything of a
// substep but the Euler update); substeps: whole substeps
enum { STAGE_FORWARD = 0, STAGE_COLLIDE = 1, STAGE_CONSTRAINTS = 2, STAGE_SOLVE = 3, STAGE_SUBSTEPS = 4 };

template <int NL>
MJ_FN void run_stage(const Model& m, const real* hull, Work& w, int stage, int nsub, int lane) {
  if (stage == STAGE_SUBSTEPS) {
    for (int s = 0; s < nsub; ++s) substep<NL>(m, hull, w, lane);
    return;
  }
  kinematics<NL>(m, w, lane);
  mass_matrix<NL>(m, w, lane);
  if (stage == STAGE_FORWARD) {
    bias_forces<NL>(m, w, lane);
    return;
  }
  collide<NL>(m, hull, w, lane);
  if (stage == STAGE_COLLIDE) return;
  make_constraints<NL>(m, w, lane);
  contact_rows<NL>(m, w, lane);
  if (stage == STAGE_CONSTRAINTS) return;
  bias_forces<NL>(m, w, lane);
  // qfrc_smooth exactly as substep() forms it (passive forces - bias + servo actuation)
  const int nv = m.nv;
  for (int i = lane; i < nv; i += NL) w.smooth[i] = -m.dof_damping[i] * w.qvel[i] - w.bias[i];
  wsync<NL>();
  if (lane == 0) {
    for (int j = 0; j < m.njnt; ++j)
      if (m.jnt_stiffness[j] != 0 && m.jnt_type[j] >= 2)
        w.smooth[m.jnt_dofadr[j]] -= m.jnt_stiffness[j] * (w.qpos[m.jnt_qposadr[j]] - m.jnt_springref[j]);
    for (int u = 0; u < m.nu; ++u) {
      real c = w.ctrl[u];
      if (m.act_ctrllimited[u]) c = clampr(c, m.act_ctrlrange[u][0], m.act_ctrlrange[u][1]);
      real f = m.act_kp[u] * c - m.act_kp[u] * w.qpos[m.act_qposadr[u]];
      if (m.act_forcelimited[u]) f = clampr(f, m.act_forcerange[u][0], m.act_forcerange[u][1]);
      w.smooth[m.act_dof[u]] += f;
    }
  }
  wsync<NL>();
  solve<NL>(m, w, lane);
}

// ---------------------------------------------------------------------------------------------- host-side readers
// capacities of this build: MAXV, LDM, MAXEFC, MAXCON, MAXHIT, MAXCAND, MAXB
inline void read_caps(int* out) {
  out[0] = MAXV; out[1] = LDM; out[2] = MAXEFC; out[3] = MAXCON; out[4] = MAXHIT; out[5] = MAXCAND; out[6] = MAXB;
}
// a new state (set_state): counters and flags of the previous one cleared, the cached broad phase invalid
inline void load_state(const Model& m, Work& w, const double* qpos, const double* qvel, const double* warm, const double* mocap_pos,
                       const double* mocap_quat, const double* ctrl) {
  for (int k = 0; k < m.nq; ++k) w.qpos[k] = (real)qpos[k];
  for (int k = 0; k < m.nv; ++k) { w.qvel[k] = (real)qvel[k]; w.warm[k] = (real)warm[k]; }
  for (int k = 0; k < 3; ++k) w.mocap_pos[k] = mocap_pos[k];
  for (int k = 0; k < 4; ++k) w.mocap_quat[k] = (real)mocap_quat[k];
  for (int k = 0; k < m.nu; ++k) w.ctrl[k] = (real)ctrl[k];
  w.broad_valid = 0;
  w.bad = 0;
  w.nefc = w.ncon = w.nhit = w.solver_iter = 0;
}
inline void read_state(const Model& m, const Work& w, double* qpos, double* qvel, double* warm) {
  for (int k = 0; k < m.nq; ++k) qpos[k] = w.qpos[k];
  for (int k = 0; k < m.nv; ++k) { qvel[k] = w.qvel[k]; warm[k] = w.warm[k]; }
}
// nefc, ncon, nhit, solver_iter, bad, ncand, broad_valid
inline void read_info(const Work& w, int* out) {
  out[0] = w.nefc; out[1] = w.ncon; out[2] = w.nhit; out[3] = w.solver_iter; out[4] = w.bad; out[5] = w.ncand; out[6] = w.broad_valid;
}
// xpos [nbody][3], xmat [nbody][9], M [nv][nv], bias [nv]
inline void read_forward(const Model& m, const Work& w, double* xpos, double* xmat, double* M, double* bias) {
  for (int b = 0; b < m.nbody; ++b) {
    for (int k = 0; k < 3; ++k) xpos[3 * b + k] = w.xpos[b][k];
    for (int k = 0; k < 9; ++k) xmat[9 * b + k] = w.xmat[b][k];
  }
  for (int i = 0; i < m.nv; ++i) {
    bias[i] = w.bias[i];
    for (int j = 0; j < m.nv; ++j) M[i * m.nv + j] = w.M[i][j];
  }
}
// hit pairs [MAXHIT][2] as geom indices, in list order; returns nhit
inline int read_hits(const Model& m, const Work& w, int* pairs) {
  const int n = w.nhit < MAXHIT ? w.nhit : MAXHIT;
  for (int k = 0; k < n; ++k) {
    pairs[2 * k] = m.pair_g1[w.hit_list[k]];
    pairs[2 * k + 1] = m.pair_g2[w.hit_list[k]];
  }
  return n;
}
// dist [MAXCON], pos [MAXCON][3], frame [MAXCON][9], geoms [MAXCON][2]; returns ncon
inline int read_contacts(const Work& w, double* dist, double* pos, double* frame, int* geoms) {
  const int n = w.ncon < MAXCON ? w.ncon : MAXCON;
  for (int c = 0; c < n; ++c) {
    dist[c] = w.con_dist[c];
    for (int k = 0; k < 3; ++k) pos[3 * c + k] = w.con_pos[c][k];
    for (int k = 0; k < 9; ++k) frame[9 * c + k] = w.con_frame[c][k];
    geoms[2 * c] = w.con_g1[c];
    geoms[2 * c + 1] = w.con_g2[c];
  }
  return n;
}
// type [MAXEFC], J [MAXEFC][nv], pos / R / D / aref [MAXEFC]; con [MAXCON][2] = (first row, dim) of each contact and
// mu [MAXCON], fri [MAXCON][5] of its cone; returns nefc
inline int read_rows(const Model& m, const Work& w, int* type, double* J, double* pos, double* R, double* D, double* aref, int* con,
                     double* mu, double* fri) {
  const int n = w.nefc < MAXEFC ? w.nefc : MAXEFC;
  for (int r = 0; r < n; ++r) {
    type[r] = w.e_type[r];
    for (int c = 0; c < m.nv; ++c) J[r * m.nv + c] = w.J[r][c];
    pos[r] = w.e_pos[r]; R[r] = w.e_R[r]; D[r] = w.e_D[r]; aref[r] = w.e_aref[r];
  }
  const int nc = w.ncon < MAXCON ? w.ncon : MAXCON;
  for (int c = 0; c < nc; ++c) {
    con[2 * c] = w.con_row[c]; con[2 * c + 1] = w.con_dim[c];
    mu[c] = w.con_mu[c];
    for (int k = 0; k < 5; ++k) fri[5 * c + k] = w.con_fri[c][k];
  }
  return n;
}
// acc, fcon, smooth [nv]; force [MAXEFC]
inline void read_solve(const Model& m, const Work& w, double* acc, double* fcon, double* smooth, double* force) {
  for (int i = 0; i < m.nv; ++i) { acc[i] = w.acc[i]; fcon[i] = w.fcon[i]; smooth[i] = w.smooth[i]; }
  const int n = w.nefc < MAXEFC ? w.nefc : MAXEFC;
  for (int r = 0; r < n; ++r) force[r] = w.e_force[r];
}

}  // namespace mj
}  // namespace earl
