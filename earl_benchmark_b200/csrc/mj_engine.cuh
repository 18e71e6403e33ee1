// mj_engine.cuh -- articulated-body engine for the EARL Sawyer tasks, one WARP per environment instance.
//
// Replaces, for the reference's sawyer_door / sawyer_peg step path, the native engine call the reference makes
// through mujoco-py: metaworld SawyerXYZEnv.step -> do_simulation -> frame_skip x sim.step()  (MuJoCo 2.1.0
// mj_step; invoked by earl_benchmark/envs/sawyer_door.py and sawyer_peg.py, which do not override step()).
// Per substep: forward kinematics, composite-rigid-body mass matrix, Newton-Euler bias forces, constraint rows
// (mocap weld, joint limits, contacts), Cholesky solve for the smooth acceleration, Newton solve of the convex
// constraint problem with exact line search, semi-implicit Euler with implicit joint damping.
//
// Execution model.  All per-env working data lives in a per-warp shared-memory workspace (`Work`).  Every
// function is called by all lanes of the warp with the same arguments:
//   * "serial" sections (kinematic chain, inertia accumulation) are executed redundantly by every lane --
//     identical values are written to identical addresses, no divergence, no shuffles;
//   * "parallel" sections are lane-strided loops `for (i = lane; i < n; i += NL)` over dofs / rows / pairs;
//   * reductions go through wsum()/wmax(), phases are separated by wsync().
// The same source compiles for the host with NL = 1 (wsum = identity, wsync = no-op), which is how the CPU test
// suite checks this file against the fp64 checker without a GPU (tests/host_emulation).  The product library
// only ever runs the NL = 32 device instantiation.
#pragma once

#include <math.h>
#include <stdint.h>

// MJ_HD: small helpers, always inlined.  MJ_FN: engine phases and the larger helpers, kept as real functions on the
// device -- with everything inlined the step kernel was ~400 KB of SASS and ran instruction-fetch bound
// (ncu: stall_no_inst 76 %); as calls the hot loop fits the instruction caches.
#if defined(__CUDACC__)
#define MJ_HD __host__ __device__ __forceinline__
#define MJ_FN __host__ __device__ __noinline__
#else
#define MJ_HD inline
#define MJ_FN inline
#endif

namespace earl {
namespace mj {

typedef float real;

#if defined(MJ_CAPSET_KITCHEN)
// Third capacity set: the Franka kitchen (23 dofs, 118 colliding geoms, friction loss on every dof, pyramidal cones).
// So far instantiated by the host build of this source only (tests/host_emulation); the device instantiation is the
// next step (DESIGN.md section 9).
constexpr int MAXB = 24;    // fused bodies incl. world
constexpr int MAXV = 24;    // dofs
constexpr int MAXQ = 24;    // generalized coordinates
constexpr int MAXJ = 24;    // joints
constexpr int MAXG = 128;   // geoms kept on the device
constexpr int MAXS = 12;    // sites kept on the device
#else
constexpr int MAXB = 12;    // fused bodies incl. world
constexpr int MAXV = 16;    // dofs
constexpr int MAXQ = 20;    // generalized coordinates
constexpr int MAXJ = 12;    // joints
constexpr int MAXG = 32;    // geoms kept on the device
constexpr int MAXS = 12;    // sites kept on the device
#endif
constexpr int MAXU = 2;     // actuators
constexpr int MAXW = 1;     // welds
constexpr int MAXEQ = 8;    // joint equalities
// joint-equality / friction-loss / pyramidal rows and capsule geoms only exist in the kitchen: the door / peg builds drop
// those branches at compile time (they cost 3.5 % of the step when left in)
#if defined(MJ_CAPSET_KITCHEN)
constexpr bool KITCHEN_ROWS = true;
constexpr bool BROAD_CACHE = true;   // cached broad phase (mj_collide.cuh: collide)
constexpr int MAXCAND = 160;         // cached candidate pairs
#else
constexpr bool KITCHEN_ROWS = false;
constexpr bool BROAD_CACHE = false;
constexpr int MAXCAND = 1;
#endif
#ifndef MJ_BROAD_SLACK
#define MJ_BROAD_SLACK 0.015f
#endif
constexpr float BROAD_SLACK = MJ_BROAD_SLACK;  // inflation of the cached broad phase (m)
// The door / peg engine is compiled twice from these sources: the primary set (earl_mj.cu) and the extra-large set of the
// redo pass (earl_mj_xl.cu).  The workspace of one environment lives in shared memory, so rows x dofs and contacts decide
// how many environments one SM keeps in flight.
#if defined(MJ_CAPSET_KITCHEN)
#if defined(MJ_CAPSET_KITCHEN_XL)
// kitchen redo pass (earl_mj_kitchen_xl.cu): the few env steps with a substep beyond the primary set's rows (half a dozen
// six-dimensional finger contacts at once: 10 rows each) or 24 contacts are re-stepped with these capacities
constexpr int MAXCON = 48;  // contacts (an arm jammed into a cabinet: 33-40 seen in 0.04 % of the env steps of a long random rollout)
constexpr int MAXEFC = 544; // constraint rows: cannot overflow before the contacts do (6 weld + 5 equality + 23 friction loss + <= 23 limits + 48 x 10)
#else
// Device: 112 rows (27.1 KB workspace, 8 environments in flight per SM); the ~0.1 % of env steps with a substep beyond
// that are re-stepped by the extra-large set.  Measured at 14,208 envs: 192 rows / 6 per SM 1.33e5 env-steps/s, 128 / 7
// 1.47e5, 112 / 8 1.54e5, 96 / 8 1.52e5.  The host build of this source (tests) has no redo pass and keeps 192 rows.
#ifndef MJK_MAXEFC
#ifdef __CUDACC__
#define MJK_MAXEFC 112
#else
#define MJK_MAXEFC 192
#endif
#endif
constexpr int MAXEFC = MJK_MAXEFC; // constraint rows (6 weld + 5 equality + 23 friction loss + limits + 4 / 10 per pyramidal contact)
constexpr int MAXCON = 24;  // contacts
#endif
constexpr int MAXHIT = 64;  // candidate pairs that survive the broad phase in one substep
constexpr int MAXPAIR = 4096; // candidate geom pairs
constexpr int MAXMG = 64;    // geoms on moving bodies (their world poses are recomputed every substep)
#else
#if defined(MJ_CAPSET_XL)
// "extra large": only used by the redo pass that re-steps the few environments whose substep overflowed the primary set
// (peg wedged in the block, gripper jammed between handle and door: > 16 contacts or > 64 rows)
constexpr int MAXEFC = 224; // constraint rows
constexpr int MAXCON = 56;  // contacts
constexpr int MAXHIT = 72;  // candidate pairs that survive the broad phase in one substep
#else
constexpr int MAXEFC = 64;  // constraint rows
constexpr int MAXCON = 16;  // contacts
constexpr int MAXHIT = 24;  // candidate pairs that survive the broad phase in one substep
#endif
constexpr int MAXPAIR = 192; // candidate geom pairs
constexpr int MAXMG = 16;    // geoms on moving bodies (their world poses are recomputed every substep)
#endif
constexpr int LDM = MAXV + 1;  // padded leading dimension of the dense nv x nv matrices

constexpr real MINVAL = 1e-15f;
constexpr real MINIMP = 0.0001f;
constexpr real MAXIMP = 0.9999f;

// constraint row types
// ROW_FRICTION: dof friction loss, |force| <= e_pos[r] (the row's residual is 0, so e_pos carries the bound after finish_row)
enum { ROW_EQ = 0, ROW_LIMIT = 1, ROW_CONE = 2, ROW_CONE_FRIC = 3, ROW_FRICTION = 4 };
MJ_HD bool is_cone_row(int tp) { return tp == ROW_CONE || tp == ROW_CONE_FRIC; }

// ------------------------------------------------------------------------------------------------ device model
// Built on the host from the serialized structure-of-arrays model (mjcf/compile.py: Model.FIELDS); plain floats.
struct Model {
  int nbody, nq, nv, njnt, ngeom, nsite, nu, nweld, npair, nhull;
  int iterations, frame_skip;
  real timestep, impratio;
  real gravity[3];
  // bodies (0 = world); parents precede children
  int body_parent[MAXB], body_jnt[MAXB];
  unsigned body_anc[MAXB];  // bit c set: body c is an ancestor of (or equal to) this body
  real body_pos[MAXB][3], body_quat[MAXB][4], body_mass[MAXB], body_ipos[MAXB][3], body_inertia[MAXB][6];
  // joints (one per moving body)
  int jnt_type[MAXJ], jnt_body[MAXJ], jnt_qposadr[MAXJ], jnt_dofadr[MAXJ], jnt_limited[MAXJ];
  real jnt_pos[MAXJ][3], jnt_axis[MAXJ][3], jnt_range[MAXJ][2], jnt_margin[MAXJ], jnt_solref[MAXJ][2], jnt_solimp[MAXJ][5];
  real jnt_stiffness[MAXJ], jnt_springref[MAXJ], jnt_qpos0[MAXJ];
  // dofs
  int dof_body[MAXV], dof_rot[MAXV], dof_parent[MAXV];
  real dof_damping[MAXV], dof_armature[MAXV], dof_invweight0[MAXV];
  real dof_frictionloss[MAXV], dof_solref_friction[MAXV][2], dof_solimp_friction[MAXV][5];
  real dof_lever[MAXV];  // bound on the motion of any geom centre per unit motion of the dof (cached broad phase)
  real qpos0[MAXQ];
  // joint equalities q1 - q1_0 = poly(q2 - q2_0) and the friction-cone type (blob version 2: kitchen)
  int neq, cone_elliptic;
  int eq_qposadr[MAXEQ][2], eq_dofadr[MAXEQ][2];
  real eq_polycoef[MAXEQ][5], eq_solref[MAXEQ][2], eq_solimp[MAXEQ][5], eq_invweight[MAXEQ];
  // sites (observation frames)
  int site_body[MAXS];
  real site_pos[MAXS][3];
  // actuators: position servos
  int act_dof[MAXU], act_qposadr[MAXU], act_ctrllimited[MAXU], act_forcelimited[MAXU];
  real act_kp[MAXU], act_ctrlrange[MAXU][2], act_forcerange[MAXU][2];
  // weld (mocap frame -> frame on a body)
  int weld_body[MAXW];
  real weld_pos[MAXW][3], weld_quat[MAXW][4], weld_relpose[MAXW][7], weld_solref[MAXW][2], weld_solimp[MAXW][5],
      weld_invweight[MAXW][2];
  // geoms
  int geom_body[MAXG], geom_type[MAXG], geom_condim[MAXG], geom_priority[MAXG], geom_hulladr[MAXG], geom_hullnum[MAXG];
  int geom_slot[MAXG];  // index into Work::mg_xpos / mg_xmat for geoms on moving bodies, -1 for static geoms
  int nmgeom, mgeom[MAXMG];
  real geom_size[MAXG][3], geom_pos[MAXG][3], geom_mat[MAXG][9], geom_friction[MAXG][3], geom_margin[MAXG], geom_gap[MAXG];
  real geom_solref[MAXG][2], geom_solimp[MAXG][5], geom_solmix[MAXG], geom_invweight0[MAXG][2], geom_rbound[MAXG];
  real geom_obb_size[MAXG][3], geom_obb_off[MAXG][3];  // bounding box in the geom frame (box: itself; cylinder: r,r,h; mesh: hull AABB)
  // candidate collision pairs (compile-time filtered: contype/conaffinity, same body, parent-child)
  unsigned char pair_g1[MAXPAIR], pair_g2[MAXPAIR];  // geom indices
  static_assert(MAXG <= 256, "pair tables hold geom indices in one byte");
  // task constants
  int obs_hand_site, obs_ree_site, obs_lee_site, obs_obj_geom, obs_obj_site;
  real mocap_low[3], mocap_high[3], action_scale, success_radius;
  real obj_init_pos[3], hand_init_pos[3];
  int grasp_site, lpad_site, rpad_site, corner_site[4];  // dense peg reward
};

// ------------------------------------------------------------------------------------------------ per-env record
// One 256-byte record per environment in HBM (array of structures: a warp reads its env as two 128-byte lines).
constexpr int REC_FLOATS = 64;
constexpr int REC_QPOS = 0;     // [0,20)
constexpr int REC_QVEL = 20;    // [20,36)
constexpr int REC_WARM = 36;    // [36,52)  qacc_warmstart
constexpr int REC_MOCAP = 52;   // 3 doubles = 6 floats [52,58)
constexpr int REC_STEPS = 58;   // u32 steps_since_reset
constexpr int REC_FLAGS = 59;   // u32: bit0 success-any, bit1 success-last, bit2 bad_state, bit3 capacity overflow
constexpr int REC_GOALROW = 60; // u32 goal row
constexpr int REC_SPARE = 61;

// ------------------------------------------------------------------------------------------------ workspace
struct Work {
  // state
  real qpos[MAXQ], qvel[MAXV], warm[MAXV], ctrl[MAXU];
  double mocap_pos[3];
  real mocap_quat[4];
  // kinematics
  real xpos[MAXB][3], xquat[MAXB][4], xmat[MAXB][9], xipos[MAXB][3];
  real dof_axis[MAXV][3], dof_anchor[MAXV][3];
  // dense matrices.  H doubles as scratch while it is idle: narrow-phase scratch during collision (mj_collide.cuh) and
  // the Newton-Euler pass (angular velocity / acceleration, linear velocity / acceleration of the body origin, wrench
  // about the body origin) between the constraint rows and the solve.
  real M[MAXV][LDM];
  union {
    real H[MAXV][LDM];
    struct { real b_w[MAXB][3], b_v[MAXB][3], b_al[MAXB][3], b_a[MAXB][3], b_F[MAXB][3], b_N[MAXB][3]; } rne;
  };
  // dof vectors
  real bias[MAXV], smooth[MAXV], acc[MAXV], Ma[MAXV], grad[MAXV], dir[MAXV], fcon[MAXV], tmp[MAXV];
  // constraint rows
  int nefc, ncon;
  // the Jacobian is written after collision; before that its storage holds the composite inertias of the mass-matrix
  // pass (about the composite CoM, world axes)
  union {
    real J[MAXEFC][MAXV];
    struct { real c_mass[MAXB], c_com[MAXB][3], c_I[MAXB][6]; } crb;
  };
  real e_pos[MAXEFC], e_aref[MAXEFC], e_D[MAXEFC], e_R[MAXEFC], e_jar[MAXEFC], e_jv[MAXEFC], e_force[MAXEFC];
  unsigned char e_type[MAXEFC], e_state[MAXEFC];
  // collision
  // world poses of the geoms on moving bodies: written and read by the collision phase only, so the same storage
  // holds the cone Hessian blocks (dim x dim, dim <= 4; middle zone) that only the solve phase touches
  union {
    struct { real mg_xpos[MAXMG][3], mg_xmat[MAXMG][9]; };
    real con_H[MAXCON][16];
  };
  int nhit;
  unsigned short hit_list[MAXHIT];
  // cached broad phase (BROAD_CACHE): candidates of the last loose pass and the travel bound used up since
  unsigned short cand_list[MAXCAND];
  int ncand, broad_valid, acc_rebuild;  // acc_rebuild: loose passes of the current env step (scheduling cost estimate)
  real broad_travel;
  // contacts
  real con_pos[MAXCON][3], con_frame[MAXCON][9], con_dist[MAXCON], con_fri[MAXCON][5], con_mu[MAXCON];
  int con_g1[MAXCON], con_g2[MAXCON], con_dim[MAXCON], con_row[MAXCON];
  // task layer
  real action[4], obs7[8];
  unsigned steps, flags, goalrow;
  real spare[3];  // record floats 61..63: self.obj_init_pos of the last reset (dense peg reward)
  // diagnostics
  int solver_iter;
  int bad;  // bit 0: numerical failure (non-positive pivot); capacity overflows: bit 1 candidate pairs, bit 2 contacts, bit 3 rows
  int acc_iter, acc_rows, acc_con, acc_mpr, acc_sup;  // summed over the substeps of one env step (acc_sup: support-function calls)
  int peak_efc, peak_con, peak_hit;                   // largest row / contact / candidate-pair count of a substep of this env step
#ifdef MJ_PHASE_TIMING
  long long phase[8], phase_t0;     // SM cycles per engine phase (profiling builds only)
#endif
};

#if defined(MJ_PHASE_TIMING) && defined(__CUDA_ARCH__)
#define MJ_PHASE_BEGIN(w) do { (w).phase_t0 = clock64(); } while (0)
#define MJ_PHASE_END(w, k) do { const long long t_ = clock64(); (w).phase[k] += t_ - (w).phase_t0; (w).phase_t0 = t_; } while (0)
#else
#define MJ_PHASE_BEGIN(w) do { } while (0)
#define MJ_PHASE_END(w, k) do { } while (0)
#endif

// ------------------------------------------------------------------------------------------------ warp primitives
template <int NL>
MJ_HD void wsync() {
#if defined(__CUDA_ARCH__)
  if (NL > 1) __syncwarp();
#endif
}
// block-wide phase barrier: keeps the warps of a block in the same engine phase, so that they share the instruction
// caches instead of each walking a different part of a large program
template <int NL>
MJ_HD void bsync() {
#if defined(__CUDA_ARCH__) && !defined(MJ_NO_PHASE_BARRIERS)
#if defined(MJ_BARRIER_DOMAINS) && MJ_BARRIER_DOMAINS > 1
  // the block's warps in MJ_BARRIER_DOMAINS groups, each with its own named barrier (fewer warps to wait for, more phases
  // resident in the instruction caches at once): used by the kitchen set (earl_mj_kitchen.cu)
  if (NL > 1) {
    const unsigned per = (blockDim.x >> 5) / MJ_BARRIER_DOMAINS;
    const unsigned dom = (threadIdx.x >> 5) / per;
    if (dom < MJ_BARRIER_DOMAINS) asm volatile("bar.sync %0, %1;" ::"r"(1u + dom), "r"(per * 32u) : "memory");
  }
#else
  if (NL > 1) __syncthreads();
#endif
#endif
}
template <int NL>
MJ_HD real wsum(real x) {
#if defined(__CUDA_ARCH__)
  if (NL > 1) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  }
#endif
  return x;
}
template <int NL>
MJ_HD double wmaxd(double x) {
#if defined(__CUDA_ARCH__)
  if (NL > 1) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = fmax(x, __shfl_xor_sync(0xffffffffu, x, o));
  }
#endif
  return x;
}
template <int NL>
MJ_HD real wmax(real x) {
#if defined(__CUDA_ARCH__)
  if (NL > 1) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = fmaxf(x, __shfl_xor_sync(0xffffffffu, x, o));
  }
#endif
  return x;
}

// ------------------------------------------------------------------------------------------------ small math
template <class T>
MJ_HD void cross3(T* r, const T* a, const T* b) {
  T x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  r[0] = x; r[1] = y; r[2] = z;
}
template <class T>
MJ_HD T dot3(const T* a, const T* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
MJ_HD float msqrt(float x) { return sqrtf(x); }
MJ_HD double msqrt(double x) { return sqrt(x); }
MJ_HD float mabs(float x) { return fabsf(x); }
MJ_HD double mabs(double x) { return fabs(x); }
MJ_HD void mulmatvec3(real* r, const real* m, const real* v) {
  real x = m[0] * v[0] + m[1] * v[1] + m[2] * v[2], y = m[3] * v[0] + m[4] * v[1] + m[5] * v[2],
       z = m[6] * v[0] + m[7] * v[1] + m[8] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}
MJ_HD void mulmatTvec3(real* r, const real* m, const real* v) {
  real x = m[0] * v[0] + m[3] * v[1] + m[6] * v[2], y = m[1] * v[0] + m[4] * v[1] + m[7] * v[2],
       z = m[2] * v[0] + m[5] * v[1] + m[8] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}
MJ_HD void mulquat(real* r, const real* a, const real* b) {
  real w = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3], x = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
       y = a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1], z = a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0];
  r[0] = w; r[1] = x; r[2] = y; r[3] = z;
}
MJ_HD void normquat(real* q) {
  real n = sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  if (n < MINVAL) { q[0] = 1; q[1] = q[2] = q[3] = 0; return; }
  real s = 1.0f / n;
  q[0] *= s; q[1] *= s; q[2] *= s; q[3] *= s;
}
MJ_HD void quat2mat(real* m, const real* q) {
  real w = q[0], x = q[1], y = q[2], z = q[3];
  m[0] = 1 - 2 * (y * y + z * z); m[1] = 2 * (x * y - w * z); m[2] = 2 * (x * z + w * y);
  m[3] = 2 * (x * y + w * z); m[4] = 1 - 2 * (x * x + z * z); m[5] = 2 * (y * z - w * x);
  m[6] = 2 * (x * z - w * y); m[7] = 2 * (y * z + w * x); m[8] = 1 - 2 * (x * x + y * y);
}
MJ_HD real clampr(real x, real lo, real hi) { return x < lo ? lo : (x > hi ? hi : x); }

// ------------------------------------------------------------------------------------------------ kinematics
// mj_kinematics + mj_comPos for the fused tree: serial chain, executed redundantly by all lanes.
template <int NL>
MJ_FN void kinematics(const Model& m, Work& w, int lane) {
  (void)lane;
  w.xpos[0][0] = w.xpos[0][1] = w.xpos[0][2] = 0;
  w.xquat[0][0] = 1; w.xquat[0][1] = w.xquat[0][2] = w.xquat[0][3] = 0;
  for (int k = 0; k < 9; ++k) w.xmat[0][k] = (k % 4 == 0) ? 1.0f : 0.0f;
  wsync<NL>();
  for (int b = 1; b < m.nbody; ++b) {
    const int p = m.body_parent[b], j = m.body_jnt[b];
    real pos[3], quat[4], R[9], t[3];
    mulmatvec3(t, w.xmat[p], m.body_pos[b]);
    for (int k = 0; k < 3; ++k) pos[k] = w.xpos[p][k] + t[k];
    mulquat(quat, w.xquat[p], m.body_quat[b]);
    const int qa = m.jnt_qposadr[j], da = m.jnt_dofadr[j], jt = m.jnt_type[j];
    if (jt == 3) {  // hinge
      quat2mat(R, quat);
      real anchor[3], axis[3], qj[4];
      mulmatvec3(t, R, m.jnt_pos[j]);
      for (int k = 0; k < 3; ++k) anchor[k] = pos[k] + t[k];
      mulmatvec3(axis, R, m.jnt_axis[j]);
      const real half = 0.5f * (w.qpos[qa] - m.jnt_qpos0[j]);
      real s, c;
#if defined(__CUDA_ARCH__)
      sincosf(half, &s, &c);
#else
      s = sinf(half); c = cosf(half);
#endif
      qj[0] = c; qj[1] = m.jnt_axis[j][0] * s; qj[2] = m.jnt_axis[j][1] * s; qj[3] = m.jnt_axis[j][2] * s;
      mulquat(quat, quat, qj);
      normquat(quat);
      quat2mat(R, quat);
      mulmatvec3(t, R, m.jnt_pos[j]);
      for (int k = 0; k < 3; ++k) {
        pos[k] = anchor[k] - t[k];
        w.dof_axis[da][k] = axis[k];
        w.dof_anchor[da][k] = anchor[k];
      }
    } else if (jt == 2) {  // slide
      quat2mat(R, quat);
      real axis[3];
      mulmatvec3(axis, R, m.jnt_axis[j]);
      const real dq = w.qpos[qa] - m.jnt_qpos0[j];
      for (int k = 0; k < 3; ++k) {
        pos[k] += axis[k] * dq;
        w.dof_axis[da][k] = axis[k];
        w.dof_anchor[da][k] = pos[k];
      }
    } else {  // free: 3 world-axis translations, then 3 body-axis rotations
      for (int k = 0; k < 3; ++k) pos[k] = w.qpos[qa + k];
      for (int k = 0; k < 4; ++k) quat[k] = w.qpos[qa + 3 + k];
      normquat(quat);
      for (int k = 0; k < 4; ++k) w.qpos[qa + 3 + k] = quat[k];  // mj_kinematics normalises quaternions in place
      quat2mat(R, quat);
      for (int a = 0; a < 3; ++a)
        for (int k = 0; k < 3; ++k) {
          w.dof_axis[da + a][k] = (a == k) ? 1.0f : 0.0f;
          w.dof_anchor[da + a][k] = pos[k];
          w.dof_axis[da + 3 + a][k] = R[3 * k + a];
          w.dof_anchor[da + 3 + a][k] = pos[k];
        }
    }
    for (int k = 0; k < 3; ++k) w.xpos[b][k] = pos[k];
    for (int k = 0; k < 4; ++k) w.xquat[b][k] = quat[k];
    for (int k = 0; k < 9; ++k) w.xmat[b][k] = R[k];
    mulmatvec3(t, R, m.body_ipos[b]);
    for (int k = 0; k < 3; ++k) w.xipos[b][k] = pos[k] + t[k];
    wsync<NL>();
  }
}

// world-frame inertia (6: xx yy zz xy xz yz) of body b about its CoM
MJ_FN void body_inertia_world(const Model& m, const Work& w, int b, real* I6) {
  const real* L = m.body_inertia[b];
  const real* R = w.xmat[b];
  const real Il[9] = {L[0], L[3], L[4], L[3], L[1], L[5], L[4], L[5], L[2]};
  real T[9];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) T[3 * i + j] = R[3 * i] * Il[j] + R[3 * i + 1] * Il[3 + j] + R[3 * i + 2] * Il[6 + j];
  real Iw[9];
  for (int i = 0; i < 3; ++i)
    for (int j = i; j < 3; ++j) Iw[3 * i + j] = T[3 * i] * R[3 * j] + T[3 * i + 1] * R[3 * j + 1] + T[3 * i + 2] * R[3 * j + 2];
  I6[0] = Iw[0]; I6[1] = Iw[4]; I6[2] = Iw[8]; I6[3] = Iw[1]; I6[4] = Iw[2]; I6[5] = Iw[5];
}
MJ_HD void sym6_mulvec(real* r, const real* I6, const real* v) {
  real x = I6[0] * v[0] + I6[3] * v[1] + I6[4] * v[2], y = I6[3] * v[0] + I6[1] * v[1] + I6[5] * v[2],
       z = I6[4] * v[0] + I6[5] * v[1] + I6[2] * v[2];
  r[0] = x; r[1] = y; r[2] = z;
}

// ------------------------------------------------------------------------------------------------ mass matrix (CRB)
// Composite inertias are kept about the composite CoM in world axes, so every vector that enters a product is a
// LOCAL difference (fp32-safe).  M[i][j] = S_j . (Ic_i S_i) for j an ancestor dof of i; + armature on the diagonal.
template <int NL>
MJ_FN void mass_matrix(const Model& m, Work& w, int lane) {
  const int nb = m.nbody, nv = m.nv;
  for (int b = 1 + lane; b < nb; b += NL) {
    w.crb.c_mass[b] = m.body_mass[b];
    for (int k = 0; k < 3; ++k) w.crb.c_com[b][k] = w.xipos[b][k];
    if (m.body_mass[b] > 0) body_inertia_world(m, w, b, w.crb.c_I[b]);
    else for (int k = 0; k < 6; ++k) w.crb.c_I[b][k] = 0;
  }
  for (int i = lane; i < nv; i += NL)
    for (int j = 0; j < nv; ++j) w.M[i][j] = 0;
  wsync<NL>();
  // accumulate children into parents (serial, leaves first)
  for (int b = nb - 1; b >= 1; --b) {
    const int p = m.body_parent[b];
    if (p <= 0) continue;
    const real m1 = w.crb.c_mass[p], m2 = w.crb.c_mass[b], mt = m1 + m2;
    if (m2 <= 0) continue;
    real c[3], d1[3], d2[3];
    for (int k = 0; k < 3; ++k) {
      c[k] = (m1 * w.crb.c_com[p][k] + m2 * w.crb.c_com[b][k]) / mt;
      d1[k] = w.crb.c_com[p][k] - c[k];
      d2[k] = w.crb.c_com[b][k] - c[k];
    }
    const real s1 = dot3(d1, d1), s2 = dot3(d2, d2);
    real I[6];
    I[0] = w.crb.c_I[p][0] + w.crb.c_I[b][0] + m1 * (s1 - d1[0] * d1[0]) + m2 * (s2 - d2[0] * d2[0]);
    I[1] = w.crb.c_I[p][1] + w.crb.c_I[b][1] + m1 * (s1 - d1[1] * d1[1]) + m2 * (s2 - d2[1] * d2[1]);
    I[2] = w.crb.c_I[p][2] + w.crb.c_I[b][2] + m1 * (s1 - d1[2] * d1[2]) + m2 * (s2 - d2[2] * d2[2]);
    I[3] = w.crb.c_I[p][3] + w.crb.c_I[b][3] - m1 * d1[0] * d1[1] - m2 * d2[0] * d2[1];
    I[4] = w.crb.c_I[p][4] + w.crb.c_I[b][4] - m1 * d1[0] * d1[2] - m2 * d2[0] * d2[2];
    I[5] = w.crb.c_I[p][5] + w.crb.c_I[b][5] - m1 * d1[1] * d1[2] - m2 * d2[1] * d2[2];
    wsync<NL>();
    w.crb.c_mass[p] = mt;
    for (int k = 0; k < 3; ++k) w.crb.c_com[p][k] = c[k];
    for (int k = 0; k < 6; ++k) w.crb.c_I[p][k] = I[k];
    wsync<NL>();
  }
  // one lane per dof i: wrench of a unit acceleration of dof i on its composite body, projected on ancestor dofs
  for (int i = lane; i < nv; i += NL) {
    const int b = m.dof_body[i];
    const real mass = w.crb.c_mass[b];
    real F[3], N[3];  // force, torque about the composite CoM
    if (m.dof_rot[i]) {
      real r[3] = {w.crb.c_com[b][0] - w.dof_anchor[i][0], w.crb.c_com[b][1] - w.dof_anchor[i][1], w.crb.c_com[b][2] - w.dof_anchor[i][2]};
      cross3(F, w.dof_axis[i], r);
      F[0] *= mass; F[1] *= mass; F[2] *= mass;
      sym6_mulvec(N, w.crb.c_I[b], w.dof_axis[i]);
    } else {
      for (int k = 0; k < 3; ++k) { F[k] = mass * w.dof_axis[i][k]; N[k] = 0; }
    }
    for (int j = i; j >= 0; j = m.dof_parent[j]) {
      real v;
      if (m.dof_rot[j]) {
        real r[3] = {w.crb.c_com[b][0] - w.dof_anchor[j][0], w.crb.c_com[b][1] - w.dof_anchor[j][1], w.crb.c_com[b][2] - w.dof_anchor[j][2]};
        real t[3];
        cross3(t, r, F);
        v = dot3(w.dof_axis[j], N) + dot3(w.dof_axis[j], t);
      } else {
        v = dot3(w.dof_axis[j], F);
      }
      w.M[i][j] = v;
      if (j != i) w.M[j][i] = v;
    }
    w.M[i][i] += m.dof_armature[i];
  }
  wsync<NL>();
}

// ------------------------------------------------------------------------------------------------ bias forces (RNE)
// Newton-Euler with world-axis vectors referred to each body's own origin; gravity enters as a base acceleration.
template <int NL>
MJ_FN void bias_forces(const Model& m, Work& w, int lane) {
  const int nb = m.nbody, nv = m.nv;
  for (int k = 0; k < 3; ++k) {
    w.rne.b_w[0][k] = 0; w.rne.b_v[0][k] = 0; w.rne.b_al[0][k] = 0; w.rne.b_a[0][k] = -m.gravity[k];
  }
  wsync<NL>();
  for (int b = 1; b < nb; ++b) {  // forward pass (serial chain, redundant across lanes)
    const int p = m.body_parent[b], j = m.body_jnt[b], da = m.jnt_dofadr[j], jt = m.jnt_type[j];
    real om[3], al[3], v[3], a[3];
    for (int k = 0; k < 3; ++k) { om[k] = w.rne.b_w[p][k]; al[k] = w.rne.b_al[p][k]; }
    if (jt == 3) {
      const real qd = w.qvel[da];
      const real* ax = w.dof_axis[da];
      const real* an = w.dof_anchor[da];
      // anchor as a point of the parent
      real r[3] = {an[0] - w.xpos[p][0], an[1] - w.xpos[p][1], an[2] - w.xpos[p][2]}, t[3], t2[3], vP[3], aP[3];
      cross3(t, om, r);
      for (int k = 0; k < 3; ++k) vP[k] = w.rne.b_v[p][k] + t[k];
      cross3(t2, om, t);
      cross3(t, al, r);
      for (int k = 0; k < 3; ++k) aP[k] = w.rne.b_a[p][k] + t[k] + t2[k];
      // joint
      cross3(t, om, ax);
      for (int k = 0; k < 3; ++k) { al[k] += t[k] * qd; om[k] += ax[k] * qd; }
      real rb[3] = {w.xpos[b][0] - an[0], w.xpos[b][1] - an[1], w.xpos[b][2] - an[2]};
      cross3(t, om, rb);
      for (int k = 0; k < 3; ++k) v[k] = vP[k] + t[k];
      cross3(t2, om, t);
      cross3(t, al, rb);
      for (int k = 0; k < 3; ++k) a[k] = aP[k] + t[k] + t2[k];
    } else if (jt == 2) {
      const real qd = w.qvel[da];
      const real* ax = w.dof_axis[da];
      real r[3] = {w.xpos[b][0] - w.xpos[p][0], w.xpos[b][1] - w.xpos[p][1], w.xpos[b][2] - w.xpos[p][2]}, t[3], t2[3], t3[3];
      cross3(t, om, r);
      for (int k = 0; k < 3; ++k) v[k] = w.rne.b_v[p][k] + t[k] + ax[k] * qd;
      cross3(t2, om, t);
      cross3(t, al, r);
      cross3(t3, om, ax);
      for (int k = 0; k < 3; ++k) a[k] = w.rne.b_a[p][k] + t[k] + t2[k] + 2 * t3[k] * qd;
    } else {  // free joint: velocities are given in the world (translation) and body (rotation) frames
      real wl[3] = {w.qvel[da + 3], w.qvel[da + 4], w.qvel[da + 5]};
      mulmatvec3(om, w.xmat[b], wl);  // world angular velocity
      for (int k = 0; k < 3; ++k) { v[k] = w.qvel[da + k]; al[k] = 0; a[k] = -m.gravity[k]; }
      // body-axis rotational dofs: axis_k_dot = om x axis_k, summed over k with qd_k gives om x om = 0
    }
    for (int k = 0; k < 3; ++k) { w.rne.b_w[b][k] = om[k]; w.rne.b_al[b][k] = al[k]; w.rne.b_v[b][k] = v[k]; w.rne.b_a[b][k] = a[k]; }
    wsync<NL>();
  }
  // wrench of each body about its own origin (parallel over bodies)
  for (int b = 1 + lane; b < nb; b += NL) {
    const real mass = m.body_mass[b];
    real F[3] = {0, 0, 0}, N[3] = {0, 0, 0};
    if (mass > 0) {
      real I6[6], c[3] = {w.xipos[b][0] - w.xpos[b][0], w.xipos[b][1] - w.xpos[b][1], w.xipos[b][2] - w.xpos[b][2]};
      body_inertia_world(m, w, b, I6);
      real t[3], t2[3], ac[3], Iw[3], Ial[3];
      cross3(t, w.rne.b_w[b], c);
      cross3(t2, w.rne.b_w[b], t);
      cross3(t, w.rne.b_al[b], c);
      for (int k = 0; k < 3; ++k) ac[k] = w.rne.b_a[b][k] + t[k] + t2[k];
      for (int k = 0; k < 3; ++k) F[k] = mass * ac[k];
      sym6_mulvec(Iw, I6, w.rne.b_w[b]);
      sym6_mulvec(Ial, I6, w.rne.b_al[b]);
      cross3(t, w.rne.b_w[b], Iw);
      cross3(t2, c, F);
      for (int k = 0; k < 3; ++k) N[k] = Ial[k] + t[k] + t2[k];
    }
    for (int k = 0; k < 3; ++k) { w.rne.b_F[b][k] = F[k]; w.rne.b_N[b][k] = N[k]; }
  }
  wsync<NL>();
  // project: dof i collects the wrenches of every body in its subtree (parallel over dofs)
  for (int i = lane; i < nv; i += NL) {
    const int bi = m.dof_body[i];
    real F[3] = {0, 0, 0}, N[3] = {0, 0, 0};  // torque about the dof anchor
    const real* an = w.dof_anchor[i];
    for (int c = bi; c < nb; ++c) {
      if (!((m.body_anc[c] >> bi) & 1u)) continue;
      real r[3] = {w.xpos[c][0] - an[0], w.xpos[c][1] - an[1], w.xpos[c][2] - an[2]}, t[3];
      cross3(t, r, w.rne.b_F[c]);
      for (int k = 0; k < 3; ++k) { F[k] += w.rne.b_F[c][k]; N[k] += w.rne.b_N[c][k] + t[k]; }
    }
    w.bias[i] = m.dof_rot[i] ? dot3(w.dof_axis[i], N) : dot3(w.dof_axis[i], F);
  }
  wsync<NL>();
}

// ------------------------------------------------------------------------------------------------ Cholesky
// In-place lower Cholesky of the n x n SPD matrix A (leading dimension LDM); row i is owned by lane i.
template <int NL>
MJ_FN int chol_factor(real (*A)[LDM], int n, int lane) {
  int ok = 1;
  for (int j = 0; j < n; ++j) {
    for (int i = j + lane; i < n; i += NL) {
      real s = A[i][j];
      for (int k = 0; k < j; ++k) s -= A[i][k] * A[j][k];
      A[i][j] = s;  // unscaled; row j's own entry is the pivot
    }
    wsync<NL>();
    const real piv = A[j][j];
    if (!(piv > MINVAL)) { ok = 0; break; }
    const real d = sqrtf(piv), inv = 1.0f / d;
    wsync<NL>();
    for (int i = j + lane; i < n; i += NL) A[i][j] = (i == j) ? d : A[i][j] * inv;
    wsync<NL>();
  }
  return ok;
}
// x <- A^-1 x given the Cholesky factor (x in shared memory)
template <int NL>
MJ_FN void chol_solve(real (*L)[LDM], int n, real* x, int lane) {
  for (int j = 0; j < n; ++j) {
    const real xj = x[j] / L[j][j];
    wsync<NL>();
    if (lane == 0) x[j] = xj;
    for (int i = j + 1 + lane; i < n; i += NL) x[i] -= L[i][j] * xj;
    wsync<NL>();
  }
  for (int j = n - 1; j >= 0; --j) {
    const real xj = x[j] / L[j][j];
    wsync<NL>();
    if (lane == 0) x[j] = xj;
    for (int i = lane; i < j; i += NL) x[i] -= L[j][i] * xj;
    wsync<NL>();
  }
}

#if defined(__CUDACC__)
// Device path of spd_solve (n <= 32): lane i owns row i of the factor in shared memory (odd leading dimension, so own-row
// and same-row accesses are conflict free); the pivot and the substitution operands travel by warp shuffle, the
// right-hand side stays in a register.  One warp barrier per column, none in the two triangular solves, and a few
// dozen instructions of code (an earlier fully unrolled all-register version was 47 KB of SASS and made the kernel
// instruction-fetch bound).
__device__ __noinline__ int spd_solve_reg(real (*A)[LDM], int n, real* x, int lane) {
  const unsigned FULL = 0xffffffffu;
  const int i = lane;
  const bool row = i < n;
  int ok = 1;
  real invd = 1.0f;  // 1 / L[i][i] of this lane's row
  for (int j = 0; j < n; ++j) {
    real s = 0.0f;
    if (row && i >= j) {
      s = A[i][j];
      for (int k = 0; k < j; ++k) s -= A[i][k] * A[j][k];
    }
    const real piv = __shfl_sync(FULL, s, j);
    if (!(piv > MINVAL)) ok = 0;
    const real inv = rsqrtf(fmaxf(piv, MINVAL));
    if (i == j) invd = inv;
    if (row && i >= j) A[i][j] = (i == j) ? piv * inv : s * inv;
    __syncwarp();
  }
  real xi = row ? x[i] : 0.0f;
  for (int j = 0; j < n; ++j) {
    if (i == j) xi *= invd;
    const real xj = __shfl_sync(FULL, xi, j);
    if (row && i > j) xi -= A[i][j] * xj;
  }
  for (int j = n - 1; j >= 0; --j) {
    if (i == j) xi *= invd;
    const real xj = __shfl_sync(FULL, xi, j);
    if (i < j) xi -= A[j][i] * xj;
  }
  if (row) x[i] = xi;
  __syncwarp();
  return ok;
}
#endif

// x <- A^-1 x for the SPD matrix A (lower triangle read, overwritten by its factor)
template <int NL>
MJ_FN int spd_solve(real (*A)[LDM], int n, real* x, int lane) {
#if defined(__CUDA_ARCH__)
  if (NL == 32) return spd_solve_reg(A, n, x, lane);
#endif
  const int ok = chol_factor<NL>(A, n, lane);
  chol_solve<NL>(A, n, x, lane);
  return ok;
}

// ------------------------------------------------------------------------------------------------ constraint rows
MJ_HD real impedance(const real* solimp, real pos, real margin) {
  real dmin = clampr(solimp[0], MINIMP, MAXIMP), dmax = clampr(solimp[1], MINIMP, MAXIMP);
  real width = solimp[2] < MINVAL ? MINVAL : solimp[2];
  real mid = clampr(solimp[3], MINIMP, MAXIMP), power = solimp[4] < 1 ? 1.0f : solimp[4];
  if (dmin == dmax || width <= MINVAL) return 0.5f * (dmin + dmax);
  real x = fabsf(pos - margin) / width, y;
  if (x >= 1) return dmax;
  if (x <= 0) return dmin;
  if (power == 1) y = x;
  else if (power == 2) y = (x <= mid) ? x * x / mid : 1 - (1 - x) * (1 - x) / (1 - mid);
#if !defined(__CUDA_ARCH__)
  else y = (x <= mid) ? powf(x, power) / powf(mid, power - 1) : 1 - powf(1 - x, power) / powf(1 - mid, power - 1);
#else
  else y = x;  // unreachable: the host rejects models whose solimp power is neither 1 nor 2 (keeps powf out of the kernel)
#endif
  return dmin + y * (dmax - dmin);
}

// aref / R / D of row r from (solref, solimp, pos, margin, diagApprox); mj_makeImpedance + mj_referenceConstraint
// `imp_pos` < 0: the impedance is evaluated at the row's own violation; >= 0: at this violation (vector residuals: the
// six rows of a weld share the impedance of the residual's Euclidean norm, engine_core_constraint.c getposdim)
// `vel_known`: J qvel of the row when the caller has it for free (rows with one or two non-zero Jacobian entries)
MJ_FN void finish_row(const Model& m, Work& w, int r, const real* solref, const real* solimp, real margin, real diag, real* R_out,
                      real imp_pos = -1.0f, const real* vel_known = nullptr) {
  real vel = 0;
  if (vel_known) vel = *vel_known;
  else for (int k = 0; k < m.nv; ++k) vel += w.J[r][k] * w.qvel[k];
  const real imp = impedance(solimp, imp_pos >= 0 ? imp_pos : w.e_pos[r], margin);
  const real dmax = clampr(solimp[1], MINIMP, MAXIMP);
  real k, b;
  if (solref[0] > 0) {
    const real tc = solref[0] < 2 * m.timestep ? 2 * m.timestep : solref[0];  // refsafe
    const real dr = solref[1];
    k = 1 / (dmax * dmax * tc * tc * dr * dr);
    b = 2 / (dmax * tc);
  } else {
    k = -solref[0] / (dmax * dmax);
    b = -solref[1] / dmax;
  }
  real R = (1 - imp) * diag / imp;
  if (R < MINVAL) R = MINVAL;
  w.e_R[r] = R;
  w.e_D[r] = 1 / R;
  w.e_aref[r] = -b * vel - k * imp * (w.e_pos[r] - margin);
  if (R_out) *R_out = R;
}

// Jacobian column of dof c for a point `pt` rigidly attached to body b (zero if c does not move b)
MJ_FN void jac_col(const Model& m, const Work& w, int b, const real* pt, int c, real* jp, real* jr) {
  if ((m.body_anc[b] >> m.dof_body[c]) & 1u) {
    if (m.dof_rot[c]) {
      real r[3] = {pt[0] - w.dof_anchor[c][0], pt[1] - w.dof_anchor[c][1], pt[2] - w.dof_anchor[c][2]};
      cross3(jp, w.dof_axis[c], r);
      jr[0] = w.dof_axis[c][0]; jr[1] = w.dof_axis[c][1]; jr[2] = w.dof_axis[c][2];
    } else {
      jp[0] = w.dof_axis[c][0]; jp[1] = w.dof_axis[c][1]; jp[2] = w.dof_axis[c][2];
      jr[0] = jr[1] = jr[2] = 0;
    }
  } else {
    jp[0] = jp[1] = jp[2] = jr[0] = jr[1] = jr[2] = 0;
  }
}

template <int NL>
MJ_FN void make_constraints(const Model& m, Work& w, int lane) {
  const int nv = m.nv;
  int r = 0;
  // --- mocap weld: 3 translational + 3 rotational rows (mj_instantiateEquality, mjEQ_WELD)
  for (int wi = 0; wi < m.nweld; ++wi) {
    const int b = m.weld_body[wi];
    const real* rel = m.weld_relpose[wi];
    real p1[3], q1[4], t[3], mq[4], mR[9], quat[4], q1c[4], quat2[4];
    mulmatvec3(t, w.xmat[b], m.weld_pos[wi]);
    for (int k = 0; k < 3; ++k) p1[k] = w.xpos[b][k] + t[k];
    mulquat(q1, w.xquat[b], m.weld_quat[wi]);
    for (int k = 0; k < 4; ++k) mq[k] = w.mocap_quat[k];
    normquat(mq);
    quat2mat(mR, mq);
    mulmatvec3(t, mR, rel);
    real cpos[6];
    for (int k = 0; k < 3; ++k) cpos[k] = (real)(w.mocap_pos[k] - (double)p1[k]) + t[k];
    mulquat(quat, mq, rel + 3);
    q1c[0] = q1[0]; q1c[1] = -q1[1]; q1c[2] = -q1[2]; q1c[3] = -q1[3];
    mulquat(quat2, q1c, quat);
    for (int k = 0; k < 3; ++k) cpos[3 + k] = quat2[1 + k];
    for (int c = lane; c < nv; c += NL) {
      real jp[3], jr[3];
      jac_col(m, w, b, p1, c, jp, jr);
      real ax[4] = {0, -jr[0], -jr[1], -jr[2]}, q2[4], q3[4];
      mulquat(q2, q1c, ax);
      mulquat(q3, q2, quat);
      for (int k = 0; k < 3; ++k) {
        w.J[r + k][c] = -jp[k];
        w.J[r + 3 + k][c] = 0.5f * q3[1 + k];
      }
    }
    for (int k = lane; k < 6; k += NL) { w.e_pos[r + k] = cpos[k]; w.e_type[r + k] = ROW_EQ; }
    wsync<NL>();
    const real cnorm = msqrt(cpos[0] * cpos[0] + cpos[1] * cpos[1] + cpos[2] * cpos[2] + cpos[3] * cpos[3] + cpos[4] * cpos[4] +
                             cpos[5] * cpos[5]);
    for (int k = lane; k < 6; k += NL)
      finish_row(m, w, r + k, m.weld_solref[wi], m.weld_solimp[wi], 0.0f, m.weld_invweight[wi][k >= 3], nullptr, cnorm);
    r += 6;
  }
  // --- joint equalities q1 - q1_0 = poly(q2 - q2_0) (mj_instantiateEquality, mjEQ_JOINT): one lane per equality
  if (KITCHEN_ROWS && m.neq > 0) {
    if (r + m.neq > MAXEFC) { if (lane == 0) w.bad |= 8; }
    else {
      for (int e = lane; e < m.neq; e += NL) {
        const int q1 = m.eq_qposadr[e][0], q2 = m.eq_qposadr[e][1], d1 = m.eq_dofadr[e][0], d2 = m.eq_dofadr[e][1];
        const real dif = w.qpos[q2] - m.qpos0[q2];
        real pw = 1, cpos = w.qpos[q1] - m.qpos0[q1], deriv = 0;
        for (int k = 0; k < 5; ++k) {
          cpos -= m.eq_polycoef[e][k] * pw;
          if (k < 4) deriv += (k + 1) * m.eq_polycoef[e][k + 1] * pw;
          pw *= dif;
        }
        const int row = r + e;
        for (int c = 0; c < nv; ++c) w.J[row][c] = c == d1 ? 1.0f : (c == d2 ? -deriv : 0.0f);
        w.e_pos[row] = cpos;
        w.e_type[row] = ROW_EQ;
        const real vel = w.qvel[d1] - deriv * w.qvel[d2];
        finish_row(m, w, row, m.eq_solref[e], m.eq_solimp[e], 0.0f, m.eq_invweight[e], nullptr, -1.0f, &vel);
      }
      r += m.neq;
    }
    wsync<NL>();
  }
  // --- dof friction loss (mj_instantiateFriction): one row per dof with frictionloss > 0, residual 0; one lane per dof
  if (KITCHEN_ROWS) {
    int nf = 0;
    for (int i = 0; i < nv; ++i) nf += m.dof_frictionloss[i] > 0;
    if (r + nf > MAXEFC) { if (lane == 0 && nf) w.bad |= 8; }
    else if (nf) {
      for (int i = lane; i < nv; i += NL) {
        if (!(m.dof_frictionloss[i] > 0)) continue;
        int k = 0;
        for (int j = 0; j < i; ++j) k += m.dof_frictionloss[j] > 0;
        const int row = r + k;
        for (int c = 0; c < nv; ++c) w.J[row][c] = c == i ? 1.0f : 0.0f;
        w.e_pos[row] = 0;
        w.e_type[row] = ROW_FRICTION;
        const real vel = w.qvel[i];
        finish_row(m, w, row, m.dof_solref_friction[i], m.dof_solimp_friction[i], 0.0f, m.dof_invweight0[i], nullptr, -1.0f, &vel);
        w.e_pos[row] = m.dof_frictionloss[i];  // from here on e_pos of a friction row is its force bound
      }
      r += nf;
    }
    wsync<NL>();
  }
  // --- joint limits (hinge / slide): candidates (joint, side) in order, one lane each; rows are allocated by a prefix
  // count over the active ones, so the row order is that of the serial loop
  const int ncand = 2 * m.njnt;
  for (int base = 0; base < ncand; base += NL) {
    const int idx = base + lane, j = idx >> 1, side = idx & 1;
    bool act = false;
    real dist = 0;
    if (idx < ncand && m.jnt_limited[j] && m.jnt_type[j] >= 2) {
      const int qa = m.jnt_qposadr[j];
      dist = side == 0 ? w.qpos[qa] - m.jnt_range[j][0] : m.jnt_range[j][1] - w.qpos[qa];
      act = dist < m.jnt_margin[j];
    }
#if defined(__CUDA_ARCH__)
    const unsigned mask = NL > 1 ? __ballot_sync(0xffffffffu, act) : (act ? 1u : 0u);
    const int before = __popc(mask & ((1u << lane) - 1u)), cnt = __popc(mask);
#else
    const int before = 0, cnt = act ? 1 : 0;
#endif
    if (act) {
      const int row = r + before;
      if (row < MAXEFC) {
        const int da = m.jnt_dofadr[j];
        const real sgn = side == 0 ? 1.0f : -1.0f;
        for (int c = 0; c < nv; ++c) w.J[row][c] = c == da ? sgn : 0.0f;
        w.e_pos[row] = dist;
        w.e_type[row] = ROW_LIMIT;
        const real vel = sgn * w.qvel[da];
        finish_row(m, w, row, m.jnt_solref[j], m.jnt_solimp[j], m.jnt_margin[j], m.dof_invweight0[da], nullptr, -1.0f, &vel);
      } else {
        w.bad |= 8;
      }
    }
    r += cnt;
    if (r > MAXEFC) r = MAXEFC;
  }
  wsync<NL>();
  w.nefc = r;
  wsync<NL>();
}

// ------------------------------------------------------------------------------------------------ convex solve
// minimise  0.5 (a - a_s)' M (a - a_s) + sum_rows s(J a - aref)   (MuJoCo "Computation": primal problem), Newton
// with exact line search.  Row cost and force for the current jar; state: 0 inactive, 1 quadratic, 2 cone zone.
MJ_HD void row_update(Work& w, int r) {
  const int tp = w.e_type[r];
  const real jar = w.e_jar[r], D = w.e_D[r];
  if (tp == ROW_EQ) { w.e_force[r] = -D * jar; w.e_state[r] = 1; }
  else if (tp == ROW_LIMIT) {
    if (jar < 0) { w.e_force[r] = -D * jar; w.e_state[r] = 1; }
    else { w.e_force[r] = 0; w.e_state[r] = 0; }
  } else if (KITCHEN_ROWS && tp == ROW_FRICTION) {  // quadratic inside |jar| < R f, linear (saturated force) outside; states 3 / 4 = saturated
    const real f = w.e_pos[r], rf = w.e_R[r] * f;
    if (jar <= -rf) { w.e_force[r] = f; w.e_state[r] = 3; }
    else if (jar >= rf) { w.e_force[r] = -f; w.e_state[r] = 4; }
    else { w.e_force[r] = -D * jar; w.e_state[r] = 1; }
  }
}

// elliptic cone of contact c at jar (+ alpha * jv when jv != null): cost, d/dalpha, d2/dalpha2; when `commit`,
// forces / zone / Hessian block are written.  Scaled variables U0 = jar0 * mu, Uj = jar_j * fri_j (engine_solver.c).
MJ_FN void cone_eval(Work& w, int c, real alpha, bool line, bool commit, real* cost, real* d1, real* d2) {
  const int r = w.con_row[c], dim = w.con_dim[c];
  const real mu = w.con_mu[c];
  const real* fri = w.con_fri[c];
  real U[4], V[4];
  U[0] = (w.e_jar[r] + (line ? alpha * w.e_jv[r] : 0.0f)) * mu;
  V[0] = line ? w.e_jv[r] * mu : 0.0f;
  real TT = 0, UV = 0, VV = 0;
  for (int j = 1; j < dim; ++j) {
    U[j] = (w.e_jar[r + j] + (line ? alpha * w.e_jv[r + j] : 0.0f)) * fri[j - 1];
    V[j] = line ? w.e_jv[r + j] * fri[j - 1] : 0.0f;
    TT += U[j] * U[j]; UV += U[j] * V[j]; VV += V[j] * V[j];
  }
  const real T = sqrtf(TT), N = U[0];
  const real Dm = w.e_D[r] / (mu * mu * (1 + mu * mu));
  real cst = 0, g = 0, h = 0;
  int zone;
  if (N >= mu * T || (T <= 0 && N >= 0)) zone = 0;                    // top: no force
  else if (mu * N + T <= 0 || (T <= 0 && N < 0)) zone = 1;            // bottom: quadratic in every row
  else zone = 2;                                                      // middle: cone
  if (zone == 1) {
    for (int j = 0; j < dim; ++j) {
      const real x = w.e_jar[r + j] + (line ? alpha * w.e_jv[r + j] : 0.0f), D = w.e_D[r + j];
      cst += 0.5f * D * x * x;
      if (line) { g += D * x * w.e_jv[r + j]; h += D * w.e_jv[r + j] * w.e_jv[r + j]; }
      if (commit) { w.e_force[r + j] = -D * x; w.e_state[r + j] = 1; }
    }
  } else if (zone == 2) {
    const real NT = N - mu * T;
    cst = 0.5f * Dm * NT * NT;
    if (line) {
      const real N1 = V[0], T1 = UV / T, T2 = (VV - T1 * T1) / T;
      g = Dm * NT * (N1 - mu * T1);
      h = Dm * ((N1 - mu * T1) * (N1 - mu * T1) - NT * mu * T2);
    }
    if (commit) {
      const real f0 = -Dm * NT * mu;
      w.e_force[r] = f0;
      for (int j = 1; j < dim; ++j) w.e_force[r + j] = -f0 / T * U[j] * fri[j - 1];
      for (int j = 0; j < dim; ++j) w.e_state[r + j] = 2;
      real* Hc = w.con_H[c];
      real scl[4];
      scl[0] = mu;
      for (int j = 1; j < dim; ++j) scl[j] = fri[j - 1];
      Hc[0] = 1;
      for (int j = 1; j < dim; ++j) Hc[j] = Hc[4 * j] = -mu * U[j] / T;
      for (int p = 1; p < dim; ++p)
        for (int q = 1; q < dim; ++q) Hc[4 * p + q] = mu * N / (TT * T) * U[p] * U[q] + (p == q ? mu * mu - mu * N / T : 0.0f);
      for (int p = 0; p < dim; ++p)
        for (int q = 0; q < dim; ++q) Hc[4 * p + q] *= Dm * scl[p] * scl[q];
    }
  } else if (commit) {
    for (int j = 0; j < dim; ++j) { w.e_force[r + j] = 0; w.e_state[r + j] = 0; }
  }
  if (cost) *cost = cst;
  if (d1) *d1 = g;
  if (d2) *d2 = h;
}

// jar = J a - aref, Ma = M a - qfrc_smooth (= M (a - a_smooth)), forces / states, gradient = Ma - J' f
template <int NL>
MJ_FN int solver_update(const Model& m, Work& w, int lane) {
  const int nv = m.nv, ne = w.nefc;
  real changed = 0;
  for (int r = lane; r < ne; r += NL) {
    real s = -w.e_aref[r];
    for (int c = 0; c < nv; ++c) s += w.J[r][c] * w.acc[c];
    w.e_jar[r] = s;
  }
  for (int i = lane; i < nv; i += NL) {
    real s = -w.smooth[i];
    for (int j = 0; j < nv; ++j) s += w.M[i][j] * w.acc[j];
    w.Ma[i] = s;
  }
  wsync<NL>();
  for (int r = lane; r < ne; r += NL)
    if (!is_cone_row(w.e_type[r])) {
      const int old = w.e_state[r];
      row_update(w, r);
      changed += (old != w.e_state[r]) ? 1.0f : 0.0f;
    }
  for (int c = lane; c < w.ncon; c += NL) {
    if (KITCHEN_ROWS && w.con_dim[c] <= 0) continue;  // pyramidal contact: its rows are plain unilateral rows
    const int old = w.e_state[w.con_row[c]];
    cone_eval(w, c, 0, false, true, nullptr, nullptr, nullptr);
    changed += (old != w.e_state[w.con_row[c]] || old == 2) ? 1.0f : 0.0f;  // the cone zone is not quadratic
  }
  changed = wsum<NL>(changed);
  wsync<NL>();
  for (int i = lane; i < nv; i += NL) {
    real s = w.Ma[i];
    for (int r = 0; r < ne; ++r) s -= w.J[r][i] * w.e_force[r];
    w.grad[i] = s;
  }
  wsync<NL>();
  return (int)changed;
}

// derivative and curvature of the 1-D cost along dir at step alpha (constraint part only)
template <int NL>
MJ_FN void line_eval(Work& w, real alpha, int lane, real* d1, real* d2) {
  real g = 0, h = 0;
  for (int r = lane; r < w.nefc; r += NL) {
    const int tp = w.e_type[r];
    if (is_cone_row(tp)) continue;
    const real x = w.e_jar[r] + alpha * w.e_jv[r], D = w.e_D[r], jv = w.e_jv[r];
    if (KITCHEN_ROWS && tp == ROW_FRICTION) {
      const real f = w.e_pos[r], rf = w.e_R[r] * f;
      if (x <= -rf) g -= f * jv;
      else if (x >= rf) g += f * jv;
      else { g += D * x * jv; h += D * jv * jv; }
    } else if (tp == ROW_EQ || x < 0) { g += D * x * jv; h += D * jv * jv; }
  }
  for (int c = lane; c < w.ncon; c += NL) {
    if (KITCHEN_ROWS && w.con_dim[c] <= 0) continue;
    real cg, ch;
    cone_eval(w, c, alpha, true, false, nullptr, &cg, &ch);
    g += cg; h += ch;
  }
  *d1 = wsum<NL>(g);
  *d2 = wsum<NL>(h);
}

template <int NL>
MJ_FN void solve(const Model& m, Work& w, int lane) {
  const int nv = m.nv, ne = w.nefc;
  if (ne == 0) {  // unconstrained: qacc = M^-1 qfrc_smooth
    for (int i = lane; i < nv; i += NL) {
      for (int j = 0; j <= i; ++j) w.H[i][j] = w.M[i][j];
      w.acc[i] = w.smooth[i];
      w.fcon[i] = 0;
    }
    wsync<NL>();
    if (!spd_solve<NL>(w.H, nv, w.acc, lane)) w.bad |= 1;
    w.solver_iter = 0;
    return;
  }
  // Start from the previous step's acceleration (qacc_warmstart).  MuJoCo starts from the cheaper of that and the
  // unconstrained acceleration; the problem is strictly convex, so the minimiser the iteration converges to is the
  // same, and skipping the comparison saves one factorisation of M and two cost evaluations per substep.
  for (int i = lane; i < nv; i += NL) w.acc[i] = w.warm[i];
  wsync<NL>();
  solver_update<NL>(m, w, lane);
  int it = 0;
  for (; it < m.iterations; ++it) {
    // Hessian = M + J' D J over active rows (+ cone blocks), lower triangle distributed over lanes
    const int npairs = nv * (nv + 1) / 2;
    for (int p = lane; p < npairs; p += NL) {
      int i = (int)((sqrtf(8.0f * p + 1.0f) - 1.0f) * 0.5f);
      while ((i + 1) * (i + 2) / 2 <= p) ++i;
      while (i * (i + 1) / 2 > p) --i;
      const int j = p - i * (i + 1) / 2;
      real s = w.M[i][j];
      for (int r = 0; r < ne; ++r)
        if (w.e_state[r] == 1) s += w.e_D[r] * w.J[r][i] * w.J[r][j];
      for (int c = 0; c < w.ncon; ++c) {
        const int r0 = w.con_row[c];
        if ((KITCHEN_ROWS && w.con_dim[c] <= 0) || w.e_state[r0] != 2) continue;
        const int dim = w.con_dim[c];
        for (int a = 0; a < dim; ++a)
          for (int b = 0; b < dim; ++b) s += w.con_H[c][4 * a + b] * w.J[r0 + a][i] * w.J[r0 + b][j];
      }
      w.H[i][j] = s;
    }
    for (int i = lane; i < nv; i += NL) w.dir[i] = -w.grad[i];
    wsync<NL>();
    if (!spd_solve<NL>(w.H, nv, w.dir, lane)) { w.bad |= 1; break; }
    // line search along dir
    for (int r = lane; r < ne; r += NL) {
      real s = 0;
      for (int c = 0; c < nv; ++c) s += w.J[r][c] * w.dir[c];
      w.e_jv[r] = s;
    }
    real g0 = 0, h0 = 0;
    for (int i = lane; i < nv; i += NL) {
      real s = 0;
      for (int j = 0; j < nv; ++j) s += w.M[i][j] * w.dir[j];
      g0 += w.dir[i] * w.Ma[i];
      h0 += w.dir[i] * s;
    }
    g0 = wsum<NL>(g0);
    h0 = wsum<NL>(h0);
    wsync<NL>();
    real alpha = 0, lo = 0, hi = -1, g, h, gstart;
    line_eval<NL>(w, 0, lane, &g, &h);
    g += g0; h += h0;
    gstart = fabsf(g);
#if defined(MJ_TRACE_DEVICE) && defined(__CUDA_ARCH__)
    if (threadIdx.x == 0) printf("  [dev] it %d  g %g h %g  (g0 %g h0 %g)\n", it, (double)g, (double)h, (double)g0, (double)h0);
#endif
    if (!(g < 0) || !(h > 0)) break;  // not a descent direction: converged to rounding
    for (int ls = 0; ls < 20; ++ls) {
      real next = alpha - g / h;
      if (hi > 0 && !(next > lo && next < hi)) next = 0.5f * (lo + hi);
      if (hi < 0 && !(next > lo)) next = 2 * alpha + 1;
      alpha = next;
      line_eval<NL>(w, alpha, lane, &g, &h);
      g += g0 + alpha * h0;
      h += h0;
      if (fabsf(g) <= 1e-6f * gstart) break;
      if (g > 0) hi = alpha; else lo = alpha;
      if (hi > 0 && hi - lo <= 1e-7f * hi) break;
    }
    real mx = 0, an = 0;
    for (int i = lane; i < nv; i += NL) {
      w.acc[i] += alpha * w.dir[i];
      mx = fmaxf(mx, fabsf(alpha * w.dir[i]));
      an = fmaxf(an, fabsf(w.acc[i]));
    }
    mx = wmax<NL>(mx);
    an = wmax<NL>(an);
    wsync<NL>();
    const int nchg = solver_update<NL>(m, w, lane);
#if defined(MJ_TRACE_DEVICE) && defined(__CUDA_ARCH__)
    if (threadIdx.x == 0) printf("  [dev] it %d alpha %g mx %g an %g nchg %d\n", it, (double)alpha, (double)mx, (double)an, nchg);
#endif
#if defined(MJ_DEBUG) && !defined(__CUDA_ARCH__)
    printf("  newton it %d alpha %g mx %g an %g g0 %g nchg %d\n", it, (double)alpha, (double)mx, (double)an, (double)gstart, nchg);
#endif
    // a full Newton step with no row changing its active set solves the problem exactly IF the cost is purely
    // quadratic there, i.e. no cone sits in its middle zone (where the cost is not quadratic and a step of length
    // ~1 can still be 1e-3 of a large step away from the minimiser); otherwise stop once the step is at the fp32
    // noise floor of the largest acceleration
    int nmid = 0;
    for (int c = 0; c < w.ncon; ++c) nmid += (!KITCHEN_ROWS || w.con_dim[c] > 0) && w.e_state[w.con_row[c]] == 2;
    const real floor_ = 1e-4f + 1e-5f * an;
    bool exact = nchg == 0 && nmid == 0 && fabsf(alpha - 1.0f) < 1e-3f;
    if (exact) {
      // ... in exact arithmetic.  The fp32 factorisation of an ill-conditioned Hessian (kN contact rows next to
      // 0.03 kg m^2 wrist joints) can leave the light dofs off by O(cond * eps) of the step: accept the shortcut only
      // if the gradient left over is small against those dofs' own inertia (H >= M, so |H^-1 g| <= max |g_i| / M_ii)
      real ge = 0;
      for (int i = lane; i < nv; i += NL) ge = fmaxf(ge, fabsf(w.grad[i]) / w.M[i][i]);
      ge = wmax<NL>(ge);
      if (ge > 10.0f * floor_) exact = false;
    }
    if (exact || mx <= floor_) { ++it; break; }
  }
  w.solver_iter = it;
  for (int i = lane; i < nv; i += NL) {
    real s = 0;
    for (int r = 0; r < ne; ++r) s += w.J[r][i] * w.e_force[r];
    w.fcon[i] = s;
  }
  wsync<NL>();
}

}  // namespace mj
}  // namespace earl
