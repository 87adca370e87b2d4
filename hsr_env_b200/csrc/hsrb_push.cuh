// Action kernel of the "sliding base + at most one free box" models (README block-push: --use-dof slide_x slide_y,
// --n-blocks 0/1; BASELINE.json configs[0], [1] and [3]).
//
// Same substep as the general kernel (hsrb_kernels.cuh / hsr_core.h, SURVEY.md App. B), laid out for the hardware:
//   * G lanes (8, 16 or 32) of a warp own one environment.  State (qpos, qvel, qacc_warmstart, ctrl, goal) is
//     replicated in the registers of the lanes for all 300 substeps; it touches HBM once per action.
//   * The robot only translates (two slides on one world-attached body): every robot geom keeps its compile-time
//     orientation and world AABB, its position is base + axis0*q0 + axis1*q1 (PushInfo tables).  The mass matrix
//     is constant and diagonal, so CRB / RNE / factorisation collapse to closed forms.
//   * Collision: one candidate pair per lane in the cull, one box corner per lane in plane-box, the hull scan of
//     the convex-convex support function across the lanes.
//   * Constraint rows live in the environment's slice of shared memory as 32-byte Jacobian rows (two 128-bit loads);
//     every solver loop is a short rolled loop over rows (rows across lanes) or over contacts (one contact per
//     lane), so the instruction footprint of a Newton iteration is a few hundred instructions instead of the
//     fully unrolled register version's ~6000 (ncu: 86 % of that kernel's stall samples were instruction fetch).
//   * Lane i < NV owns dof i: gradient component, Hessian row, Cholesky row.  The factorisation and the two
//     triangular solves are warp-shuffle exchanges between the 8 dof lanes.
//
// Replaces the loop over sim.step() in HSREnv.step (/root/reference/hsr/env.py:115-135).
#pragma once
#include "hsrb_kernels.cuh"

#ifndef PUSH_MAXCON
#define PUSH_MAXCON 8
#endif
// Block-wide barriers separate the phases of a substep: every warp of the SM runs the same code region at the same time
// (ncu: instruction-fetch stalls fell from 57 % to 7 % of the samples) and the convex-convex narrowphase jobs of all
// the block's environments go through one block-shared queue served by whole warps.
#define PUSH_MAXJOBS 96    // queue capacity per block and pair chunk; overflowing jobs run in their own group
#define PUSH_ENVJOBS 8     // queued jobs per environment and pair chunk
#define PUSH_ROWS (6 * PUSH_MAXCON)   // fixed stride of 6 rows per contact; rows >= condim are zero rows
#define PUSH_PAIRC 12      // doubles per candidate pair in PushInfo::pairc
#define PUSH_SEPMAX 32     // candidate pairs with a cached separating direction (mpr_penetration's `sep`)

// Model constants of this kernel family, filled on the host (push_fill_info) and passed by value as a kernel
// parameter (uniform constant-bank reads); the per-geom / per-pair tables are device arrays.
struct PushInfo {
  int nv;                 // 2 (no block) or 8
  int robot_body, block_body;
  float Mdiag[8];         // [m_r, m_r, m_b, m_b, m_b, I1, I2, I3]
  float damp[8];
  float axis[2][3];       // slide axes in the world frame
  double axisd[2][3];     // the same in double (geom positions)
  float gq[2];            // generalised gravity force on the slides: m_r * (g . axis)
  int act_n; int act_dof[2]; int act_q[2];
  float kp[2], gear[2], cr_lo[2], cr_hi[2], fr_lo[2], fr_hi[2];
  int ctrllimited[2], forcelimited[2];
  int limited[2];
  float range[2][2];
  double lim_k[2], lim_b[2], lim_imp[2][5], lim_diag[2];   // reference-acceleration gains / impedance of the limits
  float gravity[3];
  // tables (device pointers; host pointers in the emulated build)
  const double* gbase;    // [ngeom][3] world position of the geom with both slides at 0 (static geoms: as is)
  const double* gmatw;    // [ngeom][9] world orientation of static / robot geoms; block geoms: geom_mat (body frame)
  const float* ghalf;     // [ngeom][3] world AABB half extents of static / robot geoms
  const int* gmove;       // [ngeom] 0 static, 1 rides on the robot, 2 rides on the block
  const double* pairc;    // [npair][PUSH_PAIRC] k, b, diagApprox, solimp d0, dmax, width, mid, power (clamped as MuJoCo does), 1/width, 1/mid, 1/(1-mid)
  const double* xmat0;    // [nbody][9] compile-time body orientations (world, robot; the block's is overwritten)
  const float* verts4;    // [nvert][4] hull vertices padded to 16 bytes (128-bit loads in the support scan)
};

// Host-side table builder (also used by the emulated build).  Layout of `tab` (doubles):
//   gbase ngeom*3 | gmatw ngeom*9 | pairc npair*PUSH_PAIRC | xmat0 nbody*9 | ghalf ngeom*3 (floats, padded) | gmove ngeom (ints, padded)
struct PushTables {
  std::vector<double> tab;
  size_t off_gbase, off_gmatw, off_pairc, off_xmat0, off_ghalf, off_gmove, off_verts4;
  void point(PushInfo& f, const unsigned char* base) const {
    f.gbase = (const double*)(base + off_gbase); f.gmatw = (const double*)(base + off_gmatw);
    f.pairc = (const double*)(base + off_pairc); f.xmat0 = (const double*)(base + off_xmat0);
    f.ghalf = (const float*)(base + off_ghalf); f.gmove = (const int*)(base + off_gmove);
    f.verts4 = (const float*)(base + off_verts4);
  }
  size_t bytes() const { return tab.size() * sizeof(double); }
};

// reference-acceleration gains and clamped impedance parameters of one (solref, solimp) pair (App. B.5)
inline void push_row_consts(double timestep, const float* solref, const float* solimp, double* k, double* b, double* imp5) {
  const double MINIMP = 1e-4, MAXIMP = 0.9999;
  double tc = std::fmax((double)solref[0], 2 * timestep), dr = (double)solref[1];
  double dmax = std::fmin(std::fmax((double)solimp[1], MINIMP), MAXIMP);
  *k = 1.0 / (dmax * dmax * tc * tc * dr * dr);
  *b = 2.0 / (dmax * tc);
  imp5[0] = std::fmin(std::fmax((double)solimp[0], MINIMP), MAXIMP);
  imp5[1] = dmax;
  imp5[2] = std::fmax(1e-15, (double)solimp[2]);
  imp5[3] = std::fmin(std::fmax((double)solimp[3], MINIMP), MAXIMP);
  imp5[4] = std::fmax(1.0, (double)solimp[4]);
}

// Is the model in the family this kernel handles?  One world-attached body carrying exactly two slide joints
// (constant orientation), optionally one world-attached free box whose frame is its principal-axis frame, actuators
// only on the slides.  `m` holds host pointers.
inline bool push_fill_info(const ModelT<float>& m, PushInfo& f, PushTables& t, char* why, size_t why_len) {
  memset(&f, 0, sizeof(f));
  auto no = [&](const char* msg) { snprintf(why, why_len, "%s", msg); return false; };
  if (m.nbody != 2 && m.nbody != 3) return no("needs 1 robot body and at most 1 block");
  if (m.body_parent[1] != 0 || m.body_jntnum[1] != 2) return no("robot body must carry exactly two joints");
  for (int j = 0; j < 2; j++)
    if (m.jnt_type[j] != JNT_SLIDE || m.jnt_dofadr[j] != j || m.jnt_qposadr[j] != j) return no("robot joints must be slides");
  f.robot_body = 1; f.block_body = -1; f.nv = 2;
  if (m.nbody == 3) {
    int j = m.body_jntadr[2];
    if (m.body_parent[2] != 0 || m.body_jntnum[2] != 1 || m.jnt_type[j] != JNT_FREE) return no("second body must be a free body");
    if (m.jnt_qposadr[j] != 2 || m.jnt_dofadr[j] != 2) return no("unexpected dof layout");
    if (m.body_ipos[6] != 0 || m.body_ipos[7] != 0 || m.body_ipos[8] != 0) return no("block frame must sit at its CoM");
    if (m.body_inertia[15] != 0 || m.body_inertia[16] != 0 || m.body_inertia[17] != 0) return no("block frame must be principal");
    f.block_body = 2; f.nv = 8;
  }
  if (m.nv != f.nv || m.nu > 2) return no("unexpected nv / nu");
  if (m.ngeom > 64 || m.npair > 256) return no("too many geoms / pairs");
  // robot orientation (constant) and world-frame slide axes, in double from the fp32 model constants
  double Rr[9], bq[4] = {(double)m.body_quat[4], (double)m.body_quat[5], (double)m.body_quat[6], (double)m.body_quat[7]};
  quatnormalize(bq);
  quat2mat(bq, Rr);
  double axd[2][3];
  for (int j = 0; j < 2; j++) {
    V3<double> ax = mulv(Rr, ldg(m.jnt_axis + 3 * j));
    axd[j][0] = ax.x; axd[j][1] = ax.y; axd[j][2] = ax.z;
    f.axisd[j][0] = ax.x; f.axisd[j][1] = ax.y; f.axisd[j][2] = ax.z;
    f.axis[j][0] = (float)ax.x; f.axis[j][1] = (float)ax.y; f.axis[j][2] = (float)ax.z;
  }
  double dot01 = axd[0][0] * axd[1][0] + axd[0][1] * axd[1][1] + axd[0][2] * axd[1][2];
  if (std::fabs(dot01) > 1e-7) return no("slide axes must be orthogonal (diagonal mass matrix)");
  for (int j = 0; j < 2; j++) {
    f.Mdiag[j] = m.body_mass[1];
    f.damp[j] = m.dof_damping[j];
    f.gq[j] = m.body_mass[1] * (m.gravity[0] * f.axis[j][0] + m.gravity[1] * f.axis[j][1] + m.gravity[2] * f.axis[j][2]);
    f.limited[j] = m.jnt_limited[j];
    f.range[j][0] = m.jnt_range[2 * j]; f.range[j][1] = m.jnt_range[2 * j + 1];
    push_row_consts((double)m.timestep, m.jnt_solref + 2 * j, m.jnt_solimp + 5 * j, &f.lim_k[j], &f.lim_b[j], f.lim_imp[j]);
    f.lim_diag[j] = (double)m.dof_invweight0[j];
  }
  if (f.nv == 8) {
    for (int k = 0; k < 3; k++) { f.Mdiag[2 + k] = m.body_mass[2]; f.Mdiag[5 + k] = m.body_inertia[12 + k]; }
    for (int k = 0; k < 6; k++) f.damp[2 + k] = m.dof_damping[2 + k];
  }
  f.act_n = m.nu;
  for (int k = 0; k < m.nu; k++) {
    if (m.act_dof[k] > 1) return no("actuators must drive the slides");
    f.act_dof[k] = m.act_dof[k]; f.act_q[k] = m.act_qposadr[k];
    f.kp[k] = m.act_kp[k]; f.gear[k] = m.act_gear[k];
    f.cr_lo[k] = m.act_ctrlrange[2 * k]; f.cr_hi[k] = m.act_ctrlrange[2 * k + 1];
    f.fr_lo[k] = m.act_forcerange[2 * k]; f.fr_hi[k] = m.act_forcerange[2 * k + 1];
    f.ctrllimited[k] = m.act_ctrllimited[k]; f.forcelimited[k] = m.act_forcelimited[k];
  }
  for (int k = 0; k < 3; k++) f.gravity[k] = m.gravity[k];
  // ---- tables
  const int ng = m.ngeom, np = m.npair, nb = m.nbody;
  size_t nd = (size_t)ng * 3 + (size_t)ng * 9 + (size_t)np * PUSH_PAIRC + (size_t)nb * 9;
  t.off_gbase = 0; t.off_gmatw = sizeof(double) * ng * 3; t.off_pairc = t.off_gmatw + sizeof(double) * ng * 9;
  t.off_xmat0 = t.off_pairc + sizeof(double) * np * PUSH_PAIRC;
  t.off_ghalf = sizeof(double) * nd;
  size_t nhalf_d = ((size_t)ng * 3 * sizeof(float) + 7) / 8, nmove_d = ((size_t)ng * sizeof(int) + 7) / 8;
  t.off_gmove = t.off_ghalf + 8 * nhalf_d;
  t.off_verts4 = t.off_gmove + 8 * nmove_d;
  t.off_verts4 += (16 - t.off_verts4 % 16) % 16;
  const size_t nv4_d = ((size_t)m.nvert * 4 * sizeof(float) + 7) / 8 + 2;
  t.tab.assign(t.off_verts4 / 8 + nv4_d, 0.0);
  double* gbase = t.tab.data(); double* gmatw = gbase + ng * 3; double* pairc = gmatw + ng * 9; double* xmat0 = pairc + np * PUSH_PAIRC;
  float* ghalf = (float*)((unsigned char*)t.tab.data() + t.off_ghalf);
  int* gmove = (int*)((unsigned char*)t.tab.data() + t.off_gmove);
  float* verts4 = (float*)((unsigned char*)t.tab.data() + t.off_verts4);
  for (int i = 0; i < m.nvert; i++)
    for (int k = 0; k < 3; k++) verts4[4 * i + k] = m.hull_vert[3 * i + k];
  const double I3[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  for (int k = 0; k < 9; k++) { xmat0[k] = I3[k]; xmat0[9 + k] = Rr[k]; if (nb == 3) xmat0[18 + k] = I3[k]; }
  // robot body origin with both slides at zero: body_pos - sum_j axis_j * qpos0_j  (xpos = body_pos + axis (q - q0))
  double rb0[3];
  for (int k = 0; k < 3; k++) rb0[k] = (double)m.body_pos[3 + k] - axd[0][k] * (double)m.qpos0[0] - axd[1][k] * (double)m.qpos0[1];
  for (int gi = 0; gi < ng; gi++) {
    int b = m.geom_body[gi];
    double gm[9];
    for (int k = 0; k < 9; k++) gm[k] = (double)m.geom_mat[9 * gi + k];
    if (b == f.block_body) {
      gmove[gi] = 2;
      for (int k = 0; k < 3; k++) gbase[3 * gi + k] = (double)m.geom_pos[3 * gi + k];
      for (int k = 0; k < 9; k++) gmatw[9 * gi + k] = gm[k];
      continue;
    }
    gmove[gi] = b == 1 ? 1 : 0;
    const double* Rb = b == 1 ? Rr : I3;
    V3<double> p = mulv(Rb, ldg(m.geom_pos + 3 * gi));
    for (int k = 0; k < 3; k++) gbase[3 * gi + k] = (b == 1 ? rb0[k] : 0.0) + comp(p, k);
    mulm(Rb, gm, gmatw + 9 * gi);
    // conservative world AABB half extents, fp32 like cdof_geoms (midphase cull only)
    float Rbf[9], Rg[9];
    for (int k = 0; k < 9; k++) Rbf[k] = (float)Rb[k];
    mulm(Rbf, m.geom_mat + 9 * gi, Rg);
    const float* h = m.geom_aabb + 3 * gi;
    for (int i = 0; i < 3; i++) ghalf[3 * gi + i] = std::fabs(Rg[3 * i]) * h[0] + std::fabs(Rg[3 * i + 1]) * h[1] + std::fabs(Rg[3 * i + 2]) * h[2];
  }
  for (int pk = 0; pk < np; pk++) {
    double* c = pairc + PUSH_PAIRC * pk;
    push_row_consts((double)m.timestep, m.pair_solref + 2 * pk, m.pair_solimp + 5 * pk, c + 0, c + 1, c + 3);
    c[8] = 1.0 / c[5]; c[9] = 1.0 / c[6]; c[10] = 1.0 / (1.0 - c[6]); c[11] = 0.0;   // reciprocals for impedance5<true>
    c[2] = (double)(m.geom_invweight[m.pair_geom1[pk]] + m.geom_invweight[m.pair_geom2[pk]]);  // fp32 sum, as row setup does
  }
  why[0] = 0;
  return true;
}

namespace push {

struct Ws {  // per-environment slice of shared memory
  GT *xpos, *xmat, *gpos;
  float* gaabb;
  float *con_dist, *con_pos, *con_frame;
  int *con_pair, *con_adr, *wi;
  float *J, *Dr, *aref, *jar, *jv, *f, *L;
  float* hq;             // rank-1 Hessian terms: p, q of the cone contacts [MAXCON][16], their weights [MAXCON][2], row weights [ROWS]
  int* jq;               // queue ids of this environment's convex-convex jobs, in pair order
  float* sep;            // [min(npair, PUSH_SEPMAX)][4] separating direction + valid flag of each candidate pair
  const float* verts4;   // hull vertices of the model as float4, one copy per block (after the per-environment slices)
};

// block-shared tail of dynamic shared memory: hull vertices as float4, then the narrowphase job queue
struct Blk {
  int* ctr;        // [0] jobs queued, [1] next job to serve
  int* jobs;       // [PUSH_MAXJOBS] (group << 16) | pair
  double* res;     // [PUSH_MAXJOBS][8] hit, depth, direction, position
  unsigned char* tab;   // block-shared model tables (Tab)
};
// Block-shared copies of the model tables the substep reads (a few KB): with ~200 KB of the SM's 256 KB carved out
// as shared memory the L1 is small and L2 is flushed between actions, so a table read from global memory costs an L2
// round trip on the critical path of every substep.
struct Tab {
  const double *gbase, *gmatw, *pairc;
  const float *ghalf, *geom_rbound, *geom_size, *pair_friction, *geom_mat, *geom_aabb;
  const int *gmove, *geom_type, *geom_body, *geom_vertadr, *geom_vertnum, *pair_geom1, *pair_geom2, *pair_func, *pair_condim;
};
__host__ __device__ inline size_t tab_bytes(const ModelT<float>& m) {
  const size_t ng = m.ngeom, np = m.npair;
  size_t b = 8 * (ng * 3 + ng * 9 + np * PUSH_PAIRC);
  b += 4 * (ng * 3 + ng + ng * 3 + np * 5 + ng * 9 + ng * 3);
  b += 4 * (ng * 5 + np * 4);
  return (b + 15) & ~(size_t)15;
}
__host__ __device__ inline size_t shared_tail(const ModelT<float>& m) {
  return (size_t)m.nvert * 16 + 16 + sizeof(int) * PUSH_MAXJOBS + sizeof(double) * 8 * PUSH_MAXJOBS + tab_bytes(m);
}
__host__ __device__ inline void carve_tail(const ModelT<float>& m, unsigned char* tail, const float** verts4, Blk* b) {
  *verts4 = (const float*)tail;
  unsigned char* p = tail + (size_t)m.nvert * 16;
  b->ctr = (int*)p; p += 16;
  b->jobs = (int*)p; p += sizeof(int) * PUSH_MAXJOBS;
  b->res = (double*)p; p += sizeof(double) * 8 * PUSH_MAXJOBS;
  b->tab = p;
}

__host__ __device__ inline size_t carve(const ModelT<float>& m, Ws* w, unsigned char* base) {
  size_t off = 0;
  Ws dummy;
  if (!w) w = &dummy;
#define CARVE(field, type, n) { w->field = (type*)(base + off); off += sizeof(type) * (size_t)(n); off += (16 - off % 16) % 16; }
  const int nb = m.nbody, nc = PUSH_MAXCON, nr = PUSH_ROWS;
  CARVE(xpos, GT, nb * 3) CARVE(xmat, GT, nb * 9) CARVE(gpos, GT, m.ngeom * 3)
  CARVE(gaabb, float, m.ngeom * 3)
  CARVE(con_dist, float, nc) CARVE(con_pos, float, nc * 3) CARVE(con_frame, float, nc * 9)
  CARVE(con_pair, int, nc) CARVE(con_adr, int, nc) CARVE(wi, int, WI_COUNT)
  CARVE(J, float, nr * 8) CARVE(hq, float, 18 * nc + nr) CARVE(Dr, float, nr) CARVE(aref, float, nr) CARVE(jar, float, nr)
  CARVE(jv, float, nr) CARVE(f, float, nr) CARVE(L, float, 64) CARVE(jq, int, PUSH_ENVJOBS)
  CARVE(sep, float, 4 * (m.npair < PUSH_SEPMAX ? m.npair : PUSH_SEPMAX))
#undef CARVE
  return off;
}

struct F8 { float v[8]; };
__device__ __forceinline__ F8 ld8(const float* p) {  // 32-byte aligned row
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  F8 r; r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w; r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
  return r;
}
__device__ __forceinline__ void st8(float* p, const float* v) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}

// impedance d(|pos|) with pre-clamped parameters c = {d0, dmax, width, mid, power}  (App. B.5); INV: c[5..7] hold
// 1/width, 1/mid, 1/(1-mid) (the candidate-pair table), which takes three double divisions off every contact
template <bool INV = false>
__device__ __forceinline__ double impedance5(const double* c, double pos) {
  const double d0 = c[0], dmax = c[1], width = c[2], mid = c[3], power = c[4];
  if (d0 == dmax || width <= 1e-15) return 0.5 * (d0 + dmax);
  const double x = INV ? fabs(pos) * c[5] : fabs(pos) / width;
  if (x >= 1) return dmax;
  if (x == 0) return d0;
  double y;
  if (power == 1) y = x;
  else if (power == 2) y = x <= mid ? (INV ? c[6] : 1.0 / mid) * (x * x) : 1.0 - (INV ? c[7] : 1.0 / (1.0 - mid)) * ((1.0 - x) * (1.0 - x));
  else if (x <= mid) y = (1.0 / pow(mid, power - 1)) * pow(x, power);
  else y = 1.0 - (1.0 / pow(1 - mid, power - 1)) * pow(1 - x, power);
  return d0 + y * (dmax - d0);
}

}  // namespace push

// geometry of one geom for the shared narrowphase routines: pose from the tables / the block pose, no matrix product
// for static and robot geoms
__device__ __forceinline__ void push_load_geom(const ModelT<float>& m, const push::Tab& t, const push::Ws& s, int gi, Geom<float>& ge) {
  ge.type = t.geom_type[gi];
#pragma unroll
  for (int k = 0; k < 3; k++) ge.size[k] = t.geom_size[3 * gi + k];
  ge.verts = m.hull_vert + 3 * t.geom_vertadr[gi]; ge.nvert = t.geom_vertnum[gi];
  ge.verts4 = s.verts4 + 4 * t.geom_vertadr[gi];   // block-shared copy in shared memory
  ge.pos = ld3(s.gpos + 3 * gi);
  const double* gm = t.gmatw + 9 * gi;
  if (t.gmove[gi] == 2) mulm(s.xmat + 9 * t.geom_body[gi], gm, ge.mat);
  else {
#pragma unroll
    for (int k = 0; k < 9; k++) ge.mat[k] = gm[k];
  }
}

// ---------------------------------------------------------------------------------------------------- collision
// Candidate pairs -> bounding-sphere + world-AABB cull (one pair per lane) -> narrowphase.  Contacts are appended to
// the workspace in pair order (plane-box: corner order), exactly as the general kernel's collision() does.
#ifndef PUSH_COLLISION_ATTR
#define PUSH_COLLISION_ATTR __noinline__
#endif
template <int G>
__device__ PUSH_COLLISION_ATTR int push_collision(const ModelT<float>& m, const push::Tab& t, push::Ws& s, WS<float>& w,
                                           const DevGrp<G>& g, const push::Blk& blk, unsigned char* smem, unsigned ws_bytes, unsigned opts) {
  int ncon = 0, nrow = 0, narrow = 0, npflop = 0;
  const int gi = threadIdx.x / G;
  for (int base = 0; base < m.npair; base += 32) {
    // ---- cull up to 32 candidate pairs (G per round, one pair per lane) into this environment's job mask
    unsigned bits = 0;
    for (int k0 = 0; k0 < 32 && base + k0 < m.npair; k0 += G) {
      const int k = base + k0 + g.lane;
      bool hit = false;
      if (k < m.npair) {
        const int a = t.pair_geom1[k], b = t.pair_geom2[k];
        const V3<float> dp = cvt<float>(ld3(s.gpos + 3 * b) - ld3(s.gpos + 3 * a));
        if (t.geom_type[a] == GEOM_PLANE) {
          const double* Ma = t.gmatw + 9 * a;  // planes are static: world orientation is a table entry
          hit = dot(dp, mk<float>((float)Ma[2], (float)Ma[5], (float)Ma[8])) <= t.geom_rbound[b];
        } else {
          const float rr = t.geom_rbound[a] + t.geom_rbound[b];
          hit = dot(dp, dp) <= rr * rr;
          const float* ha = s.gaabb + 3 * a; const float* hb = s.gaabb + 3 * b;
          hit = hit && fabsf(dp.x) <= ha[0] + hb[0] && fabsf(dp.y) <= ha[1] + hb[1] && fabsf(dp.z) <= ha[2] + hb[2];
        }
      }
      bits |= ((__ballot_sync(0xffffffffu, hit) >> g.shift) & ((G == 32) ? 0xffffffffu : ((1u << G) - 1u))) << k0;   // full-warp vote, own group's bits
    }
    // ---- queue the convex-convex candidates of this environment (pair order) for the block's warps
    if (g.lane == 0) {
      unsigned bb = bits;
      int nq = 0;
      while (bb) {
        const int l = __ffs((int)bb) - 1;
        bb &= bb - 1;
        if (t.pair_func[base + l] != NP_CONVEX_CONVEX) continue;
        if (nq < PUSH_ENVJOBS) {
          // longest jobs first: a pair without a cached separating direction (in contact last time, or new) is a full
          // refinement (~11 support evaluations) and goes to the front half of the queue, a pair with one is usually a
          // single support evaluation and goes to the back half, which the warps serve afterwards
          const int pk_ = base + l;
          const bool quick = pk_ < PUSH_SEPMAX && !(opts & 1u) && s.sep[4 * pk_ + 3] == 1.f;
          int j = atomicAdd(blk.ctr + (quick ? 2 : 0), 1);
          if (j < PUSH_MAXJOBS / 2) { j += quick ? PUSH_MAXJOBS / 2 : 0; blk.jobs[j] = (gi << 16) | pk_; } else j = -1;
          s.jq[nq] = j;
        }
        nq++;
      }
    }
    __syncthreads();
    // ---- portal refinement of the queued jobs: one job per warp at a time (32 lanes scan the hull), warps take jobs
    //      dynamically, results go to the queue's result records
    {
      DevGrp<32> gw;
      int total = blk.ctr[0], slot0 = 0;
      int* next = blk.ctr + 1;
      if (total > PUSH_MAXJOBS / 2) total = PUSH_MAXJOBS / 2;
      while (true) {
        int j = 0;
        if (gw.lane == 0) j = atomicAdd(next, 1);
        j = __shfl_sync(0xffffffffu, j, 0);
        if (j >= total) {
          if (slot0) break;
          slot0 = PUSH_MAXJOBS / 2; next = blk.ctr + 3; total = blk.ctr[2];   // then the quick half
          if (total > PUSH_MAXJOBS / 2) total = PUSH_MAXJOBS / 2;
          continue;
        }
        j += slot0;
        const int code = blk.jobs[j];
        const int pk = code & 0xffff;
        push::Ws so;
        push::carve(m, &so, smem + (size_t)(code >> 16) * ws_bytes);
        so.verts4 = s.verts4;
        Geom<float> A, B;
        push_load_geom(m, t, so, t.pair_geom1[pk], A);
        push_load_geom(m, t, so, t.pair_geom2[pk], B);
        GT depth = 0; V3<GT> dir = mk<GT>(0, 0, 1), pos = mk<GT>(0, 0, 0);
        // inlined instance: the two geoms and the portal stay in registers (the out-of-line one keeps them on the local
        // stack and reloads them around every support evaluation; +16 % substeps/s)
        const bool hit = mpr_penetration_inl(A, B, (GT)m.mpr_tolerance, m.mpr_iterations, gw, depth, dir, pos,
                                         pk < PUSH_SEPMAX && !(opts & 1u) ? so.sep + 4 * pk : nullptr);
        if (gw.lane == 0) {
          double* r = blk.res + 8 * j;
          r[0] = hit ? 1.0 : 0.0; r[1] = depth; r[2] = dir.x; r[3] = dir.y; r[4] = dir.z; r[5] = pos.x; r[6] = pos.y; r[7] = pos.z;
        }
      }
    }
    __syncthreads();
    // ---- contacts of this environment in pair order (plane-box: corner order), exactly as the general kernel's
    //      collision() appends them; the environments of a warp take their k-th candidate in the same round
    int qi = 0;
    while (__any_sync(0xffffffffu, bits != 0)) {
      if (bits) {
        const int l = __ffs((int)bits) - 1;
        bits &= bits - 1;
        const int pk = base + l;
        const int func = t.pair_func[pk];
        narrow++;
        npflop += func == NP_PLANE_BOX ? 80 : (func == NP_PLANE_CONVEX ? 100 : (func == NP_BOX_BOX ? 500 : 5000));
        if (func == NP_PLANE_BOX) {
          // mjc_PlaneBox: one corner per lane; the first four penetrating corners (corner order) become contacts
          const int ga = t.pair_geom1[pk], gb = t.pair_geom2[pk];
          const double* Ma = t.gmatw + 9 * ga;
          const V3<GT> n = mk<GT>(Ma[2], Ma[5], Ma[8]);
          const V3<GT> pb = ld3(s.gpos + 3 * gb);
          const GT dist0 = dot(pb - ld3(s.gpos + 3 * ga), n);
          const int i = g.lane;
          const float* sz = t.geom_size + 3 * gb;
          const V3<GT> c = mk<GT>((i & 1) ? (GT)sz[0] : -(GT)sz[0], (i & 2) ? (GT)sz[1] : -(GT)sz[1], (i & 4) ? (GT)sz[2] : -(GT)sz[2]);
          // geom orientation in the world: table entry (static / robot geoms) or xmat(block) * geom_mat, applied to the
          // corner as matrix-vector products
          V3<GT> vec = mulv(t.gmatw + 9 * gb, c);
          if (t.gmove[gb] == 2) vec = mulv(s.xmat + 9 * t.geom_body[gb], vec);
          const GT ld = dot(n, vec);
          const bool pen = i < 8 && !(dist0 + ld > 0 || ld > 0);
          const unsigned pm = g.ballot(pen);
          const int rank = __popc(pm & ((1u << i) - 1u));
          int nh = __popc(pm);
          if (nh > 4) nh = 4;
          const int room = m.ncon_max - ncon;
          if (pen && rank < nh && rank < room) {
            const int slot = ncon + rank;
            const GT dist = dist0 + ld;
            s.con_pair[slot] = pk; s.con_dist[slot] = (float)dist;
            st3c(s.con_pos + 3 * slot, pb + vec - n * (dist * GT(0.5)));
            make_frame(n, s.con_frame + 9 * slot);
          }
          if (nh > room) { nh = room; if (g.lane == 0) s.wi[WI_FLAGS] |= FLAG_CON_OVERFLOW; }
          ncon += nh;
        } else if (func == NP_CONVEX_CONVEX && qi < PUSH_ENVJOBS && s.jq[qi] >= 0) {
          const double* r = blk.res + 8 * s.jq[qi];
          qi++;
          if (r[0] != 0.0) add_contact(m, w, g, ncon, nrow, pk, -r[1], mk<GT>(r[5], r[6], r[7]), mk<GT>(r[2], r[3], r[4]));
        } else {
          if (func == NP_CONVEX_CONVEX) qi++;   // did not fit the queue: refine here, with this group's lanes
          Geom<float> A, B;
          push_load_geom(m, t, s, t.pair_geom1[pk], A);
          push_load_geom(m, t, s, t.pair_geom2[pk], B);
          if (func == NP_PLANE_CONVEX) {
            const V3<GT> n = mcol(A.mat, 2);
            const V3<GT> p = support_d(B, -n, g);
            const GT dist = dot(p - A.pos, n);
            if (dist <= 0) add_contact(m, w, g, ncon, nrow, pk, dist, p - n * (dist * GT(0.5)), n);
          } else if (func == NP_BOX_BOX) {
            box_box(m, w, g, ncon, nrow, pk, A, B);
          } else {
            GT depth; V3<GT> dir, pos;
            if (mpr_penetration(A, B, (GT)m.mpr_tolerance, m.mpr_iterations, g, depth, dir, pos, pk < PUSH_SEPMAX && !(opts & 1u) ? s.sep + 4 * pk : nullptr))
              add_contact(m, w, g, ncon, nrow, pk, -depth, pos, dir);
          }
        }
      }
    }
    // the queue is empty again for the next chunk / substep (every thread is past the two barriers above and nothing is
    // queued before the next one)
    if (threadIdx.x == 0) { blk.ctr[0] = 0; blk.ctr[1] = 0; blk.ctr[2] = 0; blk.ctr[3] = 0; }
    if (base + 32 < m.npair) __syncthreads();
  }
  if (g.lane == 0) { s.wi[WI_NARROW] += narrow; s.wi[WI_NPFLOP] = npflop; }
  return ncon;
}

// ---------------------------------------------------------------------------------------------------- the kernel
template <int G, int NV>
__global__ void __launch_bounds__(G == 16 ? 448 : 256) hsrb_push_kernel(const __grid_constant__ KArgs a, const __grid_constant__ PushInfo fi) {
  HSRB_DYN_SMEM(smem);
  DevGrp<G> g;
  constexpr bool HASB = NV == 8;
  constexpr int SUBS = G / 8;                 // row stripes of the dof-lane loops
  const int gi = threadIdx.x / G;
  const int li = g.lane & 7;                  // dof owned by this lane
  const int sub = g.lane >> 3;                // row stripe of this lane in dof-lane loops
  push::Ws s;
  push::carve(a.m, &s, smem + (size_t)gi * a.ws_bytes);
  push::Blk blk;
  {
    // block-shared copy of the hull vertices (128-bit shared loads in the support scan; generic global loads need a
    // descriptor rebuilt from registers on every access when the warp is diverged) and the empty job queue
    unsigned char* tail = smem + (size_t)(blockDim.x / G) * a.ws_bytes;
    push::carve_tail(a.m, tail, &s.verts4, &blk);
    float* v4 = reinterpret_cast<float*>(tail);
    for (int i = threadIdx.x; i < a.m.nvert * 4; i += blockDim.x) v4[i] = fi.verts4[i];
    if (threadIdx.x == 0) { blk.ctr[0] = 0; blk.ctr[1] = 0; blk.ctr[2] = 0; blk.ctr[3] = 0; }
  }
  push::Tab t;
  {
    // block-shared copies of the model tables (doubles first: 8-byte alignment)
    unsigned char* p = blk.tab;
    const int ng = a.m.ngeom, np = a.m.npair;
#define TAB_COPY(field, type, src, n)                                                        \
  {                                                                                          \
    type* d_ = reinterpret_cast<type*>(p);                                                   \
    for (int i = threadIdx.x; i < (n); i += blockDim.x) d_[i] = (src)[i];                    \
    t.field = d_; p += sizeof(type) * (size_t)(n);                                           \
  }
    TAB_COPY(gbase, double, fi.gbase, ng * 3) TAB_COPY(gmatw, double, fi.gmatw, ng * 9) TAB_COPY(pairc, double, fi.pairc, np * PUSH_PAIRC)
    TAB_COPY(ghalf, float, fi.ghalf, ng * 3) TAB_COPY(geom_rbound, float, a.m.geom_rbound, ng)
    TAB_COPY(geom_size, float, a.m.geom_size, ng * 3) TAB_COPY(pair_friction, float, a.m.pair_friction, np * 5)
    TAB_COPY(geom_mat, float, a.m.geom_mat, ng * 9) TAB_COPY(geom_aabb, float, a.m.geom_aabb, ng * 3)
    TAB_COPY(gmove, int, fi.gmove, ng) TAB_COPY(geom_type, int, a.m.geom_type, ng) TAB_COPY(geom_body, int, a.m.geom_body, ng)
    TAB_COPY(geom_vertadr, int, a.m.geom_vertadr, ng) TAB_COPY(geom_vertnum, int, a.m.geom_vertnum, ng)
    TAB_COPY(pair_geom1, int, a.m.pair_geom1, np) TAB_COPY(pair_geom2, int, a.m.pair_geom2, np)
    TAB_COPY(pair_func, int, a.m.pair_func, np) TAB_COPY(pair_condim, int, a.m.pair_condim, np)
#undef TAB_COPY
    __syncthreads();
  }
  WS<float> w;                                // view for the shared narrowphase routines (hsr_core.h)
  w.xpos = s.xpos; w.xmat = s.xmat; w.gpos = s.gpos; w.gaabb = s.gaabb;
  w.con_dist = s.con_dist; w.con_pos = s.con_pos; w.con_frame = s.con_frame;
  w.con_pair = s.con_pair; w.con_adr = s.con_adr; w.wi = s.wi; w.sep = nullptr;
  const ModelT<float>& m = a.m;
  const int nq = m.nq;
  const float dt = m.timestep;
  const float scale = 1.0f / (m.meaninertia * (float)(NV > 1 ? NV : 1));
  const int epb = blockDim.x / G;

  // Control flow is uniform across the warp: every group runs the same number of environment rounds and substeps,
  // and the data-dependent loops (narrowphase jobs, Newton iterations) are voted on by the whole warp, so that the
  // groups of a warp execute each phase together instead of drifting apart and being issued one after the other.
  // A group without an environment (tail of the batch) or whose environment has finished its action keeps computing
  // on a copy; its results were written when it finished and nothing is stored afterwards.
  constexpr unsigned FULL = 0xffffffffu;
#ifndef PUSH_UNROLL_ROWS
#define PUSH_UNROLL_ROWS 6
#endif
  constexpr int UR = PUSH_UNROLL_ROWS;        // unroll factor of the per-dof row loops (gradient, Hessian)
  for (int env0 = blockIdx.x * epb; env0 < a.n; env0 += gridDim.x * epb) {
    const bool valid = env0 + gi < a.n;
    const int env = valid ? env0 + gi : a.n - 1;
    // ------------------------------------------------------------------ state -> registers (replicated)
    float qpos[9], qvel[8], warm[8], ctrl[2], mocap[3];
#pragma unroll
    for (int i = 0; i < 9; i++) qpos[i] = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) { qvel[i] = 0.f; warm[i] = 0.f; }
    {
      const float* st = a.state + (size_t)env * a.S;
#pragma unroll
      for (int i = 0; i < (HASB ? 9 : 2); i++) qpos[i] = st[i];
#pragma unroll
      for (int i = 0; i < NV; i++) { qvel[i] = st[nq + i]; warm[i] = st[nq + NV + i]; }
#pragma unroll
      for (int i = 0; i < 3; i++) mocap[i] = st[nq + 2 * NV + i];
      ctrl[0] = ctrl[1] = 0.f;
      if (a.ctrl)
        for (int i = 0; i < fi.act_n; i++) ctrl[i] = a.ctrl[(size_t)env * m.nu + i];
      for (int i = g.lane; i < WI_COUNT; i += G) s.wi[i] = 0;
      for (int i = g.lane; i < 4 * (m.npair < PUSH_SEPMAX ? m.npair : PUSH_SEPMAX); i += G) s.sep[i] = 0.f;   // no cached directions
      // constant part of the pose workspace: body orientations, static geoms, robot AABBs
      for (int i = g.lane; i < m.nbody * 9; i += G) s.xmat[i] = fi.xmat0[i];
      for (int i = g.lane; i < m.nbody * 3; i += G) s.xpos[i] = 0;
      for (int i = g.lane; i < m.ngeom * 3; i += G) {
        s.gpos[i] = t.gbase[i];
        s.gaabb[i] = t.ghalf[i];
      }
    }
    int n_iter = 0, n_ls = 0, sumcon = 0, sumefc = 0, kflop = 0, flags = 0;
    bool success = false;
    bool finished = !valid || a.nsub <= 0;   // results written (or nothing to write)
    int taken = 0;
    __syncwarp();
    if (valid && a.nsub <= 0) {
      // no substeps requested: the observation is the current state
      float* st = a.state + (size_t)env * a.S;
      const int nobs = nq + NV;
      for (int i = g.lane; i < nobs; i += G) if (a.obs) a.obs[(size_t)env * nobs + i] = st[i];
      if (g.lane == 0) {
        if (a.reward) a.reward[env] = 0.f;
        if (a.done) a.done[env] = 0;
        if (a.success) a.success[env] = 0;
        if (a.taken) a.taken[env] = 0;
        if (a.bad) a.bad[env] = 0;
      }
    }

    for (int sb_ = 0; sb_ < a.nsub; sb_++) {
      if (__syncthreads_and(finished)) break;
      HSR_PHASE_START(s, g);
      // ---------------------------------------------------------------- poses (B.1), geometry in double
      GT xb[3] = {0, 0, 0}, Rb[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
      if (HASB) {
        GT qd[4] = {(GT)qpos[5], (GT)qpos[6], (GT)qpos[7], (GT)qpos[8]};
        quatnormalize(qd);   // same rounding as the oracle: the narrowphase decisions downstream are discontinuous in the pose
#pragma unroll
        for (int k = 0; k < 4; k++) qpos[5 + k] = (float)qd[k];  // MuJoCo normalises qpos in place
        quat2mat(qd, Rb);
#pragma unroll
        for (int k = 0; k < 3; k++) xb[k] = (GT)qpos[2 + k];
        if (g.lane == 0) {
#pragma unroll
          for (int k = 0; k < 3; k++) s.xpos[3 * fi.block_body + k] = xb[k];
#pragma unroll
          for (int k = 0; k < 9; k++) s.xmat[9 * fi.block_body + k] = Rb[k];
        }
      }
      {
        const GT q0 = (GT)qpos[0], q1 = (GT)qpos[1];
        for (int gg = g.lane; gg < m.ngeom; gg += G) {
          const int mv = t.gmove[gg];
          if (mv == 1) {
#pragma unroll
            for (int k = 0; k < 3; k++) s.gpos[3 * gg + k] = t.gbase[3 * gg + k] + fi.axisd[0][k] * q0 + fi.axisd[1][k] * q1;
          } else if (mv == 2) {
            const V3<GT> p = mk<GT>(xb[0], xb[1], xb[2]) + mulv(Rb, ld3(t.gbase + 3 * gg));
            st3(s.gpos + 3 * gg, p);
            float Rbf[9], Rg[9];
#pragma unroll
            for (int k = 0; k < 9; k++) Rbf[k] = (float)Rb[k];
            mulm(Rbf, t.geom_mat + 9 * gg, Rg);
            const float* h = t.geom_aabb + 3 * gg;
#pragma unroll
            for (int i = 0; i < 3; i++)
              s.gaabb[3 * gg + i] = fabsf(Rg[3 * i]) * h[0] + fabsf(Rg[3 * i + 1]) * h[1] + fabsf(Rg[3 * i + 2]) * h[2];
          }
        }
      }
      __syncwarp();
      HSR_PHASE(s, g, PH_KIN);
      // ---------------------------------------------------------------- active joint limits (redundant in every lane)
      float lim_sg[2], lim_D[2], lim_aref[2];
      int nlimit = 0;
#pragma unroll
      for (int j = 0; j < 2; j++) {
        lim_sg[j] = 0.f; lim_D[j] = 0.f; lim_aref[j] = 0.f;
        if (fi.limited[j]) {
          const float q = qpos[j];
          const float dlo = q - fi.range[j][0], dhi = fi.range[j][1] - q;
          float dist = 0.f, sg = 0.f;
          if (dlo < 0) { dist = dlo; sg = 1.f; }
          else if (dhi < 0) { dist = dhi; sg = -1.f; }
          if (sg != 0.f) {
            const GT imp = push::impedance5(fi.lim_imp[j], (GT)dist);
            const GT R = fmax(GT(1e-15), (1 - imp) / imp * fi.lim_diag[j]);
            lim_sg[j] = sg; lim_D[j] = (float)(GT(1) / R);
            lim_aref[j] = (float)(-fi.lim_b[j] * (GT)(sg * qvel[j]) - fi.lim_k[j] * imp * (GT)dist);
            nlimit++;
          }
        }
      }
      // ---------------------------------------------------------------- collision (B.3)
      int ncon = push_collision<G>(m, t, s, w, g, blk, smem, a.ws_bytes, a.opts);
      __syncthreads();
      if (ncon > PUSH_MAXCON) ncon = PUSH_MAXCON;
      flags |= s.wi[WI_FLAGS];
      HSR_PHASE(s, g, PH_COLLIDE);

      // ---------------------------------------------------------------- smooth forces (closed form, B.6)
      float qs[8], as[8];  // qfrc_smooth, qacc_smooth
#pragma unroll
      for (int i = 0; i < 8; i++) { qs[i] = 0.f; as[i] = 0.f; }
#pragma unroll
      for (int j = 0; j < 2; j++) qs[j] = -fi.damp[j] * qvel[j] + fi.gq[j];
#pragma unroll
      for (int k = 0; k < 2; k++) {
        if (k < fi.act_n) {
          float c = ctrl[k];
          if (fi.ctrllimited[k]) c = fminf(fmaxf(c, fi.cr_lo[k]), fi.cr_hi[k]);
          const float qa = fi.act_q[k] == 0 ? qpos[0] : qpos[1];
          float fo = fi.kp[k] * c - fi.kp[k] * fi.gear[k] * qa;
          if (fi.forcelimited[k]) fo = fminf(fmaxf(fo, fi.fr_lo[k]), fi.fr_hi[k]);
          const float ga = fi.gear[k] * fo;
          if (fi.act_dof[k] == 0) qs[0] += ga; else qs[1] += ga;
        }
      }
      if (HASB) {
        // free box: gravity on the translational dofs, -w x (I w) on the body-frame rotational dofs
#pragma unroll
        for (int k = 0; k < 3; k++) qs[2 + k] = fi.Mdiag[2] * fi.gravity[k] - fi.damp[2 + k] * qvel[2 + k];
        const float Iw0 = fi.Mdiag[5] * qvel[5], Iw1 = fi.Mdiag[6] * qvel[6], Iw2 = fi.Mdiag[7] * qvel[7];
        qs[5] = -(qvel[6] * Iw2 - qvel[7] * Iw1) - fi.damp[5] * qvel[5];
        qs[6] = -(qvel[7] * Iw0 - qvel[5] * Iw2) - fi.damp[6] * qvel[6];
        qs[7] = -(qvel[5] * Iw1 - qvel[6] * Iw0) - fi.damp[7] * qvel[7];
      }
#pragma unroll
      for (int i = 0; i < NV; i++) as[i] = qs[i] / fi.Mdiag[i];

      // ---------------------------------------------------------------- constraint rows: one contact per lane (B.4/B.5)
      // The owning lane keeps its contact's regularisers / friction in registers; Jacobian rows go to shared memory.
      float D[6], fri[5], mu = 0.f;
      int dim = 0;
#pragma unroll
      for (int r = 0; r < 6; r++) D[r] = 0.f;
#pragma unroll
      for (int k = 0; k < 5; k++) fri[k] = 1.f;
      const int nr = 6 * ncon;  // contact rows in shared memory
      if (g.lane < ncon) {
        const int c = g.lane;
        const int pk = s.con_pair[c];
        dim = t.pair_condim[pk];
        const int g1 = t.pair_geom1[pk], g2 = t.pair_geom2[pk];
        const int b1 = t.geom_body[g1], b2 = t.geom_body[g2];
        const float sr = (float)(b2 == fi.robot_body) - (float)(b1 == fi.robot_body);
        const float sbk = (float)(b2 == fi.block_body) - (float)(b1 == fi.block_body);
        float fr[9];
#pragma unroll
        for (int k = 0; k < 9; k++) fr[k] = s.con_frame[9 * c + k];
#pragma unroll
        for (int k = 0; k < 5; k++) fri[k] = t.pair_friction[5 * pk + k];
        float rel[3] = {0.f, 0.f, 0.f};
        if (HASB) {
#pragma unroll
          for (int k = 0; k < 3; k++) rel[k] = (float)((GT)s.con_pos[3 * c + k] - xb[k]);
        }
        const double* pc = t.pairc + PUSH_PAIRC * pk;
        const GT dist = (GT)s.con_dist[c];
        const GT imp = push::impedance5<true>(pc + 3, dist);
        // regularisers: R0 = (1 - d) / d * diagApprox on the normal row, R0 / impratio on the first friction row, scaled by
        // (fri0 / fri_r)^2 on the others.  One double division for the impedance ratio; the per-row inverses D = 1 / R
        // are formed in float from D0 (relative rounding 1e-7 on a solver weight).
        const float D0 = (float)fmin(GT(1e15), imp / ((1 - imp) * pc[2]));   // 1 / max(1e-15, R0)
        const float D1 = D0 * m.impratio;
        float vel[6];
#pragma unroll
        for (int r = 0; r < 6; r++) {
          float Jr[8];
#pragma unroll
          for (int d = 0; d < 8; d++) Jr[d] = 0.f;
          if (r < dim) {
            if (r < 3) {
#pragma unroll
              for (int j = 0; j < 2; j++)
                Jr[j] = sr * (fr[3 * r] * fi.axis[j][0] + fr[3 * r + 1] * fi.axis[j][1] + fr[3 * r + 2] * fi.axis[j][2]);
            }
            if (HASB) {
#pragma unroll
              for (int k = 0; k < 3; k++) {
                const float ax0 = (float)Rb[k], ax1 = (float)Rb[3 + k], ax2 = (float)Rb[6 + k];  // body axis k, world frame
                if (r < 3) {
                  const float jp0 = ax1 * rel[2] - ax2 * rel[1], jp1 = ax2 * rel[0] - ax0 * rel[2], jp2 = ax0 * rel[1] - ax1 * rel[0];
                  Jr[2 + k] = sbk * fr[3 * r + k];
                  Jr[5 + k] = sbk * (fr[3 * r] * jp0 + fr[3 * r + 1] * jp1 + fr[3 * r + 2] * jp2);
                } else {
                  Jr[5 + k] = sbk * (fr[3 * (r - 3)] * ax0 + fr[3 * (r - 3) + 1] * ax1 + fr[3 * (r - 3) + 2] * ax2);
                }
              }
            }
          }
          float v = 0.f;
#pragma unroll
          for (int d = 0; d < NV; d++) v += Jr[d] * qvel[d];
          vel[r] = v;
          push::st8(s.J + 8 * (6 * c + r), Jr);
        }
#pragma unroll
        for (int r = 0; r < 6; r++) {
          float ar = 0.f, Dv = 0.f;
          if (r < dim) {
            if (r == 0) { Dv = D0; ar = (float)(-pc[1] * (GT)vel[0] - pc[0] * imp * dist); }
            else {
              ar = (float)(-pc[1] * (GT)vel[r]);
              Dv = r == 1 ? D1 : D1 * (fri[r - 1] * fri[r - 1]) / (fri[0] * fri[0]);
            }
          }
          D[r] = Dv;
          s.Dr[6 * c + r] = Dv; s.aref[6 * c + r] = ar;
        }
        mu = dim > 1 ? fri[0] * rsqrtf(m.impratio) : fri[0];   // fri0 * sqrt(R1 / R0)
      }
      int nefc_true = nlimit;  // MuJoCo's nefc: limit rows + condim rows per contact
      for (int c = 0; c < ncon; c++) nefc_true += t.pair_condim[s.con_pair[c]];
      sumcon += ncon; sumefc += nefc_true;
      __syncwarp();
      HSR_PHASE(s, g, PH_ROWS);

      // ---------------------------------------------------------------- Newton solver (B.7)
      // Warp-uniform control flow: every lane of the warp executes every statement of the solver; which environment
      // is still iterating only decides what is committed (x, the rows, counters).  The groups of a warp therefore
      // stay converged (a partial-mask __syncwarp / shuffle splits the warp into separately issued groups: the
      // previous version ran this section at 8-16 active threads per instruction), synchronisation is the
      // full-warp __syncwarp(), and reductions / broadcasts inside a group are full-mask shuffles whose partners stay
      // inside the group (xor offsets below G, width-G segments).
      float x[8], qfc[8];  // qacc (replicated), J^T f (replicated after the solve)
#pragma unroll
      for (int i = 0; i < 8; i++) { x[i] = 0.f; qfc[i] = 0.f; }
      int it = 0, ls_used = 0;
      int zone = 0;
      float cN = 0.f, cT = 0.f;
      auto gsum = [&](float v) -> float {
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
        return v;
      };
      int nr_w = nr;   // longest row list among the warp's environments (uniform loop bounds)
#pragma unroll
      for (int o = G; o < 32; o <<= 1) { const int t = __shfl_xor_sync(FULL, nr_w, o); nr_w = t > nr_w ? t : nr_w; }

      // jar = J xx - aref for the contact rows (rows across lanes)
      auto rows_jar = [&](const float* xx) {
        for (int r = g.lane; r < nr_w; r += G) {
          if (r < nr) {
            const push::F8 j = push::ld8(s.J + 8 * r);
            float acc = -s.aref[r];
#pragma unroll
            for (int d = 0; d < NV; d++) acc += j.v[d] * xx[d];
            s.jar[r] = acc;
          }
        }
      };
      // cone state of this lane's contact from its rows in s.jar: cost; full: zone, forces -> s.f
      auto cone = [&](bool full) -> float {
        float cost = 0.f;
        if (dim == 0) return 0.f;
        float jr[6];
        const float* pj = s.jar + 6 * g.lane;
#pragma unroll
        for (int r = 0; r < 6; r++) jr[r] = pj[r];
        int z = 0; float n_ = 0.f, t_ = 0.f;
        if (dim == 1) {
          z = jr[0] < 0 ? 1 : 0;
        } else {
          n_ = jr[0] * mu;
          float tt = 0.f;
#pragma unroll
          for (int j = 1; j < 6; j++) if (j < dim) { const float u = jr[j] * fri[j - 1]; tt += u * u; }
          t_ = sqrtf(tt);
          if (n_ >= mu * t_ || (t_ <= 0 && n_ >= 0)) z = 0;
          else if (mu * n_ + t_ <= 0 || (t_ <= 0 && n_ < 0)) z = 1;
          else z = 2;
        }
        float fo[6];
#pragma unroll
        for (int r = 0; r < 6; r++) fo[r] = 0.f;
        if (z == 1) {
#pragma unroll
          for (int r = 0; r < 6; r++) if (r < dim) { cost += 0.5f * D[r] * jr[r] * jr[r]; fo[r] = -D[r] * jr[r]; }
        } else if (z == 2) {
          const float Dm = D[0] / (mu * mu * (1 + mu * mu));
          const float NTv = n_ - mu * t_;
          cost += 0.5f * Dm * NTv * NTv;
          const float f0 = -Dm * NTv * mu;
          fo[0] = f0;
#pragma unroll
          for (int j = 1; j < 6; j++) if (j < dim) { const float U = jr[j] * fri[j - 1]; fo[j] = -f0 / t_ * U * fri[j - 1]; }
        }
        if (full) {
          zone = z; cN = n_; cT = t_;
          float* pf = s.f + 6 * g.lane;
#pragma unroll
          for (int r = 0; r < 6; r++) pf[r] = fo[r];
        }
        return cost;
      };
      auto limit_cost = [&](const float* xx) -> float {
        float cst = 0.f;
#pragma unroll
        for (int j = 0; j < 2; j++) if (lim_sg[j] != 0.f) {
          const float jr = lim_sg[j] * xx[j] - lim_aref[j];
          if (jr < 0) cst += 0.5f * lim_D[j] * jr * jr;
        }
        return cst;
      };
      auto gauss_of = [&](const float* xx) -> float {
        float gs = 0.f;
#pragma unroll
        for (int i = 0; i < NV; i++) { const float mx = fi.Mdiag[i] * xx[i]; gs += 0.5f * (mx - qs[i]) * (xx[i] - as[i]); }
        return gs;
      };

      bool solving = nefc_true != 0;
      bool finishing = false;   // converged by the improvement test: stop after the next gradient (forces of the final point)
      float cost = 0.f;
      {
        // warm start: the cheaper of qacc_smooth / qacc_warmstart (ties -> warm start); evaluated in that order so
        // that s.jar already holds the rows of the usual winner
        rows_jar(as);
        __syncwarp();
        const float cs = gsum(cone(false)) + gauss_of(as) + limit_cost(as);
        __syncwarp();
        rows_jar(warm);
        __syncwarp();
        const float cw = gsum(cone(false)) + gauss_of(warm) + limit_cost(warm);
        const bool use_warm = cw <= cs && solving;   // no constraint rows: qacc = qacc_smooth
#pragma unroll
        for (int i = 0; i < NV; i++) x[i] = use_warm ? warm[i] : as[i];
        __syncwarp();
        if (__any_sync(FULL, !use_warm)) {
          for (int r = g.lane; r < nr_w; r += G) {
            if (r < nr && !use_warm) {
              const push::F8 j = push::ld8(s.J + 8 * r);
              float acc = -s.aref[r];
#pragma unroll
              for (int d = 0; d < NV; d++) acc += j.v[d] * x[d];
              s.jar[r] = acc;
            }
          }
          __syncwarp();
        }
        cost = gsum(cone(true)) + gauss_of(x) + limit_cost(x);
        __syncwarp();
      }
      // Newton iterations: the loop is voted on by the whole warp
      while (__any_sync(FULL, solving)) {
        bool stop = !solving;
        // ---- gradient component of this lane's dof: M x - qfrc_smooth - J^T f
        float myx = 0.f, myqs = 0.f, myM = 0.f;
#pragma unroll
        for (int i = 0; i < NV; i++) if (li == i) { myx = x[i]; myqs = qs[i]; myM = fi.Mdiag[i]; }
        float qf = 0.f;
#pragma unroll UR
        for (int r = sub; r < nr_w; r += SUBS) if (r < nr) qf += s.J[8 * r + li] * s.f[r];
#pragma unroll
        for (int o = 8; o < G; o <<= 1) qf += __shfl_xor_sync(FULL, qf, o);
        bool lim_act[2];
#pragma unroll
        for (int j = 0; j < 2; j++) {
          lim_act[j] = false;
          if (lim_sg[j] != 0.f) {
            const float jr = lim_sg[j] * x[j] - lim_aref[j];
            lim_act[j] = jr < 0;
            if (lim_act[j] && li == j) qf += lim_sg[j] * (-lim_D[j] * jr);
          }
        }
        const float grad = (li < NV) ? myM * myx - myqs - qf : 0.f;
        float gn = grad * grad;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) gn += __shfl_xor_sync(FULL, gn, o);
        gn = sqrtf(gn);
        if (finishing || (it > 0 && scale * gn < m.tolerance) || it >= m.iterations) stop = true;
        float qfg[8];   // qfrc_constraint of the current point, replicated (committed when this environment stops)
#pragma unroll
        for (int i = 0; i < 8; i++) qfg[i] = (i < NV) ? __shfl_sync(FULL, qf, i, G) : 0.f;
        if (__any_sync(FULL, !stop)) {
          // ---- Hessian J^T (cone Hessians) J as a sum of weighted outer products of Jacobian rows.  Quadratic-zone
          //      contact: sum_r D_r J_r J_r^T.  Cone-zone contact (U_a = jar_a s_a, u = U / T, s_0 = mu, s_a = fri_a-1,
          //      k = mu (N - mu T) / T):  Dm (p p^T + k q q^T) - Dm k sum_{a>=1} s_a^2 J_a J_a^T
          //      with p = mu J_0 - mu sum_{a>=1} u_a s_a J_a and q = sum_{a>=1} u_a s_a J_a -- the 6x6 cone block
          //      Dm S (v v^T - k (I_t - u u^T)) S of the row formulation, v = e_0 - mu u, never formed.
          float* const PQ = s.hq; float* const wpq = s.hq + 16 * PUSH_MAXCON; float* const wrow = wpq + 2 * PUSH_MAXCON;
          {
            float wr_[6], wp = 0.f, wq = 0.f;
#pragma unroll
            for (int r = 0; r < 6; r++) wr_[r] = (zone == 1 && r < dim) ? D[r] : 0.f;
            if (zone == 2) {
              const float Dm = D[0] / (mu * mu * (1 + mu * mu)), NTv = cN - mu * cT, invT = 1.0f / cT;
              const float kap = mu * NTv * invT;
              const float* pj = s.jar + 6 * g.lane;
              float pv[8], qv[8];
              {
                const push::F8 j = push::ld8(s.J + 8 * (6 * g.lane));
#pragma unroll
                for (int d = 0; d < 8; d++) { pv[d] = mu * j.v[d]; qv[d] = 0.f; }
              }
#pragma unroll
              for (int aa = 1; aa < 6; aa++) if (aa < dim) {
                const float sa = fri[aa - 1];
                const float cq = pj[aa] * sa * invT * sa, cp = -mu * cq;
                const push::F8 j = push::ld8(s.J + 8 * (6 * g.lane + aa));
#pragma unroll
                for (int d = 0; d < 8; d++) { pv[d] += cp * j.v[d]; qv[d] += cq * j.v[d]; }
                wr_[aa] = -Dm * kap * sa * sa;
              }
              wp = Dm; wq = Dm * kap;
              push::st8(PQ + 16 * g.lane, pv); push::st8(PQ + 16 * g.lane + 8, qv);
            }
            if (g.lane < PUSH_MAXCON) {
#pragma unroll
              for (int r = 0; r < 6; r++) wrow[6 * g.lane + r] = wr_[r];
              wpq[2 * g.lane] = wp; wpq[2 * g.lane + 1] = wq;
            }
          }
          __syncwarp();
          float Hr[8];
#pragma unroll
          for (int j = 0; j < 8; j++) Hr[j] = 0.f;
#pragma unroll UR
          for (int r = sub; r < nr_w; r += SUBS) {
            if (r < nr) {
              const float ji = s.J[8 * r + li] * wrow[r];
              const push::F8 jv_ = push::ld8(s.J + 8 * r);
#pragma unroll
              for (int j = 0; j < 8; j++) Hr[j] += ji * jv_.v[j];
            }
          }
          for (int c = sub; 6 * c < nr_w; c += SUBS) {
            if (6 * c < nr && wpq[2 * c] != 0.f) {
              const float pi_ = PQ[16 * c + li] * wpq[2 * c], qi_ = PQ[16 * c + 8 + li] * wpq[2 * c + 1];
              const push::F8 pv = push::ld8(PQ + 16 * c), qv = push::ld8(PQ + 16 * c + 8);
#pragma unroll
              for (int j = 0; j < 8; j++) Hr[j] += pi_ * pv.v[j] + qi_ * qv.v[j];
            }
          }
#pragma unroll
          for (int o = 8; o < G; o <<= 1)
#pragma unroll
            for (int j = 0; j < 8; j++) Hr[j] += __shfl_xor_sync(FULL, Hr[j], o);
#pragma unroll
          for (int j = 0; j < 8; j++) if (li == j) {
            Hr[j] += (j < NV) ? fi.Mdiag[j] : 1.0f;
            if (j < 2 && lim_act[j]) Hr[j] += lim_D[j];
          }
          // ---- Cholesky H = L L^T: lane i holds row i; column k is finished by a broadcast of the pivot and one
          //      shuffle per trailing column
          float inv_diag = 1.f;
#pragma unroll
          for (int k = 0; k < 8; k++) {
            float dkk = __shfl_sync(FULL, Hr[k], k, G);
            if (!(dkk > 1e-15f)) { dkk = 1e-15f; if (!stop) flags |= FLAG_CHOL; }
            const float lkk = sqrtf(dkk);
            const float inv = 1.0f / lkk;
            const float lik = (li == k) ? lkk : Hr[k] * inv;   // L[i][k] for i >= k
            Hr[k] = lik;
            if (li == k) inv_diag = inv;
#pragma unroll
            for (int j = k + 1; j < 8; j++) {
              const float ljk = __shfl_sync(FULL, lik, j, G);
              Hr[j] -= lik * ljk;                               // meaningful for i >= j
            }
          }
          // ---- forward solve L y = -grad
          float acc = -grad, y = 0.f;
#pragma unroll
          for (int k = 0; k < 8; k++) {
            const float yk = __shfl_sync(FULL, acc * inv_diag, k, G);
            if (li == k) y = yk;
            acc -= Hr[k] * yk;                                  // meaningful for i > k
          }
          // ---- backward solve L^T s = y: column k of L gathered through shared memory
          __syncwarp();
          if (sub == 0) push::st8(s.L + 8 * li, Hr);
          __syncwarp();
          float Lc[8];
#pragma unroll
          for (int i = 0; i < 8; i++) Lc[i] = s.L[8 * i + li];   // L[i][li], meaningful for i >= li
          acc = y;
          float sv = 0.f;
#pragma unroll
          for (int k = 7; k >= 0; k--) {
            const float xk = __shfl_sync(FULL, acc * inv_diag, k, G);
            if (li == k) sv = xk;
            acc -= Lc[k] * xk;                                  // meaningful for li < k
          }
          float srch[8];
#pragma unroll
          for (int i = 0; i < 8; i++) srch[i] = (i < NV) ? __shfl_sync(FULL, sv, i, G) : 0.f;
          float sn = 0.f, dec = 0.f;
          {
            float dd = (li < NV) ? -grad * sv : 0.f;
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) dd += __shfl_xor_sync(FULL, dd, o);
            dec = dd;
          }
#pragma unroll
          for (int i = 0; i < NV; i++) sn += srch[i] * srch[i];
          sn = sqrtf(sn);
          if (!(sn >= 1e-15f)) stop = true;                     // also catches the garbage direction of a stopped group
          // ---- jv = J search (rows across lanes)
          for (int r = g.lane; r < nr_w; r += G) {
            if (r < nr) {
              const push::F8 j = push::ld8(s.J + 8 * r);
              float accv = 0.f;
#pragma unroll
              for (int d = 0; d < NV; d++) accv += j.v[d] * srch[d];
              s.jv[r] = accv;
            }
          }
          __syncwarp();
          const float gtol = m.tolerance * m.ls_tolerance * sn / scale;
          // ---- exact line search: root of the 1-D derivative (safeguarded Newton with bracketing)
          float q1 = 0.f, q2 = 0.f;
#pragma unroll
          for (int i = 0; i < NV; i++) {
            const float mv = fi.Mdiag[i] * srch[i];
            q1 += srch[i] * (fi.Mdiag[i] * x[i] - qs[i]); q2 += 0.5f * srch[i] * mv;
          }
          float lq[10];
          {
            float uu = 0.f, uv = 0.f, vv = 0.f, Q1 = 0.f, Q2 = 0.f, j0 = 0.f, v0 = 0.f;
            if (dim > 0) {
              const float* pj = s.jar + 6 * g.lane; const float* pv = s.jv + 6 * g.lane;
              j0 = pj[0]; v0 = pv[0];
#pragma unroll
              for (int r = 0; r < 6; r++) if (r < dim) {
                const float xx = pj[r], v = pv[r], Dv = D[r];
                Q1 += Dv * xx * v; Q2 += 0.5f * Dv * v * v;
                if (r > 0) { const float u = xx * fri[r - 1], sv2 = v * fri[r - 1]; uu += u * u; uv += u * sv2; vv += sv2 * sv2; }
              }
            }
            if (dim == 1) { lq[0] = j0; lq[1] = v0; lq[8] = 1.f; lq[9] = -1.f; }
            else { lq[0] = j0 * mu; lq[1] = v0 * mu; lq[8] = mu; lq[9] = dim > 0 ? D[0] / (mu * mu * (1 + mu * mu)) : 0.f; }
            lq[2] = uu; lq[3] = uv; lq[4] = vv; lq[5] = 0.f; lq[6] = Q1; lq[7] = Q2;
          }
          // derivative of the cost along the search direction and its slope at alpha; select-only arithmetic (no divergent
          // branches: the zones of the four environments' contacts differ).  A lane without a contact has all-zero
          // coefficients and lands in the "top" zone (no force); an inactive limit has sg = D = aref = 0.
          auto ls_eval = [&](float alpha, float& d1, float& d2) {
            const float mu_ = lq[8], Dm = lq[9];
            const float N = lq[0] + alpha * lq[1];
            const float tsq = lq[2] + alpha * (2 * lq[3] + alpha * lq[4]);
            const float rT = tsq > 0 ? rsqrtf(tsq) : 0.f;     // 1 / T (used in the cone zone only, where T > 0)
            const float Tn = tsq * rT;
            const bool quad = Dm < 0;                          // condim-1 contact: half-line instead of a cone
            const bool top = quad ? !(N < 0) : ((N >= mu_ * Tn) || (Tn <= 0 && N >= 0));
            const bool bottom = quad ? (N < 0) : ((mu_ * N + Tn <= 0) || (Tn <= 0 && N < 0));
            const float NTv = N - mu_ * Tn;
            const float T1 = (lq[3] + alpha * lq[4]) * rT;
            const float T2 = (lq[4] - T1 * T1) * rT;
            const float tt = lq[1] - mu_ * T1;
            const float lm1 = Dm * NTv * tt, lm2 = Dm * (tt * tt - NTv * mu_ * T2);
            const float lb1 = lq[6] + 2 * alpha * lq[7], lb2 = 2 * lq[7];
            float l1 = top ? 0.f : (bottom ? lb1 : lm1), l2 = top ? 0.f : (bottom ? lb2 : lm2);
            l1 = gsum(l1); l2 = gsum(l2);
#pragma unroll
            for (int j = 0; j < 2; j++) {
              const float xv = lim_sg[j] * srch[j];
              const float xx = lim_sg[j] * x[j] - lim_aref[j] + alpha * xv;
              const float dd = xx < 0 ? lim_D[j] : 0.f;
              l1 += dd * xx * xv; l2 += dd * xv * xv;
            }
            d1 = l1 + q1 + 2 * alpha * q2;
            d2 = l2 + 2 * q2;
          };
          float alpha = 0.f;
          {
            float d1, d2;
            ls_eval(0.f, d1, d2);
            int nev = 1;
            float lo = 0.f, hi = -1.f, dlo = d1, dhi = 0.f;
            const float rel = 3.4526698e-4f;  // sqrt(FLT_EPSILON)
            bool conv = fabsf(d1) < gtol;
            bool searching = !stop && !conv;                    // this environment still refines its step
#pragma unroll 1
            for (int lit = 0; lit < m.ls_iterations; lit++) {
              float nxt = alpha;
              bool tiny = false;
              if (searching) {
                const float step = d2 > 1e-15f ? -d1 / d2 : (d1 < 0 ? 1.f : -1.f);
                nxt = alpha + step;
                if (hi >= 0 && !(lo < nxt && nxt < hi)) nxt = 0.5f * (lo + hi);
                if (nxt <= 0 && hi < 0) nxt = alpha * 0.5f;
                if (nxt == alpha) searching = false;
                tiny = fabsf(nxt - alpha) <= rel * fabsf(nxt);
              }
              if (!__any_sync(FULL, searching)) break;
              float e1, e2;
              ls_eval(searching ? nxt : alpha, e1, e2);
              if (searching) {
                alpha = nxt; d1 = e1; d2 = e2;
                nev++;
                if (d1 < 0) { if (alpha > lo) { lo = alpha; dlo = d1; } }
                else if (hi < 0 || alpha < hi) { hi = alpha; dhi = d1; }
                conv = fabsf(d1) < gtol || tiny;
                if (conv) searching = false;
              }
            }
            if (!stop) ls_used += nev;
            if (!conv) {
              if (hi >= 0 && (lo <= 0 || fabsf(dhi) < fabsf(dlo))) alpha = (lo > 0 || fabsf(dhi) < fabsf(dlo)) ? hi : 0.f;
              else alpha = lo;
            }
          }
          if (alpha == 0.f) stop = true;
          if (!stop) {
#pragma unroll
            for (int i = 0; i < NV; i++) x[i] += alpha * srch[i];
          }
          for (int r = g.lane; r < nr_w; r += G) if (r < nr && !stop) s.jar[r] += alpha * s.jv[r];
          __syncwarp();
          const float newcost = gsum(cone(true)) + gauss_of(x) + limit_cost(x);   // stopped groups: unchanged rows, same result
          __syncwarp();
          if (!stop) {
            const float old = cost;
            cost = newcost;
            it++;
            const float improvement = alpha < 2.f ? alpha * (1.f - 0.5f * alpha) * dec : old - cost;
            if (scale * improvement < m.tolerance) finishing = true;   // the next pass computes J^T f of this point and stops
          }
        }
        if (solving && stop) {
#pragma unroll
          for (int i = 0; i < NV; i++) qfc[i] = qfg[i];
          solving = false;
        }
      }
      __syncthreads();
      HSR_PHASE(s, g, PH_SOLVE);
      n_iter += it; n_ls += ls_used;
      kflop += algorithmic_flops(m, false, ncon, nefc_true, it, ls_used, s.wi[WI_NPFLOP]);   // slides + free box: M is constant

      // ---------------------------------------------------------------- goal test on the poses of this forward pass
      bool reached = false;
      if (HASB && a.cfg.has_goal) {
        const GT dx = xb[0] - (GT)mocap[0], dy = xb[1] - (GT)mocap[1], dz = xb[2] - (GT)mocap[2];
        reached = sqrt(dx * dx + dy * dy + dz * dz) < (GT)a.cfg.geofence;
      }
      // ---------------------------------------------------------------- Euler with implicit joint damping (B.8)
#pragma unroll
      for (int i = 0; i < NV; i++) {
        const float ai = m.any_damping ? (qs[i] + qfc[i]) / (fi.Mdiag[i] + dt * fi.damp[i]) : x[i];
        warm[i] = x[i];
        qvel[i] += dt * ai;
        if (!(fabsf(qvel[i]) < 1e6f)) flags |= FLAG_BAD_NUM;
      }
      qpos[0] += dt * qvel[0]; qpos[1] += dt * qvel[1];
      if (HASB) {
#pragma unroll
        for (int k = 0; k < 3; k++) qpos[2 + k] += dt * qvel[2 + k];
        const float om0 = qvel[5], om1 = qvel[6], om2 = qvel[7];
        const float ang = sqrtf(om0 * om0 + om1 * om1 + om2 * om2);
        quatnormalize(qpos + 5);
        if (ang * dt > 1e-15f) {
          // rotation by ang * dt about omega: dq = [cos h, sin(h) / ang * omega], h = ang dt / 2.  Below h = 0.5 rad per
          // substep (ang < 500 rad/s) the series of cos h and sin(h) / h are exact to 1e-9 and need neither the range
          // reduction of sinf / cosf nor the division by ang.
          const float hh = 0.5f * ang * dt;
          float ch, sn_;
          if (hh < 0.5f) {
            const float h2 = hh * hh;
            ch = 1.f + h2 * (-0.5f + h2 * (4.1666667e-2f + h2 * (-1.3888889e-3f + h2 * (2.4801587e-5f - h2 * 2.7557319e-7f))));
            sn_ = 0.5f * dt * (1.f + h2 * (-1.6666667e-1f + h2 * (8.3333333e-3f + h2 * (-1.9841270e-4f + h2 * 2.7557319e-6f))));
          } else {
            ch = cosf(hh); sn_ = sinf(hh) / ang;
          }
          float dq[4] = {ch, sn_ * om0, sn_ * om1, sn_ * om2};
          quatmul(qpos + 5, dq, qpos + 5);
        }
        quatnormalize(qpos + 5);
      }
      __syncwarp();
      HSR_PHASE(s, g, PH_EULER);
      if (!finished) {
        taken++;
        if (reached) success = true;
        if (reached || sb_ == a.nsub - 1) {
          // ---------------------------------------------------------------- results: HBM once per action
          finished = true;
          float* st = a.state + (size_t)env * a.S;
          const int nobs = nq + NV;
          for (int i = g.lane; i < nq + 2 * NV; i += G) {
            float v = 0.f;
#pragma unroll
            for (int k = 0; k < (HASB ? 9 : 2); k++) if (i == k) v = qpos[k];
#pragma unroll
            for (int k = 0; k < NV; k++) { if (i == nq + k) v = qvel[k]; if (i == nq + NV + k) v = warm[k]; }
            st[i] = v;
            if (a.obs && i < nobs) a.obs[(size_t)env * nobs + i] = v;
          }
          if (g.lane == 0) {
            if (a.reward) a.reward[env] = success ? 1.0f : 0.0f;
            if (a.done) a.done[env] = success ? 1 : 0;
            if (a.success) a.success[env] = success ? 1 : 0;
            if (a.taken) a.taken[env] = taken;
            if (a.bad) a.bad[env] = (unsigned char)flags;
            atomicAdd(a.stats + ST_SUBSTEPS, (unsigned long long)taken);
            atomicAdd(a.stats + ST_ITERS, (unsigned long long)n_iter);
            atomicAdd(a.stats + ST_NARROW, (unsigned long long)s.wi[WI_NARROW]);
            atomicAdd(a.stats + ST_LSEVAL, (unsigned long long)n_ls);
            atomicAdd(a.stats + ST_CONTACTS, (unsigned long long)sumcon);
            atomicAdd(a.stats + ST_ROWS, (unsigned long long)sumefc);
            atomicAdd(a.stats + ST_FLOPS, (unsigned long long)kflop);
            if (flags) atomicAdd(a.stats + ST_BAD, 1ull);
#ifdef HSRB_PHASE_CLOCKS
            for (int k = 0; k < PH_COUNT; k++) atomicAdd(a.stats + ST_PHASE0 + k, (unsigned long long)s.wi[WI_PHASE0 + k]);
#endif
          }
        }
      }
    }
    __syncwarp();
  }
}

// host side (hsrb_push.cu): p.lanes picks G, p.fam->nv picks NV
cudaError_t hsrb_push_prepare(const Plan& p, int* bps);
cudaError_t hsrb_push_launch(const Plan& p, const KArgs& a, cudaStream_t s);
