// Transition derivatives (hsrb_transition_fd, MuJoCo's mjd_transitionFD): finite-difference A = dx'/dx and B = dx'/du of
// x' = nsub substeps of the general path's substep() from each environment's resident state, ctrl held.
//
// x = (dq, qvel) has 2 nv coordinates, dq the tangent-space displacement of qpos (a free joint: 3 position + 3 rotation),
// u = ctrl[nu].  Coordinate c of an environment: c < nv position dof c, c < 2 nv velocity dof c - nv, else ctrl c - 2 nv.
// Run r of an environment: r = 0 the nominal input; r = 1 + c * S + s (S = 2 centered, 1 forward; s = 0 the + side, 1 the
// - side) the input with coordinate c perturbed.  In forward mode a ctrl run whose + side the ctrl-limit rule refuses takes
// the - side (fd_side).
//
// Two launches.  hsrb_fd_kernel: one (environment, run) job per group of G lanes, the lean layout of the general path
// (one warp per block, 32 / G workspaces, grid-stride), jobs environment-major so that one environment's runs share a block
// and its state row.  Each job: load_state (the resident qacc_warmstart, an empty separating-direction cache), the caller's
// ctrl, the perturbation (fd_perturb, lane 0), the multipliers, nsub x substep(); then x' (qpos | qvel), the run's flags
// and the realised perturbation h (double) go to its scratch row.  hsrb_fd_form_kernel: one thread per (environment,
// column) forms the column in double from the scratch rows and rounds it to fp32 once; one more thread per environment
// writes next_obs and bad_state.  Nothing is written back to the state and no work counter moves.
#pragma once
#include <cstring>

#include "hsrb_kernels.cuh"

struct FdArgs {
  KArgs k;               // model (ncon_max / nefc_max: the general plan's), n, S, ws_bytes, state, ctrl (nullable), params
  float eps;
  double rot_c, rot_s;   // cos(eps / 2), sin(eps / 2) in double, computed once on the host (the rotation perturbation)
  int centered, nsub, nruns;
  float* scratch;        // [n, nruns, fd_row(m)]: x' (nq + nv floats) | flags (int bits) | h (double, two words)
  // outputs (nullable): A [n, 2nv, 2nv]; B [n, 2nv, nu]; next_obs [n, nq + nv]; bad [n]
  float* A; float* B; float* next_obs; unsigned char* bad;
};

template <typename T> HSR_HD int fd_row(const ModelT<T>& m) { return m.nq + m.nv + 3; }
template <typename T> HSR_HD int fd_nruns(const ModelT<T>& m, bool centered) { return 1 + (centered ? 2 : 1) * (2 * m.nv + m.nu); }

// x +- eps in fp32; when the rounded value equals x, the next float in that direction, so that no column divides by 0
HSR_HD float fd_nudge(float x, float eps, int side) {
  const float y = side > 0 ? x + eps : x - eps;
  return y != x ? y : nextafterf(x, side > 0 ? FLT_MAX : -FLT_MAX);
}

// MuJoCo's ctrl-limit rule: side `side` of ctrl i may be used only if both u and the nudged u lie within a limited
// actuator's ctrlrange
template <typename T>
HSR_HD bool fd_ctrl_ok(const ModelT<T>& m, int i, float u, float eps, int side) {
  if (!m.act_ctrllimited[i]) return true;
  const float lo = (float)m.act_ctrlrange[2 * i], hi = (float)m.act_ctrlrange[2 * i + 1], un = fd_nudge(u, eps, side);
  return u >= lo && u <= hi && un >= lo && un <= hi;
}

// MuJoCo's mju_subQuat: the axis-angle vector of conj(qb) (x) qa.  For nearby quaternions the vector part of the product is
// a cancellation of O(1) terms, so every product is rounded on its own (mul_rn): a fused multiply-add would change the small
// result by far more than an fp32 ulp of the column it feeds.  Only atan2 then differs between the device and the host.
HSR_HD void fd_subquat(const double* qa, const double* qb, double* res) {
  const double d[4] = {mul_rn(qb[0], qa[0]) + mul_rn(qb[1], qa[1]) + mul_rn(qb[2], qa[2]) + mul_rn(qb[3], qa[3]),
                       mul_rn(qb[0], qa[1]) - mul_rn(qb[1], qa[0]) - mul_rn(qb[2], qa[3]) + mul_rn(qb[3], qa[2]),
                       mul_rn(qb[0], qa[2]) + mul_rn(qb[1], qa[3]) - mul_rn(qb[2], qa[0]) - mul_rn(qb[3], qa[1]),
                       mul_rn(qb[0], qa[3]) - mul_rn(qb[1], qa[2]) + mul_rn(qb[2], qa[1]) - mul_rn(qb[3], qa[0])};
  double ax[3] = {d[1], d[2], d[3]};
  const double s = sqrt(mul_rn(ax[0], ax[0]) + mul_rn(ax[1], ax[1]) + mul_rn(ax[2], ax[2]));
  if (s < 1e-15) { ax[0] = 1; ax[1] = 0; ax[2] = 0; }
  else { const double inv = 1 / s; ax[0] *= inv; ax[1] *= inv; ax[2] *= inv; }
  double speed = 2 * atan2(s, d[0]);
  if (speed > 3.14159265358979323846) speed -= 2 * 3.14159265358979323846;
  for (int k = 0; k < 3; k++) res[k] = ax[k] * speed;
}

// side (+1 / -1) of run r > 0; u the environment's ctrl of that coordinate (read only for ctrl coordinates)
template <typename T>
HSR_HD int fd_side(const ModelT<T>& m, int r, bool centered, float eps, float u) {
  const int S = centered ? 2 : 1, c = (r - 1) / S;
  if (centered) return (r - 1) % S == 0 ? 1 : -1;
  return c >= 2 * m.nv && !fd_ctrl_ok(m, c - 2 * m.nv, u, eps, 1) ? -1 : 1;
}

// The input of run r: perturbs qpos / qvel / ctrl (the fp32 values of the resident state and the caller's ctrl) in place
// and returns the realised perturbation h, in double from the fp32 values used (0 for the nominal run r = 0).
// Scalars: fd_nudge.  Rotation k of a free joint: q+- = normalize(q (x) [cos(eps/2), +-sin(eps/2) e_k]) in double (the
// local-frame convention of euler_lane0), rounded to fp32, h = component k of mju_subQuat(q+-, q).  The products are rounded
// one by one (mul_rn), so the perturbed quaternion has the same bits on the device, the host and in numpy.
template <typename T>
HSR_HD double fd_perturb(const ModelT<T>& m, int r, bool centered, float eps, double rot_c, double rot_s, float* qpos,
                         float* qvel, float* ctrl) {
  if (r == 0) return 0.0;
  const int S = centered ? 2 : 1, c = (r - 1) / S, nv = m.nv;
  const int side = fd_side(m, r, centered, eps, c >= 2 * nv ? ctrl[c - 2 * nv] : 0.f);
  float* x;
  if (c >= 2 * nv) x = ctrl + (c - 2 * nv);
  else if (c >= nv) x = qvel + (c - nv);
  else {
    const int j = m.dof_jnt[c], a = m.jnt_qposadr[j], k = c - m.jnt_dofadr[j];
    if (m.jnt_type[j] == JNT_FREE && k >= 3) {
      float* q = qpos + a + 3;
      const double q0[4] = {(double)q[0], (double)q[1], (double)q[2], (double)q[3]};
      const double s = side > 0 ? rot_s : -rot_s, e[3] = {k == 3 ? s : 0.0, k == 4 ? s : 0.0, k == 5 ? s : 0.0};
      double p[4] = {mul_rn(q0[0], rot_c) - mul_rn(q0[1], e[0]) - mul_rn(q0[2], e[1]) - mul_rn(q0[3], e[2]),
                     mul_rn(q0[0], e[0]) + mul_rn(q0[1], rot_c) + mul_rn(q0[2], e[2]) - mul_rn(q0[3], e[1]),
                     mul_rn(q0[0], e[1]) - mul_rn(q0[1], e[2]) + mul_rn(q0[2], rot_c) + mul_rn(q0[3], e[0]),
                     mul_rn(q0[0], e[2]) + mul_rn(q0[1], e[1]) - mul_rn(q0[2], e[0]) + mul_rn(q0[3], rot_c)};
      const double n = sqrt(mul_rn(p[0], p[0]) + mul_rn(p[1], p[1]) + mul_rn(p[2], p[2]) + mul_rn(p[3], p[3]));
      double qp[4], h3[3];
      for (int i = 0; i < 4; i++) { q[i] = (float)(p[i] / n); qp[i] = (double)q[i]; }
      fd_subquat(qp, q0, h3);
      return h3[k - 3];
    }
    x = qpos + a + k;
  }
  const float x0 = *x;
  *x = fd_nudge(x0, eps, side);
  return (double)*x - (double)x0;
}

template <int G, bool PARAMS>
__global__ void __launch_bounds__(32) hsrb_fd_kernel(const __grid_constant__ FdArgs f) {
  HSRB_DYN_SMEM(smem);
  const KArgs& a = f.k;
  DevGrp<G> g;
  const int gpb = 32 / G;
  const int gi = threadIdx.x / G;
  WS<float> w;
  ws_carve<float>(a.m, &w, smem + (size_t)gi * a.ws_bytes);
  const int nx = a.m.nq + a.m.nv, R = fd_row(a.m);
  const long long jobs = (long long)a.n * f.nruns;
  for (long long jb = (long long)blockIdx.x * gpb + gi; jb < jobs; jb += (long long)gridDim.x * gpb) {
    const int env = (int)(jb / f.nruns), r = (int)(jb % f.nruns);
    load_state<G>(a, w, g, env);
    for (int i = g.lane; i < a.m.nu; i += G) w.ctrl[i] = a.ctrl ? a.ctrl[(size_t)env * a.m.nu + i] : 0.f;
    g.sync();
    double h = 0;
    if (g.lane == 0) h = fd_perturb(a.m, r, f.centered != 0, f.eps, f.rot_c, f.rot_s, w.qpos, w.qvel, w.ctrl);
    g.sync();
    typename ScaleOf<PARAMS>::type sc;
    load_scale(sc, a, env);
    for (int s = 0; s < f.nsub; s++) substep(a.m, w, g, sc);
    float* row = f.scratch + (size_t)jb * R;
    for (int i = g.lane; i < nx; i += G) row[i] = w.qpos[i];   // qpos | qvel are contiguous in the workspace
    if (g.lane == 0) {
      row[nx] = __int_as_float(w.wi[WI_FLAGS]);
      memcpy(row + nx + 1, &h, sizeof(double));
    }
    g.sync();   // the group's reads of the workspace are done before the next job's load_state
  }
}

// the realised perturbation h of a scratch row
HSR_HD double fd_h(const float* row, int nx) {
  double h;
  memcpy(&h, row + nx + 1, sizeof(double));
  return h;
}

// One thread per (environment, column c < 2nv + nu); thread c = 2nv + nu of an environment writes next_obs and bad.
// Output row i of the column: d+- = x'+- (-) x'0 in double, plain differences except a free joint's rotation rows, which
// take mju_subQuat(q'+-, q'0); centered (d+ - d-) / (h+ - h-), one-sided d / h, rounded to fp32 once.
template <bool CENTERED>
__global__ void __launch_bounds__(128) hsrb_fd_form_kernel(const __grid_constant__ FdArgs f) {
  const ModelT<float>& m = f.k.m;
  const int nq = m.nq, nv = m.nv, nu = m.nu, nxs = 2 * nv, ncol = nxs + nu, nx = nq + nv, R = fd_row(m);
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)f.k.n * (ncol + 1)) return;
  const int env = (int)(t / (ncol + 1)), c = (int)(t % (ncol + 1));
  const float* base = f.scratch + (size_t)env * f.nruns * R;
  if (c == ncol) {
    if (f.next_obs) for (int i = 0; i < nx; i++) f.next_obs[(size_t)env * nx + i] = base[i];
    if (f.bad) {
      int fl = 0;
      for (int r = 0; r < f.nruns; r++) fl |= __float_as_int(base[(size_t)r * R + nx]);
      f.bad[env] = (unsigned char)fl;
    }
    return;
  }
  float* out = c < nxs ? (f.A ? f.A + (size_t)env * nxs * nxs + c : nullptr) : (f.B ? f.B + (size_t)env * nxs * nu + (c - nxs) : nullptr);
  if (!out) return;
  const int ostride = c < nxs ? nxs : nu;
  // the runs of column c and MuJoCo's ctrl-limit rule
  const int S = CENTERED ? 2 : 1, rp = 1 + c * S, rm = CENTERED ? rp + 1 : rp;
  bool usep = true, usem = CENTERED;
  if (c >= nxs) {
    const float u = f.k.ctrl ? f.k.ctrl[(size_t)env * nu + (c - nxs)] : 0.f;
    const bool okp = fd_ctrl_ok(m, c - nxs, u, f.eps, 1), okm = fd_ctrl_ok(m, c - nxs, u, f.eps, -1);
    usep = okp;
    usem = CENTERED ? okm : !okp && okm;   // forward mode: run rp went to the - side (fd_side)
  }
  const float *x0 = base, *xp = base + (size_t)rp * R, *xm = base + (size_t)rm * R;
  const double hp = fd_h(xp, nx), hm = fd_h(xm, nx);
  auto col = [&](double dp, double dm) -> float {
    if (usep && usem) return (float)((dp - dm) / (hp - hm));
    if (usep) return (float)(dp / hp);
    if (usem) return (float)(dm / hm);
    return 0.f;
  };
  auto sub = [&](const float* x, int i) { return (double)x[i] - (double)x0[i]; };
  for (int j = 0; j < m.njnt; j++) {
    const int a = m.jnt_qposadr[j], v = m.jnt_dofadr[j];
    if (m.jnt_type[j] == JNT_FREE) {
      for (int k = 0; k < 3; k++) out[(size_t)(v + k) * ostride] = col(sub(xp, a + k), sub(xm, a + k));
      double q0[4], qp[4], qm[4], dp[3], dm[3];
      for (int k = 0; k < 4; k++) { q0[k] = x0[a + 3 + k]; qp[k] = xp[a + 3 + k]; qm[k] = xm[a + 3 + k]; }
      fd_subquat(qp, q0, dp);
      fd_subquat(qm, q0, dm);
      for (int k = 0; k < 3; k++) out[(size_t)(v + 3 + k) * ostride] = col(dp[k], dm[k]);
    } else {
      out[(size_t)v * ostride] = col(sub(xp, a), sub(xm, a));
    }
  }
  for (int i = 0; i < nv; i++) out[(size_t)(nv + i) * ostride] = col(sub(xp, nq + i), sub(xm, nq + i));
}

// host side (hsrb_fd.cu), in the general kernel's plan p: p.lanes picks G, f.k.params the instance with parameters.
// prepare: the shared-memory limit of the instances and the resident blocks per SM of the run kernel at p.smem
cudaError_t hsrb_fd_prepare(const Plan& p, int* bps);
cudaError_t hsrb_fd_launch(const Plan& p, const FdArgs& f, int grid, cudaStream_t s);
