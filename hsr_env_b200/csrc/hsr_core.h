// One physics substep (mj_step semantics, SURVEY.md Appendix B) for one environment, executed
// cooperatively by a group of G lanes.  The same source is compiled
//   * by nvcc for sm_100a with T=float and G in {4,8,16,32} lanes of a warp per environment
//     (hsrb_kernels.cu; the per-environment workspace WS<T> lives in shared memory for all substeps), and
//   * by g++ with G=1 (oracle/cpu_port.cpp, T=double) as the CPU baseline / host-side cross-check.
//
// Replaces the body of sim.step() at /root/reference/hsr/env.py:123 (MuJoCo's mj_step, not in the tree).
//
// Execution model inside a group: values held in registers are computed redundantly and are bit-identical on
// all lanes (butterfly reductions preserve this); every workspace address is written by exactly one lane in a
// phase and phases are separated by g.sync().
#pragma once
#include <cfloat>
#include <cmath>
#include <cstdint>

#include "hsr_model.h"

// HSR_HDN: out-of-line on the device (one copy of the big routines), HSR_HDC: out-of-line only in translation units
// that define HSR_COMPACT (the register-resident kernels, whose own code is large; measured +10 % there, -20 % in
// the shared-memory kernel, where the extra calls spill the workspace pointer table).
#if defined(__CUDACC__)
#define HSR_HD __host__ __device__ __forceinline__
#define HSR_HDN __host__ __device__ __noinline__
#if defined(HSR_COMPACT)
#define HSR_HDC __host__ __device__ __noinline__
#else
#define HSR_HDC __host__ __device__ __forceinline__
#endif
#else
#define HSR_HDC inline
#define HSR_HD inline
#define HSR_HDN inline
#endif

#if defined(HSR_SCAN_NOISE) && !defined(__CUDA_ARCH__)
static thread_local unsigned long long hsr_scan_noise_seed = 0;   // 0 = off
#endif

namespace hsr {

// Geometry precision.  Body / geom poses, the narrowphase and the goal distance are evaluated in double whatever
// the state / solver type T is: a contact distance is a difference of O(0.3 m) positions and is multiplied by the
// contact stiffness (k ~ 5e3 s^-2) and the constraint weight before it reaches the 1 kg block whose inertia is
// ~3e-4 kg m^2, so the 3e-8 m resolution of fp32 positions shows up as ~1 rad/s^2 in qacc.  Inputs (qpos, model
// constants) are fp32 on the device and are exactly representable in double, so this stage has no input error.
// It is a few hundred flops per substep; the solver (the bulk of the arithmetic) stays in T.
using GT = double;

using std::cos; using std::fabs; using std::fmax; using std::fmin; using std::pow; using std::sin; using std::sqrt;

template <typename T> struct Lim;
template <> struct Lim<float> {
  HSR_HD static float eps() { return FLT_EPSILON; }
  HSR_HD static float minval() { return 1e-15f; }
};
template <> struct Lim<double> {
  HSR_HD static double eps() { return DBL_EPSILON; }
  HSR_HD static double minval() { return 1e-15; }
};

// ------------------------------------------------------------------------------------------------ per-environment parameters
// Multipliers of model constants (DESIGN 4.3b), applied once where the constant is read, as a rounded product that no later
// multiply-add absorbs: a scale of 1 reads the model's bits, a power of two reads the bits of a model whose arrays were scaled.
//   [PRM_FRICTION] pair_friction (all five), [PRM_BLOCK_MASS] body_mass and body_inertia of the bodies in block_body,
//   [PRM_GAIN] act_kp, [PRM_DAMPING] dof_damping.
// The stages take the policy as a template argument: NoScale (the default) reads the model as it is and compiles to the
// code without parameters; EnvScale holds one environment's multipliers.
enum { PRM_FRICTION = 0, PRM_BLOCK_MASS, PRM_GAIN, PRM_DAMPING, PRM_COUNT };
HSR_HD float mul_rn(float v, float s) {
#if defined(__CUDA_ARCH__)
  return __fmul_rn(v, s);
#else
  volatile float p = v * s;   // stored: never contracted into a later multiply-add
  return p;
#endif
}
HSR_HD double mul_rn(double v, double s) {
#if defined(__CUDA_ARCH__)
  return __dmul_rn(v, s);
#else
  volatile double p = v * s;
  return p;
#endif
}
struct NoScale {
  template <typename T> HSR_HD const T* friction(const T* f, T*) const { return f; }
  template <typename T> HSR_HD T block(const ModelT<T>&, int, T v) const { return v; }
  template <typename T> HSR_HD const T* inertia(const ModelT<T>& m, int b, T*) const { return m.body_inertia + 6 * b; }
  template <typename T> HSR_HD T gain(T v) const { return v; }
  template <typename T> HSR_HD T damping(T v) const { return v; }
  HSR_HD float scale(int) const { return 1.f; }
  HSR_HD void unit(int) {}
};
struct EnvScale {
  float s[PRM_COUNT];
  // the five coefficients of a pair, scaled into buf
  template <typename T> HSR_HD const T* friction(const T* f, T* buf) const {
    for (int k = 0; k < 5; k++) buf[k] = mul_rn(f[k], (T)s[PRM_FRICTION]);
    return buf;
  }
  // a mass or inertia entry of body b
  template <typename T> HSR_HD T block(const ModelT<T>& m, int b, T v) const {
    for (int k = 0; k < m.nblock; k++)
      if (m.block_body[k] == b) return mul_rn(v, (T)s[PRM_BLOCK_MASS]);
    return v;
  }
  // the six inertia entries of body b, scaled into buf
  template <typename T> HSR_HD const T* inertia(const ModelT<T>& m, int b, T* buf) const {
    for (int k = 0; k < 6; k++) buf[k] = block(m, b, m.body_inertia[6 * b + k]);
    return buf;
  }
  template <typename T> HSR_HD T gain(T v) const { return mul_rn(v, (T)s[PRM_GAIN]); }
  template <typename T> HSR_HD T damping(T v) const { return mul_rn(v, (T)s[PRM_DAMPING]); }
  HSR_HD float scale(int k) const { return s[k]; }
  HSR_HD void unit(int k) { s[k] = 1.f; }
};

enum { FLAG_CON_OVERFLOW = 1, FLAG_BAD_NUM = 2, FLAG_CHOL = 4 };
enum { WI_NCON = 0, WI_NEFC = 1, WI_NLIMIT = 2, WI_FLAGS = 3, WI_ITER = 4, WI_NARROW = 5, WI_LSEVAL = 6, WI_KFLOP = 7,
       WI_SUMCON = 8, WI_SUMEFC = 9, WI_NPFLOP = 10, WI_TLAST = 11, WI_PHASE0 = 12, WI_COUNT = 20 };
enum { PH_KIN = 0, PH_CRB, PH_SMOOTH, PH_COLLIDE, PH_ROWS, PH_SOLVE, PH_EULER, PH_COUNT };
// per-phase cycle counters (lane 0, clock64), compiled in only with -DHSRB_PHASE_CLOCKS (tools/gpu_phases.sh)
#if defined(HSRB_PHASE_CLOCKS) && defined(__CUDA_ARCH__)
#define HSR_PHASE(w, g, id)                                                             \
  do {                                                                                  \
    if ((g).lane == 0) {                                                                \
      int t_ = (int)clock64();                                                          \
      (w).wi[WI_PHASE0 + (id)] += (t_ - (w).wi[WI_TLAST]) >> 4;                         \
      (w).wi[WI_TLAST] = t_;                                                            \
    }                                                                                   \
  } while (0)
#define HSR_PHASE_START(w, g) do { if ((g).lane == 0) (w).wi[WI_TLAST] = (int)clock64(); } while (0)
#else
#define HSR_PHASE(w, g, id) do { } while (0)
#define HSR_PHASE_START(w, g) do { } while (0)
#endif
#define HSR_LSQ 10
#define HSR_MAXJOBS 16   // convex-convex narrowphase jobs an environment can queue per substep (phase-locked general kernel)

// ------------------------------------------------------------------------------------------------ groups
struct HostGrp {
  static constexpr int G = 1;
  int lane = 0;
  template <typename T> HSR_HD T sum(T x) const { return x; }
  template <typename T> HSR_HD void argmax(T&, int&) const {}
  HSR_HD unsigned ballot(bool p) const { return p ? 1u : 0u; }
  HSR_HD double max(double x) const { return x; }
  HSR_HD int min(int x) const { return x; }
  template <typename T> HSR_HD T bcast(T x, int) const { return x; }
  HSR_HD void sync() const {}
};

#if defined(__CUDACC__)
template <int G_>
struct DevGrp {
  static constexpr int G = G_;
  int lane;       // lane inside the group
  unsigned mask;  // member mask of the group inside its warp
  int shift;      // first warp lane of the group
  __device__ __forceinline__ DevGrp() {
    int wl = threadIdx.x & 31;
    lane = wl % G_;
    shift = wl - lane;
    mask = (G_ == 32) ? 0xffffffffu : (((1u << G_) - 1u) << shift);
  }
  template <typename T> __device__ __forceinline__ T sum(T x) const {
#pragma unroll
    for (int o = G_ / 2; o > 0; o >>= 1) x += __shfl_xor_sync(mask, x, o);
    return x;
  }
  // full warp, float keys: two warp reductions (redux.sync) on an order-preserving integer image of the key instead of
  // five shuffle rounds; ties go to the lowest index like the butterfly below
  __device__ __forceinline__ void argmax(float& v, int& i) const {
#ifndef HSR_NO_REDUX
    if (G_ == 32) {
      const unsigned u = __float_as_uint(v);
      const unsigned key = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
      const unsigned best = __reduce_max_sync(0xffffffffu, key);
      i = __reduce_min_sync(0xffffffffu, key == best ? i : 0x7fffffff);
      const unsigned b = (best & 0x80000000u) ? (best & 0x7fffffffu) : ~best;
      v = __uint_as_float(b);
      return;
    }
#endif
#pragma unroll
    for (int o = G_ / 2; o > 0; o >>= 1) {
      float ov = __shfl_xor_sync(mask, v, o);
      int oi = __shfl_xor_sync(mask, i, o);
      if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
    }
  }
  template <typename T> __device__ __forceinline__ void argmax(T& v, int& i) const {
#pragma unroll
    for (int o = G_ / 2; o > 0; o >>= 1) {
      T ov = __shfl_xor_sync(mask, v, o);
      int oi = __shfl_xor_sync(mask, i, o);
      if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
    }
  }
  __device__ __forceinline__ unsigned ballot(bool p) const {
    unsigned b = __ballot_sync(mask, p) >> shift;
    return (G_ == 32) ? b : (b & ((1u << G_) - 1u));
  }
  __device__ __forceinline__ double max(double x) const {
#pragma unroll
    for (int o = G_ / 2; o > 0; o >>= 1) { const double t = __shfl_xor_sync(mask, x, o); x = t > x ? t : x; }
    return x;
  }
  __device__ __forceinline__ int min(int x) const {
#pragma unroll
    for (int o = G_ / 2; o > 0; o >>= 1) { const int t = __shfl_xor_sync(mask, x, o); x = t < x ? t : x; }
    return x;
  }
  template <typename T> __device__ __forceinline__ T bcast(T x, int src) const { return __shfl_sync(mask, x, src, G_); }   // value of lane `src` of the group
  __device__ __forceinline__ void sync() const { __syncwarp(mask); }
};
#endif

// ------------------------------------------------------------------------------------------------ vec3
template <typename T> struct V3 { T x, y, z; };
template <typename T> HSR_HD V3<T> mk(T x, T y, T z) { V3<T> v; v.x = x; v.y = y; v.z = z; return v; }
template <typename T> HSR_HD V3<T> ld3(const T* p) { return mk<T>(p[0], p[1], p[2]); }
template <typename T> HSR_HD V3<GT> ldg(const T* p) { return mk<GT>((GT)p[0], (GT)p[1], (GT)p[2]); }
template <typename T, typename U> HSR_HD V3<T> cvt(V3<U> v) { return mk<T>((T)v.x, (T)v.y, (T)v.z); }
template <typename T, typename U> HSR_HD void st3c(T* p, V3<U> v) { p[0] = (T)v.x; p[1] = (T)v.y; p[2] = (T)v.z; }
template <typename T> HSR_HD void st3(T* p, V3<T> v) { p[0] = v.x; p[1] = v.y; p[2] = v.z; }
template <typename T> HSR_HD V3<T> operator+(V3<T> a, V3<T> b) { return mk<T>(a.x + b.x, a.y + b.y, a.z + b.z); }
template <typename T> HSR_HD V3<T> operator-(V3<T> a, V3<T> b) { return mk<T>(a.x - b.x, a.y - b.y, a.z - b.z); }
template <typename T> HSR_HD V3<T> operator-(V3<T> a) { return mk<T>(-a.x, -a.y, -a.z); }
template <typename T> HSR_HD V3<T> operator*(V3<T> a, T s) { return mk<T>(a.x * s, a.y * s, a.z * s); }
template <typename T> HSR_HD T dot(V3<T> a, V3<T> b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
template <typename T> HSR_HD V3<T> cross(V3<T> a, V3<T> b) {
  return mk<T>(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
template <typename T> HSR_HD T norm(V3<T> a) { return sqrt(dot(a, a)); }
template <typename T> HSR_HD V3<T> normalized(V3<T> a) {
#if defined(__CUDA_ARCH__)
  return a * (T)rsqrt(dot(a, a));   // one special-function sequence instead of sqrt + divide (<= 2 ulp of T)
#else
  return a * (T(1) / norm(a));
#endif
}
template <typename T> HSR_HD T comp(V3<T> a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }
// 3x3 row-major helpers
template <typename T> HSR_HD V3<T> mcol(const T* R, int k) { return mk<T>(R[k], R[3 + k], R[6 + k]); }
template <typename T> HSR_HD V3<T> mulv(const T* R, V3<T> v) {
  return mk<T>(R[0] * v.x + R[1] * v.y + R[2] * v.z, R[3] * v.x + R[4] * v.y + R[5] * v.z,
               R[6] * v.x + R[7] * v.y + R[8] * v.z);
}
template <typename T> HSR_HD V3<T> multv(const T* R, V3<T> v) {  // R^T v
  return mk<T>(R[0] * v.x + R[3] * v.y + R[6] * v.z, R[1] * v.x + R[4] * v.y + R[7] * v.z,
               R[2] * v.x + R[5] * v.y + R[8] * v.z);
}
template <typename T> HSR_HD void mulm(const T* A, const T* B, T* C) {  // C = A B
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}
template <typename T> HSR_HD void quat2mat(const T* q, T* R) {
  T w = q[0], x = q[1], y = q[2], z = q[3];
  R[0] = w * w + x * x - y * y - z * z; R[1] = 2 * (x * y - w * z); R[2] = 2 * (x * z + w * y);
  R[3] = 2 * (x * y + w * z); R[4] = w * w - x * x + y * y - z * z; R[5] = 2 * (y * z - w * x);
  R[6] = 2 * (x * z - w * y); R[7] = 2 * (y * z + w * x); R[8] = w * w - x * x - y * y + z * z;
}
template <typename T> HSR_HD void quatmul(const T* a, const T* b, T* r) {
  T r0 = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3];
  T r1 = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
  T r2 = a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1];
  T r3 = a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0];
  r[0] = r0; r[1] = r1; r[2] = r2; r[3] = r3;
}
template <typename T> HSR_HD void quatnormalize(T* q) {
  T n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  if (n < Lim<T>::minval()) { q[0] = 1; q[1] = q[2] = q[3] = 0; return; }
  T inv = T(1) / n;
  q[0] *= inv; q[1] *= inv; q[2] *= inv; q[3] *= inv;
}

// ------------------------------------------------------------------------------------------------ workspace
template <typename T>
struct WS {
  GT *xpos, *xquat, *xmat, *xipos, *anchor, *axis, *gpos, *com;
  T *qpos, *qvel, *warm, *ctrl, *mocap;
  T *cdof, *cinert, *binert;
  T *cvel, *cacc, *cfrc;   // RNE scratch [nbody][6] each (shared memory on the device: local arrays would live in L2)
  GT* trig;                // [njnt][2] cos, sin of the hinge joints' half angles (computed one joint per lane)
  T *M, *L, *H;
  T *qfrc_smooth, *qacc_smooth, *qacc, *Ma, *grad, *search, *Mv, *tmpv, *invd;
  T *gaabb;
  T *con_dist, *con_pos, *con_frame, *con_mu;
  T *J, *D, *aref, *jar, *jv, *force;
  T *wrow, *PQ, *wpq;   // Hessian as weighted outer products: row weights [ne], cone vectors p | q [nc][2][nv], their weights [nc][2]
  T *lsq;
  int *con_pair, *con_adr, *con_zone;
  int* wi;
  float* sep;   // [npair][4] cached separating direction + valid flag of each candidate pair (mpr_penetration's `sep`)
  GT* jres;     // [HSR_MAXJOBS][8] phase-locked kernel: results of this environment's convex-convex jobs (hit, depth, dir, pos)
  unsigned* cand;   // [8] phase-locked kernel: candidate pairs that passed the cull (bit mask, npair <= 256)
};

// Carve the workspace out of `base` (nullptr: just return the size in bytes).
template <typename T>
HSR_HD size_t ws_carve(const ModelT<T>& m, WS<T>* w, unsigned char* base) {
  size_t off = 0;
  WS<T> dummy;
  if (!w) w = &dummy;
#define CARVE(field, type, n) { w->field = (type*)(base + off); off += sizeof(type) * (size_t)(n); }
  int nv = m.nv, nb = m.nbody, nc = m.ncon_max, ne = m.nefc_max;
  CARVE(xpos, GT, nb * 3) CARVE(xquat, GT, nb * 4) CARVE(xmat, GT, nb * 9) CARVE(xipos, GT, nb * 3)
  CARVE(anchor, GT, m.njnt * 3) CARVE(axis, GT, m.njnt * 3) CARVE(gpos, GT, m.ngeom * 3) CARVE(com, GT, nb * 3)
  CARVE(trig, GT, m.njnt * 2)
  CARVE(qpos, T, m.nq) CARVE(qvel, T, nv) CARVE(warm, T, nv) CARVE(ctrl, T, m.nu > 0 ? m.nu : 1) CARVE(mocap, T, 3)
  CARVE(cdof, T, nv * 6) CARVE(cinert, T, nb * 10) CARVE(binert, T, nb * 10)
  CARVE(cvel, T, nb * 6) CARVE(cacc, T, nb * 6) CARVE(cfrc, T, nb * 6)
  CARVE(M, T, nv * nv) CARVE(L, T, nv * nv) CARVE(H, T, nv * nv)
  CARVE(qfrc_smooth, T, nv) CARVE(qacc_smooth, T, nv) CARVE(qacc, T, nv) CARVE(Ma, T, nv) CARVE(grad, T, nv)
  CARVE(search, T, nv) CARVE(Mv, T, nv) CARVE(tmpv, T, nv) CARVE(invd, T, nv)
  CARVE(gaabb, T, m.ngeom * 3)
  CARVE(con_dist, T, nc) CARVE(con_pos, T, nc * 3) CARVE(con_frame, T, nc * 9) CARVE(con_mu, T, nc)
  CARVE(J, T, ne * nv) CARVE(wrow, T, ne) CARVE(PQ, T, 2 * nc * nv) CARVE(wpq, T, 2 * nc) CARVE(D, T, ne) CARVE(aref, T, ne) CARVE(jar, T, ne) CARVE(jv, T, ne)
  CARVE(force, T, ne) CARVE(lsq, T, nc * HSR_LSQ)
  CARVE(con_pair, int, nc) CARVE(con_adr, int, nc) CARVE(con_zone, int, nc) CARVE(wi, int, WI_COUNT)
  CARVE(sep, float, 4 * m.npair)
  off += (8 - off % 8) % 8;
  CARVE(jres, GT, 8 * HSR_MAXJOBS) CARVE(cand, unsigned, 8)
#undef CARVE
  off += (16 - off % 16) % 16;
  return off;
}

// ------------------------------------------------------------------------------------------------ B.1 kinematics
// 10-number spatial inertia about the reference point (tree CoM): Ixx Iyy Izz Ixy Ixz Iyz  m*cx m*cy m*cz  m
template <typename T> HSR_HD void inert_mul(const T* I, const T* v, T* f) {  // f = I * v,  v=[ang;lin], f=[torque;force]
  V3<T> w = ld3(v), vo = ld3(v + 3), mc = ld3(I + 6);
  V3<T> fl = vo * I[9] + cross(w, mc);
  V3<T> fa = mk<T>(I[0] * w.x + I[3] * w.y + I[4] * w.z, I[3] * w.x + I[1] * w.y + I[5] * w.z,
                   I[4] * w.x + I[5] * w.y + I[2] * w.z) + cross(mc, vo);
  st3(f, fa); st3(f + 3, fl);
}

// cos / sin of the hinge joints' half angles, one joint per lane (the serial chain of kinematics_lane0 then only multiplies)
template <typename T, typename Grp>
HSR_HD void kinematics_trig(const ModelT<T>& m, WS<T>& w, const Grp& g) {
  for (int j = g.lane; j < m.njnt; j += Grp::G) {
    if (m.jnt_type[j] != JNT_HINGE) continue;
    const GT h = ((GT)w.qpos[m.jnt_qposadr[j]] - (GT)m.qpos0[m.jnt_qposadr[j]]) * GT(0.5);
    w.trig[2 * j] = cos(h); w.trig[2 * j + 1] = sin(h);
  }
  g.sync();
}

template <typename T, typename Sc = NoScale>
HSR_HDC void kinematics_lane0(const ModelT<T>& m, WS<T>& w, const Sc& sc = Sc()) {
  // world
  for (int k = 0; k < 3; k++) { w.xpos[k] = 0; w.xipos[k] = 0; }
  for (int k = 0; k < 9; k++) w.xmat[k] = (k % 4 == 0) ? GT(1) : GT(0);
  w.xquat[0] = 1; w.xquat[1] = w.xquat[2] = w.xquat[3] = 0;
  for (int k = 0; k < 10; k++) { w.binert[k] = 0; }
  for (int b = 1; b < m.nbody; b++) {
    int p = m.body_parent[b];
    int j0 = m.body_jntadr[b], nj = m.body_jntnum[b];
    GT pos[3], quat[4], R[9];
    if (nj == 1 && m.jnt_type[j0] == JNT_FREE) {
      int a = m.jnt_qposadr[j0];
      for (int k = 0; k < 3; k++) pos[k] = (GT)w.qpos[a + k];
      for (int k = 0; k < 4; k++) quat[k] = (GT)w.qpos[a + 3 + k];
      quatnormalize(quat);
      for (int k = 0; k < 4; k++) w.qpos[a + 3 + k] = (T)quat[k];  // MuJoCo normalises qpos in place
      for (int k = 0; k < 3; k++) w.anchor[3 * j0 + k] = pos[k];
      quat2mat(quat, R);
    } else {
      V3<GT> pp = ld3(w.xpos + 3 * p) + mulv(w.xmat + 9 * p, ldg(m.body_pos + 3 * b));
      st3(pos, pp);
      GT bq[4] = {(GT)m.body_quat[4 * b], (GT)m.body_quat[4 * b + 1], (GT)m.body_quat[4 * b + 2], (GT)m.body_quat[4 * b + 3]};
      quatmul(w.xquat + 4 * p, bq, quat);
      quat2mat(quat, R);
      for (int j = j0; j < j0 + nj; j++) {
        V3<GT> anc = ld3(pos) + mulv(R, ldg(m.jnt_pos + 3 * j));
        V3<GT> ax = mulv(R, ldg(m.jnt_axis + 3 * j));
        st3(w.anchor + 3 * j, anc); st3(w.axis + 3 * j, ax);
        GT q = (GT)w.qpos[m.jnt_qposadr[j]] - (GT)m.qpos0[m.jnt_qposadr[j]];
        if (m.jnt_type[j] == JNT_SLIDE) {
          st3(pos, ld3(pos) + ax * q);
        } else {
          const GT sn = w.trig[2 * j + 1];
          GT dq[4] = {w.trig[2 * j], sn * (GT)m.jnt_axis[3 * j], sn * (GT)m.jnt_axis[3 * j + 1], sn * (GT)m.jnt_axis[3 * j + 2]};
          quatmul(quat, dq, quat);
          quat2mat(quat, R);
          st3(pos, anc - mulv(R, ldg(m.jnt_pos + 3 * j)));
        }
      }
      quatnormalize(quat);
      quat2mat(quat, R);
    }
    for (int k = 0; k < 3; k++) w.xpos[3 * b + k] = pos[k];
    for (int k = 0; k < 4; k++) w.xquat[4 * b + k] = quat[k];
    for (int k = 0; k < 9; k++) w.xmat[9 * b + k] = R[k];
    V3<GT> cg = ld3(pos) + mulv(R, ldg(m.body_ipos + 3 * b));
    st3(w.xipos + 3 * b, cg);
  }
  // Centre of mass of every kinematic tree.  All spatial quantities of a tree (motion axes, inertias, bias forces,
  // contact Jacobians) are expressed about its CoM instead of the world origin, as MuJoCo does: about the origin
  // the parallel-axis term m |c|^2 (4e-2 for a block 0.2 m away) swamps the block's own 3e-4 kg m^2 inertia and
  // fp32 loses 1e-5 of it.  The two formulations are the same mathematics.
  for (int b = 0; b < m.nbody; b++) { w.com[3 * b] = 0; w.com[3 * b + 1] = 0; w.com[3 * b + 2] = 0; }
  for (int r = 1; r < m.nbody; r++) {
    if (m.body_root[r] != r) continue;
    V3<GT> acc = mk<GT>(0, 0, 0);
    GT mt = 0;
    for (int b = r; b < m.nbody; b++)
      if (m.body_root[b] == r) { acc = acc + ld3(w.xipos + 3 * b) * (GT)sc.block(m, b, m.body_mass[b]); mt += (GT)sc.block(m, b, m.body_mass[b]); }
    if (mt > 0) acc = acc * (GT(1) / mt);
    for (int b = r; b < m.nbody; b++)
      if (m.body_root[b] == r) st3(w.com + 3 * b, acc);
  }
  for (int b = 1; b < m.nbody; b++) {
    // spatial inertia about the tree CoM (solver precision)
    const GT* R = w.xmat + 9 * b;
    V3<T> c = cvt<T>(ld3(w.xipos + 3 * b) - ld3(w.com + 3 * b));
    T Rt_[9];
    for (int k = 0; k < 9; k++) Rt_[k] = (T)R[k];
    T ibuf[6];
    const T* ib = sc.inertia(m, b, ibuf);
    T Ib[9] = {ib[0], ib[3], ib[4], ib[3], ib[1], ib[5], ib[4], ib[5], ib[2]};
    T tmp[9], Iw[9], Rt[9];
    for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) Rt[3 * i + j] = Rt_[3 * j + i];
    mulm(Rt_, Ib, tmp); mulm(tmp, Rt, Iw);
    T mass = sc.block(m, b, m.body_mass[b]);
    T cc = dot(c, c);
    T* I = w.binert + 10 * b;
    I[0] = Iw[0] + mass * (cc - c.x * c.x); I[1] = Iw[4] + mass * (cc - c.y * c.y); I[2] = Iw[8] + mass * (cc - c.z * c.z);
    I[3] = Iw[1] - mass * c.x * c.y; I[4] = Iw[2] - mass * c.x * c.z; I[5] = Iw[5] - mass * c.y * c.z;
    I[6] = mass * c.x; I[7] = mass * c.y; I[8] = mass * c.z; I[9] = mass;
  }
  // composite inertias (leaf -> root)
  for (int k = 0; k < 10 * m.nbody; k++) w.cinert[k] = w.binert[k];
  for (int b = m.nbody - 1; b > 0; b--) {
    int p = m.body_parent[b];
    if (p > 0) for (int k = 0; k < 10; k++) w.cinert[10 * p + k] += w.cinert[10 * b + k];
  }
}

// B.2 (part): motion axes about the tree CoM, [ang; lin]; geom centres + world AABB half extents
template <typename T, typename Grp>
HSR_HDC void cdof_geoms(const ModelT<T>& m, WS<T>& w, const Grp& g) {
  for (int j = g.lane; j < m.njnt; j += Grp::G) {
    int a = m.jnt_dofadr[j], b = m.jnt_body[j], t = m.jnt_type[j];
    if (t == JNT_FREE) {
      V3<GT> xp = ld3(w.xpos + 3 * b) - ld3(w.com + 3 * b);
      for (int k = 0; k < 3; k++) {
        T* c = w.cdof + 6 * (a + k);
        for (int i = 0; i < 6; i++) c[i] = (i == 3 + k) ? T(1) : T(0);
        V3<GT> ax = mcol(w.xmat + 9 * b, k);
        T* cr = w.cdof + 6 * (a + 3 + k);
        st3c(cr, ax); st3c(cr + 3, cross(xp, ax));
      }
    } else if (t == JNT_SLIDE) {
      T* c = w.cdof + 6 * a;
      c[0] = c[1] = c[2] = 0; st3c(c + 3, ld3(w.axis + 3 * j));
    } else {
      T* c = w.cdof + 6 * a;
      V3<GT> ax = ld3(w.axis + 3 * j);
      st3c(c, ax); st3c(c + 3, cross(ld3(w.anchor + 3 * j) - ld3(w.com + 3 * b), ax));
    }
  }
  for (int gi = g.lane; gi < m.ngeom; gi += Grp::G) {
    int b = m.geom_body[gi];
    const GT* R = w.xmat + 9 * b;
    st3(w.gpos + 3 * gi, ld3(w.xpos + 3 * b) + mulv(R, ldg(m.geom_pos + 3 * gi)));
    // conservative world AABB half extents (midphase cull only): solver precision
    T Rb[9], Rg[9];
    for (int k = 0; k < 9; k++) Rb[k] = (T)R[k];
    mulm(Rb, m.geom_mat + 9 * gi, Rg);
    const T* h = m.geom_aabb + 3 * gi;
    for (int i = 0; i < 3; i++)
      w.gaabb[3 * gi + i] = fabs(Rg[3 * i]) * h[0] + fabs(Rg[3 * i + 1]) * h[1] + fabs(Rg[3 * i + 2]) * h[2];
  }
}

// B.2: dense joint-space inertia by the composite-rigid-body method; one dof row per lane
template <typename T, typename Grp>
HSR_HDC void mass_matrix(const ModelT<T>& m, WS<T>& w, const Grp& g) {
  int nv = m.nv;
  for (int i = g.lane; i < nv; i += Grp::G) {
    T f[6];
    inert_mul(w.cinert + 10 * m.dof_body[i], w.cdof + 6 * i, f);
    for (int j = 0; j < nv; j++) if (j > i || !((m.body_dofmask[m.dof_body[i]] >> j) & 1u)) w.M[i * nv + j] = 0;
    int j = i;
    while (j >= 0) {
      const T* c = w.cdof + 6 * j;
      T v = c[0] * f[0] + c[1] * f[1] + c[2] * f[2] + c[3] * f[3] + c[4] * f[4] + c[5] * f[5];
      w.M[i * nv + j] = v;
      j = m.dof_parent[j];
    }
  }
  g.sync();
  // mirror to the upper triangle (each lane mirrors its own rows' transposes)
  for (int i = g.lane; i < nv; i += Grp::G)
    for (int j = i + 1; j < nv; j++) w.M[i * nv + j] = w.M[j * nv + i];
}

// dense Cholesky A = L L^T (lower, in place) and solves; serial (lane 0)
template <typename T> HSR_HDC bool chol_factor(T* A, int n) {
  bool ok = true;
  for (int k = 0; k < n; k++) {
    T d = A[k * n + k];
    for (int j = 0; j < k; j++) d -= A[k * n + j] * A[k * n + j];
    if (!(d > Lim<T>::minval())) { d = Lim<T>::minval(); ok = false; }
    d = sqrt(d);
    A[k * n + k] = d;
    T inv = T(1) / d;
    for (int i = k + 1; i < n; i++) {
      T s = A[i * n + k];
      for (int j = 0; j < k; j++) s -= A[i * n + j] * A[k * n + j];
      A[i * n + k] = s * inv;
    }
  }
  return ok;
}
template <typename T> HSR_HDC void chol_solve(const T* L, int n, T* x) {
  for (int i = 0; i < n; i++) {
    T s = x[i];
    for (int j = 0; j < i; j++) s -= L[i * n + j] * x[j];
    x[i] = s / L[i * n + i];
  }
  for (int i = n - 1; i >= 0; i--) {
    T s = x[i];
    for (int j = i + 1; j < n; j++) s -= L[j * n + i] * x[j];
    x[i] = s / L[i * n + i];
  }
}

// The same factorisation / solves with the lanes of a group sharing the rows (A in the environment's shared-memory
// workspace).  Column k: every row i >= k forms its dot product with row k in the serial routine's order (so L is
// bit-identical to chol_factor's), then the rows below the diagonal are scaled.  The solves are column-oriented: once
// x[i] is final the lanes subtract its column from the remaining entries.  With one lane (host port) this is the
// serial algorithm.
template <typename T> HSR_HD T rsqrt_t(T x) {
#if defined(__CUDA_ARCH__)
  return (T)rsqrt(x);
#else
  return T(1) / sqrt(x);
#endif
}
// `invd` (n entries) receives the reciprocals of the diagonal of L: the solves multiply instead of dividing.
// n <= G (one row per lane: every kernel layout with nv <= lanes per environment, and the host port's G = 1 through
// the other branch): lane i keeps its running element in a register, the pivot travels by a group broadcast instead of
// through shared memory: one barrier per column instead of three, no division, no square root + division pair.
template <typename T, typename Grp> HSR_HDC bool chol_factor_g(T* A, int n, T* invd, const Grp& g) {
  bool ok = true;
  if (Grp::G > 1 && n <= Grp::G) {
    const int i = g.lane;
    for (int k = 0; k < n; k++) {
      T s = 0;
      if (i >= k && i < n) {
        s = A[i * n + k];
        for (int j = 0; j < k; j++) s -= A[i * n + j] * A[k * n + j];
      }
      T d = g.bcast(s, k);
      if (!(d > Lim<T>::minval())) { d = Lim<T>::minval(); ok = false; }
      const T rs = rsqrt_t(d);
      if (i >= k && i < n) A[i * n + k] = (i == k) ? d * rs : s * rs;
      if (i == k) invd[k] = rs;
      g.sync();
    }
    return ok;
  }
  for (int k = 0; k < n; k++) {
    for (int i = k + g.lane; i < n; i += Grp::G) {
      T s = A[i * n + k];
      for (int j = 0; j < k; j++) s -= A[i * n + j] * A[k * n + j];
      A[i * n + k] = s;
    }
    g.sync();
    T d = A[k * n + k];
    if (!(d > Lim<T>::minval())) { d = Lim<T>::minval(); ok = false; }
    const T rs = rsqrt_t(d);
    g.sync();   // every lane has read the pivot
    for (int i = k + g.lane; i < n; i += Grp::G) A[i * n + k] = (i == k) ? d * rs : A[i * n + k] * rs;
    if (g.lane == 0) invd[k] = rs;
    g.sync();
  }
  return ok;
}
template <typename T, typename Grp> HSR_HDC void chol_solve_g(const T* L, int n, const T* invd, T* x, const Grp& g) {
  if (Grp::G > 1 && n <= Grp::G) {
    // lane r keeps x[r] in a register; the finished component travels by a group broadcast
    const int r = g.lane;
    T xr = r < n ? x[r] : T(0);
    for (int i = 0; i < n; i++) {        // L y = b
      const T xi = g.bcast(xr, i) * invd[i];
      if (r == i) xr = xi;
      else if (r > i && r < n) xr -= L[r * n + i] * xi;
    }
    for (int i = n - 1; i >= 0; i--) {   // L^T x = y
      const T xi = g.bcast(xr, i) * invd[i];
      if (r == i) xr = xi;
      else if (r < i) xr -= L[i * n + r] * xi;
    }
    if (r < n) x[r] = xr;
    g.sync();
    return;
  }
  for (int i = 0; i < n; i++) {        // L y = b
    const T xi = x[i] * invd[i];
    g.sync();
    if (g.lane == 0) x[i] = xi;
    for (int r = i + 1 + g.lane; r < n; r += Grp::G) x[r] -= L[r * n + i] * xi;
    g.sync();
  }
  for (int i = n - 1; i >= 0; i--) {   // L^T x = y
    const T xi = x[i] * invd[i];
    g.sync();
    if (g.lane == 0) x[i] = xi;
    for (int r = g.lane; r < i; r += Grp::G) x[r] -= L[i * n + r] * xi;
    g.sync();
  }
}

// ------------------------------------------------------------------------------------------------ B.6 smooth dynamics
template <typename T> HSR_HD void cross_motion(const T* v, const T* s, T* r) {
  V3<T> va = ld3(v), vl = ld3(v + 3), sa = ld3(s), sl = ld3(s + 3);
  st3(r, cross(va, sa)); st3(r + 3, cross(va, sl) + cross(vl, sa));
}
template <typename T> HSR_HD void cross_force(const T* v, const T* f, T* r) {
  V3<T> va = ld3(v), vl = ld3(v + 3), fa = ld3(f), fl = ld3(f + 3);
  st3(r, cross(va, fa) + cross(vl, fl)); st3(r + 3, cross(va, fl));
}

// lane 0: RNE bias, passive, actuation -> qfrc_smooth
template <typename T, typename Sc = NoScale>
HSR_HDC void smooth_lane0(const ModelT<T>& m, WS<T>& w, const Sc& sc = Sc()) {
  int nv = m.nv;
  T (*cvel)[6] = reinterpret_cast<T(*)[6]>(w.cvel);
  T (*cacc)[6] = reinterpret_cast<T(*)[6]>(w.cacc);
  T (*cfrc)[6] = reinterpret_cast<T(*)[6]>(w.cfrc);
  for (int k = 0; k < 6; k++) { cvel[0][k] = 0; cacc[0][k] = 0; cfrc[0][k] = 0; }
  cacc[0][3] = -m.gravity[0]; cacc[0][4] = -m.gravity[1]; cacc[0][5] = -m.gravity[2];
  for (int b = 1; b < m.nbody; b++) {
    int p = m.body_parent[b];
    T v[6], a[6], t[6];
    for (int k = 0; k < 6; k++) { v[k] = cvel[p][k]; a[k] = cacc[p][k]; }
    for (int j = m.body_jntadr[b]; j < m.body_jntadr[b] + m.body_jntnum[b]; j++) {
      int d0 = m.jnt_dofadr[j];
      if (m.jnt_type[j] == JNT_FREE) {
        for (int k = 0; k < 3; k++) for (int i = 0; i < 6; i++) v[i] += w.cdof[6 * (d0 + k) + i] * w.qvel[d0 + k];
        T vt[6];
        for (int i = 0; i < 6; i++) vt[i] = v[i];
        for (int k = 3; k < 6; k++) {
          cross_motion(vt, w.cdof + 6 * (d0 + k), t);
          for (int i = 0; i < 6; i++) { a[i] += t[i] * w.qvel[d0 + k]; v[i] += w.cdof[6 * (d0 + k) + i] * w.qvel[d0 + k]; }
        }
      } else {
        cross_motion(v, w.cdof + 6 * d0, t);
        for (int i = 0; i < 6; i++) { a[i] += t[i] * w.qvel[d0]; v[i] += w.cdof[6 * d0 + i] * w.qvel[d0]; }
      }
    }
    T Ia[6], Iv[6];
    inert_mul(w.binert + 10 * b, a, Ia);
    inert_mul(w.binert + 10 * b, v, Iv);
    cross_force(v, Iv, t);
    for (int k = 0; k < 6; k++) { cvel[b][k] = v[k]; cacc[b][k] = a[k]; cfrc[b][k] = Ia[k] + t[k]; }
  }
  for (int b = m.nbody - 1; b > 0; b--) {
    int p = m.body_parent[b];
    if (p > 0) for (int k = 0; k < 6; k++) cfrc[p][k] += cfrc[b][k];
  }
  for (int i = 0; i < nv; i++) {
    const T* c = w.cdof + 6 * i;
    const T* f = cfrc[m.dof_body[i]];
    T bias = c[0] * f[0] + c[1] * f[1] + c[2] * f[2] + c[3] * f[3] + c[4] * f[4] + c[5] * f[5];
    w.qfrc_smooth[i] = -sc.damping(m.dof_damping[i]) * w.qvel[i] - bias;
  }
  for (int a = 0; a < m.nu; a++) {
    T c = w.ctrl[a];
    if (m.act_ctrllimited[a]) c = fmin(fmax(c, m.act_ctrlrange[2 * a]), m.act_ctrlrange[2 * a + 1]);
    T f = sc.gain(m.act_kp[a]) * c - sc.gain(m.act_kp[a]) * m.act_gear[a] * w.qpos[m.act_qposadr[a]];
    if (m.act_forcelimited[a]) f = fmin(fmax(f, m.act_forcerange[2 * a]), m.act_forcerange[2 * a + 1]);
    w.qfrc_smooth[m.act_dof[a]] += m.act_gear[a] * f;
  }
}
// factor M -> L and qacc_smooth = M^-1 qfrc_smooth, rows across the lanes of the group
template <typename T, typename Grp>
HSR_HD void smooth_solve(const ModelT<T>& m, WS<T>& w, const Grp& g) {
  const int nv = m.nv;
  for (int k = g.lane; k < nv * nv; k += Grp::G) w.L[k] = w.M[k];
  for (int i = g.lane; i < nv; i += Grp::G) w.qacc_smooth[i] = w.qfrc_smooth[i];
  g.sync();
  if (!chol_factor_g(w.L, nv, w.invd, g) && g.lane == 0) w.wi[WI_FLAGS] |= FLAG_CHOL;
  chol_solve_g(w.L, nv, w.invd, w.qacc_smooth, g);
}

// ------------------------------------------------------------------------------------------------ B.3 collision
template <typename T> struct Geom {
  int type; T size[3]; const T* verts; int nvert; V3<GT> pos; GT mat[9];   // size by value: read on every support call
  const T* verts4 = nullptr;  // optional copy of the hull vertices with a stride of 4 (16-byte aligned): 128-bit loads
};

template <typename T>
HSR_HD void load_geom(const ModelT<T>& m, const WS<T>& w, int gi, Geom<T>& ge) {
  ge.type = m.geom_type[gi];
  for (int k = 0; k < 3; k++) ge.size[k] = m.geom_size[3 * gi + k];
  ge.verts = m.hull_vert + 3 * m.geom_vertadr[gi]; ge.nvert = m.geom_vertnum[gi];
  ge.pos = ld3(w.gpos + 3 * gi);
  GT gm[9];
  for (int k = 0; k < 9; k++) gm[k] = (GT)m.geom_mat[9 * gi + k];
  mulm(w.xmat + 9 * m.geom_body[gi], gm, ge.mat);
}

template <typename T> HSR_HD void make_frame(V3<GT> n, T* fr) {
  n = normalized(n);
  V3<GT> t = (n.y > GT(-0.5) && n.y < GT(0.5)) ? mk<GT>(0, 1, 0) : mk<GT>(0, 0, 1);
  t = t - n * dot(n, t);
  t = normalized(t);
  st3c(fr, n); st3c(fr + 3, t); st3c(fr + 6, cross(n, t));
}

template <typename T, typename Grp>
HSR_HDC void add_contact(const ModelT<T>& m, WS<T>& w, const Grp& g, int& ncon, int& nrow, int pair, GT dist, V3<GT> pos,
                        V3<GT> n) {
  int dim = m.pair_condim[pair];
  if (ncon >= m.ncon_max || nrow + dim > m.nefc_max) {
    if (g.lane == 0) w.wi[WI_FLAGS] |= FLAG_CON_OVERFLOW;
    return;
  }
  if (g.lane == 0) {
    w.con_pair[ncon] = pair; w.con_dist[ncon] = (T)dist; st3c(w.con_pos + 3 * ncon, pos);
    make_frame(n, w.con_frame + 9 * ncon);
    w.con_adr[ncon] = nrow;
  }
  ncon++; nrow += dim;
}

template <typename T> struct Sup { V3<T> v, v1, v2; };

template <typename T> HSR_HD bool is_zero(T x) { return fabs(x) < Lim<T>::eps(); }
template <typename T> HSR_HD bool ccd_eq(T a, T b) {
  T ab = fabs(a - b);
  if (ab < Lim<T>::eps()) return true;
  a = fabs(a); b = fabs(b);
  return ab < Lim<T>::eps() * (b > a ? b : a);
}

// squared distance from the origin to triangle (a,b,c) with the closest point q
template <typename T> HSR_HD T origin_tri_dist2(V3<T> a, V3<T> b, V3<T> c, V3<T>& q) {
  V3<T> ab = b - a, ac = c - a, ap = -a;
  T d1 = dot(ab, ap), d2 = dot(ac, ap);
  if (d1 <= 0 && d2 <= 0) { q = a; return dot(q, q); }
  V3<T> bp = -b;
  T d3 = dot(ab, bp), d4 = dot(ac, bp);
  if (d3 >= 0 && d4 <= d3) { q = b; return dot(q, q); }
  T vc = d1 * d4 - d3 * d2;
  V3<T> cp = -c;
  T d5 = dot(ab, cp), d6 = dot(ac, cp);
  if (vc <= 0 && d1 >= 0 && d3 <= 0) { q = a + ab * (d1 / (d1 - d3)); return dot(q, q); }
  if (d6 >= 0 && d5 <= d6) { q = c; return dot(q, q); }
  T vb = d5 * d2 - d1 * d6, va = d3 * d6 - d5 * d4;
  if (vb <= 0 && d2 >= 0 && d6 <= 0) { q = a + ac * (d2 / (d2 - d6)); return dot(q, q); }
  if (va <= 0 && (d4 - d3) >= 0 && (d5 - d6) >= 0) { q = b + (c - b) * ((d4 - d3) / ((d4 - d3) + (d5 - d6))); return dot(q, q); }
  T den = T(1) / (va + vb + vc);
  q = a + ab * (vb * den) + ac * (vc * den);
  return dot(q, q);
}

// Support point for the portal refinement, evaluated in double whatever T is: the decisions of the refinement
// compare triple products of vectors that shrink with the penetration depth against libccd's DBL_EPSILON-scale
// thresholds, which fp32 cannot resolve (a 0.1 mm contact came out with a different face normal).  Only the
// vertex scan of a hull (the bulk of the work) runs in T; its result is an index, i.e. exact.
// Support ties (oracle/mjstep.py support()): a local direction component within SUPPORT_TIE of zero counts as positive,
// and among the hull vertices whose support is within SUPPORT_TIE of the maximum the lowest index wins.  Face-aligned
// directions are structural in this path (the portal refinement converges to face normals, resting contacts line up
// with box axes); with plain comparisons the winner is rounding noise and differs between implementations (fp64 numpy,
// fp64 g++, CUDA with FMA contraction), moving the contact point across the face.
#define HSR_SUPPORT_TIE 1e-12
// the vertex scan runs in T; vertices within this distance of the scanned maximum are re-evaluated in double
template <typename T> HSR_HD T scan_slack(T best) { return sizeof(T) == 4 ? T(1e-6) * (T(1) + fabs(best)) : T(HSR_SUPPORT_TIE); }
// <v, l> in double, evaluated left to right without contraction (the same number on every implementation)
HSR_HD double dot3_exact(double x, double y, double z, double lx, double ly, double lz) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(__dadd_rn(__dmul_rn(x, lx), __dmul_rn(y, ly)), __dmul_rn(z, lz));
#else
  volatile double a = x * lx, b = y * ly, c = z * lz;
  volatile double ab = a + b;
  return ab + c;
#endif
}

// argmax_i <v_i, l> over the n vertices of a hull (stride `st` floats / Ts per vertex), lanes of the group striding over
// the vertices: scan in T tracking each lane's best and second-best value; when exactly one vertex of the whole group is
// within the slack of the scanned maximum (the usual case) that vertex wins; otherwise the candidates are re-evaluated
// in double and the lowest index within HSR_SUPPORT_TIE of the maximum wins.
template <typename T> HSR_HD void load_vert(const T* p, int st, T& x, T& y, T& z) { (void)st; x = p[0]; y = p[1]; z = p[2]; }
#if defined(__CUDACC__)
template <> HSR_HD void load_vert<float>(const float* p, int st, float& x, float& y, float& z) {
  if (st == 4) { const float4 a = *reinterpret_cast<const float4*>(p); x = a.x; y = a.y; z = a.z; }   // 16-byte vertices: one 128-bit load
  else { x = p[0]; y = p[1]; z = p[2]; }
}
#endif
template <typename T, typename Grp>
HSR_HD int hull_argmax(const T* __restrict__ v, int st, int n, V3<double> dl, const Grp& g) {
  const T lx = (T)dl.x, ly = (T)dl.y, lz = (T)dl.z;
  T best = -FLT_MAX, second = -FLT_MAX;
  int bi = 0x7fffffff;
  for (int i = g.lane; i < n; i += Grp::G) {
    T px, py, pz;
    load_vert(v + (size_t)st * i, st, px, py, pz);
    T val = px * lx + py * ly + pz * lz;
#if defined(HSR_SCAN_NOISE) && !defined(__CUDA_ARCH__)
    // ORACLE-SIDE ONLY (oracle/cpu_port.cpp): relative noise of the size of an fp32 rounding error on the scanned
    // support values, to find the states whose result depends on how a near-tie between hull vertices is rounded
    // (tests/golden/make_golden.py `sensitive`)
    if (hsr_scan_noise_seed) {
      hsr_scan_noise_seed = hsr_scan_noise_seed * 6364136223846793005ull + 1442695040888963407ull;
      val += (T)(fabs((double)val) * 2.4e-7 * ((double)(hsr_scan_noise_seed >> 40) / 16777216.0 - 0.5));
    }
#endif
    if (val > best) bi = i;
    second = fmax(second, fmin(best, val));
    best = fmax(best, val);
  }
  T gbest = best;
  int gbi = bi;
  g.argmax(gbest, gbi);
  const T cut = gbest - scan_slack(gbest);
  const unsigned involved = g.ballot(best >= cut);            // lanes holding a candidate
  const unsigned multi = g.ballot(second >= cut);             // lanes holding more than one
  if (multi == 0 && (involved & (involved - 1)) == 0) return gbi;
  if (multi == 0) {
    // tie between vertices of different lanes, one candidate per lane (the usual tie: a face of the hull): the lanes'
    // best vertices in double, lowest index within HSR_SUPPORT_TIE of the maximum
    double dv = -DBL_MAX;
    if (best >= cut) {
      T px, py, pz;
      load_vert(v + (size_t)st * bi, st, px, py, pz);
      dv = dot3_exact((double)px, (double)py, (double)pz, dl.x, dl.y, dl.z);
    }
    const double dmax = g.max(dv);
    return g.min(dv >= dmax - HSR_SUPPORT_TIE ? bi : 0x7fffffff);
  }
  // some lane holds several candidates: re-scan, candidates in double
  double dbest = -DBL_MAX;
  if (best >= cut) {
    for (int i = g.lane; i < n; i += Grp::G) {
      T px, py, pz;
      load_vert(v + (size_t)st * i, st, px, py, pz);
      const T val = px * lx + py * ly + pz * lz;
      if (val >= cut) { const double d = dot3_exact((double)px, (double)py, (double)pz, dl.x, dl.y, dl.z); if (d > dbest) dbest = d; }
    }
  }
  dbest = g.max(dbest);
  int mi = 0x7fffffff;
  if (best >= cut) {
    for (int i = g.lane; i < n; i += Grp::G) {
      T px, py, pz;
      load_vert(v + (size_t)st * i, st, px, py, pz);
      const T val = px * lx + py * ly + pz * lz;
      if (val >= cut && i < mi && dot3_exact((double)px, (double)py, (double)pz, dl.x, dl.y, dl.z) >= dbest - HSR_SUPPORT_TIE) mi = i;
    }
  }
  return g.min(mi);
}

template <typename T, typename Grp>
HSR_HD V3<double> support_d(const Geom<T>& ge, V3<double> d, const Grp& g) {
  typedef double W;
  const W* R = ge.mat;
  V3<W> dl = multv(R, d), res;
  const W tie = -HSR_SUPPORT_TIE;
  if (ge.type == GEOM_BOX) {
    res = mk<W>(dl.x >= tie ? (W)ge.size[0] : -(W)ge.size[0], dl.y >= tie ? (W)ge.size[1] : -(W)ge.size[1],
                dl.z >= tie ? (W)ge.size[2] : -(W)ge.size[2]);
  } else if (ge.type == GEOM_CYLINDER) {
    W n = sqrt(dl.x * dl.x + dl.y * dl.y);
    res = mk<W>(0, 0, dl.z >= tie ? (W)ge.size[1] : -(W)ge.size[1]);
    if (n > 1e-15) { res.x = dl.x / n * (W)ge.size[0]; res.y = dl.y / n * (W)ge.size[0]; }
#if defined(__CUDACC__)
  } else if (ge.verts4) {
    const int bi = hull_argmax<float>(ge.verts4, 4, ge.nvert, dl, g);
    res = mk<W>((W)ge.verts4[4 * bi], (W)ge.verts4[4 * bi + 1], (W)ge.verts4[4 * bi + 2]);
#endif
  } else {
    const int bi = hull_argmax<T>(ge.verts, 3, ge.nvert, dl, g);
    res = mk<W>((W)ge.verts[3 * bi], (W)ge.verts[3 * bi + 1], (W)ge.verts[3 * bi + 2]);
  }
  return ge.pos + mulv(R, res);
}

// support point of the Minkowski difference g1 - g2 along d (inlined: the out-of-line part is the hull scan)
template <typename T, typename Grp>
HSR_HD void mpr_support(const Geom<T>& g1, const Geom<T>& g2, V3<double> d, const Grp& g, Sup<double>& s) {
  s.v1 = support_d(g1, d, g); s.v2 = support_d(g2, -d, g); s.v = s.v1 - s.v2;
}

// Minkowski Portal Refinement penetration query (libccd ccdMPRPenetration as used by mjc_Convex).
//
// `sep` (optional, 4 floats: direction + flag; flag 1 = direction valid, 2 = the pair was in contact, 0 = nothing
// known) caches a separating direction of the pair between calls: a
// direction d with max <a - b, d> < 0 proves the shapes disjoint, so a later call first spends one support
// evaluation on the cached direction and returns "no contact" if it still separates (same decision as the full
// query, which can only end without contact for disjoint shapes); every exit of the query that has such a
// direction in hand stores it.  Callers without temporal coherence pass nullptr.
template <typename T, typename Grp>
HSR_HD bool mpr_penetration_inl(const Geom<T>& g1, const Geom<T>& g2, GT tol, int max_iter, const Grp& g, GT& depth_,
                                V3<GT>& pdir_, V3<GT>& ppos_, float* sep = nullptr);
// out-of-line instance (one copy per group type); callers on a hot path with the geoms in registers use _inl directly
template <typename T, typename Grp>
HSR_HDN bool mpr_penetration(const Geom<T>& g1, const Geom<T>& g2, GT tol, int max_iter, const Grp& g, GT& depth_,
                             V3<GT>& pdir_, V3<GT>& ppos_, float* sep = nullptr) {
  return mpr_penetration_inl(g1, g2, tol, max_iter, g, depth_, pdir_, ppos_, sep);
}
template <typename T, typename Grp>
HSR_HD bool mpr_penetration_inl(const Geom<T>& g1, const Geom<T>& g2, GT tol, int max_iter, const Grp& g, GT& depth_,
                                V3<GT>& pdir_, V3<GT>& ppos_, float* sep) {
  typedef double W;
  auto sup = [&](V3<W> d) { Sup<W> s; mpr_support(g1, g2, d, g, s); return s; };
  auto miss = [&](V3<W> d) {   // disjoint along d: remember the direction
    if (sep && g.lane == 0) { sep[0] = (float)d.x; sep[1] = (float)d.y; sep[2] = (float)d.z; sep[3] = 1.f; }
    return false;
  };
  if (sep && sep[3] == 1.f) {
    V3<W> dc = normalized(mk<W>((W)sep[0], (W)sep[1], (W)sep[2]));
    Sup<W> sc = sup(dc);
    W dtc = dot(sc.v, dc);
    if (dtc < 0 && !is_zero(dtc)) return false;
    g.sync();
    if (g.lane == 0) sep[3] = 0.f;
  }
  auto reach_tol = [&](const Sup<W>& v1, const Sup<W>& v2, const Sup<W>& v3, const Sup<W>& v4, V3<W> d) {
    W dv4 = dot(v4.v, d);
    W d1 = dv4 - dot(v1.v, d), d2 = dv4 - dot(v2.v, d), d3 = dv4 - dot(v3.v, d);
    W mn = fmin(d1, fmin(d2, d3));
    return ccd_eq(mn, tol) || mn < tol;
  };
  auto expand = [&](const Sup<W>& v0, Sup<W>& v1, Sup<W>& v2, Sup<W>& v3, const Sup<W>& v4) {
    V3<W> v4v0 = cross(v4.v, v0.v);
    if (dot(v1.v, v4v0) > 0) {
      if (dot(v2.v, v4v0) > 0) v1 = v4; else v3 = v4;
    } else {
      if (dot(v3.v, v4v0) > 0) v2 = v4; else v1 = v4;
    }
  };
  auto finish = [&](W depth, V3<W> dir, V3<W> pos) {
    depth_ = depth; pdir_ = dir; ppos_ = pos;
    if (sep && g.lane == 0) sep[3] = 2.f;   // in contact: the next query of this pair is a long one (job ordering)
    return true;
  };
  const W eps = Lim<W>::eps();
  Sup<W> v0, v1, v2, v3, v4;
  v0.v1 = g1.pos; v0.v2 = g2.pos;
  v0.v = v0.v1 - v0.v2;
  if (fabs(v0.v.x) < eps && fabs(v0.v.y) < eps && fabs(v0.v.z) < eps) v0.v.x += eps * 10;
  V3<W> d = normalized(-v0.v);
  v1 = sup(d);
  W dt = dot(v1.v, d);
  if (is_zero(dt) || dt < 0) return dt < 0 && !is_zero(dt) ? miss(d) : false;
  d = cross(v0.v, v1.v);
  if (is_zero(dot(d, d))) {
    if (fabs(v1.v.x) < eps && fabs(v1.v.y) < eps && fabs(v1.v.z) < eps) return false;
    W dep = norm(v1.v);
    return finish(dep, v1.v * (W(1) / dep), (v1.v1 + v1.v2) * W(0.5));
  }
  d = normalized(d);
  v2 = sup(d);
  dt = dot(v2.v, d);
  if (is_zero(dt) || dt < 0) return dt < 0 && !is_zero(dt) ? miss(d) : false;
  d = normalized(cross(v1.v - v0.v, v2.v - v0.v));
  if (dot(d, v0.v) > 0) { Sup<W> t = v1; v1 = v2; v2 = t; d = -d; }
  for (int guard = 0; guard < 64; guard++) {
    v3 = sup(d);
    dt = dot(v3.v, d);
    if (is_zero(dt) || dt < 0) return dt < 0 && !is_zero(dt) ? miss(d) : false;
    bool cont = false;
    dt = dot(cross(v1.v, v3.v), v0.v);
    if (dt < 0 && !is_zero(dt)) { v2 = v3; cont = true; }
    if (!cont) {
      dt = dot(cross(v3.v, v2.v), v0.v);
      if (dt < 0 && !is_zero(dt)) { v1 = v3; cont = true; }
    }
    if (!cont) break;
    d = normalized(cross(v1.v - v0.v, v2.v - v0.v));
  }
  // refine the portal until it encapsulates the origin
  for (int guard = 0; guard < 256; guard++) {
    d = normalized(cross(v2.v - v1.v, v3.v - v1.v));
    dt = dot(d, v1.v);
    if (is_zero(dt) || dt > 0) break;
    v4 = sup(d);
    dt = dot(v4.v, d);
    if (!(is_zero(dt) || dt > 0)) return miss(d);
    if (reach_tol(v1, v2, v3, v4, d)) return false;
    expand(v0, v1, v2, v3, v4);
  }
  // find penetration
  int it = 0;
  while (true) {
    d = normalized(cross(v2.v - v1.v, v3.v - v1.v));
    v4 = sup(d);
    if (reach_tol(v1, v2, v3, v4, d) || it > max_iter) {
      V3<W> q;
      W d2 = origin_tri_dist2(v1.v, v2.v, v3.v, q);
      W dep = sqrt(d2);
      if (is_zero(dep)) return false;
      V3<W> dir = q * (W(1) / norm(q));
      W b0 = dot(cross(v1.v, v2.v), v3.v), b1 = dot(cross(v3.v, v2.v), v0.v), b2 = dot(cross(v0.v, v1.v), v3.v),
        b3 = dot(cross(v2.v, v1.v), v0.v);
      W s = b0 + b1 + b2 + b3;
      if (is_zero(s) || s < 0) {
        b0 = 0; b1 = dot(cross(v2.v, v3.v), d); b2 = dot(cross(v3.v, v1.v), d); b3 = dot(cross(v1.v, v2.v), d);
        s = b1 + b2 + b3;
      }
      W inv = W(1) / s;
      V3<W> p1 = (v0.v1 * b0 + v1.v1 * b1 + v2.v1 * b2 + v3.v1 * b3) * inv;
      V3<W> p2 = (v0.v2 * b0 + v1.v2 * b1 + v2.v2 * b2 + v3.v2 * b3) * inv;
      return finish(dep, dir, (p1 + p2) * W(0.5));
    }
    expand(v0, v1, v2, v3, v4);
    it++;
  }
}

// Box-box manifold (SAT over 15 axes, face clipping with <=8 points, or one edge-edge contact); see oracle box_box.
template <typename T, typename Grp>
HSR_HDN void box_box(const ModelT<T>& m, WS<T>& w, const Grp& g, int& ncon, int& nrow, int pair, const Geom<T>& A,
                     const Geom<T>& B) {
  const GT* R1 = A.mat; const GT* R2 = B.mat;
  const GT s1[3] = {(GT)A.size[0], (GT)A.size[1], (GT)A.size[2]}, s2[3] = {(GT)B.size[0], (GT)B.size[1], (GT)B.size[2]};
  V3<GT> p1 = A.pos, p2 = B.pos, d = p2 - p1;
  GT C[9], Q[9];
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) {
    C[3 * i + j] = dot(mcol(R1, i), mcol(R2, j)); Q[3 * i + j] = fabs(C[3 * i + j]) + GT(1e-10);
  }
  V3<GT> dl1 = multv(R1, d), dl2 = multv(R2, d);
  GT best = -FLT_MAX; int code = -1; V3<GT> n = mk<GT>(0, 0, 1);
  for (int i = 0; i < 3; i++) {
    GT dd = comp(dl1, i);
    GT sep = fabs(dd) - (s1[i] + Q[3 * i] * s2[0] + Q[3 * i + 1] * s2[1] + Q[3 * i + 2] * s2[2]);
    if (sep > 0) return;
    if (sep > best) { best = sep; code = i; n = mcol(R1, i) * (dd >= 0 ? GT(1) : GT(-1)); }
  }
  for (int i = 0; i < 3; i++) {
    GT dd = comp(dl2, i);
    GT sep = fabs(dd) - (s2[i] + Q[i] * s1[0] + Q[3 + i] * s1[1] + Q[6 + i] * s1[2]);
    if (sep > 0) return;
    if (sep > best) { best = sep; code = 3 + i; n = mcol(R2, i) * (dd >= 0 ? GT(1) : GT(-1)); }
  }
  GT ebest = -FLT_MAX; int ecode = -1; V3<GT> en = n;
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) {
    V3<GT> ax = cross(mcol(R1, i), mcol(R2, j));
    GT ln = norm(ax);
    if (ln < GT(1e-4)) continue;
    ax = ax * (GT(1) / ln);
    int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
    GT ra = s1[i1] * fabs(dot(mcol(R1, i1), ax)) + s1[i2] * fabs(dot(mcol(R1, i2), ax));
    GT rb = s2[j1] * fabs(dot(mcol(R2, j1), ax)) + s2[j2] * fabs(dot(mcol(R2, j2), ax));
    GT dd = dot(d, ax);
    GT sep = fabs(dd) - (ra + rb);
    if (sep > 0) return;
    if (sep > ebest) { ebest = sep; ecode = 6 + 3 * i + j; en = ax * (dd >= 0 ? GT(1) : GT(-1)); }
  }
  if (ecode >= 0 && GT(1.05) * ebest > best) { best = ebest; code = ecode; n = en; }
  if (code >= 6) {
    int i = (code - 6) / 3, j = (code - 6) % 3;
    V3<GT> pa = p1, pb = p2;
    for (int k = 0; k < 3; k++) {
      if (k != i) pa = pa + mcol(R1, k) * (s1[k] * (dot(mcol(R1, k), n) > 0 ? GT(1) : GT(-1)));
      if (k != j) pb = pb - mcol(R2, k) * (s2[k] * (dot(mcol(R2, k), n) > 0 ? GT(1) : GT(-1)));
    }
    V3<GT> ua = mcol(R1, i), ub = mcol(R2, j), ww = pa - pb;
    GT a_ = dot(ua, ua), b_ = dot(ua, ub), c_ = dot(ub, ub), d_ = dot(ua, ww), e_ = dot(ub, ww);
    GT den = a_ * c_ - b_ * b_;
    GT ta = (b_ * e_ - c_ * d_) / den, tb = (a_ * e_ - b_ * d_) / den;
    ta = fmin(fmax(ta, -s1[i]), s1[i]); tb = fmin(fmax(tb, -s2[j]), s2[j]);
    V3<GT> ca = pa + ua * ta, cb = pb + ub * tb;
    add_contact(m, w, g, ncon, nrow, pair, best, (ca + cb) * GT(0.5), n);
    return;
  }
  const GT *Rr, *sr, *Ri, *si; V3<GT> pr, pi, nr; int ax;
  if (code < 3) { pr = p1; Rr = R1; sr = s1; pi = p2; Ri = R2; si = s2; nr = n; ax = code; }
  else { pr = p2; Rr = R2; sr = s2; pi = p1; Ri = R1; si = s1; nr = -n; ax = code - 3; }
  V3<GT> dots = multv(Ri, nr);
  int k = 0;
  if (fabs(dots.y) > fabs(comp(dots, k))) k = 1;
  if (fabs(dots.z) > fabs(comp(dots, k))) k = 2;
  GT sgn = comp(dots, k) > 0 ? GT(-1) : GT(1);
  V3<GT> fc = pi + mcol(Ri, k) * (si[k] * sgn);
  int k1 = (k + 1) % 3, k2 = (k + 2) % 3;
  V3<GT> u = mcol(Ri, k1) * si[k1], v = mcol(Ri, k2) * si[k2];
  V3<GT> poly[16], tmp[16];
  int np = 4;
  poly[0] = fc + u + v; poly[1] = fc - u + v; poly[2] = fc - u - v; poly[3] = fc + u - v;
  int a1 = (ax + 1) % 3, a2 = (ax + 2) % 3;
  for (int side = 0; side < 4; side++) {
    int axis_id = side < 2 ? a1 : a2;
    GT sg = (side & 1) ? GT(-1) : GT(1);
    V3<GT> pn = mcol(Rr, axis_id) * sg;
    GT off = dot(pn, pr) + sr[axis_id];
    int nn = 0;
    for (int q = 0; q < np; q++) {
      V3<GT> Aq = poly[q], Bq = poly[(q + 1) % np];
      GT da = dot(pn, Aq) - off, db = dot(pn, Bq) - off;
      if (da <= 0) tmp[nn++] = Aq;
      if ((da < 0 && db > 0) || (db < 0 && da > 0)) tmp[nn++] = Aq + (Bq - Aq) * (da / (da - db));
    }
    np = nn;
    for (int q = 0; q < np; q++) poly[q] = tmp[q];
    if (np == 0) return;
  }
  GT face_off = dot(nr, pr) + sr[ax];
  int cnt = 0;
  for (int q = 0; q < np && cnt < 8; q++) {
    GT dep = face_off - dot(nr, poly[q]);
    if (dep < 0) continue;
    add_contact(m, w, g, ncon, nrow, pair, -dep, poly[q] + nr * (dep * GT(0.5)), n);
    cnt++;
  }
}

// Narrowphase of one candidate pair that passed the culls (mjc_PlaneBox / plane-convex / box-box / mjc_Convex).
template <typename T, typename Grp>
HSR_HD void narrow_pair(const ModelT<T>& m, WS<T>& w, const Grp& g, int pk, int& ncon, int& nrow, int& npflop) {
  Geom<T> A, B;
  load_geom(m, w, m.pair_geom1[pk], A);
  load_geom(m, w, m.pair_geom2[pk], B);
  int func = m.pair_func[pk];
  npflop += func == NP_PLANE_BOX ? 80 : (func == NP_PLANE_CONVEX ? 100 : (func == NP_BOX_BOX ? 500 : 5000));
  if (func == NP_PLANE_BOX) {
    V3<GT> n = mcol(A.mat, 2);
    GT dist0 = dot(B.pos - A.pos, n);
    int cnt = 0;
    for (int i = 0; i < 8 && cnt < 4; i++) {
      V3<GT> sz = mk<GT>((i & 1) ? (GT)B.size[0] : -(GT)B.size[0], (i & 2) ? (GT)B.size[1] : -(GT)B.size[1],
                         (i & 4) ? (GT)B.size[2] : -(GT)B.size[2]);
      V3<GT> vec = mulv(B.mat, sz);
      GT ld = dot(n, vec);
      if (dist0 + ld > 0 || ld > 0) continue;
      GT dist = dist0 + ld;
      add_contact(m, w, g, ncon, nrow, pk, dist, B.pos + vec - n * (dist * GT(0.5)), n);
      cnt++;
    }
  } else if (func == NP_PLANE_CONVEX) {
    V3<GT> n = mcol(A.mat, 2);
    V3<GT> p = support_d(B, -n, g);
    GT dist = dot(p - A.pos, n);
    if (dist <= 0) add_contact(m, w, g, ncon, nrow, pk, dist, p - n * (dist * GT(0.5)), n);
  } else if (func == NP_BOX_BOX) {
    box_box(m, w, g, ncon, nrow, pk, A, B);
  } else {
    GT depth; V3<GT> dir, pos;
#if !defined(HSR_COMPACT)   // shared-memory kernel: the inlined query keeps the geoms in registers (C3 +4 %)
    float* sp = nullptr;
#if defined(__CUDA_ARCH__)
    sp = w.sep + 4 * pk;       // device only: the host port stays the plain query
#endif
    if (mpr_penetration_inl(A, B, (GT)m.mpr_tolerance, m.mpr_iterations, g, depth, dir, pos, sp))
#else
    if (mpr_penetration(A, B, (GT)m.mpr_tolerance, m.mpr_iterations, g, depth, dir, pos))
#endif
      add_contact(m, w, g, ncon, nrow, pk, -depth, pos, dir);
  }
}

// Candidate pairs -> bounding sphere + conservative world-AABB cull -> narrowphase.  Returns #contacts;
// nrow is advanced by the constraint rows the contacts will occupy.
template <typename T, typename Grp>
HSR_HDC int collision(const ModelT<T>& m, WS<T>& w, const Grp& g, int& nrow) {
  int ncon = 0;
  int narrow = 0, npflop = 0;
  for (int base = 0; base < m.npair; base += Grp::G) {
    int k = base + g.lane;
    bool hit = false;
    if (k < m.npair) {
      int a = m.pair_geom1[k], b = m.pair_geom2[k];
      V3<T> dp = cvt<T>(ld3(w.gpos + 3 * b) - ld3(w.gpos + 3 * a));
      if (m.geom_type[a] == GEOM_PLANE) {
        Geom<T> P;
        load_geom(m, w, a, P);
        hit = dot(dp, cvt<T>(mcol(P.mat, 2))) <= m.geom_rbound[b];
      } else {
        T rr = m.geom_rbound[a] + m.geom_rbound[b];
        hit = dot(dp, dp) <= rr * rr;
        const T* ha = w.gaabb + 3 * a; const T* hb = w.gaabb + 3 * b;
        hit = hit && fabs(dp.x) <= ha[0] + hb[0] && fabs(dp.y) <= ha[1] + hb[1] && fabs(dp.z) <= ha[2] + hb[2];
      }
    }
    unsigned bits = g.ballot(hit);
    while (bits) {
      int l = 0;
      while (!((bits >> l) & 1u)) l++;
      bits &= bits - 1;
      narrow++;
      narrow_pair(m, w, g, base + l, ncon, nrow, npflop);
    }
  }
  if (g.lane == 0) { w.wi[WI_NARROW] += narrow; w.wi[WI_NPFLOP] = npflop; }
  return ncon;
}

// The same collision stage in two halves for the phase-locked kernel (hsrb_step_lock_kernel, 32 lanes per environment):
// the cull leaves a bit mask of the candidate pairs in w.cand; between the halves the convex-convex candidates are
// refined by ANY warp of the block (block-shared job queue) into w.jres; the second half appends the contacts in pair
// order exactly as collision() does, taking the queued pairs' results from w.jres.
template <typename T, typename Grp>
HSR_HD void collision_cull(const ModelT<T>& m, WS<T>& w, const Grp& g) {
  static_assert(Grp::G == 32 || Grp::G == 1, "one ballot = 32 candidate pairs");
  for (int base = 0; base < m.npair; base += 32) {
    unsigned bits = 0;
    for (int k0 = 0; k0 < 32; k0 += Grp::G) {
      int k = base + k0 + g.lane;
      bool hit = false;
      if (k < m.npair) {
        int a = m.pair_geom1[k], b = m.pair_geom2[k];
        V3<T> dp = cvt<T>(ld3(w.gpos + 3 * b) - ld3(w.gpos + 3 * a));
        if (m.geom_type[a] == GEOM_PLANE) {
          Geom<T> P;
          load_geom(m, w, a, P);
          hit = dot(dp, cvt<T>(mcol(P.mat, 2))) <= m.geom_rbound[b];
        } else {
          T rr = m.geom_rbound[a] + m.geom_rbound[b];
          hit = dot(dp, dp) <= rr * rr;
          const T* ha = w.gaabb + 3 * a; const T* hb = w.gaabb + 3 * b;
          hit = hit && fabs(dp.x) <= ha[0] + hb[0] && fabs(dp.y) <= ha[1] + hb[1] && fabs(dp.z) <= ha[2] + hb[2];
        }
      }
      bits |= g.ballot(hit) << k0;
    }
    if (g.lane == 0) w.cand[base >> 5] = bits;
  }
  g.sync();
}
template <typename T, typename Grp>
HSR_HD int collision_assemble(const ModelT<T>& m, WS<T>& w, const Grp& g, int& nrow) {
  int ncon = 0, narrow = 0, npflop = 0, kc = 0;
  for (int base = 0; base < m.npair; base += 32) {
    unsigned bits = w.cand[base >> 5];
    while (bits) {
      int l = 0;
      while (!((bits >> l) & 1u)) l++;
      bits &= bits - 1;
      const int pk = base + l;
      narrow++;
      if (m.pair_func[pk] == NP_CONVEX_CONVEX && kc < HSR_MAXJOBS) {
        const GT* r = w.jres + 8 * kc;
        kc++;
        npflop += 5000;
        if (r[0] != 0) add_contact(m, w, g, ncon, nrow, pk, -r[1], mk<GT>(r[5], r[6], r[7]), mk<GT>(r[2], r[3], r[4]));
      } else {
        if (m.pair_func[pk] == NP_CONVEX_CONVEX) kc++;
        narrow_pair(m, w, g, pk, ncon, nrow, npflop);
      }
    }
  }
  if (g.lane == 0) { w.wi[WI_NARROW] += narrow; w.wi[WI_NPFLOP] = npflop; }
  return ncon;
}

// ------------------------------------------------------------------------------------------------ B.4 / B.5
// Row parameters are evaluated in double and rounded once: R = (1 - imp)/imp * diag cancels three digits of imp.
template <typename T> HSR_HD GT impedance(const T* solimp, GT pos) {
  const GT MINIMP = 1e-4, MAXIMP = 0.9999;
  GT d0 = fmin(fmax((GT)solimp[0], MINIMP), MAXIMP), dmax = fmin(fmax((GT)solimp[1], MINIMP), MAXIMP);
  GT width = fmax(GT(1e-15), (GT)solimp[2]), mid = fmin(fmax((GT)solimp[3], MINIMP), MAXIMP), power = fmax(GT(1), (GT)solimp[4]);
  if (d0 == dmax || width <= GT(1e-15)) return GT(0.5) * (d0 + dmax);
  GT x = fabs(pos) / width;
  if (x >= 1) return dmax;
  if (x == 0) return d0;
  GT y;
  if (power == 1) y = x;
  else if (x <= mid) y = (GT(1) / pow(mid, power - 1)) * pow(x, power);
  else y = GT(1) - (GT(1) / pow(1 - mid, power - 1)) * pow(1 - x, power);
  return d0 + y * (dmax - d0);
}

// reference acceleration + regulariser of one scalar row
template <typename T>
HSR_HDC void row_params(const ModelT<T>& m, const T* solref, const T* solimp, T pos_, T vel, T diag, bool friction_row,
                       GT& R, T& aref) {
  GT pos = (GT)pos_;
  GT tc = fmax((GT)solref[0], 2 * (GT)m.timestep), dr = (GT)solref[1];
  GT dmax = fmin(fmax((GT)solimp[1], GT(1e-4)), GT(0.9999));
  GT imp = impedance(solimp, pos);
  R = fmax(GT(1e-15), (1 - imp) / imp * (GT)diag);
  GT k = friction_row ? GT(0) : GT(1) / (dmax * dmax * tc * tc * dr * dr);
  GT b = GT(2) / (dmax * tc);
  aref = (T)(-b * (GT)vel - k * imp * pos);
}

// rows: active joint limits (joint order) then contacts (elliptic, dim rows each)
template <typename T, typename Grp, typename Sc = NoScale>
HSR_HDC void make_constraint(const ModelT<T>& m, WS<T>& w, const Grp& g, int nlimit, int ncon, const Sc& sc = Sc()) {
  int nv = m.nv;
  // limit rows (recomputed by every lane; lane 0 writes)
  if (g.lane == 0) {
    int r = 0;
    for (int j = 0; j < m.njnt; j++) {
      if (!m.jnt_limited[j] || m.jnt_type[j] == JNT_FREE) continue;
      T q = w.qpos[m.jnt_qposadr[j]];
      int dof = m.jnt_dofadr[j];
      for (int side = 0; side < 2; side++) {
        T dist = side == 0 ? q - m.jnt_range[2 * j] : m.jnt_range[2 * j + 1] - q;
        if (dist < 0) {
          T sg = side == 0 ? T(1) : T(-1);
          for (int d = 0; d < nv; d++) w.J[r * nv + d] = (d == dof) ? sg : T(0);
          GT R; T aref;
          row_params(m, m.jnt_solref + 2 * j, m.jnt_solimp + 5 * j, dist, sg * w.qvel[dof], m.dof_invweight0[dof], false, R, aref);
          w.D[r] = (T)(GT(1) / R); w.aref[r] = aref;
          r++;
        }
      }
    }
  }
  // contact Jacobians: dof columns across lanes
  for (int c = 0; c < ncon; c++) {
    int pk = w.con_pair[c];
    int dim = m.pair_condim[pk], r0 = w.con_adr[c];
    uint32_t m1 = m.body_dofmask[m.geom_body[m.pair_geom1[pk]]], m2 = m.body_dofmask[m.geom_body[m.pair_geom2[pk]]];
    V3<GT> p = ldg(w.con_pos + 3 * c);
    const T* fr = w.con_frame + 9 * c;
    for (int d = g.lane; d < nv; d += Grp::G) {
      T sg = T((m2 >> d) & 1u) - T((m1 >> d) & 1u);
      const T* cd = w.cdof + 6 * d;
      V3<T> jr = ld3(cd) * sg;
      V3<T> rel = cvt<T>(p - ld3(w.com + 3 * m.dof_body[d]));  // contact point relative to the dof's tree CoM
      V3<T> jp = (ld3(cd + 3) + cross(ld3(cd), rel)) * sg;
      for (int r = 0; r < dim; r++)
        w.J[(r0 + r) * nv + d] = r < 3 ? dot(ld3(fr + 3 * r), jp) : dot(ld3(fr + 3 * (r - 3)), jr);
    }
  }
  g.sync();
  // per-contact row parameters: one contact per lane
  for (int c = g.lane; c < ncon; c += Grp::G) {
    int pk = w.con_pair[c];
    int dim = m.pair_condim[pk], r0 = w.con_adr[c];
    T fbuf[5];
    const T* fri = sc.friction(m.pair_friction + 5 * pk, fbuf);
    T diag = m.geom_invweight[m.pair_geom1[pk]] + m.geom_invweight[m.pair_geom2[pk]];
    GT R0 = 0;
    for (int r = 0; r < dim; r++) {
      T vel = 0;
      for (int d = 0; d < nv; d++) vel += w.J[(r0 + r) * nv + d] * w.qvel[d];
      GT R; T aref;
      row_params(m, m.pair_solref + 2 * pk, m.pair_solimp + 5 * pk, r == 0 ? w.con_dist[c] : T(0), vel, diag, r > 0, R, aref);
      if (r == 0) R0 = R;
      else if (r == 1) R = R0 / (GT)m.impratio;
      else R = (R0 / (GT)m.impratio) * (GT)fri[0] * (GT)fri[0] / ((GT)fri[r - 1] * (GT)fri[r - 1]);
      w.D[r0 + r] = (T)(GT(1) / R); w.aref[r0 + r] = aref;
    }
    w.con_mu[c] = dim > 1 ? (T)((GT)fri[0] * sqrt((R0 / (GT)m.impratio) / R0)) : fri[0];
  }
  (void)nlimit;
}

// ------------------------------------------------------------------------------------------------ B.7 solver
// zone of an elliptic contact given jar rows x: 0 top (no force), 1 bottom (quadratic), 2 middle (cone)
template <typename T>
HSR_HD int cone_zone(const T* x, int dim, T mu, const T* fri, T& N, T& Tn) {
  N = x[0] * mu;
  T tt = 0;
  for (int j = 1; j < dim; j++) { T u = x[j] * fri[j - 1]; tt += u * u; }
  Tn = sqrt(tt);
  if (N >= mu * Tn || (Tn <= 0 && N >= 0)) return 0;
  if (mu * N + Tn <= 0 || (Tn <= 0 && N < 0)) return 1;
  return 2;
}

// constraint cost of the current w.jar (rows across lanes / one contact per lane).  full: also the forces and the pieces
// of the Hessian J^T (cone Hessians) J as a sum of weighted outer products of Jacobian rows (no ne x nv matrix W):
//   quadratic zone / active limit:  sum_r D_r J_r J_r^T                                            -> w.wrow
//   cone zone (U_a = jar_a s_a, u = U / T, s_0 = mu, s_a = fri_a-1, k = mu (N - mu T) / T):
//       Dm (p p^T + k q q^T) - Dm k sum_{a>=1} s_a^2 J_a J_a^T,  p = mu J_0 - mu sum_{a>=1} u_a s_a J_a,  q = sum_{a>=1} u_a s_a J_a
//   i.e. the 6x6 cone block Dm S (v v^T - k (I_t - u u^T)) S of the row formulation, v = e_0 - mu u, never formed.
template <typename T, typename Grp, typename Sc = NoScale>
HSR_HDC T constraint_update(const ModelT<T>& m, WS<T>& w, const Grp& g, int nlimit, int ncon, bool full, const Sc& sc = Sc()) {
  int nv = m.nv;
  T cost = 0;
  for (int i = g.lane; i < nlimit; i += Grp::G) {
    T x = w.jar[i];
    bool act = x < 0;
    if (act) cost += T(0.5) * w.D[i] * x * x;
    if (full) {
      w.force[i] = act ? -w.D[i] * x : T(0);
      w.wrow[i] = act ? w.D[i] : T(0);
    }
  }
  for (int c = g.lane; c < ncon; c += Grp::G) {
    int pk = w.con_pair[c];
    int dim = m.pair_condim[pk], r0 = w.con_adr[c];
    T fbuf[5];
    const T* fri = sc.friction(m.pair_friction + 5 * pk, fbuf);
    T mu = w.con_mu[c];
    const T* x = w.jar + r0;
    T N, Tn;
    int zone;
    if (dim == 1) { zone = x[0] < 0 ? 1 : 0; N = x[0]; Tn = 0; }
    else zone = cone_zone(x, dim, mu, fri, N, Tn);
    if (full) { w.con_zone[c] = zone; w.wpq[2 * c] = 0; w.wpq[2 * c + 1] = 0; }
    if (zone == 0) {
      if (full) for (int r = 0; r < dim; r++) { w.force[r0 + r] = 0; w.wrow[r0 + r] = 0; }
    } else if (zone == 1) {
      for (int r = 0; r < dim; r++) {
        T D = w.D[r0 + r];
        cost += T(0.5) * D * x[r] * x[r];
        if (full) { w.force[r0 + r] = -D * x[r]; w.wrow[r0 + r] = D; }
      }
    } else {
      T Dm = w.D[r0] / (mu * mu * (1 + mu * mu));
      T NT = N - mu * Tn;
      cost += T(0.5) * Dm * NT * NT;
      if (full) {
        T f0 = -Dm * NT * mu;
        w.force[r0] = f0;
        T invT = T(1) / Tn;
        T kap = mu * NT * invT;
        T cq[6];
        w.wrow[r0] = 0;
        for (int j = 1; j < dim; j++) {
          T sa = fri[j - 1];
          T U = x[j] * sa;
          w.force[r0 + j] = -f0 * invT * U * sa;
          cq[j] = U * invT * sa;
          w.wrow[r0 + j] = -Dm * kap * sa * sa;
        }
        T* P = w.PQ + (size_t)2 * c * nv;
        T* Qv = P + nv;
        for (int d = 0; d < nv; d++) {
          T q = 0;
          for (int j = 1; j < dim; j++) q += cq[j] * w.J[(r0 + j) * nv + d];
          Qv[d] = q;
          P[d] = mu * w.J[r0 * nv + d] - mu * q;
        }
        w.wpq[2 * c] = Dm; w.wpq[2 * c + 1] = Dm * kap;
      }
    }
  }
  return g.sum(cost);
}

// jar = J x - aref (rows across lanes), Ma = M x (dofs across lanes); returns the Gauss term
template <typename T, typename Grp>
HSR_HDC T residuals(const ModelT<T>& m, WS<T>& w, const Grp& g, const T* x, int nefc) {
  int nv = m.nv;
  for (int r = g.lane; r < nefc; r += Grp::G) {
    T s = -w.aref[r];
    for (int d = 0; d < nv; d++) s += w.J[r * nv + d] * x[d];
    w.jar[r] = s;
  }
  T gauss = 0;
  for (int i = g.lane; i < nv; i += Grp::G) {
    T s = 0;
    for (int d = 0; d < nv; d++) s += w.M[i * nv + d] * x[d];
    w.Ma[i] = s;
    gauss += T(0.5) * (s - w.qfrc_smooth[i]) * (x[i] - w.qacc_smooth[i]);
  }
  return g.sum(gauss);
}

template <typename T, typename Grp>
HSR_HDC void ls_eval(const ModelT<T>& m, const WS<T>& w, const Grp& g, int nlimit, int ncon, T alpha, T q1, T q2, T& c,
                    T& d1, T& d2) {
  T lc = 0, l1 = 0, l2 = 0;
  for (int i = g.lane; i < nlimit; i += Grp::G) {
    T x = w.jar[i] + alpha * w.jv[i];
    if (x < 0) { T D = w.D[i]; lc += T(0.5) * D * x * x; l1 += D * x * w.jv[i]; l2 += D * w.jv[i] * w.jv[i]; }
  }
  for (int cc = g.lane; cc < ncon; cc += Grp::G) {
    const T* q = w.lsq + HSR_LSQ * cc;
    // q: U0 V0 UU UV VV  Q0 Q1 Q2  mu Dm
    T mu = q[8];
    T N = q[0] + alpha * q[1];
    T tsq = q[2] + alpha * (2 * q[3] + alpha * q[4]);
    T Tn = tsq > 0 ? sqrt(tsq) : T(0);
    bool top = (N >= mu * Tn) || (Tn <= 0 && N >= 0);
    bool bottom = (mu * N + Tn <= 0) || (Tn <= 0 && N < 0);
    if (q[9] < 0) { top = !(N < 0); bottom = N < 0; }  // dim-1 contact: plain unilateral row
    if (top) continue;
    if (bottom) {
      lc += q[5] + alpha * (q[6] + alpha * q[7]); l1 += q[6] + 2 * alpha * q[7]; l2 += 2 * q[7];
      continue;
    }
    T Dm = q[9];
    T NT = N - mu * Tn;
    T N1 = q[1];
    T T1 = (q[3] + alpha * q[4]) / Tn;
    T T2 = q[4] / Tn - T1 * T1 / Tn;
    lc += T(0.5) * Dm * NT * NT;
    l1 += Dm * NT * (N1 - mu * T1);
    l2 += Dm * ((N1 - mu * T1) * (N1 - mu * T1) - NT * mu * T2);
  }
  c = g.sum(lc) + alpha * q1 + alpha * alpha * q2;
  d1 = g.sum(l1) + q1 + 2 * alpha * q2;
  d2 = g.sum(l2) + 2 * q2;
}

// exact line search along w.search (safeguarded Newton on the 1-D derivative with bracketing)
template <typename T, typename Grp, typename Sc = NoScale>
HSR_HDC T linesearch(const ModelT<T>& m, WS<T>& w, const Grp& g, int nlimit, int ncon, T gtol, const Sc& sc = Sc()) {
  int nv = m.nv;
  T a1 = 0, a2 = 0;
  for (int i = g.lane; i < nv; i += Grp::G) {
    a1 += w.search[i] * (w.Ma[i] - w.qfrc_smooth[i]);
    a2 += T(0.5) * w.search[i] * w.Mv[i];
  }
  T q1 = g.sum(a1), q2 = g.sum(a2);
  for (int c = g.lane; c < ncon; c += Grp::G) {
    int pk = w.con_pair[c];
    int dim = m.pair_condim[pk], r0 = w.con_adr[c];
    T fbuf[5];
    const T* fri = sc.friction(m.pair_friction + 5 * pk, fbuf);
    T mu = w.con_mu[c];
    T* q = w.lsq + HSR_LSQ * c;
    T uu = 0, uv = 0, vv = 0, Q0 = 0, Q1 = 0, Q2 = 0;
    for (int r = 0; r < dim; r++) {
      T x = w.jar[r0 + r], v = w.jv[r0 + r], D = w.D[r0 + r];
      Q0 += T(0.5) * D * x * x; Q1 += D * x * v; Q2 += T(0.5) * D * v * v;
      if (r > 0) { T u = x * fri[r - 1], s = v * fri[r - 1]; uu += u * u; uv += u * s; vv += s * s; }
    }
    if (dim == 1) { q[0] = w.jar[r0]; q[1] = w.jv[r0]; q[8] = 1; q[9] = -1; }
    else { q[0] = w.jar[r0] * mu; q[1] = w.jv[r0] * mu; q[8] = mu; q[9] = w.D[r0] / (mu * mu * (1 + mu * mu)); }
    q[2] = uu; q[3] = uv; q[4] = vv; q[5] = Q0; q[6] = Q1; q[7] = Q2;
  }
  g.sync();
  // Root of the 1-D derivative by safeguarded Newton with bracketing.  The cost is convex along the search
  // direction, so only the derivative is consulted: comparing cost values (a difference of O(1e3) numbers that
  // agree to 7 digits near convergence) is rounding noise in fp32 and used to end the solve one iteration early.
  T c0, d1, d2;
  ls_eval(m, w, g, nlimit, ncon, T(0), q1, q2, c0, d1, d2);
  int nev = 1;
  T lo = 0, hi = -1, dlo = d1, dhi = 0, alpha = 0;
  const T rel = sqrt(Lim<T>::eps());
  bool conv = fabs(d1) < gtol;
  for (int it = 0; it < m.ls_iterations && !conv; it++) {
    T step = d2 > Lim<T>::minval() ? -d1 / d2 : (d1 < 0 ? T(1) : T(-1));
    T nxt = alpha + step;
    if (hi >= 0 && !(lo < nxt && nxt < hi)) nxt = T(0.5) * (lo + hi);
    if (nxt <= 0 && hi < 0) nxt = alpha * T(0.5);
    if (nxt == alpha) break;
    bool tiny = fabs(nxt - alpha) <= rel * fabs(nxt);
    alpha = nxt;
    T c;
    ls_eval(m, w, g, nlimit, ncon, alpha, q1, q2, c, d1, d2);
    nev++;
    if (d1 < 0) { if (alpha > lo) { lo = alpha; dlo = d1; } }
    else if (hi < 0 || alpha < hi) { hi = alpha; dhi = d1; }
    conv = fabs(d1) < gtol || tiny;
  }
  if (g.lane == 0) w.wi[WI_LSEVAL] += nev;
  if (conv) return alpha;
  // not converged within ls_iterations: the bracket end with the smaller |derivative| (lo = 0 means no descent)
  if (hi >= 0 && (lo <= 0 || fabs(dhi) < fabs(dlo))) return lo > 0 || fabs(dhi) < fabs(dlo) ? hi : T(0);
  return lo;
}

// Newton solver on the primal convex cost; on exit w.qacc, w.force (and w.tmpv = J^T force) are final.
// The Newton solver in three pieces, so that a kernel whose warps lock-step through the passes (hsrb_step_lock_kernel: one
// block vote per pass keeps every warp of the block in the same code region) can drive the loop itself:
//   newton_begin (warm start, cost of the starting point) -> while (newton_pass) -> newton_end (J^T f, counters).
template <typename T> struct NewtonState { T cost, scale; int it; };
template <typename T, typename Grp, typename Sc = NoScale>
HSR_HDC bool newton_begin(const ModelT<T>& m, WS<T>& w, const Grp& g, int nlimit, int ncon, int nefc, NewtonState<T>& ns,
                          const Sc& sc = Sc()) {
  int nv = m.nv;
  ns.it = 0; ns.cost = 0; ns.scale = T(1) / (m.meaninertia * T(nv > 1 ? nv : 1));
  if (nefc == 0) {
    for (int i = g.lane; i < nv; i += Grp::G) { w.qacc[i] = w.qacc_smooth[i]; w.tmpv[i] = 0; }
    g.sync();
    return false;
  }
  // warm start: lower cost of qacc_warmstart / qacc_smooth
  T gw = residuals(m, w, g, w.warm, nefc);
  g.sync();
  T cw = constraint_update(m, w, g, nlimit, ncon, false, sc) + gw;
  g.sync();
  T gs = residuals(m, w, g, w.qacc_smooth, nefc);
  g.sync();
  T cs = constraint_update(m, w, g, nlimit, ncon, false, sc) + gs;
  bool use_warm = cw <= cs;
  for (int i = g.lane; i < nv; i += Grp::G) w.qacc[i] = use_warm ? w.warm[i] : w.qacc_smooth[i];
  g.sync();
  T gauss = use_warm ? residuals(m, w, g, w.qacc, nefc) : gs;
  g.sync();
  ns.cost = constraint_update(m, w, g, nlimit, ncon, true, sc) + gauss;
  g.sync();
  return true;
}
// one pass: gradient, convergence tests, Hessian, Newton direction, line search, update; false = the solver has stopped
template <typename T, typename Grp, typename Sc = NoScale>
HSR_HDC bool newton_pass(const ModelT<T>& m, WS<T>& w, const Grp& g, int nlimit, int ncon, int nefc, NewtonState<T>& ns,
                         const Sc& sc = Sc()) {
  const int nv = m.nv;
  const T scale = ns.scale;
  {
    // gradient (dofs across lanes) and Hessian H = M + J^T W (lower triangle entries across lanes)
    T gn = 0;
    for (int i = g.lane; i < nv; i += Grp::G) {
      T s = w.Ma[i] - w.qfrc_smooth[i];
      for (int r = 0; r < nefc; r++) s -= w.J[r * nv + i] * w.force[r];
      w.grad[i] = s; gn += s * s;
    }
    gn = sqrt(g.sum(gn));
    if (ns.it > 0 && scale * gn < m.tolerance) return false;
    if (ns.it >= m.iterations) return false;
    int ntri = nv * (nv + 1) / 2;
    for (int e = g.lane; e < ntri; e += Grp::G) {
      int a = 0, rem = e;
      while (rem > a) { rem -= a + 1; a++; }
      int b = rem;  // a >= b
      T s = w.M[a * nv + b];
      for (int r = 0; r < nefc; r++) {
        const T wr = w.wrow[r];
        if (wr != 0) s += wr * w.J[r * nv + a] * w.J[r * nv + b];
      }
      for (int c = 0; c < ncon; c++) {
        const T wp = w.wpq[2 * c];
        if (wp != 0) {
          const T* P = w.PQ + (size_t)2 * c * nv;
          s += wp * P[a] * P[b] + w.wpq[2 * c + 1] * P[nv + a] * P[nv + b];
        }
      }
      w.H[a * nv + b] = s;
    }
    for (int i = g.lane; i < nv; i += Grp::G) w.search[i] = -w.grad[i];
    g.sync();
    if (!chol_factor_g(w.H, nv, w.invd, g) && g.lane == 0) w.wi[WI_FLAGS] |= FLAG_CHOL;
    chol_solve_g(w.H, nv, w.invd, w.search, g);
    T sn = 0, dec = 0;
    for (int i = g.lane; i < nv; i += Grp::G) { sn += w.search[i] * w.search[i]; dec -= w.grad[i] * w.search[i]; }
    sn = sqrt(g.sum(sn));
    dec = g.sum(dec);  // Newton decrement^2 = grad^T H^-1 grad
    if (sn < Lim<T>::minval()) return false;
    for (int i = g.lane; i < nv; i += Grp::G) {
      T s = 0;
      for (int d = 0; d < nv; d++) s += w.M[i * nv + d] * w.search[d];
      w.Mv[i] = s;
    }
    for (int r = g.lane; r < nefc; r += Grp::G) {
      T s = 0;
      for (int d = 0; d < nv; d++) s += w.J[r * nv + d] * w.search[d];
      w.jv[r] = s;
    }
    g.sync();
    T gtol = m.tolerance * m.ls_tolerance * sn / scale;
    T alpha = linesearch(m, w, g, nlimit, ncon, gtol, sc);
    if (alpha == 0) return false;
    T gsum = 0;
    for (int i = g.lane; i < nv; i += Grp::G) {
      w.qacc[i] += alpha * w.search[i]; w.Ma[i] += alpha * w.Mv[i];
      gsum += T(0.5) * (w.Ma[i] - w.qfrc_smooth[i]) * (w.qacc[i] - w.qacc_smooth[i]);
    }
    for (int r = g.lane; r < nefc; r += Grp::G) w.jar[r] += alpha * w.jv[r];
    gsum = g.sum(gsum);
    g.sync();
    T old = ns.cost;
    ns.cost = constraint_update(m, w, g, nlimit, ncon, true, sc) + gsum;
    g.sync();
    ns.it++;
    // improvement of this step.  The reference tests old - cost; in fp32 that difference of two large numbers
    // is rounding noise near convergence, so the quadratic-model prediction alpha (1 - alpha/2) grad^T H^-1 grad
    // is used instead (equal to old - cost to second order, free of cancellation); the measured difference is
    // kept only where the model does not apply (alpha >= 2).
    T improvement = alpha < T(2) ? alpha * (T(1) - T(0.5) * alpha) * dec : old - ns.cost;
    if (scale * improvement < m.tolerance) return false;
  }
  return true;
}
template <typename T, typename Grp>
HSR_HDC void newton_end(const ModelT<T>& m, WS<T>& w, const Grp& g, int nefc, const NewtonState<T>& ns) {
  const int nv = m.nv;
  for (int i = g.lane; i < nv; i += Grp::G) {
    T s = 0;
    for (int r = 0; r < nefc; r++) s += w.J[r * nv + i] * w.force[r];
    w.tmpv[i] = s;
  }
  if (g.lane == 0) w.wi[WI_ITER] += ns.it;
  g.sync();
}
template <typename T, typename Grp, typename Sc = NoScale>
HSR_HDC void solve_newton(const ModelT<T>& m, WS<T>& w, const Grp& g, int nlimit, int ncon, int nefc, const Sc& sc = Sc()) {
  NewtonState<T> ns;
  if (!newton_begin(m, w, g, nlimit, ncon, nefc, ns, sc)) return;
  while (newton_pass(m, w, g, nlimit, ncon, nefc, ns, sc)) {}
  newton_end(m, w, g, nefc, ns);
}

// ------------------------------------------------------------------------------------------------ B.8 Euler
// qacc_int = (M + dt*diag(damping))^-1 (qfrc_smooth + qfrc_constraint) -> w.grad, rows across the lanes of the group
template <typename T, typename Grp, typename Sc = NoScale>
HSR_HD void euler_solve(const ModelT<T>& m, WS<T>& w, const Grp& g, const Sc& sc = Sc()) {
  const int nv = m.nv;
  const T dt = m.timestep;
  T* x = w.grad;  // scratch
  if (m.any_damping) {
    for (int k = g.lane; k < nv * nv; k += Grp::G) { const int i = k / nv; w.H[k] = w.M[k] + ((k - i * nv == i) ? dt * sc.damping(m.dof_damping[i]) : T(0)); }
    for (int i = g.lane; i < nv; i += Grp::G) x[i] = w.qfrc_smooth[i] + w.tmpv[i];
    g.sync();
    if (!chol_factor_g(w.H, nv, w.invd, g) && g.lane == 0) w.wi[WI_FLAGS] |= FLAG_CHOL;
    chol_solve_g(w.H, nv, w.invd, x, g);
  } else {
    for (int i = g.lane; i < nv; i += Grp::G) x[i] = w.qacc[i];
    g.sync();
  }
}
// lane 0: semi-implicit Euler with the accelerations of euler_solve
template <typename T>
HSR_HDC void euler_lane0(const ModelT<T>& m, WS<T>& w) {
  int nv = m.nv;
  T dt = m.timestep;
  T* x = w.grad;
  bool bad = false;
  for (int i = 0; i < nv; i++) {
    w.warm[i] = w.qacc[i];
    w.qvel[i] += dt * x[i];
    if (!(fabs(w.qvel[i]) < T(1e6))) bad = true;
  }
  for (int j = 0; j < m.njnt; j++) {
    int a = m.jnt_qposadr[j], v = m.jnt_dofadr[j];
    if (m.jnt_type[j] == JNT_FREE) {
      for (int k = 0; k < 3; k++) w.qpos[a + k] += dt * w.qvel[v + k];
      V3<T> om = ld3(w.qvel + v + 3);
      T ang = norm(om);
      quatnormalize(w.qpos + a + 3);
      if (ang * dt > Lim<T>::minval()) {
        T h = T(0.5) * ang * dt, s = sin(h) / ang;
        T dq[4] = {cos(h), s * om.x, s * om.y, s * om.z};
        quatmul(w.qpos + a + 3, dq, w.qpos + a + 3);
      }
      quatnormalize(w.qpos + a + 3);
    } else {
      w.qpos[a] += dt * w.qvel[v];
    }
  }
  if (bad) w.wi[WI_FLAGS] |= FLAG_BAD_NUM;
}

// ------------------------------------------------------------------------------------------------ one substep
// Algorithmic flop count of one substep: the stage formulas of SURVEY.md §8(d) evaluated with the substep's actual
// contact / row / iteration / line-search counts (what bench.py's FP32 roofline numerator is made of).
template <typename T>
HSR_HD bool model_articulated(const ModelT<T>& m) {  // any joint other than world-attached slides / free joints => M varies with qpos
  bool articulated = false;
  for (int j = 0; j < m.njnt; j++)
    if (m.jnt_type[j] == JNT_HINGE || m.body_parent[m.jnt_body[j]] > 0) articulated = true;
  return articulated;
}
template <typename T>
HSR_HD int algorithmic_flops(const ModelT<T>& m, bool articulated, int nc, int ne, int it, int ls, int npflop) {
  int nv = m.nv, nb = m.nbody - 1, nfree = m.nblock;
  int f = 100 * nb + 60 * m.ngeom;                                   // FK + geom frames
  if (articulated) f += 60 * nb + 20 * nv + nv * nv * nv / 3;          // CRB + factorisation
  f += 9 * m.npair + npflop;                                           // broadphase + narrowphase
  f += 150 * nc + 2 * ne * nv + 60 * nc;                               // contact frames, Jacobian, row parameters
  f += 10 * nv + (articulated ? 150 * nb : 0);                         // passive + bias + actuation + qacc_smooth
  if (ne > 0) {
    f += 2 * (2 * ne * nv + 50 * nc + 4 * nv);                         // warm-start cost comparison
    int its = it > 0 ? it : 1;
    f += its * (50 * nc + ne * nv * nv + nv * nv * nv / 3 + 2 * ne * nv + 2 * nv * nv + 2 * ne * nv + 6 * ne);
    f += ls * 70 * nc;                                                 // line-search evaluations
  }
  f += 6 * nv + 60 * nfree + 10;                                       // Euler, quaternion integration, goal test
  return f;
}
template <typename T>
HSR_HDC int algorithmic_flops(const ModelT<T>& m, int nc, int ne, int it, int ls, int npflop) {
  return algorithmic_flops(m, model_articulated(m), nc, ne, it, ls, npflop);
}

// mj_forward up to and including the constraint solve (sim.forward(), /root/reference/hsr/env.py:176)
template <typename T, typename Grp, typename Sc = NoScale>
HSR_HDC void forward(const ModelT<T>& m, WS<T>& w, const Grp& g, const Sc& sc = Sc()) {
  HSR_PHASE_START(w, g);
  kinematics_trig(m, w, g);
  if (g.lane == 0) kinematics_lane0(m, w, sc);
  g.sync();
  HSR_PHASE(w, g, PH_KIN);
  cdof_geoms(m, w, g);
  g.sync();
  mass_matrix(m, w, g);
  g.sync();
  HSR_PHASE(w, g, PH_CRB);
  if (g.lane == 0) smooth_lane0(m, w, sc);
  g.sync();
  smooth_solve(m, w, g);
  HSR_PHASE(w, g, PH_SMOOTH);
  // active joint limits (uniform count)
  int nlimit = 0;
  for (int j = 0; j < m.njnt; j++) {
    if (!m.jnt_limited[j] || m.jnt_type[j] == JNT_FREE) continue;
    T q = w.qpos[m.jnt_qposadr[j]];
    if (q - m.jnt_range[2 * j] < 0) nlimit++;
    if (m.jnt_range[2 * j + 1] - q < 0) nlimit++;
  }
  int nrow = nlimit;
  int ncon = collision(m, w, g, nrow);
  g.sync();
  HSR_PHASE(w, g, PH_COLLIDE);
  make_constraint(m, w, g, nlimit, ncon, sc);
  int it0 = w.wi[WI_ITER], ls0 = w.wi[WI_LSEVAL];
  g.sync();
  if (g.lane == 0) { w.wi[WI_NCON] = ncon; w.wi[WI_NEFC] = nrow; w.wi[WI_NLIMIT] = nlimit; }
  g.sync();
  HSR_PHASE(w, g, PH_ROWS);
  solve_newton(m, w, g, nlimit, ncon, nrow, sc);
  HSR_PHASE(w, g, PH_SOLVE);
  if (g.lane == 0) {
    w.wi[WI_SUMCON] += ncon; w.wi[WI_SUMEFC] += nrow;
    w.wi[WI_KFLOP] += algorithmic_flops(m, ncon, nrow, w.wi[WI_ITER] - it0, w.wi[WI_LSEVAL] - ls0, w.wi[WI_NPFLOP]);
  }
  g.sync();
}

// mj_step (sim.step(), /root/reference/hsr/env.py:123)
template <typename T, typename Grp, typename Sc = NoScale>
HSR_HD void substep(const ModelT<T>& m, WS<T>& w, const Grp& g, const Sc& sc = Sc()) {
  forward(m, w, g, sc);
  euler_solve(m, w, g, sc);
  if (g.lane == 0) euler_lane0(m, w);
  g.sync();
  HSR_PHASE(w, g, PH_EULER);
}

// all(in_range(*goal)) on the body positions of the last forward pass
// (HSREnv.step / in_range / distance_between, /root/reference/hsr/env.py:126,137-147,231-232; strict <).
// ngoal == 0: the env_wrapper form (every block within `geofence` of the goal point, SURVEY App. C #2);
// otherwise the list of GoalSpecs: endpoints are body positions, the per-environment goal point or fixed points.
template <typename T>
HSR_HD V3<GT> goal_endpoint(const EnvCfg<T>& cfg, const WS<T>& w, int code) {
  if (code >= 0) return ld3(w.xpos + 3 * code);
  if (code == GOAL_EP_POINT) return mk<GT>((GT)w.mocap[0], (GT)w.mocap[1], (GT)w.mocap[2]);
  const T* p = cfg.fixed_pt[-2 - code];
  return mk<GT>((GT)p[0], (GT)p[1], (GT)p[2]);
}
template <typename T>
HSR_HD bool goal_reached(const ModelT<T>& m, const EnvCfg<T>& cfg, const WS<T>& w) {
  if (!cfg.has_goal) return false;
  bool all = true;
  if (cfg.ngoal > 0) {
    for (int k = 0; k < cfg.ngoal; k++) {
      V3<GT> d = goal_endpoint(cfg, w, cfg.goal_a[k]) - goal_endpoint(cfg, w, cfg.goal_b[k]);
      all = all && (sqrt(dot(d, d)) < (GT)cfg.goal_dist[k]);
    }
    return all;
  }
  if (m.nblock == 0) return false;
  for (int k = 0; k < m.nblock; k++) {
    const GT* p = w.xpos + 3 * m.block_body[k];
    GT dx = p[0] - (GT)w.mocap[0], dy = p[1] - (GT)w.mocap[1], dz = p[2] - (GT)w.mocap[2];
    GT dist = sqrt(dx * dx + dy * dy + dz * dz);
    all = all && (dist < (GT)cfg.geofence);
  }
  return all;
}

// HSREnv.step inner loop (/root/reference/hsr/env.py:118-131): up to nsub substeps, goal test after every
// substep, freeze at the first success.  Returns the number of substeps executed.
template <typename T, typename Grp, typename Sc = NoScale>
HSR_HD int env_action(const ModelT<T>& m, const EnvCfg<T>& cfg, WS<T>& w, const Grp& g, int nsub, bool& success,
                      const Sc& sc = Sc()) {
  int taken = 0;
  success = false;
  for (int s = 0; s < nsub; s++) {
    substep(m, w, g, sc);
    taken++;
    if (goal_reached(m, cfg, w)) { success = true; break; }
  }
  return taken;
}

// Flat per-stage dump of the last forward pass (teacher-forced parity tests); layout mirrored in
// hsr_env_b200/debug_layout.py.  Values are converted to double.
template <typename T>
HSR_HD size_t debug_size(const ModelT<T>& m) {
  return 4 + (size_t)m.nbody * 3 + (size_t)m.nv * m.nv + 3 * (size_t)m.nv + (size_t)m.ncon_max * 14 +
         (size_t)m.nefc_max * (m.nv + 3) + (size_t)m.nq + m.nv;
}
template <typename T>
HSR_HDC void debug_dump(const ModelT<T>& m, const WS<T>& w, double* o) {
  size_t k = 0;
  int nv = m.nv;
  o[k++] = w.wi[WI_NCON]; o[k++] = w.wi[WI_NEFC]; o[k++] = w.wi[WI_NLIMIT]; o[k++] = w.wi[WI_ITER];
  for (int i = 0; i < m.nbody * 3; i++) o[k++] = (double)w.xpos[i];
  for (int i = 0; i < nv * nv; i++) o[k++] = (double)w.M[i];
  for (int i = 0; i < nv; i++) o[k++] = (double)w.qfrc_smooth[i];
  for (int i = 0; i < nv; i++) o[k++] = (double)w.qacc_smooth[i];
  for (int i = 0; i < nv; i++) o[k++] = (double)w.qacc[i];
  for (int c = 0; c < m.ncon_max; c++) {
    bool on = c < w.wi[WI_NCON];
    o[k++] = on ? (double)w.con_pair[c] : -1.0;
    o[k++] = on ? (double)w.con_dist[c] : 0.0;
    for (int i = 0; i < 3; i++) o[k++] = on ? (double)w.con_pos[3 * c + i] : 0.0;
    for (int i = 0; i < 9; i++) o[k++] = on ? (double)w.con_frame[9 * c + i] : 0.0;
  }
  for (int r = 0; r < m.nefc_max; r++) {
    bool on = r < w.wi[WI_NEFC];
    for (int d = 0; d < nv; d++) o[k++] = on ? (double)w.J[r * nv + d] : 0.0;
    o[k++] = on ? (double)w.D[r] : 0.0;
    o[k++] = on ? (double)w.aref[r] : 0.0;
    o[k++] = on ? (double)w.force[r] : 0.0;
  }
  for (int i = 0; i < m.nq; i++) o[k++] = (double)w.qpos[i];
  for (int i = 0; i < nv; i++) o[k++] = (double)w.qvel[i];
}

// ------------------------------------------------------------------------------------------------ resets
HSR_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
  for (int r = 0; r < 10; r++) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// uniform float32 in [lo, hi): lo + u*(hi-lo) with u = (x>>8)*2^-24, evaluated in fp32 without FMA contraction
HSR_HD float uniform32(uint32_t x, float lo, float hi) {
  float u = (float)(x >> 8) * (1.0f / 16777216.0f);
#if defined(__CUDA_ARCH__)
  return __fadd_rn(lo, __fmul_rn(u, __fsub_rn(hi, lo)));
#else
  volatile float span = hi - lo;
  volatile float prod = u * span;
  return lo + prod;
#endif
}

// mj_resetData + HSREnv.reset_model (/root/reference/hsr/mujoco_env.py:83-85, hsr/env.py:158-177) for one env.
// Philox4x32-10, key = (seed_lo, global env id), counter = (episode, draw block, seed_hi, 0).  lane 0 only.
template <typename T>
HSR_HDC void reset_lane0(const ModelT<T>& m, const EnvCfg<T>& cfg, WS<T>& w, uint64_t seed, uint32_t env_id,
                        uint32_t episode) {
  for (int i = 0; i < m.nq; i++) w.qpos[i] = m.qpos0[i];
  for (int i = 0; i < m.nv; i++) { w.qvel[i] = 0; w.warm[i] = 0; }
  for (int i = 0; i < m.nu; i++) w.ctrl[i] = 0;
  for (int k = 0; k < 3; k++) w.mocap[k] = m.mocap_pos0[k];
  uint32_t r[4];
  uint32_t k0 = (uint32_t)seed, k1 = env_id, c2 = (uint32_t)(seed >> 32);
  if (cfg.has_goal) {
    philox4x32_10(episode, 0, c2, 0, k0, k1, r);
    for (int k = 0; k < 3; k++) w.mocap[k] = (T)uniform32(r[k], (float)cfg.goal_lo[k], (float)cfg.goal_hi[k]);
    for (int b = 0; b < m.nblock && cfg.has_block; b++) {
      int body = m.block_body[b];
      int a = m.jnt_qposadr[m.body_jntadr[body]];
      float s[4];
      for (int tries = 0; tries < 16; tries++) {
        philox4x32_10(episode, 1 + b * 16 + tries, c2, 0, k0, k1, r);
        for (int k = 0; k < 4; k++) s[k] = uniform32(r[k], (float)cfg.block_lo[k], (float)cfg.block_hi[k]);
        bool ok = true;
        if (cfg.min_sep > 0)
          for (int o = 0; o < b; o++) {
            int ao = m.jnt_qposadr[m.body_jntadr[m.block_body[o]]];
            T dx = (T)s[0] - w.qpos[ao], dy = (T)s[1] - w.qpos[ao + 1];
            if (dx * dx + dy * dy < cfg.min_sep * cfg.min_sep) ok = false;
          }
        if (ok) break;
      }
      w.qpos[a] = (T)s[0]; w.qpos[a + 1] = (T)s[1];
      w.qpos[a + 3] = w.qpos[a + 4] = w.qpos[a + 5] = w.qpos[a + 6] = 0;
      w.qpos[a + 3 + cfg.qidx0] = (T)s[2]; w.qpos[a + 3 + cfg.qidx1] = (T)s[3];
    }
  }
  // HSREnv.new_state (/root/reference/hsr/env.py:149-156): qpos slices of the joints that have a start space,
  // draw block 4096 + 2 s + (0, 1) of the environment's stream (independent of the goal / block draws above; applied last, as new_state is)
  for (int s = 0; s < cfg.nstart; s++) {
    const int a = cfg.start_adr[s], wd = cfg.start_width[s];
    for (int k = 0; k < wd; k++) {
      if ((k & 3) == 0) philox4x32_10(episode, 4096 + 2 * s + (k >> 2), c2, 0, k0, k1, r);
      w.qpos[a + k] = (T)uniform32(r[k & 3], (float)cfg.start_lo[s][k], (float)cfg.start_hi[s][k]);
    }
  }
}

// The per-environment multipliers (PRM_*) a reset draws when the handle has parameter ranges: U[lo, hi) from draw block
// 8192 of the same stream as reset_lane0 (same key, same episode), which reset_lane0 never reads.
HSR_HD void sample_env_params(const float* lo, const float* hi, uint64_t seed, uint32_t env_id, uint32_t episode, float* out) {
  uint32_t r[4];
  philox4x32_10(episode, 8192, (uint32_t)(seed >> 32), 0, (uint32_t)seed, env_id, r);
  for (int k = 0; k < PRM_COUNT; k++) out[k] = uniform32(r[k], lo[k], hi[k]);
}

}  // namespace hsr
