// Warp-per-environment action kernel of the "sliding base + at most one free box" models (README block-push:
// --use-dof slide_x slide_y, --n-blocks 0/1; BASELINE.json configs[0], [1] and [3]).
//
// Same substep as hsrb_push.cuh / the general kernel (SURVEY.md App. B), laid out for occupancy instead of for
// register residency:
//   * ONE WARP owns one environment; a block is up to 28 independent warps (no block barrier after the table copy),
//     so every environment advances at its own pace: a substep costs its own Newton iterations and its own narrowphase
//     queries, not those of the slowest environment of a lock-stepped block (measured on the bench workload: mean 1.3
//     Newton iterations per environment-substep, 5.3 for the slowest of 32).
//   * <= 72 registers per thread (28 warps = 28 environments resident per SM, 7 per scheduler: the dependent chains
//     of one warp are hidden behind the other six instead of behind a barrier).  State, poses, contacts, constraint
//     rows, solver vectors and the portal of the convex-convex query live in the warp's 5 KB slice of shared memory;
//     registers only hold what a phase is working on.
//   * Lane roles: lane k = candidate pair k (cull), box corner k (plane-box), hull vertices k, k+32, ... (support
//     scan), constraint row r = k, k+32 (Jacobian products), constraint group k (one contact or one joint limit: cone
//     state, line-search coefficients), and dof k & 7 with row stripe k >> 3 (gradient, Hessian row, Cholesky row).
//   * Joint limits are ordinary one-row groups, rows are packed (condim rows per contact).
//
// Replaces the loop over sim.step() in HSREnv.step (/root/reference/hsr/env.py:115-135).
#pragma once
#include "hsrb_push.cuh"

#ifndef WPE_MAXCON
#define WPE_MAXCON 8                       // contacts per environment (as the lock-step kernel)
#endif
#define WPE_GROUPS (WPE_MAXCON + 2)        // constraint groups: contacts + the two slide limits
#define WPE_SLOTS (6 * WPE_GROUPS)         // six row slots per group (rows >= the group's dimension are zero rows)
#define WPE_MAXROW (6 * WPE_MAXCON + 2)    // MuJoCo's nefc at capacity
#define WPE_MAXBG 2                        // geoms riding on the block
#define WPE_MAXGEOM 24                     // capacities of the fixed shared-memory layout (c2_push: 18 geoms, 21 pairs)
#define WPE_MAXPAIR 24
#define WPE_ENVJOBS 7                      // phase-locked variant: convex-convex jobs an environment can queue per substep
#ifndef WPE_MAXWARPS
#define WPE_MAXWARPS 28
#endif

namespace wpe {

// Fixed layouts: every field sits at a compile-time offset from ONE base address, so a shared-memory access is an
// LDS / STS with an immediate offset and no table of pointers lives in registers (the first version carried ~50 of them
// and spilled through local memory on every phase).
struct alignas(16) Tab {   // block-shared model tables (one copy per block)
  double gbase[WPE_MAXGEOM * 3];
  double gmatw[WPE_MAXGEOM * 9];
  double pairc[WPE_MAXPAIR * PUSH_PAIRC];
  float ghalf[WPE_MAXGEOM * 3];
  float geom_rbound[WPE_MAXGEOM];
  float geom_size[WPE_MAXGEOM * 3];
  float pair_friction[WPE_MAXPAIR * 5];
  float bgeom_mat[WPE_MAXBG * 9];            // geom_mat (body frame) of the geoms riding on the block
  float geom_aabb[WPE_MAXGEOM * 3];
  int gmove[WPE_MAXGEOM], geom_type[WPE_MAXGEOM], geom_vertadr[WPE_MAXGEOM], geom_vertnum[WPE_MAXGEOM];
  int pair_geom1[WPE_MAXPAIR], pair_geom2[WPE_MAXPAIR], pair_func[WPE_MAXPAIR], pair_condim[WPE_MAXPAIR];
  float pair_sr[WPE_MAXPAIR], pair_sb[WPE_MAXPAIR];   // sign of the pair's contact Jacobian on the robot / block dofs
};

struct alignas(16) Slice {   // per-warp (= per-environment) slice
  double xb[4], Rb[10], bmat[9 * WPE_MAXBG], gpos[WPE_MAXGEOM * 3], portal[48], mres[8];   // portal: 5 vertices x 9 + the current direction
  float qpos[12], qvel[8], warm[8], mocap[4], ctrl[4];
  float baabb[4 * WPE_MAXBG];                                  // world AABB half extents of the block geoms (the others: Tab::ghalf)
  float qs[8], as[8], x[8], qfc[8], srch[8];
  float con_dist[WPE_MAXCON], con_pos[WPE_MAXCON * 3], con_frame[WPE_MAXCON * 9];
  int con_pair[WPE_MAXCON], con_adr[WPE_MAXCON], wi[4];
  int acc[8];                                                  // per-action counters of the environment (lane 0): registers would stay live across every call
  float jres[WPE_ENVJOBS * 14 + 2];                                // phase-locked variant: results of this environment's convex-convex jobs (hit, dist, pos, frame)
  float J[WPE_SLOTS * 8];                                       // 32-byte Jacobian rows
  float Dr[WPE_SLOTS], aref[WPE_SLOTS], rsc[WPE_SLOTS], jar[WPE_SLOTS], jv[WPE_SLOTS], f[WPE_SLOTS], wrow[WPE_SLOTS];   // per row slot (rsc: mu on row 0, friction[j-1] on row j)
  float PQ[16 * WPE_GROUPS], wpq[2 * WPE_GROUPS + 4], L[64];
  float sep[4 * WPE_MAXPAIR];
};

// phase-locked variant: block-shared queue of the convex-convex narrowphase jobs of the block's environments; long jobs
// (no cached separating direction: a full portal refinement) fill it from the front, quick ones from the back, the warps
// pop from the front
#define WPE_MAXTEAMS 4
struct alignas(16) Queue {
  int cnt[WPE_MAXTEAMS][4];                   // per team: [0] long jobs, [1] quick jobs, [2] next to serve
  int jobs[WPE_MAXWARPS * WPE_ENVJOBS];       // (owner warp << 16) | (slot << 8) | pair; team k owns a contiguous share
};

static_assert(offsetof(Slice, J) % 16 == 0 && offsetof(Slice, PQ) % 16 == 0 && offsetof(Slice, L) % 16 == 0 && offsetof(Slice, qpos) % 16 == 0 &&
              offsetof(Slice, qvel) % 16 == 0 && offsetof(Slice, qs) % 16 == 0 && offsetof(Slice, x) % 16 == 0 && offsetof(Slice, srch) % 16 == 0 &&
              offsetof(Slice, warm) % 16 == 0 && offsetof(Slice, as) % 16 == 0 && sizeof(Slice) % 16 == 0,
              "128-bit shared-memory accesses (push::ld8 / st8) need 16-byte aligned fields");
__host__ __device__ inline size_t slice_bytes() { return sizeof(Slice); }
// block-shared tail after the slices: the tables, the job queue, then the hull vertices as float4
__host__ __device__ inline size_t shared_tail(const ModelT<float>& m) { return sizeof(Tab) + sizeof(Queue) + (size_t)m.nvert * 16 + 16; }

}  // namespace wpe

// kernel + device routines: only in the translation unit that owns them (hsrb_wpe.cu, the emulated build)
#if defined(HSRB_WPE_IMPL)
namespace wpe {

typedef V3<double> V3d;

// -DWPE_CHAIN_CLOCKS: cycle counters of the sections of ONE environment's dependent chain (lane 0 of every warp, clock64
// deltas accumulated with fire-and-forget atomics); read with hsrb_debug_chain_clocks().  Meant for the free-running
// variant with one warp per SM (n = 148), where a section's cycles are its latency without contention.
#if defined(WPE_CHAIN_CLOCKS)
__device__ unsigned long long wpe_ck_cyc[32], wpe_ck_cnt[32];
#define WPE_CK_DECL long long ck_last = clock64()
#define WPE_CK_RESET() do { ck_last = clock64(); } while (0)
#define WPE_CK(id) do { if ((threadIdx.x & 31) == 0) { const long long t_ = clock64(); atomicAdd(&wpe::wpe_ck_cyc[id], (unsigned long long)(t_ - ck_last)); atomicAdd(&wpe::wpe_ck_cnt[id], 1ull); } ck_last = clock64(); } while (0)
#else
#define WPE_CK_DECL do { } while (0)
#define WPE_CK_RESET() do { } while (0)
#define WPE_CK(id) do { } while (0)
#endif

// Barriers of a TEAM of warps (phase-locked variant): the block's warps form 1, 2 or 4 teams that lock-step
// independently of each other (named barriers 1 + team), so that while one team waits for its slowest member the others
// keep the SM busy.  nthreads = warps of the team x 32.
#if defined(HSRB_SIMT_EMU)
__device__ __forceinline__ void team_sync(int team, int nthreads) { emu::named_barrier(1 + team, nthreads); }
__device__ __forceinline__ bool team_and(int team, int nthreads, bool p) { return emu::named_vote(1 + team, nthreads, p, true); }
#else
__device__ __forceinline__ void team_sync(int team, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(1 + team), "r"(nthreads) : "memory");
}
__device__ __forceinline__ bool team_and(int team, int nthreads, bool p) {
  unsigned r;
  asm volatile(
      "{\n\t.reg .pred q, r;\n\tsetp.ne.u32 q, %3, 0;\n\tbar.red.and.pred r, %1, %2, q;\n\tselp.u32 %0, 1, 0, r;\n\t}"
      : "=r"(r) : "r"(1 + team), "r"(nthreads), "r"((unsigned)p) : "memory");
  return r != 0;
}
#endif

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// world orientation of a geom: table entry (static / robot geoms) or the per-substep product for block geoms
__device__ __forceinline__ const double* geom_mat(const Tab& t, const Slice& s, int gi, int gb0) {
  return t.gmove[gi] == 2 ? s.bmat + 9 * (gi - gb0) : t.gmatw + 9 * gi;
}

#ifndef WPE_SUPPORT_ATTR
#define WPE_SUPPORT_ATTR __forceinline__   // inlined at its two call sites in mpr: no call-site spills on the refinement chain (+1-3 %)
#endif
// support point of geom gi along d (world frame); hull scan in fp32 over the 32 lanes, everything else in double
// (same arithmetic as hsr::support_d)
// (s: the slice of the environment the geom belongs to)
__device__ WPE_SUPPORT_ATTR V3d support(const Tab& t, const Slice& s, const float* verts4, int gi, int gb0, V3d d) {
  WPE_CK_DECL;
  const double* R = geom_mat(t, s, gi, gb0);
  const V3d dl = multv(R, d);
  const int type = t.geom_type[gi];
  const float* sz = t.geom_size + 3 * gi;
  V3d res;
  const double tie = -HSR_SUPPORT_TIE;   // support ties: hsr_core.h
  if (type == GEOM_BOX) {
    res = mk<double>(dl.x >= tie ? (double)sz[0] : -(double)sz[0], dl.y >= tie ? (double)sz[1] : -(double)sz[1],
                     dl.z >= tie ? (double)sz[2] : -(double)sz[2]);
  } else if (type == GEOM_CYLINDER) {
    const double n = sqrt(dl.x * dl.x + dl.y * dl.y);
    res = mk<double>(0, 0, dl.z >= tie ? (double)sz[1] : -(double)sz[1]);
    if (n > 1e-15) { res.x = dl.x / n * (double)sz[0]; res.y = dl.y / n * (double)sz[0]; }
  } else {
    const DevGrp<32> gw;
    const float* v4 = verts4 + 4 * t.geom_vertadr[gi];
    WPE_CK(22);
    const int bi = hull_argmax<float>(v4, 4, t.geom_vertnum[gi], dl, gw);
    WPE_CK(23);
    res = mk<double>((double)v4[4 * bi], (double)v4[4 * bi + 1], (double)v4[4 * bi + 2]);
  }
  const V3d out_ = ld3(s.gpos + 3 * gi) + mulv(R, res);
  WPE_CK(type == GEOM_BOX ? 25 : 24);
  return out_;
}

// portal vertex k of the warp's scratch: 9 doubles  v = v1 - v2 | v1 (on geom 1) | v2 (on geom 2)
__device__ __forceinline__ V3d pv(const Slice& s, int k) { return ld3(s.portal + 9 * k); }
__device__ __forceinline__ void pcopy(Slice& s, int dst, int src) {
  const int lane = threadIdx.x & 31;
  __syncwarp();
  if (lane < 9) s.portal[9 * dst + lane] = s.portal[9 * src + lane];
  __syncwarp();
}

// Minkowski portal refinement (libccd ccdMPRPenetration as used by mjc_Convex), the decisions and the arithmetic of
// hsr::mpr_penetration_inl, restructured around ONE support evaluation site (a state machine) with the portal in shared
// memory: a few hundred instructions of code and a handful of live doubles instead of five 9-double vertices in
// registers.  `sep`: cached separating direction of the pair (see hsr::mpr_penetration_inl).  Result -> s.mres.
// o: the slice of the environment the pair belongs to (poses, cached direction); s: the executing warp's slice (portal
// scratch, result) - the same slice unless the warp serves another environment's job (phase-locked variant).
__device__ __noinline__ bool mpr(const Tab& t, const Slice& o, Slice& s, const float* verts4, int g1, int g2, int gb0, double tol,
                                 int max_iter, float* sep) {
  double* const out7 = s.mres;   // depth, direction, position (written by lane 0)
  double* const P = s.portal;    // P[9 k ..]: portal vertex k = v | v1 | v2 (k = 0 .. 4), P[45 .. 47]: the current direction
  const int lane = threadIdx.x & 31;
  enum { S_CACHE = 0, S_V1, S_V2, S_DISCOVER, S_REFINE, S_PENETRATE };
  const double eps = DBL_EPSILON;
  int state = S_V1;
  V3d dcur;   // the current direction (loop-carried in registers: support() is inlined, there is no call to keep registers free for)
  {
    V3d v0 = ld3(o.gpos + 3 * g1) - ld3(o.gpos + 3 * g2);
    if (fabs(v0.x) < eps && fabs(v0.y) < eps && fabs(v0.z) < eps) v0.x += eps * 10;
    V3d d;
    if (sep && (sep[3] == 1.f || sep[3] < 0.f)) {
      state = S_CACHE;
      d = normalized(mk<double>((double)sep[0], (double)sep[1], (double)sep[2]));
    } else {
      d = normalized(-v0);
    }
    __syncwarp();
    if (lane == 0) { st3(P, v0); st3(P + 3, ld3(o.gpos + 3 * g1)); st3(P + 6, ld3(o.gpos + 3 * g2)); }
    __syncwarp();
    dcur = d;
  }
  int guard = 0, it = 0;
  WPE_CK_DECL;
// publish the next direction and go round again
#define WPE_NEXT_DIR() { dcur = d; WPE_CK(21); continue; }
#pragma unroll 1
  while (true) {
    // ---- the support evaluation: portal vertex 4 <- support of (g1 - g2) along the current direction.  support() is inlined:
    //      the direction and the two support points stay in registers (through shared memory and two warp barriers per
    //      iteration when support() was a call: +2 % with them in registers)
    const V3d a1 = support(t, o, verts4, g1, gb0, dcur);
    const V3d a2 = support(t, o, verts4, g2, gb0, -dcur);
    const V3d v4 = a1 - a2;
    __syncwarp();   // every lane is done with the previous contents of portal vertex 4
    if (lane == 0) { st3(P + 36, v4); st3(P + 39, a1); st3(P + 42, a2); }   // read by others only through pcopy (which synchronises first)
    WPE_CK(20);
    V3d d = dcur;
    const V3d v0 = ld3(P);
    double dt = dot(v4, d);
    bool enter_refine = false;
    if (state == S_CACHE) {
      if (dt < 0 && !is_zero(dt)) {                        // the cached direction still separates the pair, by -dt
        if (lane == 0) sep[3] = (float)(dt * 0.999);       // remaining gap along it (negative flag = valid direction with a gap budget)
        return false;
      }
      if (lane == 0) sep[3] = 0.f;
      state = S_V1;
      d = normalized(-v0);
      WPE_NEXT_DIR();
    }
    if (state <= S_DISCOVER) {
      if (is_zero(dt) || dt < 0) {                         // origin outside the support plane: disjoint (or touching)
        if (dt < 0 && !is_zero(dt) && sep && lane == 0) { sep[0] = (float)d.x; sep[1] = (float)d.y; sep[2] = (float)d.z; sep[3] = (float)(dt * 0.999); }
        return false;
      }
    }
    if (state == S_V1) {
      pcopy(s, 1, 4);
      d = cross(v0, v4);
      if (is_zero(dot(d, d))) {
        if (fabs(v4.x) < eps && fabs(v4.y) < eps && fabs(v4.z) < eps) return false;
        const double dep = norm(v4);
        const V3d dir = v4 * (1.0 / dep), pos = (a1 + a2) * 0.5;
        if (lane == 0) {
          out7[0] = dep; out7[1] = dir.x; out7[2] = dir.y; out7[3] = dir.z; out7[4] = pos.x; out7[5] = pos.y; out7[6] = pos.z;
          if (sep) sep[3] = 2.f;
        }
        __syncwarp();
        return true;
      }
      d = normalized(d);
      state = S_V2;
      WPE_NEXT_DIR();
    }
    if (state == S_V2) {
      pcopy(s, 2, 4);
      const V3d v1 = pv(s, 1);
      d = normalized(cross(v1 - v0, v4 - v0));
      if (dot(d, v0) > 0) {                                // swap v1 and v2
        pcopy(s, 2, 1); pcopy(s, 1, 4);
        d = -d;
      }
      state = S_DISCOVER; guard = 0;
      WPE_NEXT_DIR();
    }
    if (state == S_DISCOVER) {
      pcopy(s, 3, 4);
      const V3d v1 = pv(s, 1), v2 = pv(s, 2);
      bool cont = false;
      dt = dot(cross(v1, v4), v0);
      if (dt < 0 && !is_zero(dt)) { pcopy(s, 2, 3); cont = true; }
      if (!cont) {
        dt = dot(cross(v4, v2), v0);
        if (dt < 0 && !is_zero(dt)) { pcopy(s, 1, 3); cont = true; }
      }
      guard++;
      if (cont && guard < 64) {
        const V3d w1 = pv(s, 1), w2 = pv(s, 2);
        d = normalized(cross(w1 - v0, w2 - v0));
        WPE_NEXT_DIR();
      }
      state = S_REFINE; guard = 0;
      enter_refine = true;
    }
    if (state == S_REFINE && !enter_refine) {
      if (!(is_zero(dt) || dt > 0)) {                      // the new support point does not pass the origin: disjoint
        if (sep && lane == 0) { sep[0] = (float)d.x; sep[1] = (float)d.y; sep[2] = (float)d.z; sep[3] = (float)(dt * 0.999); }
        return false;
      }
    }
    if (state == S_PENETRATE || (state == S_REFINE && !enter_refine)) {
      // reach_tol + expand are common to the refinement and the penetration loop
      const V3d v1 = pv(s, 1), v2 = pv(s, 2), v3 = pv(s, 3);
      const double d1 = dt - dot(v1, d), d2 = dt - dot(v2, d), d3 = dt - dot(v3, d);
      const double mn = fmin(d1, fmin(d2, d3));
      const bool reach = ccd_eq(mn, tol) || mn < tol;
      if (state == S_REFINE) {
        if (reach) return false;
      } else if (reach || it > max_iter) {
        V3d q;
        const double dd2 = origin_tri_dist2(v1, v2, v3, q);
        const double dep = sqrt(dd2);
        if (is_zero(dep)) return false;
        const V3d dir = q * (1.0 / norm(q));
        double b0 = dot(cross(v1, v2), v3), b1 = dot(cross(v3, v2), v0), b2 = dot(cross(v0, v1), v3), b3 = dot(cross(v2, v1), v0);
        double sm = b0 + b1 + b2 + b3;
        if (is_zero(sm) || sm < 0) {
          b0 = 0; b1 = dot(cross(v2, v3), d); b2 = dot(cross(v3, v1), d); b3 = dot(cross(v1, v2), d);
          sm = b1 + b2 + b3;
        }
        const double inv = 1.0 / sm;
        const double* P = s.portal;
        const V3d p1 = (ld3(P + 3) * b0 + ld3(P + 12) * b1 + ld3(P + 21) * b2 + ld3(P + 30) * b3) * inv;
        const V3d p2 = (ld3(P + 6) * b0 + ld3(P + 15) * b1 + ld3(P + 24) * b2 + ld3(P + 33) * b3) * inv;
        const V3d pos = (p1 + p2) * 0.5;
        if (lane == 0) {
          out7[0] = dep; out7[1] = dir.x; out7[2] = dir.y; out7[3] = dir.z; out7[4] = pos.x; out7[5] = pos.y; out7[6] = pos.z;
          if (sep) sep[3] = 2.f;
        }
        __syncwarp();
        return true;
      }
      // expand the portal with v4
      const V3d v4v0 = cross(v4, v0);
      int repl;
      if (dot(v1, v4v0) > 0) repl = dot(v2, v4v0) > 0 ? 1 : 3;
      else repl = dot(v3, v4v0) > 0 ? 2 : 1;
      pcopy(s, repl, 4);
      if (state == S_REFINE) guard++; else it++;
    }
    // ---- next direction: the portal's normal
    {
      const V3d v1 = pv(s, 1), v2 = pv(s, 2), v3 = pv(s, 3);
      d = normalized(cross(v2 - v1, v3 - v1));
      if (state == S_REFINE) {
        const double dv = dot(d, v1);
        if (is_zero(dv) || dv > 0 || guard >= 256) state = S_PENETRATE;   // the portal encloses the origin ray
      }
    }
    WPE_NEXT_DIR();
  }
#undef WPE_NEXT_DIR
}

}  // namespace wpe

// ---------------------------------------------------------------------------------------------------- the kernel
// LOCK = false: free-running warps (no block barrier after the table copy).
// LOCK = true:  the same code with block barriers between the phases of a substep and around every pass of the solver loop,
//               so that the 28 warps of the block run the same few-KB code region at the same time (instruction cache) while
//               each still owns one environment; a phase then lasts as long as its slowest warp.
// per-phase cycle counters of the phase-locked variant (thread 0 of block 0, clock64 before and after each block barrier),
// compiled in only with -DHSRB_PHASE_CLOCKS.  Slots (names of hsrb_stats): kinematics = poses + limits + cull + queueing,
// mass_matrix = wait at the barrier before the job service, smooth = this warp's share of the job service, collision = wait
// for the last job, rows = contact assembly + smooth forces + constraint rows + this warp's solver passes, solver = wait
// for the slowest warp's solver, euler = goal test + integration
#if defined(HSRB_PHASE_CLOCKS)
#define WPE_PH(id) do { if (LOCK && threadIdx.x == 0) { const long long t_ = clock64(); ph[id] += (unsigned long long)(t_ - tlast) >> 4; tlast = t_; } } while (0)
#else
#define WPE_PH(id) do { } while (0)
#endif
template <bool LOCK>
__global__ void __launch_bounds__(32 * WPE_MAXWARPS, 1) hsrb_wpe_kernel_t(const __grid_constant__ KArgs a, const __grid_constant__ PushInfo fi) {
  HSRB_DYN_SMEM(smem);
  constexpr unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const ModelT<float>& m = a.m;
  // ---- block-shared: model tables + hull vertices as float4 (one copy per block), after the warps' slices
  wpe::Tab& tw = *reinterpret_cast<wpe::Tab*>(smem + (size_t)wpb * sizeof(wpe::Slice));
  wpe::Queue& Q = *reinterpret_cast<wpe::Queue*>(smem + (size_t)wpb * sizeof(wpe::Slice) + sizeof(wpe::Tab));
  float* const v4w = reinterpret_cast<float*>(smem + (size_t)wpb * sizeof(wpe::Slice) + sizeof(wpe::Tab) + sizeof(wpe::Queue));
  {
    const int ng = m.ngeom, np = m.npair;
    for (int i = threadIdx.x; i < m.nvert * 4; i += blockDim.x) v4w[i] = fi.verts4[i];
#define TAB_COPY(field, src, n) for (int i = threadIdx.x; i < (n); i += blockDim.x) tw.field[i] = (src)[i];
    TAB_COPY(gbase, fi.gbase, ng * 3) TAB_COPY(gmatw, fi.gmatw, ng * 9) TAB_COPY(pairc, fi.pairc, np * PUSH_PAIRC)
    TAB_COPY(ghalf, fi.ghalf, ng * 3) TAB_COPY(geom_rbound, m.geom_rbound, ng)
    TAB_COPY(geom_size, m.geom_size, ng * 3) TAB_COPY(pair_friction, m.pair_friction, np * 5)
    TAB_COPY(geom_aabb, m.geom_aabb, ng * 3)
    {
      int gb0_ = ng;
      for (int i = ng - 1; i >= 0; i--) if (fi.gmove[i] == 2) gb0_ = i;
      for (int i = threadIdx.x; i < (ng - gb0_) * 9 && i < WPE_MAXBG * 9; i += blockDim.x) tw.bgeom_mat[i] = m.geom_mat[9 * gb0_ + i];
    }
    TAB_COPY(gmove, fi.gmove, ng) TAB_COPY(geom_type, m.geom_type, ng)
    TAB_COPY(geom_vertadr, m.geom_vertadr, ng) TAB_COPY(geom_vertnum, m.geom_vertnum, ng)
    TAB_COPY(pair_geom1, m.pair_geom1, np) TAB_COPY(pair_geom2, m.pair_geom2, np)
    TAB_COPY(pair_func, m.pair_func, np) TAB_COPY(pair_condim, m.pair_condim, np)
#undef TAB_COPY
    for (int k = threadIdx.x; k < np; k += blockDim.x) {
      const int b1 = m.geom_body[m.pair_geom1[k]], b2 = m.geom_body[m.pair_geom2[k]];
      tw.pair_sr[k] = (float)(b2 == fi.robot_body) - (float)(b1 == fi.robot_body);
      tw.pair_sb[k] = (float)(b2 == fi.block_body) - (float)(b1 == fi.block_body);
    }
    if (threadIdx.x < 4 * WPE_MAXTEAMS) (&Q.cnt[0][0])[threadIdx.x] = 0;
    __syncthreads();   // the only block barrier of the free-running variant
  }
  const wpe::Tab& t = tw;
  const float* const verts4 = v4w;
  wpe::Slice& s = *reinterpret_cast<wpe::Slice*>(smem + (size_t)wib * sizeof(wpe::Slice));
  const int NV = fi.nv;
  const bool HASB = NV == 8;
  const int nq = m.nq;
  const float dt = m.timestep;
  const float scale = 1.0f / (m.meaninertia * (float)(NV > 1 ? NV : 1));
  const int li = lane & 7, sub = lane >> 3;   // dof owned by this lane, row stripe of this lane
  int gb0 = m.ngeom;                          // first geom riding on the block
  for (int i = m.ngeom - 1; i >= 0; i--) if (t.gmove[i] == 2) gb0 = i;
  const float Mi = li < NV ? fi.Mdiag[li] : 1.0f, dampi = li < NV ? fi.damp[li] : 0.f;
  const bool use_sep = !(a.opts & 1u);
  const bool use_gap = use_sep && !(a.opts & 0x10000u);   // opts bit 16: no gap budget (every cached direction is re-checked every substep)
  float blk_radius = 0.f;   // farthest point of the block's geoms from its body origin
  for (int i = gb0; i < m.ngeom; i++) {
    const double* o3 = t.gbase + 3 * i;
    blk_radius = fmaxf(blk_radius, (float)sqrt(o3[0] * o3[0] + o3[1] * o3[1] + o3[2] * o3[2]) * 1.001f + t.geom_rbound[i]);
  }
  // teams of the phase-locked variant: opts bits 4..7 = number of teams (0 -> 1); the warps of a team are contiguous
  int nteam = LOCK ? (int)((a.opts >> 4) & 15u) : 1;
  if (nteam < 1 || nteam > WPE_MAXTEAMS || wpb % nteam != 0) nteam = 1;
  const int wpt = wpb / nteam, team = wib / wpt, tthreads = 32 * wpt;
  int* const qcnt = Q.cnt[team];
#if !defined(HSRB_SIMT_EMU)
  // experiment: opts bits 8..15 = start stagger of team k in units of 4 us x k (teams that start in phase stay in phase on
  // uniform work and then compete for the same pipes in every phase)
  if (LOCK && team > 0 && ((a.opts >> 8) & 255u)) {
    const long long t0 = clock64(), wait = (long long)((a.opts >> 8) & 255u) * 4 * 1965 * team;
    while (clock64() - t0 < wait) __nanosleep(1000);
  }
#endif
  int* const qjobs = Q.jobs + team * wpt * WPE_ENVJOBS;
  const int qcap = wpt * WPE_ENVJOBS;
#if defined(WPE_DEBUG_JOBS)
  long long dbg_long = 0, dbg_quick = 0; int dbg_nlong = 0, dbg_nquick = 0, dbg_hits = 0, dbg_jobs_total = 0, dbg_long_total = 0, dbg_sub = 0;
#endif
#if defined(HSRB_PHASE_CLOCKS)
  unsigned long long ph[PH_COUNT] = {0, 0, 0, 0, 0, 0, 0};
  long long tlast = clock64();
#endif

#pragma unroll 1
  for (int wave0 = 0; wave0 < a.n; wave0 += gridDim.x * wpb) {
    // launch slot r -> block r % grid, warp r / grid: with a.order sorted by predicted work (heaviest first) the warps of a
    // block are ordered by weight, so the heavy environments of the block share a team and the light teams do not wait for them
    const int slot = wave0 + wib * (int)gridDim.x + (int)blockIdx.x;
    const bool valid = slot < a.n;
    const int env = valid ? (a.order ? a.order[slot] : slot) : 0;
    if (!LOCK && !valid) break;
    // ------------------------------------------------------------------ state -> shared memory
    if (valid) {
      const float* st = a.state + (size_t)env * a.S;
      if (lane < 12) s.qpos[lane] = (lane < nq) ? st[lane] : 0.f;
      if (lane < 8) {
        s.qvel[lane] = lane < NV ? st[nq + lane] : 0.f;
        s.warm[lane] = lane < NV ? st[nq + NV + lane] : 0.f;
        s.qfc[lane] = 0.f;
      }
      if (lane < 3) s.mocap[lane] = st[nq + 2 * NV + lane];
      if (lane < 2) s.ctrl[lane] = (a.ctrl && lane < fi.act_n) ? a.ctrl[(size_t)env * m.nu + lane] : 0.f;
      if (lane < 4) s.wi[lane] = 0;
      for (int i = lane; i < 4 * m.npair; i += 32) s.sep[i] = 0.f;     // no cached separating directions
      for (int i = lane; i < m.ngeom * 3; i += 32) s.gpos[i] = t.gbase[i];
      if (lane < 3) s.xb[lane] = 0;
      if (lane < 9) s.Rb[lane] = (lane % 4 == 0) ? 1.0 : 0.0;
    }
    int flags = 0;
    enum { A_ITER = 0, A_LS, A_CON, A_EFC, A_KFLOP, A_NARROW, A_HIT };   // s.acc slots
    if (lane < 8) s.acc[lane] = 0;
#if defined(WPE_CHAIN_CLOCKS)
    const long long ck_env0 = clock64();
#endif
    bool success = false;
    int taken = 0;
    bool finished = !valid || a.nsub <= 0;
    __syncwarp();

#pragma unroll 1
    for (int sb_ = 0; sb_ < a.nsub; sb_++) {
      if (LOCK) { if (wpe::team_and(team, tthreads, finished)) break; }
      else if (finished) break;
#if defined(HSRB_PHASE_CLOCKS)
      if (LOCK && threadIdx.x == 0) tlast = clock64();
#endif
      int nlimit = 0, ncon = 0, nefc = 0, narrow = 0, npflop = 0, ngrp = 0, nslot = 0, gdim = 0, nskip = 0;
      unsigned bits = 0;                // candidate pairs of this environment that passed the cull
      int it = 0, ls_used = 0;
      WPE_CK_DECL;
      if (!finished) {
      // ---------------------------------------------------------------- poses (B.1), geometry in double
      if (HASB) {
        double qd[4] = {(double)s.qpos[5], (double)s.qpos[6], (double)s.qpos[7], (double)s.qpos[8]};
        quatnormalize(qd);   // same rounding as the oracle: the narrowphase decisions downstream are discontinuous in the pose
        double Rb[9];
        quat2mat(qd, Rb);
        __syncwarp();
        if (lane < 4) s.qpos[5 + lane] = (float)qd[lane];  // MuJoCo normalises qpos in place
        if (lane < 3) s.xb[lane] = (double)s.qpos[2 + lane];
        if (lane == 0) {
#pragma unroll
          for (int k = 0; k < 9; k++) s.Rb[k] = Rb[k];
        }
        __syncwarp();
      }
      {
        const double q0 = (double)s.qpos[0], q1 = (double)s.qpos[1];
        for (int gg = lane; gg < m.ngeom; gg += 32) {
          const int mv = t.gmove[gg];
          if (mv == 1) {
#pragma unroll
            for (int k = 0; k < 3; k++) s.gpos[3 * gg + k] = t.gbase[3 * gg + k] + fi.axisd[0][k] * q0 + fi.axisd[1][k] * q1;
          } else if (mv == 2) {
            const double* Rb = s.Rb;
            const wpe::V3d p = ld3(s.xb) + mulv(Rb, ld3(t.gbase + 3 * gg));
            st3(s.gpos + 3 * gg, p);
            mulm(Rb, t.gmatw + 9 * gg, s.bmat + 9 * (gg - gb0));
            float Rbf[9], Rg[9];
#pragma unroll
            for (int k = 0; k < 9; k++) Rbf[k] = (float)Rb[k];
            mulm(Rbf, t.bgeom_mat + 9 * (gg - gb0), Rg);
            const float* h = t.geom_aabb + 3 * gg;
#pragma unroll
            for (int i = 0; i < 3; i++)
              s.baabb[4 * (gg - gb0) + i] = fabsf(Rg[3 * i]) * h[0] + fabsf(Rg[3 * i + 1]) * h[1] + fabsf(Rg[3 * i + 2]) * h[2];
          }
        }
      }
      __syncwarp();
      WPE_CK(0);
      // ---------------------------------------------------------------- active joint limits: groups 0 .. nlimit-1
      {
        bool act = false;
        float sg = 0.f, Dv = 0.f, ar = 0.f;
        if (lane < 2 && fi.limited[lane]) {
          const float q = s.qpos[lane];
          const float dlo = q - fi.range[lane][0], dhi = fi.range[lane][1] - q;
          float dist = 0.f;
          if (dlo < 0) { dist = dlo; sg = 1.f; }
          else if (dhi < 0) { dist = dhi; sg = -1.f; }
          if (sg != 0.f) {
            act = true;
            const double imp = push::impedance5(fi.lim_imp[lane], (double)dist);
            const double R = fmax(1e-15, (1 - imp) / imp * fi.lim_diag[lane]);
            Dv = (float)(1.0 / R);
            ar = (float)(-fi.lim_b[lane] * (double)(sg * s.qvel[lane]) - fi.lim_k[lane] * imp * (double)dist);
          }
        }
        const unsigned lm = __ballot_sync(FULL, act);
        nlimit = __popc(lm);
        if (act) {
          const int gslot = 6 * __popc(lm & ((1u << lane) - 1u));
          const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int r = 0; r < 6; r++) {
            float4* jp = reinterpret_cast<float4*>(s.J + 8 * (gslot + r));
            jp[0] = (r == 0) ? make_float4(lane == 0 ? sg : 0.f, lane == 1 ? sg : 0.f, 0.f, 0.f) : z4;
            jp[1] = z4;
            s.Dr[gslot + r] = r == 0 ? Dv : 0.f; s.aref[gslot + r] = r == 0 ? ar : 0.f; s.rsc[gslot + r] = r == 0 ? 1.f : 0.f;
          }
        }
      }
      // ---------------------------------------------------------------- collision (B.3): contacts in pair order
      // cull: one candidate pair per lane (npair <= 32 for this kernel: WPE_MAXPAIR)
      nefc = nlimit;
      {
        const int k = lane;
        bool hit = false;
        if (k < m.npair) {
          const int ga = t.pair_geom1[k], gb = t.pair_geom2[k];
          const V3<float> dp = cvt<float>(ld3(s.gpos + 3 * gb) - ld3(s.gpos + 3 * ga));
          if (t.geom_type[ga] == GEOM_PLANE) {
            const double* Ma = t.gmatw + 9 * ga;  // planes are static: world orientation is a table entry
            hit = dot(dp, mk<float>((float)Ma[2], (float)Ma[5], (float)Ma[8])) <= t.geom_rbound[gb];
          } else {
            const float rr = t.geom_rbound[ga] + t.geom_rbound[gb];
            hit = dot(dp, dp) <= rr * rr;
            const float* ha = t.gmove[ga] == 2 ? s.baabb + 4 * (ga - gb0) : t.ghalf + 3 * ga;
            const float* hb = t.gmove[gb] == 2 ? s.baabb + 4 * (gb - gb0) : t.ghalf + 3 * gb;
            hit = hit && fabsf(dp.x) <= ha[0] + hb[0] && fabsf(dp.y) <= ha[1] + hb[1] && fabsf(dp.z) <= ha[2] + hb[2];
          }
        }
        // Temporal coherence, exact: a convex-convex pair whose cached separating direction had a gap g after its last
        // support evaluation is still separated along that direction while g exceeds the displacement any point of the two
        // bodies can have made since (robot: a translation of dt |v|; block: dt |v| + dt |w| r); such a pair needs no
        // support evaluation at all - the query could only answer "no contact".  The flag of the cache holds -g.
        bool skip = false;
        if (use_gap && k < m.npair && t.pair_func[k] == NP_CONVEX_CONVEX) {
          float f = s.sep[4 * k + 3];
          if (f < 0.f) {
            const float moved = dt * 1.001f * (fabsf(s.qvel[0]) + fabsf(s.qvel[1]) + fabsf(s.qvel[2]) + fabsf(s.qvel[3]) + fabsf(s.qvel[4]) +
                                               (fabsf(s.qvel[5]) + fabsf(s.qvel[6]) + fabsf(s.qvel[7])) * blk_radius) + 5e-8f;
            f += moved;
            if (f < -1e-6f) skip = hit; else f = 1.f;   // budget used up: the next query re-measures the gap with one support evaluation
            s.sep[4 * k + 3] = f;
          }
        }
        bits = __ballot_sync(FULL, hit && !skip);
        nskip = __popc(__ballot_sync(FULL, skip));
      }
      WPE_CK(1);
      if (LOCK && lane == 0) {
        // queue this environment's convex-convex candidates for the block's warps: a pair without a cached separating
        // direction (in contact last time, or new) is a full refinement (~11 support evaluations) and goes to the front,
        // a pair with one is usually a single support evaluation and goes to the back
        unsigned bb = bits;
        int kc = 0;
        while (bb) {
          const int pk = __ffs((int)bb) - 1;
          bb &= bb - 1;
          if (t.pair_func[pk] != NP_CONVEX_CONVEX) continue;
          if (kc < WPE_ENVJOBS) {
            const bool quick = use_sep && (s.sep[4 * pk + 3] == 1.f || s.sep[4 * pk + 3] < 0.f);
            const int code = (wib << 16) | (kc << 8) | pk;
            if (quick) qjobs[qcap - 1 - atomicAdd(&qcnt[1], 1)] = code;
            else qjobs[atomicAdd(&qcnt[0], 1)] = code;
          }
          kc++;
        }
      }
      }
      if (LOCK) {
        WPE_PH(PH_KIN);
        wpe::team_sync(team, tthreads);
        WPE_PH(PH_CRB);
        // ---- every warp of the block (finished ones included) serves jobs: the owner's poses, this warp's portal scratch
        // (a team without jobs in this substep - the usual case for light environments since the gap budget - skips the
        //  service and its closing barrier: the counters are not written again before the next two team barriers)
        const int nlong = qcnt[0], njobs = nlong + qcnt[1];
        if (njobs > 0 || (a.opts & 0x20000u)) {   // opts bit 17: always run the service and its barrier (experiments)
#pragma unroll 1
        while (true) {
          int j = 0;
          if (lane == 0) j = atomicAdd(&qcnt[2], 1);
          j = __shfl_sync(FULL, j, 0);
          if (j >= njobs) break;
          const int code = j < nlong ? qjobs[j] : qjobs[qcap - 1 - (j - nlong)];
#if defined(WPE_DEBUG_JOBS)
          const long long tj0 = clock64();
#endif
          const int pk = code & 255;
          wpe::Slice& o = *reinterpret_cast<wpe::Slice*>(smem + (size_t)(code >> 16) * sizeof(wpe::Slice));
          const bool hitc = wpe::mpr(t, o, s, verts4, t.pair_geom1[pk], t.pair_geom2[pk], gb0, (double)m.mpr_tolerance, m.mpr_iterations,
                                     use_sep ? o.sep + 4 * pk : nullptr);
          if (lane == 0) {
            float* r = o.jres + 14 * ((code >> 8) & 255);
            r[0] = hitc ? 1.f : 0.f;
            if (hitc) {
              const double* r7 = s.mres;
              r[1] = (float)(-r7[0]); r[2] = (float)r7[4]; r[3] = (float)r7[5]; r[4] = (float)r7[6];
              make_frame(mk<double>(r7[1], r7[2], r7[3]), r + 5);
            }
          }
          __syncwarp();
#if defined(WPE_DEBUG_JOBS)
          if (threadIdx.x == 0) { const long long dtj = clock64() - tj0; if (j < nlong) { dbg_long += dtj; dbg_nlong++; if (hitc) dbg_hits++; } else { dbg_quick += dtj; dbg_nquick++; } }
#endif
        }
#if defined(WPE_DEBUG_JOBS)
        if (threadIdx.x == 0) { dbg_jobs_total += njobs; dbg_long_total += nlong; dbg_sub++; }
#endif
        WPE_PH(PH_SMOOTH);
        wpe::team_sync(team, tthreads);
        WPE_PH(PH_COLLIDE);
        if (wib == team * wpt && lane < 3) qcnt[lane] = 0;   // empty again; the next jobs are queued after the solver's barrier
        }
      }
      if (!finished) {
      {
        int kc = 0;
#pragma unroll 1
        while (bits) {
          const int pk = __ffs((int)bits) - 1;
          bits &= bits - 1;
          const int func = t.pair_func[pk];
          const int ga = t.pair_geom1[pk], gb = t.pair_geom2[pk];
          const int dim = t.pair_condim[pk];
          narrow++;
          npflop += func == NP_PLANE_BOX ? 80 : (func == NP_PLANE_CONVEX ? 100 : (func == NP_BOX_BOX ? 500 : 5000));
          if (func == NP_PLANE_BOX) {
            // mjc_PlaneBox: one corner per lane; the first four penetrating corners (corner order) become contacts
            const double* Ma = t.gmatw + 9 * ga;
            const wpe::V3d n = mk<double>(Ma[2], Ma[5], Ma[8]);
            const wpe::V3d pb = ld3(s.gpos + 3 * gb);
            const double dist0 = dot(pb - ld3(s.gpos + 3 * ga), n);
            const int i = lane;
            const float* sz = t.geom_size + 3 * gb;
            const wpe::V3d c = mk<double>((i & 1) ? (double)sz[0] : -(double)sz[0], (i & 2) ? (double)sz[1] : -(double)sz[1],
                                          (i & 4) ? (double)sz[2] : -(double)sz[2]);
            const wpe::V3d vec = mulv(wpe::geom_mat(t, s, gb, gb0), c);
            const double ld = dot(n, vec);
            const bool pen = i < 8 && !(dist0 + ld > 0 || ld > 0);
            const unsigned pm = __ballot_sync(FULL, pen);
            const int rank = __popc(pm & ((1u << i) - 1u));
            int nh = __popc(pm);
            if (nh > 4) nh = 4;
            const int room = WPE_MAXCON - ncon;
            if (pen && rank < nh && rank < room) {
              const int slot = ncon + rank;
              const double dist = dist0 + ld;
              s.con_pair[slot] = pk; s.con_dist[slot] = (float)dist;
              st3c(s.con_pos + 3 * slot, pb + vec - n * (dist * 0.5));
              make_frame(n, s.con_frame + 9 * slot);
            }
            if (nh > room) { nh = room; flags |= FLAG_CON_OVERFLOW; }
            ncon += nh; nefc += nh * dim;
            WPE_CK(2);
          } else if (func == NP_CONVEX_CONVEX && LOCK && kc < WPE_ENVJOBS) {
            // the job's result record (written by the warp that served it)
            const float* r = s.jres + 14 * kc;
            kc++;
            if (r[0] != 0.f) {
              if (lane == 0) s.acc[A_HIT]++;   // convex-convex contacts over the action (full portal refinements: the long jobs)
              if (ncon >= WPE_MAXCON) flags |= FLAG_CON_OVERFLOW;
              else {
                if (lane == 0) s.con_pair[ncon] = pk;
                if (lane == 1) s.con_dist[ncon] = r[1];
                if (lane >= 2 && lane < 5) s.con_pos[3 * ncon + lane - 2] = r[lane];
                if (lane >= 5 && lane < 14) s.con_frame[9 * ncon + lane - 5] = r[lane];
                ncon++; nefc += dim;
              }
            }
          } else if (func == NP_CONVEX_CONVEX || func == NP_PLANE_CONVEX) {
            bool hitc;
            kc++;
            WPE_CK_RESET();
            const float sf_ = use_sep ? s.sep[4 * pk + 3] : 0.f;
            if (func == NP_PLANE_CONVEX) {
              const double* Ma = t.gmatw + 9 * ga;
              const wpe::V3d n = mk<double>(Ma[2], Ma[5], Ma[8]);
              const wpe::V3d p = wpe::support(t, s, verts4, gb, gb0, -n);
              const double dist = dot(p - ld3(s.gpos + 3 * ga), n);
              hitc = dist <= 0;
              const wpe::V3d pos = p - n * (dist * 0.5);
              __syncwarp();
              if (lane == 0) { double* r7 = s.mres; r7[0] = -dist; r7[1] = n.x; r7[2] = n.y; r7[3] = n.z; r7[4] = pos.x; r7[5] = pos.y; r7[6] = pos.z; }
              __syncwarp();
            } else {
              hitc = wpe::mpr(t, s, s, verts4, ga, gb, gb0, (double)m.mpr_tolerance, m.mpr_iterations, use_sep ? s.sep + 4 * pk : nullptr);
            }
            if (hitc) {
              if (func == NP_CONVEX_CONVEX && lane == 0) s.acc[A_HIT]++;
              if (ncon >= WPE_MAXCON) flags |= FLAG_CON_OVERFLOW;
              else {
                if (lane == 0) {
                  const double* r7 = s.mres;
                  s.con_pair[ncon] = pk; s.con_dist[ncon] = (float)(-r7[0]);
                  s.con_pos[3 * ncon] = (float)r7[4]; s.con_pos[3 * ncon + 1] = (float)r7[5]; s.con_pos[3 * ncon + 2] = (float)r7[6];
                  make_frame(mk<double>(r7[1], r7[2], r7[3]), s.con_frame + 9 * ncon);
                }
                ncon++; nefc += dim;
              }
            }
            WPE_CK(hitc ? 3 : (sf_ == 1.f ? 4 : 5));
          } else {   // box-box (block against the pan): hsr_core.h, rare
            WS<float> w;                                // view for hsr::box_box / add_contact
            w.gpos = s.gpos; w.gaabb = nullptr; w.con_dist = s.con_dist; w.con_pos = s.con_pos; w.con_frame = s.con_frame;
            w.con_pair = s.con_pair; w.con_adr = s.con_adr; w.wi = s.wi; w.sep = nullptr;
            const DevGrp<32> g;
            Geom<float> A, B;
            A.type = GEOM_BOX; B.type = GEOM_BOX; A.verts = B.verts = nullptr; A.nvert = B.nvert = 0;
#pragma unroll
            for (int q = 0; q < 3; q++) { A.size[q] = t.geom_size[3 * ga + q]; B.size[q] = t.geom_size[3 * gb + q]; }
            A.pos = ld3(s.gpos + 3 * ga); B.pos = ld3(s.gpos + 3 * gb);
            const double* RA = wpe::geom_mat(t, s, ga, gb0); const double* RB = wpe::geom_mat(t, s, gb, gb0);
#pragma unroll
            for (int q = 0; q < 9; q++) { A.mat[q] = RA[q]; B.mat[q] = RB[q]; }
            int nrow_ = nefc;
            box_box(m, w, g, ncon, nrow_, pk, A, B);   // capacities: the host sets m.ncon_max / m.nefc_max to this kernel's
            nefc = nrow_;
            __syncwarp();
            flags |= s.wi[WI_FLAGS];
            WPE_CK(18);
          }
        }
      }
      __syncwarp();
      ngrp = nlimit + ncon;
      nslot = 6 * ngrp;
      narrow += nskip; npflop += 5000 * nskip;   // pairs settled by the gap budget still count as the reference's narrowphase work
      if (lane == 0) { s.acc[A_NARROW] += narrow; s.acc[A_CON] += ncon; s.acc[A_EFC] += nefc; }

      WPE_CK_RESET();
      // ---------------------------------------------------------------- smooth forces (closed form, B.6): dof lanes
      if (lane < 8) {
        float q = 0.f;
        const float v = s.qvel[lane];
        if (lane < 2) {
          q = -fi.damp[lane] * v + fi.gq[lane];
          for (int k = 0; k < fi.act_n; k++) {
            if (fi.act_dof[k] != lane) continue;
            float c = s.ctrl[k];
            if (fi.ctrllimited[k]) c = fminf(fmaxf(c, fi.cr_lo[k]), fi.cr_hi[k]);
            float fo = fi.kp[k] * c - fi.kp[k] * fi.gear[k] * s.qpos[fi.act_q[k]];
            if (fi.forcelimited[k]) fo = fminf(fmaxf(fo, fi.fr_lo[k]), fi.fr_hi[k]);
            q += fi.gear[k] * fo;
          }
        } else if (HASB) {
          if (lane < 5) q = fi.Mdiag[2] * fi.gravity[lane - 2] - fi.damp[lane] * v;
          else {
            // free box: -w x (I w) on the body-frame rotational dofs
            const int i0 = lane - 5, i1 = (i0 + 1) % 3, i2 = (i0 + 2) % 3;
            const float w1 = s.qvel[5 + i1], w2 = s.qvel[5 + i2];
            q = -(w1 * (fi.Mdiag[5 + i2] * w2) - w2 * (fi.Mdiag[5 + i1] * w1)) - fi.damp[lane] * v;
          }
        }
        s.qs[lane] = q;
        s.as[lane] = lane < NV ? q / fi.Mdiag[lane] : 0.f;
      }
      WPE_CK(6);
      // ---------------------------------------------------------------- constraint rows (B.4/B.5): lane = (contact, row), five contacts per round
      if (lane < nlimit) gdim = 1;
      else if (lane < ngrp) gdim = t.pair_condim[s.con_pair[lane - nlimit]];
      {
        const int cl = (lane * 43) >> 8, r = lane - 6 * cl;   // lane / 6, lane % 6
#pragma unroll 1
        for (int c0 = 0; c0 < ncon; c0 += 5) {
          const int c = c0 + cl;
          if (lane < 30 && c < ncon) {
            const int pk = s.con_pair[c];
            const int gd = t.pair_condim[pk];
            float Jr[8];
#pragma unroll
            for (int d = 0; d < 8; d++) Jr[d] = 0.f;
            float Dv = 0.f, ar = 0.f, rs = 0.f;
            if (r < gd) {
              const float sr = t.pair_sr[pk], sbk = t.pair_sb[pk];
              const float* frr = s.con_frame + 9 * c + 3 * (r < 3 ? r : r - 3);
              const float f0 = frr[0], f1 = frr[1], f2 = frr[2];
              const float* fri = t.pair_friction + 5 * pk;
              const double* pc = t.pairc + PUSH_PAIRC * pk;
              const double dist = (double)s.con_dist[c];
              const double imp = push::impedance5<true>(pc + 3, dist);
              const float D0 = (float)fmin(1e15, imp / ((1 - imp) * pc[2]));   // 1 / max(1e-15, R0)
              const float D1 = D0 * m.impratio;
              float w0 = f0, w1 = f1, w2 = f2;   // rotational rows: the frame axis itself; translational: rel x f
              if (r < 3) {
                Jr[0] = sr * (f0 * fi.axis[0][0] + f1 * fi.axis[0][1] + f2 * fi.axis[0][2]);
                Jr[1] = sr * (f0 * fi.axis[1][0] + f1 * fi.axis[1][1] + f2 * fi.axis[1][2]);
                if (HASB) {
                  const float r0 = (float)((double)s.con_pos[3 * c] - s.xb[0]), r1 = (float)((double)s.con_pos[3 * c + 1] - s.xb[1]),
                              r2 = (float)((double)s.con_pos[3 * c + 2] - s.xb[2]);
                  Jr[2] = sbk * f0; Jr[3] = sbk * f1; Jr[4] = sbk * f2;
                  w0 = r1 * f2 - r2 * f1; w1 = r2 * f0 - r0 * f2; w2 = r0 * f1 - r1 * f0;   // f . (axis x rel) = axis . (rel x f)
                }
              }
              if (HASB) {
#pragma unroll
                for (int q = 0; q < 3; q++)   // body axis q of the block in the world frame = column q of Rb
                  Jr[5 + q] = sbk * ((float)s.Rb[q] * w0 + (float)s.Rb[3 + q] * w1 + (float)s.Rb[6 + q] * w2);
              }
              const push::F8 qv8 = push::ld8(s.qvel);
              float vel = 0.f;
#pragma unroll
              for (int d = 0; d < 8; d++) vel += Jr[d] * qv8.v[d];
              if (r == 0) { Dv = D0; ar = (float)(-pc[1] * (double)vel - pc[0] * imp * dist); rs = gd > 1 ? fri[0] * rsqrtf(m.impratio) : 1.f; }   // rs: mu = fri0 * sqrt(R1 / R0)
              else {
                ar = (float)(-pc[1] * (double)vel);
                Dv = r == 1 ? D1 : D1 * (fri[r - 1] * fri[r - 1]) / (fri[0] * fri[0]);
                rs = fri[r - 1];
              }
            }
            const int slot_ = 6 * (nlimit + c) + r;
            push::st8(s.J + 8 * slot_, Jr);
            s.Dr[slot_] = Dv; s.aref[slot_] = ar; s.rsc[slot_] = rs;
          }
        }
      }
      __syncwarp();
      WPE_CK(7);

      // ---------------------------------------------------------------- Newton solver (B.7)
      // One loop whose body appears once in the instruction stream: [rows at the point] -> cost / forces / zones ->
      // bookkeeping of the phase -> Newton step.  Phases: 0 cost at qacc_smooth, 1 cost at qacc_warmstart (the usual
      // winner, evaluated last so that its rows and forces are in place), 2 back to qacc_smooth when it won, 3.. Newton.
      if (ngrp == 0) {
        if (lane < 8) { s.x[lane] = s.as[lane]; s.qfc[lane] = 0.f; }
        __syncwarp();
      }
      }
      {
        bool solving = !finished && ngrp != 0;
        int zone = 0;
        float cN = 0.f, cT = 0.f;
        int phase = 0;
        const float* xp = s.warm;
        float cost = 0.f, alpha = 0.f, dec = 0.f;
        bool finishing = false;   // converged by the improvement test: stop after the next gradient (forces of the final point)
#pragma unroll 1
        while (true) {
#if defined(WPE_PASS_LOCK)
          if (LOCK) { if (!__syncthreads_or(solving)) break; }   // every solver pass in lock-step (measured: slower)
          else if (!solving) break;
#else
          if (!solving) break;   // the warps run their passes freely inside the solver phase (one barrier after the loop)
#endif
          if (!solving) continue;
          const bool dual = phase == 0;   // both starting points in one pass: lanes 0..15 at qacc_warmstart, lanes 16..31 at qacc_smooth
          if (dual) {
            // jar = J warm - aref, and J as - aref into the (still unused) jv slots
            const push::F8 xw = push::ld8(s.warm), xa = push::ld8(s.as);
            for (int r = lane; r < nslot; r += 32) {
              const push::F8 j = push::ld8(s.J + 8 * r);
              float accw = -s.aref[r], acca = accw;
#pragma unroll
              for (int d = 0; d < 8; d++) { accw += j.v[d] * xw.v[d]; acca += j.v[d] * xa.v[d]; }
              s.jar[r] = accw; s.jv[r] = acca;
            }
            __syncwarp();
            WPE_CK(8);
          } else if (phase < 3) {
            // jar = J x - aref (row slots across lanes)
            const push::F8 xv = push::ld8(xp);
            for (int r = lane; r < nslot; r += 32) {
              const push::F8 j = push::ld8(s.J + 8 * r);
              float acc = -s.aref[r];
#pragma unroll
              for (int d = 0; d < 8; d++) acc += j.v[d] * xv.v[d];
              s.jar[r] = acc;
            }
            __syncwarp();
            WPE_CK(8);
          }
          // ---- cost of the point: Gauss term on the dof lanes, cone / half-line state of each group on its lane
          //      (zone, forces -> s.f)
          float cl = 0.f;
          if (lane < 8) { const float xi = xp[lane]; cl = 0.5f * (Mi * xi - s.qs[lane]) * (xi - s.as[lane]); }   // zero at qacc_smooth
          const int gl = dual ? (lane & 15) : lane;                                 // group of this lane
          const int gd_ = dual ? __shfl_sync(FULL, gdim, lane & 15) : gdim;
          if (gl < ngrp) {
            const float* pj = ((dual && lane >= 16) ? s.jv : s.jar) + 6 * gl; const float* pD = s.Dr + 6 * gl; const float* ps = s.rsc + 6 * gl;
            float jr[6], Dv[6], rs[6];
#pragma unroll
            for (int r = 0; r < 6; r++) { jr[r] = pj[r]; Dv[r] = pD[r]; rs[r] = ps[r]; }
            const float mu = rs[0];
            int z; float n_ = 0.f, t_ = 0.f;
            if (gd_ == 1) {
              z = jr[0] < 0 ? 1 : 0;
            } else {
              n_ = jr[0] * mu;
              float tt = 0.f;
#pragma unroll
              for (int j = 1; j < 6; j++) { const float u = jr[j] * rs[j]; tt += u * u; }
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
              for (int r = 0; r < 6; r++) { cl += 0.5f * Dv[r] * jr[r] * jr[r]; fo[r] = -Dv[r] * jr[r]; }
            } else if (z == 2) {
              const float Dm = Dv[0] / (mu * mu * (1 + mu * mu));
              const float NTv = n_ - mu * t_;
              cl += 0.5f * Dm * NTv * NTv;
              const float f0 = -Dm * NTv * mu;
              fo[0] = f0;
              const float f0t = -f0 / t_;
#pragma unroll
              for (int j = 1; j < 6; j++) fo[j] = f0t * (jr[j] * rs[j]) * rs[j];
            }
            if (lane < 16) {   // (the qacc_smooth half of a dual pass only needs the cost)
              float* pf = s.f + 6 * gl;
#pragma unroll
              for (int r = 0; r < 6; r++) pf[r] = fo[r];
            }
            zone = z; cN = n_; cT = t_;
          }
          float c;
          if (dual) {   // sums of the two half-warps
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) cl += __shfl_xor_sync(FULL, cl, o);
            c = cl;
          } else c = wpe::warp_sum(cl);
          __syncwarp();
          WPE_CK(9);
          if (dual) {
            const float cw = __shfl_sync(FULL, c, 0), cs = __shfl_sync(FULL, c, 16);
            c = cw;
            const bool use_warm = cw <= cs;   // ties -> warm start
            if (lane < 8) s.x[lane] = use_warm ? s.warm[lane] : s.as[lane];
            __syncwarp();
            xp = s.x;
            if (!use_warm) { phase = 2; continue; }
            cost = c; phase = 3;
          } else if (phase == 2) {
            cost = c; phase = 3;
          } else {
            const float old = cost;
            cost = c;
            it++;
            const float improvement = alpha < 2.f ? alpha * (1.f - 0.5f * alpha) * dec : old - cost;
            if (scale * improvement < m.tolerance) finishing = true;   // the next pass computes J^T f of this point and stops
          }
          // ---- gradient component of this lane's dof: M x - qfrc_smooth - J^T f   (row stripes: r = sub, sub + 4, ...)
          float qf = 0.f;
#pragma unroll 2
          for (int r = sub; r < nslot; r += 4) qf += s.J[8 * r + li] * s.f[r];
          qf += __shfl_xor_sync(FULL, qf, 8);
          qf += __shfl_xor_sync(FULL, qf, 16);
          const float xi = s.x[li];
          const float grad = (li < NV) ? Mi * xi - s.qs[li] - qf : 0.f;
          float gn = grad * grad;
#pragma unroll
          for (int o = 1; o < 8; o <<= 1) gn += __shfl_xor_sync(FULL, gn, o);
          gn = sqrtf(gn);
          WPE_CK(10);
          if (finishing || (it > 0 && scale * gn < m.tolerance) || it >= m.iterations) {
            if (lane < 8) s.qfc[lane] = qf;
            solving = false;
            continue;
          }
          // ---- Hessian J^T (cone Hessians) J as a sum of weighted outer products of Jacobian rows (see hsrb_push.cuh):
          //      quadratic-zone group: sum_r D_r J_r J_r^T;  cone-zone contact: Dm (p p^T + k q q^T) - Dm k sum_{a>=1} s_a^2 J_a J_a^T
          if (lane < ngrp) {
            const float* pD = s.Dr + 6 * lane; const float* ps = s.rsc + 6 * lane;
            float wr_[6], wp = 0.f, wq = 0.f;
#pragma unroll
            for (int r = 0; r < 6; r++) wr_[r] = zone == 1 ? pD[r] : 0.f;
            if (zone == 2) {
              const float mu = ps[0];
              const float Dm = pD[0] / (mu * mu * (1 + mu * mu)), NTv = cN - mu * cT, invT = 1.0f / cT;
              const float kap = mu * NTv * invT;
              const float* pj = s.jar + 6 * lane;
              float pvv[8], qv[8];
              {
                const push::F8 j = push::ld8(s.J + 8 * (6 * lane));
#pragma unroll
                for (int d = 0; d < 8; d++) { pvv[d] = mu * j.v[d]; qv[d] = 0.f; }
              }
#pragma unroll
              for (int aa = 1; aa < 6; aa++) {
                const float sa = ps[aa];
                const float cq = pj[aa] * sa * invT * sa, cp = -mu * cq;
                const push::F8 j = push::ld8(s.J + 8 * (6 * lane + aa));
#pragma unroll
                for (int d = 0; d < 8; d++) { pvv[d] += cp * j.v[d]; qv[d] += cq * j.v[d]; }
                wr_[aa] = -Dm * kap * sa * sa;
              }
              wp = Dm; wq = Dm * kap;
              push::st8(s.PQ + 16 * lane, pvv); push::st8(s.PQ + 16 * lane + 8, qv);
            }
            float* pw = s.wrow + 6 * lane;
#pragma unroll
            for (int r = 0; r < 6; r++) pw[r] = wr_[r];
            s.wpq[2 * lane] = wp; s.wpq[2 * lane + 1] = wq;
          }
          __syncwarp();
          float Hr[8];
#pragma unroll
          for (int j = 0; j < 8; j++) Hr[j] = 0.f;
#pragma unroll 2
          for (int r = sub; r < nslot; r += 4) {
            const float ji = s.J[8 * r + li] * s.wrow[r];
            const push::F8 jv_ = push::ld8(s.J + 8 * r);
#pragma unroll
            for (int j = 0; j < 8; j++) Hr[j] += ji * jv_.v[j];
          }
          for (int c = sub; c < ngrp; c += 4) {
            const float wpc = s.wpq[2 * c];
            if (wpc != 0.f) {
              const float pi_ = s.PQ[16 * c + li] * wpc, qi_ = s.PQ[16 * c + 8 + li] * s.wpq[2 * c + 1];
              const push::F8 pv_ = push::ld8(s.PQ + 16 * c), qv_ = push::ld8(s.PQ + 16 * c + 8);
#pragma unroll
              for (int j = 0; j < 8; j++) Hr[j] += pi_ * pv_.v[j] + qi_ * qv_.v[j];
            }
          }
#pragma unroll
          for (int j = 0; j < 8; j++) {
            Hr[j] += __shfl_xor_sync(FULL, Hr[j], 8);
            Hr[j] += __shfl_xor_sync(FULL, Hr[j], 16);
          }
#pragma unroll
          for (int j = 0; j < 8; j++) if (li == j) Hr[j] += Mi;
          WPE_CK(11);
          // ---- Cholesky H = L L^T: lane i holds row i; column k is finished by a broadcast of the pivot and one
          //      shuffle per trailing column (the four 8-lane segments of the warp work redundantly)
          float inv_diag = 1.f;
#pragma unroll
          for (int k = 0; k < 8; k++) {
            float dkk = __shfl_sync(FULL, Hr[k], k, 8);
            if (!(dkk > 1e-15f)) { dkk = 1e-15f; flags |= FLAG_CHOL; }
            const float inv = rsqrtf(dkk);
            const float lkk = dkk * inv;
            const float lik = (li == k) ? lkk : Hr[k] * inv;   // L[i][k] for i >= k
            Hr[k] = lik;
            if (li == k) inv_diag = inv;
#pragma unroll
            for (int j = k + 1; j < 8; j++) {
              const float ljk = __shfl_sync(FULL, lik, j, 8);
              Hr[j] -= lik * ljk;                               // meaningful for i >= j
            }
          }
          // ---- forward solve L y = -grad
          float acc = -grad, y = 0.f;
#pragma unroll
          for (int k = 0; k < 8; k++) {
            const float yk = __shfl_sync(FULL, acc * inv_diag, k, 8);
            if (li == k) y = yk;
            acc -= Hr[k] * yk;                                  // meaningful for i > k
          }
          // ---- backward solve L^T s = y: column k of L gathered through shared memory
          __syncwarp();
          if (sub == 0) push::st8(s.L + 8 * li, Hr);
          __syncwarp();
          acc = y;
          float sv = 0.f;
#pragma unroll
          for (int k = 7; k >= 0; k--) {
            const float xk = __shfl_sync(FULL, acc * inv_diag, k, 8);
            if (li == k) sv = xk;
            acc -= s.L[8 * k + li] * xk;                        // L[k][li], meaningful for li < k
          }
          if (li >= NV) sv = 0.f;
          if (sub == 0) s.srch[li] = sv;
          float sn = sv * sv, q1 = sv * (Mi * xi - s.qs[li]), q2 = 0.5f * sv * (Mi * sv);
          dec = -grad * sv;
#pragma unroll
          for (int o = 1; o < 8; o <<= 1) {
            dec += __shfl_xor_sync(FULL, dec, o); sn += __shfl_xor_sync(FULL, sn, o);
            q1 += __shfl_xor_sync(FULL, q1, o); q2 += __shfl_xor_sync(FULL, q2, o);
          }
          sn = sqrtf(sn);
          __syncwarp();
          WPE_CK(12);
          if (!(sn >= 1e-15f)) {
            if (lane < 8) s.qfc[lane] = qf;
            solving = false;
            continue;
          }
          // ---- jv = J search (row slots across lanes)
          {
            const push::F8 sv8 = push::ld8(s.srch);
            for (int r = lane; r < nslot; r += 32) {
              const push::F8 j = push::ld8(s.J + 8 * r);
              float accv = 0.f;
#pragma unroll
              for (int d = 0; d < 8; d++) accv += j.v[d] * sv8.v[d];
              s.jv[r] = accv;
            }
          }
          __syncwarp();
          const float gtol = m.tolerance * m.ls_tolerance * sn / scale;
          // ---- exact line search: root of the 1-D derivative (safeguarded Newton with bracketing); the group lanes hold
          //      the coefficients of their group's cost along the search direction
          float l0 = 0.f, l1c = 0.f, l2c = 0.f, l3 = 0.f, l4 = 0.f, l6 = 0.f, l7 = 0.f, l9 = 0.f, mu_ = 1.f;
          if (lane < ngrp) {
            const float* pj = s.jar + 6 * lane; const float* pvv = s.jv + 6 * lane; const float* pD = s.Dr + 6 * lane;
            const float* ps = s.rsc + 6 * lane;
            float uu = 0.f, uv = 0.f, vv = 0.f, Q1 = 0.f, Q2 = 0.f;
#pragma unroll
            for (int r = 0; r < 6; r++) {
              const float xx = pj[r], v = pvv[r], Dv = pD[r];
              Q1 += Dv * xx * v; Q2 += 0.5f * Dv * v * v;
              if (r > 0) { const float u = xx * ps[r], sv2 = v * ps[r]; uu += u * u; uv += u * sv2; vv += sv2 * sv2; }
            }
            mu_ = ps[0];
            l0 = pj[0] * mu_; l1c = pvv[0] * mu_;
            l9 = gdim == 1 ? -1.f : pD[0] / (mu_ * mu_ * (1 + mu_ * mu_));
            l2c = uu; l3 = uv; l4 = vv; l6 = Q1; l7 = Q2;
          }
          {
            // At alpha = 0 the derivative along the Newton direction is grad . s = -dec and its slope s^T H s = dec (H s = -grad):
            // no evaluation needed; the first trial point is the full Newton step.
            WPE_CK(13);
            float d1 = -dec, d2 = dec, nxt = 0.f;
            int nev = 1;
            float lo = 0.f, hi = -1.f, dlo = d1, dhi = 0.f;
            const float rel = 3.4526698e-4f;  // sqrt(FLT_EPSILON)
            bool conv = fabsf(d1) < gtol, tiny = false;
            alpha = 0.f;
#pragma unroll 1
            while (!conv && nev <= m.ls_iterations) {
              const float step = d2 > 1e-15f ? -d1 / d2 : (d1 < 0 ? 1.f : -1.f);
              nxt = alpha + step;
              if (hi >= 0 && !(lo < nxt && nxt < hi)) nxt = 0.5f * (lo + hi);
              if (nxt <= 0 && hi < 0) nxt = alpha * 0.5f;
              if (nxt == alpha) break;
              tiny = fabsf(nxt - alpha) <= rel * fabsf(nxt);
              // derivative of the cost along the search direction and its slope at nxt
              {
                const float N = l0 + nxt * l1c;
                const float tsq = l2c + nxt * (2 * l3 + nxt * l4);
                const float rT = tsq > 0 ? rsqrtf(tsq) : 0.f;     // 1 / T (used in the cone zone only, where T > 0)
                const float Tn = tsq * rT;
                const bool quad = l9 < 0;                          // one-row group: half-line instead of a cone
                const bool top = quad ? !(N < 0) : ((N >= mu_ * Tn) || (Tn <= 0 && N >= 0));
                const bool bottom = quad ? (N < 0) : ((mu_ * N + Tn <= 0) || (Tn <= 0 && N < 0));
                const float NTv = N - mu_ * Tn;
                const float T1 = (l3 + nxt * l4) * rT;
                const float T2 = (l4 - T1 * T1) * rT;
                const float tt = l1c - mu_ * T1;
                const float lm1 = l9 * NTv * tt, lm2 = l9 * (tt * tt - NTv * mu_ * T2);
                const float lb1 = l6 + 2 * nxt * l7, lb2 = 2 * l7;
                float e1 = top ? 0.f : (bottom ? lb1 : lm1), e2 = top ? 0.f : (bottom ? lb2 : lm2);
                if (lane >= ngrp) { e1 = 0.f; e2 = 0.f; }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) { e1 += __shfl_xor_sync(FULL, e1, o); e2 += __shfl_xor_sync(FULL, e2, o); }
                d1 = e1 + q1 + 2 * nxt * q2;
                d2 = e2 + 2 * q2;
              }
              alpha = nxt;
              if (d1 < 0) { if (alpha > lo) { lo = alpha; dlo = d1; } }
              else if (hi < 0 || alpha < hi) { hi = alpha; dhi = d1; }
              conv = fabsf(d1) < gtol || tiny;
              nev++;
              WPE_CK(14);
            }
            ls_used += nev;
            if (!conv) {
              if (hi >= 0 && (lo <= 0 || fabsf(dhi) < fabsf(dlo))) alpha = (lo > 0 || fabsf(dhi) < fabsf(dlo)) ? hi : 0.f;
              else alpha = lo;
            }
          }
          if (alpha == 0.f) {
            if (lane < 8) s.qfc[lane] = qf;
            solving = false;
            continue;
          }
          if (lane < 8) s.x[lane] += alpha * s.srch[lane];
          for (int r = lane; r < nslot; r += 32) s.jar[r] += alpha * s.jv[r];
          __syncwarp();
          WPE_CK(16);
        }
        __syncwarp();
      }
      WPE_PH(PH_ROWS);
      if (LOCK) wpe::team_sync(team, tthreads);
      WPE_PH(PH_SOLVE);
      if (!finished) {
      WPE_CK_RESET();
      if (lane == 0) {
        s.acc[A_ITER] += it; s.acc[A_LS] += ls_used;
        s.acc[A_KFLOP] += algorithmic_flops(m, false, ncon, nefc, it, ls_used, npflop);   // slides + free box: M is constant
      }

      // ---------------------------------------------------------------- goal test on the poses of this forward pass
      bool reached = false;
      if (HASB && a.cfg.has_goal) {
        const double dx = s.xb[0] - (double)s.mocap[0], dy = s.xb[1] - (double)s.mocap[1], dz = s.xb[2] - (double)s.mocap[2];
        reached = sqrt(dx * dx + dy * dy + dz * dz) < (double)a.cfg.geofence;
      }
      // ---------------------------------------------------------------- Euler with implicit joint damping (B.8)
      bool bad = false;
      if (lane < NV) {
        const float xi = s.x[lane];
        const float ai = m.any_damping ? (s.qs[lane] + s.qfc[lane]) / (Mi + dt * dampi) : xi;
        s.warm[lane] = xi;
        const float v = s.qvel[lane] + dt * ai;
        s.qvel[lane] = v;
        if (!(fabsf(v) < 1e6f)) bad = true;
        if (lane < 5) s.qpos[lane] += dt * v;
      }
      if (__any_sync(FULL, bad)) flags |= FLAG_BAD_NUM;
      __syncwarp();
      if (HASB) {
        const float om0 = s.qvel[5], om1 = s.qvel[6], om2 = s.qvel[7];
        const float ang = sqrtf(om0 * om0 + om1 * om1 + om2 * om2);
        float qq[4] = {s.qpos[5], s.qpos[6], s.qpos[7], s.qpos[8]};
        quatnormalize(qq);
        if (ang * dt > 1e-15f) {
          // rotation by ang * dt about omega: dq = [cos h, sin(h) / ang * omega], h = ang dt / 2 (series below h = 0.5 rad)
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
          quatmul(qq, dq, qq);
        }
        quatnormalize(qq);
        __syncwarp();
        if (lane < 4) s.qpos[5 + lane] = qq[lane];
        __syncwarp();
      }
      WPE_CK(17);
      taken++;
      if (reached) success = true;
      if (reached || sb_ == a.nsub - 1) finished = true;
      }
      WPE_PH(PH_EULER);
    }
    // ------------------------------------------------------------------ results: HBM once per action
    if (valid) {
      __syncwarp();
      float* st = a.state + (size_t)env * a.S;
      const int nobs = nq + NV;
      for (int i = lane; i < nq + 2 * NV; i += 32) {
        const float v = i < nq ? s.qpos[i] : (i < nq + NV ? s.qvel[i - nq] : s.warm[i - nq - NV]);
        st[i] = v;
        if (a.obs && i < nobs) a.obs[(size_t)env * nobs + i] = v;
      }
      if (lane == 0) {
        if (a.reward) a.reward[env] = success ? 1.0f : 0.0f;
        if (a.done) a.done[env] = success ? 1 : 0;
        if (a.success) a.success[env] = success ? 1 : 0;
        if (a.taken) a.taken[env] = taken;
        if (a.bad) a.bad[env] = (unsigned char)flags;
        // work estimate in k-cycles of an uncontended warp (tools/chain_clocks.py): fixed part, Newton iterations, refinements, rows
#if defined(WPE_CHAIN_CLOCKS)
        if (a.work) a.work[env] = (int)((clock64() - ck_env0) >> 10);   // measured: k-cycles of this environment's action
#else
        if (a.work) a.work[env] = 20 * taken + 7 * s.acc[A_ITER] + 30 * s.acc[A_HIT] + s.acc[A_CON];
#endif
        atomicAdd(a.stats + ST_SUBSTEPS, (unsigned long long)taken);
        atomicAdd(a.stats + ST_ITERS, (unsigned long long)s.acc[A_ITER]);
        atomicAdd(a.stats + ST_NARROW, (unsigned long long)s.acc[A_NARROW]);
        atomicAdd(a.stats + ST_LSEVAL, (unsigned long long)s.acc[A_LS]);
        atomicAdd(a.stats + ST_CONTACTS, (unsigned long long)s.acc[A_CON]);
        atomicAdd(a.stats + ST_ROWS, (unsigned long long)s.acc[A_EFC]);
        atomicAdd(a.stats + ST_FLOPS, (unsigned long long)s.acc[A_KFLOP]);
        if (flags) atomicAdd(a.stats + ST_BAD, 1ull);
      }
      __syncwarp();
    }
  }
#if defined(HSRB_PHASE_CLOCKS)
  if (LOCK && threadIdx.x == 0 && blockIdx.x == 0)
    for (int k = 0; k < PH_COUNT; k++) atomicAdd(a.stats + ST_PHASE0 + k, ph[k]);
#endif
#if defined(WPE_DEBUG_JOBS)
  if (LOCK && threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == 77))
    printf("block %d: substeps %d, jobs/substep %.1f (long %.1f); warp 0 served %d long jobs (%d hits) at %.0f cycles each, %d quick at %.0f cycles each\n",
           blockIdx.x, dbg_sub, (double)dbg_jobs_total / dbg_sub, (double)dbg_long_total / dbg_sub, dbg_nlong, dbg_hits, dbg_nlong ? (double)dbg_long / dbg_nlong : 0.0,
           dbg_nquick, dbg_nquick ? (double)dbg_quick / dbg_nquick : 0.0);
#endif
}
#endif  // HSRB_WPE_IMPL
