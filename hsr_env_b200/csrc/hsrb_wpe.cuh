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
  // per-block constants read where they are used instead of being held in registers across the substep
  int gb0;                                   // first geom riding on the block
  float blk_radius;                          // farthest point of the block's geoms from its body origin
  int wpt;                                   // warps per team (phase-locked variant)
  unsigned char team[WPE_MAXWARPS];          // team of each warp
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
// Shared memory of a block: [Tab | Queue | slice 0 .. wpb-1 | hull vertices as float4].  The tables and the queue sit at
// offset 0, so their fields are LDS / STS with absolute addresses and no register holds their base; a slice is one 32-bit
// offset from the warp index.
constexpr unsigned SMEM_HEAD = (unsigned)(sizeof(Tab) + sizeof(Queue));
static_assert(SMEM_HEAD % 16 == 0, "the slices start 16-byte aligned");
// block-shared bytes besides the slices: the tables, the job queue and the hull vertices
__host__ __device__ inline size_t shared_tail(const ModelT<float>& m) { return SMEM_HEAD + (size_t)m.nvert * 16 + 16; }

}  // namespace wpe

// kernel + device routines: only in the translation unit that owns them (hsrb_wpe.cu, the emulated build)
#if defined(HSRB_WPE_IMPL)
namespace wpe {

typedef V3<double> V3d;

__device__ __forceinline__ unsigned char* smem_base() {
  HSRB_DYN_SMEM(smem);
  return smem;
}
__device__ __forceinline__ Tab& tab() { return *reinterpret_cast<Tab*>(smem_base()); }
__device__ __forceinline__ Queue& queue() { return *reinterpret_cast<Queue*>(smem_base() + sizeof(Tab)); }
__device__ __forceinline__ Slice& slice(int w) { return *reinterpret_cast<Slice*>(smem_base() + SMEM_HEAD + (unsigned)w * (unsigned)sizeof(Slice)); }
__device__ __forceinline__ float* hull_verts4() {
  return reinterpret_cast<float*>(smem_base() + SMEM_HEAD + (blockDim.x >> 5) * (unsigned)sizeof(Slice));
}

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
// ow: the warp whose slice holds the environment the pair belongs to (poses, cached direction o.sep + 4 sepk, none if
// sepk < 0); s: the executing warp's slice (portal scratch, result) - the same slice unless the warp serves another
// environment's job (phase-locked variant).  Every argument is one 32-bit register: the tables, the slices and the hull
// vertices are addressed from the fixed shared-memory layout, so the call carries no 64-bit pointers.  `inline`: both wpe
// translation units (hsrb_wpe.cu, hsrb_wpe_params.cu) define it.
inline __device__ __noinline__ bool mpr(int ow, int g1, int g2, int gb0, float tol_f, int max_iter, int sepk) {
  const Tab& t = tab();
  const Slice& o = slice(ow);
  Slice& s = slice(threadIdx.x >> 5);
  const float* const verts4 = hull_verts4();
  float* const sep = sepk >= 0 ? slice(ow).sep + 4 * sepk : nullptr;
  const double tol = (double)tol_f;
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

__device__ __forceinline__ int* team_jobs(Queue& Q, const Tab& t, int w) { return Q.jobs + t.team[w] * t.wpt * WPE_ENVJOBS; }

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
#define WPE_ROLLOUT 0
#define WPE_ENTRY hsrb_wpe_kernel_t
#define WPE_PARAMS false
#include "hsrb_wpe_kernel.cuh"
#undef WPE_ENTRY
#undef WPE_PARAMS
// the instance with per-environment parameters (hsrb_wpe_params.cu)
#define WPE_ENTRY hsrb_wpe_params_kernel_t
#define WPE_PARAMS true
#include "hsrb_wpe_kernel.cuh"
#undef WPE_ENTRY
#undef WPE_PARAMS
#undef WPE_ROLLOUT
// the open-loop rollout instances (hsrb_rollout: K actions per environment in one launch; hsrb_wpe_rollout.cu)
#define WPE_ROLLOUT 1
#define WPE_ENTRY hsrb_wpe_rollout_kernel_t
#define WPE_PARAMS false
#include "hsrb_wpe_kernel.cuh"
#undef WPE_ENTRY
#undef WPE_PARAMS
#define WPE_ENTRY hsrb_wpe_rollout_params_kernel_t
#define WPE_PARAMS true
#include "hsrb_wpe_kernel.cuh"
#undef WPE_ENTRY
#undef WPE_PARAMS
#undef WPE_ROLLOUT
#endif  // HSRB_WPE_IMPL

// host side (hsrb_wpe.cu): p.lock picks the instance; a.params the instance with parameters (hsrb_wpe_params.cu)
cudaError_t hsrb_wpe_prepare(const Plan& p, int* bps);
cudaError_t hsrb_wpe_params_prepare(const Plan& p);
cudaError_t hsrb_wpe_params_launch(const Plan& p, const KArgs& a, cudaStream_t s);
cudaError_t hsrb_wpe_launch(const Plan& p, const KArgs& a, cudaStream_t s);
// the phase-locked instances with the action loop (hsrb_wpe_rollout.cu): nact actions in one launch
cudaError_t hsrb_wpe_rollout_prepare();
cudaError_t hsrb_wpe_rollout_launch(const Plan& p, const KArgs& a, int nact, cudaStream_t s);
