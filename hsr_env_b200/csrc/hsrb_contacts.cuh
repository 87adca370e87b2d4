// The contact query (hsrb_contacts): mj_forward on each environment's current resident state, then a read of data.contact,
// mj_contactForce and the per-body sum of the contact wrenches (the cfrc_ext part that contacts make).
//
// Per environment: load_state, the caller's ctrl (NULL: zeros), the environment's multipliers, forward() of hsr_core.h - the
// stages MODE_DEBUG of hsrb_step_kernel runs before its Euler step - and then
//   * the contact rows, lanes striding over contacts: pair, dist, pos, frame (con_frame, row 0 the normal from geom1 to geom2)
//     and force (the contact's efc_force rows in the contact frame: normal, two tangential, torsional, two rolling; rows
//     past the pair's condim are 0);
//   * the body wrenches, lanes striding over bodies, each summing the contacts in order in double: (force, torque) in world
//     axes, torque about the body's centre of mass xipos.  A contact adds +f to body2 (of pair_geom2) and -f to body1,
//     MuJoCo's cfrc_ext sign; the world body 0 receives its reactions, so the rows sum to zero.
// Nothing is written back: no store_state (qacc_warmstart included, which mj_forward would update), no work counters.
//
// Layout: the lean launch of the general path (configure() in hsrb_api.cu): G lanes per environment, one warp per block,
// 32 / G workspaces of ws_bytes in shared memory, a grid-stride loop.
#pragma once
#include "hsrb_kernels.cuh"

struct ConArgs {
  KArgs k;              // model (ncon_max / nefc_max: the general plan's), n, S, ws_bytes, state, ctrl (nullable), params
  int C;                // rows per environment of the per-contact outputs (max_contacts)
  // outputs (nullable): count [N]; pair [N, C]; dist [N, C]; pos [N, C, 3]; frame [N, C, 9]; force [N, C, 6];
  // wrench [N, nbody, 6]; bad [N]
  int* count; int* pair; float* dist; float* pos; float* frame; float* force; float* wrench; unsigned char* bad;
};

// The wrench (force, torque about xipos) of the first ncon contacts on body b, in double, in contact order
template <typename T>
__device__ __forceinline__ void contact_wrench(const ModelT<T>& m, const WS<T>& w, int ncon, int b, GT* out6) {
  GT f[3] = {0, 0, 0}, t[3] = {0, 0, 0};
  const GT* xi = w.xipos + 3 * b;
  for (int c = 0; c < ncon; c++) {
    const int pk = w.con_pair[c];
    const int b1 = m.geom_body[m.pair_geom1[pk]], b2 = m.geom_body[m.pair_geom2[pk]];
    const GT sg = (GT)(b == b2) - (GT)(b == b1);
    if (sg == 0) continue;
    const int dim = m.pair_condim[pk], r0 = w.con_adr[c];
    const T* fr = w.con_frame + 9 * c;
    GT F[6];
    for (int r = 0; r < 6; r++) F[r] = r < dim ? (GT)w.force[r0 + r] : GT(0);
    GT fc[3], tc[3], d[3];
    for (int k = 0; k < 3; k++) {
      fc[k] = F[0] * (GT)fr[k] + F[1] * (GT)fr[3 + k] + F[2] * (GT)fr[6 + k];
      tc[k] = F[3] * (GT)fr[k] + F[4] * (GT)fr[3 + k] + F[5] * (GT)fr[6 + k];
      d[k] = (GT)w.con_pos[3 * c + k] - xi[k];
    }
    const GT tx = tc[0] + d[1] * fc[2] - d[2] * fc[1];
    const GT ty = tc[1] + d[2] * fc[0] - d[0] * fc[2];
    const GT tz = tc[2] + d[0] * fc[1] - d[1] * fc[0];
    f[0] += sg * fc[0]; f[1] += sg * fc[1]; f[2] += sg * fc[2];
    t[0] += sg * tx; t[1] += sg * ty; t[2] += sg * tz;
  }
  for (int k = 0; k < 3; k++) { out6[k] = f[k]; out6[3 + k] = t[k]; }
}

template <int G, bool PARAMS>
__global__ void __launch_bounds__(32) hsrb_contacts_kernel(const __grid_constant__ ConArgs c) {
  HSRB_DYN_SMEM(smem);
  const KArgs& a = c.k;
  DevGrp<G> g;
  const int gpb = 32 / G;
  const int gi = threadIdx.x / G;
  WS<float> w;
  ws_carve<float>(a.m, &w, smem + (size_t)gi * a.ws_bytes);
  for (int env = blockIdx.x * gpb + gi; env < a.n; env += gridDim.x * gpb) {
    load_state<G>(a, w, g, env);
    for (int i = g.lane; i < a.m.nu; i += G) w.ctrl[i] = a.ctrl ? a.ctrl[(size_t)env * a.m.nu + i] : 0.f;
    g.sync();
    typename ScaleOf<PARAMS>::type sc;
    load_scale(sc, a, env);
    forward(a.m, w, g, sc);
    const int ncon = w.wi[WI_NCON];
    // contact rows: the first min(ncon, C) are contacts, the rest padding (pair -1, zeros)
    for (int i = g.lane; i < c.C; i += G) {
      const bool on = i < ncon;
      const size_t r = (size_t)env * c.C + i;
      if (c.pair) c.pair[r] = on ? w.con_pair[i] : -1;
      if (c.dist) c.dist[r] = on ? w.con_dist[i] : 0.f;
      if (c.pos) for (int k = 0; k < 3; k++) c.pos[3 * r + k] = on ? w.con_pos[3 * i + k] : 0.f;
      if (c.frame) for (int k = 0; k < 9; k++) c.frame[9 * r + k] = on ? w.con_frame[9 * i + k] : 0.f;
      if (c.force) {
        const int dim = on ? a.m.pair_condim[w.con_pair[i]] : 0, r0 = on ? w.con_adr[i] : 0;
        for (int k = 0; k < 6; k++) c.force[6 * r + k] = k < dim ? w.force[r0 + k] : 0.f;
      }
    }
    if (c.wrench)
      for (int b = g.lane; b < a.m.nbody; b += G) {
        GT wr[6];
        contact_wrench(a.m, w, ncon, b, wr);
        float* o = c.wrench + ((size_t)env * a.m.nbody + b) * 6;
        for (int k = 0; k < 6; k++) o[k] = (float)wr[k];
      }
    if (g.lane == 0) {
      if (c.count) c.count[env] = ncon;
      if (c.bad) c.bad[env] = (unsigned char)w.wi[WI_FLAGS];
    }
    g.sync();   // the group's reads of the workspace are done before the next environment's load_state
  }
}

// host side (hsrb_contacts.cu), in the general kernel's plan p: p.lanes picks G, c.k.params the instance with parameters
cudaError_t hsrb_contacts_prepare(const Plan& p);
cudaError_t hsrb_contacts_launch(const Plan& p, const ConArgs& c, cudaStream_t s);
