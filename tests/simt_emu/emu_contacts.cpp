// TEST INFRASTRUCTURE: the contact query kernel (hsrb_contacts.cuh) and, on the same inputs, the MODE_DEBUG launch of the
// general action kernel (hsrb_debug_substep's dump), on the CPU through the SIMT emulator (simt_emu.h).  Build:
// tests/test_contacts_emu.py.  Never linked into the product.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "../../hsr_env_b200/csrc/hsrb_contacts.cuh"

namespace {
template <int G, bool P>
void run_contacts(const ConArgs& c, int grid, size_t smem) {
  emu::launch(grid, 32, smem, [&]() { hsrb_contacts_kernel<G, P>(c); });
}
template <int G, bool P>
void run_debug(const KArgs& a, int grid, size_t smem) {
  emu::launch(grid, 32, smem, [&]() { hsrb_step_kernel<G, true, P>(a); });
}
// xipos of the forward pass (kinematics_lane0's centres of mass), which neither launch writes out
template <int G, bool P>
void run_xipos(const KArgs& a, double* out, int grid, size_t smem) {
  emu::launch(grid, 32, smem, [&]() {
    HSRB_DYN_SMEM(smem_);
    DevGrp<G> g;
    const int gpb = 32 / G, gi = threadIdx.x / G;
    WS<float> w;
    ws_carve<float>(a.m, &w, smem_ + (size_t)gi * a.ws_bytes);
    for (int env = blockIdx.x * gpb + gi; env < a.n; env += gridDim.x * gpb) {
      load_state<G>(a, w, g, env);
      g.sync();
      typename ScaleOf<P>::type sc;
      load_scale(sc, a, env);
      kinematics_trig(a.m, w, g);
      if (g.lane == 0) kinematics_lane0(a.m, w, sc);
      g.sync();
      if (g.lane == 0) for (int i = 0; i < 3 * a.m.nbody; i++) out[(size_t)env * 3 * a.m.nbody + i] = w.xipos[i];
      g.sync();
    }
  });
}
template <int G>
void run_all(bool P, const ConArgs& c, const KArgs& d, double* xipos, int grid, size_t smem) {
  if (P) run_contacts<G, true>(c, grid, smem); else run_contacts<G, false>(c, grid, smem);
  if (d.dump) { if (P) run_debug<G, true>(d, grid, smem); else run_debug<G, false>(d, grid, smem); }
  if (xipos) { if (P) run_xipos<G, true>(c.k, xipos, grid, smem); else run_xipos<G, false>(c.k, xipos, grid, smem); }
}
}  // namespace

// G lanes per environment, one warp per block; ncon_max / nefc_max > 0 replace the model's capacities (hsrb_config).
// state [n, S] is the query's input (and must come back unchanged); ctrl [n, nu] or null (zeros); params [n, PRM_COUNT] or
// null.  Outputs of the query (nullable, C = max_contacts): count, pair, dist, pos, frame, force, wrench, bad, stats
// [ST_COUNT].  dump [n, debug_size] (nullable): MODE_DEBUG on a copy of the state with the same ctrl and params, its
// bad_state in dbg_bad.  xipos [n, nbody, 3] (nullable).
extern "C" int emu_contacts(const void* blob, size_t bytes, int G, int n, int ncon_max, int nefc_max, int C, float* state,
                            const float* ctrl, const float* params, int* count, int* pair, float* dist, float* pos, float* frame,
                            float* force, float* wrench, unsigned char* bad, unsigned long long* stats, double* dump,
                            unsigned char* dbg_bad, double* xipos) {
  HostModel<float> hm;
  std::string err;
  if (!hm.parse(blob, bytes, err)) { fprintf(stderr, "emu_contacts: %s\n", err.c_str()); return -1; }
  const ModelT<float>& m = hm.m;
  const int S = m.nq + 2 * m.nv + 3;
  std::vector<float> prm(params ? params : (const float*)nullptr, params ? params + (size_t)n * PRM_COUNT : (const float*)nullptr);
  ConArgs c;
  memset(&c, 0, sizeof(c));
  KArgs& a = c.k;
  a.m = m;
  if (ncon_max > 0) a.m.ncon_max = ncon_max;
  if (nefc_max > 0) a.m.nefc_max = nefc_max;
  a.cfg.qidx0 = 0; a.cfg.qidx1 = 2;
  a.n = n; a.S = S; a.stats = stats;
  a.ws_bytes = (unsigned)ws_carve<float>(a.m, nullptr, nullptr);
  a.state = state; a.ctrl = ctrl; a.params = params ? prm.data() : nullptr;
  c.C = C; c.count = count; c.pair = pair; c.dist = dist; c.pos = pos; c.frame = frame; c.force = force; c.wrench = wrench; c.bad = bad;
  // the debug launch: a copy of the state (it advances it), its own counters
  std::vector<float> st2(state, state + (size_t)n * S);
  std::vector<unsigned long long> st_dbg(ST_COUNT, 0);
  std::vector<unsigned char> done(n), succ(n);
  std::vector<float> obs((size_t)n * (m.nq + m.nv)), reward(n);
  std::vector<int> tk(n);
  KArgs d = a;
  d.mode = MODE_DEBUG; d.nsub = 1; d.state = st2.data(); d.stats = st_dbg.data();
  d.dump = dump; d.dump_stride = (unsigned)debug_size(a.m);
  d.obs = obs.data(); d.reward = reward.data(); d.done = done.data(); d.success = succ.data(); d.taken = tk.data(); d.bad = dbg_bad;
  const int gpb = 32 / G;
  const int grid = (n + gpb - 1) / gpb;
  const size_t smem = (size_t)a.ws_bytes * gpb;
  const bool P = params != nullptr;
  if (G == 4) run_all<4>(P, c, d, xipos, grid, smem); else if (G == 8) run_all<8>(P, c, d, xipos, grid, smem);
  else if (G == 16) run_all<16>(P, c, d, xipos, grid, smem); else if (G == 32) run_all<32>(P, c, d, xipos, grid, smem);
  else return -3;
  return 0;
}
