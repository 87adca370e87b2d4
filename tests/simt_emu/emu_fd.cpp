// TEST INFRASTRUCTURE: the transition-derivative kernels (hsrb_fd.cuh) and, on every run's perturbed input, the general
// action kernel (MODE_DEBUG for one substep, a STEP launch without goal for more), on the CPU through the SIMT emulator
// (simt_emu.h).  Build: tests/test_transition_fd_emu.py.  Never linked into the product.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "../../hsr_env_b200/csrc/hsrb_fd.cuh"

namespace {
template <int G, bool P>
void run_fd(const FdArgs& f, int grid, size_t smem) {
  emu::launch(grid, 32, smem, [&]() { hsrb_fd_kernel<G, P>(f); });
}
template <int G, bool P>
void run_ref(const KArgs& a, int grid, size_t smem) {
  emu::launch(grid, 32, smem, [&]() { hsrb_step_kernel<G, true, P>(a); });
}
template <int G>
void run_all(bool P, const FdArgs& f, int grid, const KArgs* ref, int rgrid, size_t smem) {
  if (P) run_fd<G, true>(f, grid, smem); else run_fd<G, false>(f, grid, smem);
  if (ref) { if (P) run_ref<G, true>(*ref, rgrid, smem); else run_ref<G, false>(*ref, rgrid, smem); }
}
}  // namespace

// G lanes per environment, one warp per block, at most grid_cap blocks (0: one job per group, no grid stride).  state [n, S]
// is the input (and must come back unchanged); ctrl [n, nu] or null (zeros); params [n, PRM_COUNT] or null.  Outputs
// (nullable): A, B, next_obs, bad, stats [ST_COUNT] (the kernels' counters), scratch [n * nruns * fd_row] (the scratch
// rows), inputs [n, nruns, nq + nv + nu] and h [n, nruns] (each run's perturbed input, fd_perturb on the host);
// ref [n * nruns, nq + nv] and ref_bad [n * nruns]: the general action kernel on those inputs (warm start and mocap of the
// resident state, the environment's multipliers).
extern "C" int emu_fd(const void* blob, size_t bytes, int G, int n, int nsub, int centered, float eps, double rot_c,
                      double rot_s, int grid_cap, float* state, const float* ctrl, const float* params, float* A, float* B,
                      float* next_obs, unsigned char* bad, unsigned long long* stats, float* scratch, float* inputs,
                      double* h, float* ref, unsigned char* ref_bad) {
  HostModel<float> hm;
  std::string err;
  if (!hm.parse(blob, bytes, err)) { fprintf(stderr, "emu_fd: %s\n", err.c_str()); return -1; }
  const ModelT<float>& m = hm.m;
  const int S = m.nq + 2 * m.nv + 3, nx = m.nq + m.nv, nu = m.nu, nruns = fd_nruns(m, centered != 0);
  const size_t jobs = (size_t)n * nruns;
  std::vector<float> scr(jobs * fd_row(m), -7.f);
  FdArgs f;
  memset(&f, 0, sizeof(f));
  KArgs& a = f.k;
  a.m = m;
  a.cfg.qidx0 = 0; a.cfg.qidx1 = 2;
  a.n = n; a.S = S; a.stats = stats;
  a.ws_bytes = (unsigned)ws_carve<float>(a.m, nullptr, nullptr);
  a.state = state; a.ctrl = ctrl; a.params = const_cast<float*>(params);
  f.eps = eps; f.rot_c = rot_c; f.rot_s = rot_s; f.centered = centered; f.nsub = nsub; f.nruns = nruns;
  f.scratch = scr.data(); f.A = A; f.B = B; f.next_obs = next_obs; f.bad = bad;
  // the perturbed inputs of every run, and the reference launch on them
  std::vector<float> st2(jobs * S), c2(jobs * (nu > 0 ? nu : 1), 0.f), p2(params ? jobs * PRM_COUNT : 0);
  std::vector<double> hh(jobs);
  for (size_t j = 0; j < jobs; j++) {
    const int e = (int)(j / nruns), r = (int)(j % nruns);
    float* s = st2.data() + j * S;
    for (int i = 0; i < S; i++) s[i] = state[(size_t)e * S + i];
    float* u = c2.data() + j * nu;
    for (int i = 0; i < nu; i++) u[i] = ctrl ? ctrl[(size_t)e * nu + i] : 0.f;
    if (params) for (int k = 0; k < PRM_COUNT; k++) p2[j * PRM_COUNT + k] = params[(size_t)e * PRM_COUNT + k];
    hh[j] = fd_perturb(m, r, centered != 0, eps, rot_c, rot_s, s, s + m.nq, u);
    if (inputs) {
      float* o = inputs + j * (nx + nu);
      for (int i = 0; i < nx; i++) o[i] = s[i];
      for (int i = 0; i < nu; i++) o[nx + i] = u[i];
    }
    if (h) h[j] = hh[j];
  }
  KArgs d;
  std::vector<unsigned long long> st_ref(ST_COUNT, 0);
  std::vector<float> obs(jobs * nx), reward(jobs);
  std::vector<unsigned char> done(jobs), succ(jobs), rbad(jobs);
  std::vector<int> tk(jobs);
  std::vector<double> dump;
  if (ref) {
    d = a;
    memset(&d.cfg, 0, sizeof(d.cfg));   // no goal: the derivative is of the physics, not of the action's freeze
    d.cfg.qidx0 = 0; d.cfg.qidx1 = 2;
    d.n = (int)jobs; d.state = st2.data(); d.ctrl = c2.data(); d.params = params ? p2.data() : nullptr; d.stats = st_ref.data();
    d.nsub = nsub; d.mode = nsub == 1 ? MODE_DEBUG : MODE_STEP;
    if (nsub == 1) {
      d.dump_stride = (unsigned)debug_size(a.m);
      dump.resize(jobs * d.dump_stride);
      d.dump = dump.data();
    }
    d.obs = obs.data(); d.reward = reward.data(); d.done = done.data(); d.success = succ.data(); d.taken = tk.data(); d.bad = rbad.data();
  }
  const int gpb = 32 / G;
  int grid = (int)((jobs + gpb - 1) / gpb);
  if (grid_cap > 0 && grid > grid_cap) grid = grid_cap;
  const int rgrid = (int)((jobs + gpb - 1) / gpb);
  const size_t smem = (size_t)a.ws_bytes * gpb;
  const bool P = params != nullptr;
  const KArgs* rp = ref ? &d : nullptr;
  if (G == 4) run_all<4>(P, f, grid, rp, rgrid, smem); else if (G == 8) run_all<8>(P, f, grid, rp, rgrid, smem);
  else if (G == 16) run_all<16>(P, f, grid, rp, rgrid, smem); else if (G == 32) run_all<32>(P, f, grid, rp, rgrid, smem);
  else return -3;
  const long long threads = (long long)n * (2 * m.nv + nu + 1);
  emu::launch((int)((threads + 127) / 128), 128, 0, [&]() {
    if (centered) hsrb_fd_form_kernel<true>(f); else hsrb_fd_form_kernel<false>(f);
  });
  if (scratch) memcpy(scratch, scr.data(), scr.size() * sizeof(float));
  if (ref) {
    for (size_t j = 0; j < jobs; j++) {
      for (int i = 0; i < nx; i++) ref[j * nx + i] = st2[j * S + i];
      ref_bad[j] = rbad[j];
    }
  }
  return 0;
}
