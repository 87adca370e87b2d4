// The body of the phase-locked general kernel, included by hsrb_kernels.cuh once per entry point: LOCK_ENTRY names the
// __global__ template <bool PARAMS>, LOCK_ROLLOUT = 1 (hsrb_rollout) takes the number of actions nact as a parameter after
// KArgs and runs the per-slot body, from the state load to the results, once per action: action k reads ctrl row
// k * n + env and writes output row k * n + env.
template <bool PARAMS = false>   // true: STEP launches with a.params
#if LOCK_ROLLOUT
__global__ void __launch_bounds__(32 * HSRB_LOCK_MAXWARPS) LOCK_ENTRY(const __grid_constant__ KArgs a, const int nact) {
#else
__global__ void __launch_bounds__(32 * HSRB_LOCK_MAXWARPS) LOCK_ENTRY(const __grid_constant__ KArgs a) {
#endif
  HSRB_DYN_SMEM(smem);
  typedef DevGrp<32> Grp;
  const Grp g;
  const int wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const ModelT<float>& m = a.m;
  WS<float> w;
  ws_carve<float>(m, &w, smem + (size_t)wib * a.ws_bytes);
  LockQueue& Q = *reinterpret_cast<LockQueue*>(smem + (size_t)wpb * a.ws_bytes);
  if (threadIdx.x < 4) Q.cnt[threadIdx.x] = 0;
  __syncthreads();
  const int nobs = m.nq + m.nv;
  const int qcap = wpb * HSR_MAXJOBS;
  for (int env0 = blockIdx.x * wpb; env0 < a.n; env0 += gridDim.x * wpb) {
    const int env = env0 + wib;
    const bool valid = env < a.n;
#if LOCK_ROLLOUT
    // the environment's actions one after the other (invalid slots too: they take part in the block barriers), each from
    // the state row the previous one wrote, as hsrb_step would run them
#pragma unroll 1
    for (int k = 0; k < nact; k++) {
    const size_t krow = (size_t)k * (size_t)a.n;
#define LOCK_ROW(e) (krow + (size_t)(e))
#else
#define LOCK_ROW(e) (e)
#endif
    typename ScaleOf<PARAMS>::type sc;
    if (valid) {
      load_scale(sc, a, env);
      load_state<32>(a, w, g, env);
      for (int i = g.lane; i < m.nu; i += 32) w.ctrl[i] = a.ctrl ? a.ctrl[(size_t)LOCK_ROW(env) * m.nu + i] : 0.f;
    }
    g.sync();
    bool success = false, finished = !valid || a.nsub <= 0;
    int taken = 0;
    for (int sb = 0; sb < a.nsub; sb++) {
      if (__syncthreads_and(finished)) break;
      int nlimit = 0, nrow = 0, ncon = 0, it0 = 0, ls0 = 0;
      // PH: block barriers between ALL phases (not only around the job service), PL: one block vote per Newton pass - the
      // warps of the block then run the same code region at the same time (the instruction stream of a substep of this
      // kernel is several hundred KB; free-running warps spent half of their stall samples waiting for instructions).
      // a.opts bit 1 / bit 2 switch them off (experiments)
      const bool PH = !(a.opts & 2u), PL = !(a.opts & 4u);
      if (!finished) {
        HSR_PHASE_START(w, g);
        kinematics_trig(m, w, g);
        if (g.lane == 0) kinematics_lane0(m, w, sc);
        g.sync();
        HSR_PHASE(w, g, PH_KIN);
      }
      if (PH) __syncthreads();
      if (!finished) {
        cdof_geoms(m, w, g);
        g.sync();
        mass_matrix(m, w, g);
        g.sync();
        HSR_PHASE(w, g, PH_CRB);
      }
      if (PH) __syncthreads();
      if (!finished) {
        if (g.lane == 0) smooth_lane0(m, w, sc);
        g.sync();
        smooth_solve(m, w, g);
        HSR_PHASE(w, g, PH_SMOOTH);
      }
      if (PH) __syncthreads();
      if (!finished) {
        for (int j = 0; j < m.njnt; j++) {
          if (!m.jnt_limited[j] || m.jnt_type[j] == JNT_FREE) continue;
          const float q = w.qpos[m.jnt_qposadr[j]];
          if (q - m.jnt_range[2 * j] < 0) nlimit++;
          if (m.jnt_range[2 * j + 1] - q < 0) nlimit++;
        }
        nrow = nlimit;
        collision_cull(m, w, g);
        // queue the convex-convex candidates: long jobs (no cached separating direction) from the front, quick ones from the back
        if (g.lane == 0) {
          int kc = 0;
          for (int base = 0; base < m.npair; base += 32) {
            unsigned bb = w.cand[base >> 5];
            while (bb) {
              const int pk = base + __ffs((int)bb) - 1;
              bb &= bb - 1;
              if (m.pair_func[pk] != NP_CONVEX_CONVEX) continue;
              if (kc < HSR_MAXJOBS) {
                const int code = (wib << 16) | (kc << 8) | pk;
                if (w.sep[4 * pk + 3] == 1.f) Q.jobs[qcap - 1 - atomicAdd(&Q.cnt[1], 1)] = code;
                else Q.jobs[atomicAdd(&Q.cnt[0], 1)] = code;
              }
              kc++;
            }
          }
        }
      }
      __syncthreads();
      {
        // every warp serves jobs: the owner's poses and separating-direction cache, this warp's registers
        const int nlong = Q.cnt[0], njobs = nlong + Q.cnt[1];
        while (true) {
          int j = 0;
          if (g.lane == 0) j = atomicAdd(&Q.cnt[2], 1);
          j = __shfl_sync(0xffffffffu, j, 0);
          if (j >= njobs) break;
          const int code = j < nlong ? Q.jobs[j] : Q.jobs[qcap - 1 - (j - nlong)];
          const int pk = code & 255;
          WS<float> wo;
          ws_carve<float>(m, &wo, smem + (size_t)(code >> 16) * a.ws_bytes);
          Geom<float> A, B;
          load_geom(m, wo, m.pair_geom1[pk], A);
          load_geom(m, wo, m.pair_geom2[pk], B);
          GT depth = 0; V3<GT> dir = mk<GT>(0, 0, 1), pos = mk<GT>(0, 0, 0);
          const bool hit = mpr_penetration_inl(A, B, (GT)m.mpr_tolerance, m.mpr_iterations, g, depth, dir, pos, wo.sep + 4 * pk);
          if (g.lane == 0) {
            GT* r = wo.jres + 8 * ((code >> 8) & 255);
            r[0] = hit ? 1.0 : 0.0; r[1] = depth; r[2] = dir.x; r[3] = dir.y; r[4] = dir.z; r[5] = pos.x; r[6] = pos.y; r[7] = pos.z;
          }
          g.sync();
        }
      }
      __syncthreads();
      if (threadIdx.x < 3) Q.cnt[threadIdx.x] = 0;
      if (!finished) {
        ncon = collision_assemble(m, w, g, nrow);
        g.sync();
        HSR_PHASE(w, g, PH_COLLIDE);
      }
      if (PH) __syncthreads();
      if (!finished) {
        make_constraint(m, w, g, nlimit, ncon, sc);
        it0 = w.wi[WI_ITER]; ls0 = w.wi[WI_LSEVAL];
        g.sync();
        if (g.lane == 0) { w.wi[WI_NCON] = ncon; w.wi[WI_NEFC] = nrow; w.wi[WI_NLIMIT] = nlimit; }
        g.sync();
        HSR_PHASE(w, g, PH_ROWS);
      }
      if (PH) __syncthreads();
      if (PL) {
        NewtonState<float> ns;
        bool act = !finished && newton_begin(m, w, g, nlimit, ncon, nrow, ns, sc);
        const bool solved = act;
        while (__syncthreads_or(act)) {
          if (act) act = newton_pass(m, w, g, nlimit, ncon, nrow, ns, sc);
        }
        if (solved) newton_end(m, w, g, nrow, ns);
      } else if (!finished) {
        solve_newton(m, w, g, nlimit, ncon, nrow, sc);
      }
      if (!finished) {
        HSR_PHASE(w, g, PH_SOLVE);
        if (g.lane == 0) {
          w.wi[WI_SUMCON] += ncon; w.wi[WI_SUMEFC] += nrow;
          w.wi[WI_KFLOP] += algorithmic_flops(m, ncon, nrow, w.wi[WI_ITER] - it0, w.wi[WI_LSEVAL] - ls0, w.wi[WI_NPFLOP]);
        }
        g.sync();
      }
      __syncthreads();
      if (!finished) {
        euler_solve(m, w, g, sc);
        if (g.lane == 0) euler_lane0(m, w);
        g.sync();
        HSR_PHASE(w, g, PH_EULER);
        taken++;
        if (goal_reached(m, a.cfg, w)) success = true;
        if (success || sb == a.nsub - 1) finished = true;
      }
    }
    if (valid) {
      store_state<32>(a, w, g, env);
      if (a.obs) for (int i = g.lane; i < nobs; i += 32) a.obs[(size_t)LOCK_ROW(env) * nobs + i] = w.qpos[i];
      if (g.lane == 0) {
        const int flags = w.wi[WI_FLAGS];
        if (a.reward) a.reward[LOCK_ROW(env)] = success ? 1.0f : 0.0f;
        if (a.done) a.done[LOCK_ROW(env)] = success ? 1 : 0;
        if (a.success) a.success[LOCK_ROW(env)] = success ? 1 : 0;
        if (a.taken) a.taken[LOCK_ROW(env)] = taken;
        if (a.bad) a.bad[LOCK_ROW(env)] = (unsigned char)flags;
        atomicAdd(a.stats + ST_SUBSTEPS, (unsigned long long)taken);
        atomicAdd(a.stats + ST_ITERS, (unsigned long long)w.wi[WI_ITER]);
        atomicAdd(a.stats + ST_NARROW, (unsigned long long)w.wi[WI_NARROW]);
        atomicAdd(a.stats + ST_LSEVAL, (unsigned long long)w.wi[WI_LSEVAL]);
        atomicAdd(a.stats + ST_CONTACTS, (unsigned long long)w.wi[WI_SUMCON]);
        atomicAdd(a.stats + ST_ROWS, (unsigned long long)w.wi[WI_SUMEFC]);
        atomicAdd(a.stats + ST_FLOPS, (unsigned long long)w.wi[WI_KFLOP]);
#ifdef HSRB_PHASE_CLOCKS
        for (int k = 0; k < PH_COUNT; k++) atomicAdd(a.stats + ST_PHASE0 + k, (unsigned long long)w.wi[WI_PHASE0 + k]);
#endif
        if (flags) atomicAdd(a.stats + ST_BAD, 1ull);
      }
    }
    __syncthreads();
#if LOCK_ROLLOUT
    }
#endif
#undef LOCK_ROW
  }
}
