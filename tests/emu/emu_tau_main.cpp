// emu_tau_main.cpp -- builds libtrex_emu_tau.so: the emulator of emu_extf_main.cpp plus the TAU instances of the front and tail
// phases (joint torque control, the library's trex_config.actuation = TREX_ACTUATION_TORQUE).  TEST INFRASTRUCTURE ONLY.
//
// The wrench emulator is included as it is.  A handle switched to torque mode (emu_set_torque_mode) steps through emu_tau_step4,
// which runs the TAU instances -- together with the ENVP instances when the handle has parameter rows and the EXTF instances
// when it has a wrench record or a push schedule; every other handle is forwarded to emu_extf_step4 of the included emulator.
#include "emu_extf_main.cpp"

// torque-mode handles and their torque bound (the model's motor_max_torque, as trex_create rounds it)
static std::mutex g_tau_lock;
static std::unordered_map<void*, float> g_tau;
static bool tau_of(void* h, float* bound) {
  std::lock_guard<std::mutex> g(g_tau_lock);
  auto it = g_tau.find(h);
  if (it == g_tau.end()) return false;
  *bound = it->second;
  return true;
}

// one env step (or reset when force_reset) on n (1..4) consecutive environment records, as emu_extf_main.cpp's step4x, with the
// front and tail phases of the TAU instances (the solve phases are the shared ones)
template <bool ENVP, bool EXTF>
static void step4t(Emu* e, Envp* p, Extf* x, float tau_max, int n, float* rec, const float* action, float* obs, float* reward,
                   uint8_t* done, float* aux, int force_reset, long long env_id0) {
  // The library keeps element 30 (the motor impulse bound) at 0 in torque mode, on create, on a set and on a randomized reset
  // (trex_capi.cu: imp_dt()).  The emulator imposes that here instead of running those paths, so its rows say nothing about
  // them; the GPU tests check the library's.
  if (ENVP) {
    p->dt = 0.0;
    for (int i = 0; i < 4; i++) p->rows[i][trex_host::ENVP_MAX_IMPULSE] = 0.0f;
  }
  float* rows = ENVP ? &p->rows[0][0] : nullptr;
  const float* mdl = e->T.mdl.data();
  const int* mdli = e->T.mdli.data();
  const float* tasks = e->T.tasks.data();
  const float* cp = e->T.cand_p.data();
  const int* cl = e->T.cand_lane.data();
  const float* com = e->T.com.data();
  const trex::PushSchedule* push = EXTF ? &x->push : nullptr;
  if (!force_reset) {
    for (int r = 0; r < e->P.n_sub; r++) {
      int envs[TREX_NCLASS][4] = {}, cnt[TREX_NCLASS] = {};
      int dres[4] = {0, 0, 0, 0};
      if (e->packed && n == 4) {
        pthread_barrier_t bar;
        pthread_barrier_init(&bar, nullptr, 4);
        g_emu_cta_barrier = &bar;
        e->solves[3]++;
        std::thread th[4];
        for (int i = 0; i < 4; i++)
          th[i] = std::thread([=, &dres]() {
            dres[i] = 255 & trex::front_phase<true, ENVP, EXTF, true>(
                                e->P, mdl, mdli, tasks, cp, cl, e->slabs[i], rec + i * TREX_STATE_STRIDE,
                                e->deferred ? e->work + i * TREX_WORK_STRIDE : nullptr, action + i * trex::NJ, r == 0, e->slabs, i, 0xf,
                                e->deferred ? e->workh + i * TREX_HEAVY_STRIDE : nullptr, ENVP ? rows + i * TREX_ENVP_DIM : nullptr,
                                EXTF ? x->rec[i] : nullptr, com, push, env_id0 + i, tau_max);
          });
        for (int i = 0; i < 4; i++) th[i].join();
        g_emu_cta_barrier = nullptr;
        pthread_barrier_destroy(&bar);
      } else {
        for (int i = 0; i < n; i++)
          dres[i] = 255 & trex::front_phase<false, ENVP, EXTF, true>(
                              e->P, mdl, mdli, tasks, cp, cl, e->S, rec + i * TREX_STATE_STRIDE,
                              e->deferred ? e->work + i * TREX_WORK_STRIDE : nullptr, action + i * trex::NJ, r == 0, nullptr, 0, 0,
                              e->deferred ? e->workh + i * TREX_HEAVY_STRIDE : nullptr, ENVP ? rows + i * TREX_ENVP_DIM : nullptr,
                              EXTF ? x->rec[i] : nullptr, com, push, env_id0 + i, tau_max);
      }
      for (int i = 0; i < n; i++) {
        const int d = dres[i];
        e->solves[d == 0 ? 0 : (d == 1 ? 1 : (d < 1 + TREX_CLASS_HEAVY ? 2 : 4))]++;
        if (d) { int& c = cnt[d - 1]; envs[d - 1][e->pack_reverse ? 3 - c : c] = i; c++; }
      }
      for (int d = 0; d < TREX_NCLASS; d++) {
        if (!cnt[d]) continue;
        const int pending = e->pack_reverse ? (((1 << cnt[d]) - 1) << (4 - cnt[d])) : ((1 << cnt[d]) - 1);
        tmem_t tm4 = {e->tmem};
        if (d == 0) trex::solve_phase<0, false, ENVP>(e->P, e->scratch, e->work, rec, envs[0], pending, tm4, rows);
        else if (d < TREX_CLASS_HEAVY && e->solve_tmem) trex::solve_phase<TREX_KC, true, ENVP>(e->P, e->scratch, e->work, rec, envs[d], pending, tm4, rows);
        else if (d < TREX_CLASS_HEAVY) trex::solve_phase<TREX_KC, false, ENVP>(e->P, e->scratch, e->work, rec, envs[d], pending, tm4, rows);
        else {
          int hv[4], nh = 0;
          for (int g = 0; g < 4; g++)
            if (pending & (1 << g)) hv[nh++] = envs[d][g];
          for (int i = 0; i < nh; i += 2) {
            const bool two = i + 1 < nh;
            int pair[2] = {hv[i], two ? hv[i + 1] : 0};
            int pend = two ? 3 : 1;
            if (e->pack_reverse && !two) { pair[1] = pair[0]; pair[0] = 0; pend = 2; }
            tmem_t tm = {e->tmem};
            if (e->heavy_tmem) trex::heavy_phase<true, ENVP>(e->P, e->scratch2, tm, e->work, e->workh, rec, pair, pend, rows);
            else trex::heavy_phase<false, ENVP>(e->P, e->scratch2, tm, e->work, e->workh, rec, pair, pend, rows);
          }
        }
      }
    }
  }
  for (int i = 0; i < n; i++)
    trex::tail_phase<ENVP, true>(e->P, mdl, mdli, tasks, cp, cl, e->S, rec + i * TREX_STATE_STRIDE, obs ? obs + i * 75 : nullptr,
                                 reward ? reward + i : nullptr, done ? done + i : nullptr, aux ? aux + i * TREX_AUX_STRIDE : nullptr,
                                 force_reset != 0, env_id0 + i, ENVP ? rows + i * TREX_ENVP_DIM : nullptr,
                                 ENVP && p->ranges_on ? p->ranges : nullptr, ENVP ? p->dt : 0.0,
                                 force_reset ? nullptr : action + i * trex::NJ, tau_max);
}

extern "C" {
void emu_tau_step4(void* h, int n, float* rec, const float* action, float* obs, float* reward, uint8_t* done, float* aux,
                   int force_reset, long long env_id0) {
  float tau_max;
  if (!tau_of(h, &tau_max)) return emu_extf_step4(h, n, rec, action, obs, reward, done, aux, force_reset, env_id0);
  Emu* e = (Emu*)h;
  Envp* p = envp_of(h);
  Extf* x = extf_of(h, false);
  if (p && x) step4t<true, true>(e, p, x, tau_max, n, rec, action, obs, reward, done, aux, force_reset, env_id0);
  else if (p) step4t<true, false>(e, p, nullptr, tau_max, n, rec, action, obs, reward, done, aux, force_reset, env_id0);
  else if (x) step4t<false, true>(e, nullptr, x, tau_max, n, rec, action, obs, reward, done, aux, force_reset, env_id0);
  else step4t<false, false>(e, nullptr, nullptr, tau_max, n, rec, action, obs, reward, done, aux, force_reset, env_id0);
}
// from now on the handle runs the TAU instances: its uniform motor settings become kp = kd = 0 and impulse bound 0, as
// trex_create builds them for a torque-mode handle
void emu_set_torque_mode(void* h) {
  Emu* e = (Emu*)h;
  e->P.kp = 0.0f; e->P.kd = 0.0f; e->P.max_impulse = 0.0f;
  std::lock_guard<std::mutex> g(g_tau_lock);
  g_tau[h] = (float)e->T.params[trex_host::P_MAX_TORQUE];
}
void emu_tau_forget(void* h) {
  std::lock_guard<std::mutex> g(g_tau_lock);
  g_tau.erase(h);
}
}
