// emu_extf_main.cpp -- builds libtrex_emu_extf.so: the emulator of emu_envp_main.cpp plus the EXTF instances of the front
// phase (external wrenches and the push schedule, the library's trex_config.external_forces = 1).  TEST INFRASTRUCTURE ONLY.
//
// The parameter emulator is included as it is.  A handle given a wrench record (emu_set_external_forces) or a push schedule
// steps through emu_extf_step4, which runs the EXTF instances -- together with the ENVP instances when the handle also has
// parameter rows; every other handle is forwarded to emu_step4 of the included emulator.
#include "emu_envp_main.cpp"

// wrench state of a handle that runs the EXTF instances
struct Extf {
  alignas(16) float rec[4][TREX_EXTF_DIM];  // records [6][32] of the (up to four) environments of emu_step4
  trex::PushSchedule push = {};
};
static std::mutex g_extf_lock;
static std::unordered_map<void*, Extf*> g_extf;
static Extf* extf_of(void* h, bool create) {
  std::lock_guard<std::mutex> g(g_extf_lock);
  auto it = g_extf.find(h);
  if (it != g_extf.end()) return it->second;
  if (!create) return nullptr;
  Extf* x = new Extf();
  memset(x->rec, 0, sizeof x->rec);
  g_extf[h] = x;
  return x;
}

// one env step (or reset when force_reset) on n (1..4) consecutive environment records, as emu_envp_main.cpp's step4, with the
// front phase of the EXTF instances (the solve and tail phases take no wrench)
template <bool ENVP>
static void step4x(Emu* e, Envp* p, Extf* x, int n, float* rec, const float* action, float* obs, float* reward, uint8_t* done,
                   float* aux, int force_reset, long long env_id0) {
  float* rows = ENVP ? &p->rows[0][0] : nullptr;
  const float* mdl = e->T.mdl.data();
  const int* mdli = e->T.mdli.data();
  const float* tasks = e->T.tasks.data();
  const float* cp = e->T.cand_p.data();
  const int* cl = e->T.cand_lane.data();
  const float* com = e->T.com.data();
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
            dres[i] = 255 & trex::front_phase<true, ENVP, true>(e->P, mdl, mdli, tasks, cp, cl, e->slabs[i], rec + i * TREX_STATE_STRIDE,
                                                    e->deferred ? e->work + i * TREX_WORK_STRIDE : nullptr, action + i * trex::NJ, r == 0,
                                                    e->slabs, i, 0xf, e->deferred ? e->workh + i * TREX_HEAVY_STRIDE : nullptr,
                                                    ENVP ? rows + i * TREX_ENVP_DIM : nullptr, x->rec[i], com, &x->push, env_id0 + i);
          });
        for (int i = 0; i < 4; i++) th[i].join();
        g_emu_cta_barrier = nullptr;
        pthread_barrier_destroy(&bar);
      } else {
        for (int i = 0; i < n; i++)
          dres[i] = 255 & trex::front_phase<false, ENVP, true>(e->P, mdl, mdli, tasks, cp, cl, e->S, rec + i * TREX_STATE_STRIDE,
                                                  e->deferred ? e->work + i * TREX_WORK_STRIDE : nullptr, action + i * trex::NJ, r == 0,
                                                  nullptr, 0, 0, e->deferred ? e->workh + i * TREX_HEAVY_STRIDE : nullptr,
                                                  ENVP ? rows + i * TREX_ENVP_DIM : nullptr, x->rec[i], com, &x->push, env_id0 + i);
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
    trex::tail_phase<ENVP>(e->P, mdl, mdli, tasks, cp, cl, e->S, rec + i * TREX_STATE_STRIDE, obs ? obs + i * 75 : nullptr,
                           reward ? reward + i : nullptr, done ? done + i : nullptr, aux ? aux + i * TREX_AUX_STRIDE : nullptr,
                           force_reset != 0, env_id0 + i, ENVP ? rows + i * TREX_ENVP_DIM : nullptr,
                           ENVP && p->ranges_on ? p->ranges : nullptr, ENVP ? p->dt : 0.0);
}

extern "C" {
void emu_extf_step4(void* h, int n, float* rec, const float* action, float* obs, float* reward, uint8_t* done, float* aux,
                    int force_reset, long long env_id0) {
  Extf* x = extf_of(h, false);
  if (!x) return emu_step4(h, n, rec, action, obs, reward, done, aux, force_reset, env_id0);
  if (Envp* p = envp_of(h)) step4x<true>((Emu*)h, p, x, n, rec, action, obs, reward, done, aux, force_reset, env_id0);
  else step4x<false>((Emu*)h, nullptr, x, n, rec, action, obs, reward, done, aux, force_reset, env_id0);
}
// from now on the handle runs the EXTF instances, with wrenches [n][26][6] (the library's user layout) for environments 0..n-1
// of emu_step4 (the records of the others keep their values)
void emu_set_external_forces(void* h, const float* wrench, int n) {
  Extf* x = extf_of(h, true);
  for (int i = 0; i < n && i < 4; i++)
    for (int c = 0; c < 6; c++)
      for (int L = 0; L < 32; L++) x->rec[i][c * 32 + L] = L < trex_topo::NB ? wrench[(i * trex_topo::NB + L) * 6 + c] : 0.0f;
}
void emu_get_external_forces(void* h, float* wrench, int n) {
  Extf* x = extf_of(h, false);
  for (int i = 0; x && i < n && i < 4; i++)
    for (int c = 0; c < 6; c++)
      for (int L = 0; L < trex_topo::NB; L++) wrench[(i * trex_topo::NB + L) * 6 + c] = x->rec[i][c * 32 + L];
}
// push schedule (on = 0: off), validated as trex_set_push_schedule does: 0, or -1 with the reason in emu_last_error
int emu_set_push_schedule(void* h, int on, int body, int interval, int duration, int first_step, float probability, float force_min,
                          float force_max) {
  Extf* x = extf_of(h, true);
  if (!on) { x->push.on = 0; return 0; }
  if (const char* why = trex_host::check_push_schedule(body, interval, duration, first_step, probability, force_min, force_max)) {
    snprintf(g_err, sizeof g_err, "%s", why);
    return -1;
  }
  trex::PushSchedule s = {};
  s.on = 1; s.lane = body; s.interval = interval; s.duration = duration; s.first_step = first_step;
  s.probability = probability; s.force_min = force_min; s.force_max = force_max;
  trex_host::push_directions(s.dir);
  x->push = s;
  return 0;
}
// the COM table as the kernels read it: [3][32]
void emu_body_com(void* h, float* out) { memcpy(out, ((Emu*)h)->T.com.data(), 3 * 32 * sizeof(float)); }
void emu_extf_forget(void* h) {
  std::lock_guard<std::mutex> g(g_extf_lock);
  auto it = g_extf.find(h);
  if (it != g_extf.end()) { delete it->second; g_extf.erase(it); }
}
}
