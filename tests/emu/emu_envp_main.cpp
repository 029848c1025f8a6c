// emu_envp_main.cpp -- builds libtrex_emu_envp.so: the emulator of emu_main.cpp plus the ENVP instances of the product kernels
// (per-environment dynamics parameters, the library's trex_config.env_params = 1).  TEST INFRASTRUCTURE ONLY.
//
// The emulator is included as it is; its three entry points that step or free a handle are renamed here and wrapped, so that a
// handle given parameter rows (emu_set_env_params) runs the ENVP instances and every other handle the uniform ones.
#define emu_step4 emu_step4_uniform
#define emu_step emu_step_uniform
#define emu_destroy emu_destroy_uniform
#include "emu_main.cpp"
#undef emu_step4
#undef emu_step
#undef emu_destroy

#include <mutex>
#include <unordered_map>

// parameter state of a handle that runs the ENVP instances
struct Envp {
  alignas(16) float rows[4][TREX_ENVP_DIM];     // rows of the (up to four) environments of emu_step4
  alignas(16) float ranges[2 * TREX_ENVP_DIM];  // randomizer lo [32] | hi [32]
  int ranges_on = 0;
  double dt = 0.0;                              // physics substep in double (the impulse bound of a row)
};
static std::mutex g_envp_lock;
static std::unordered_map<void*, Envp*> g_envp;
static Envp* envp_of(void* h) {
  std::lock_guard<std::mutex> g(g_envp_lock);
  auto it = g_envp.find(h);
  return it == g_envp.end() ? nullptr : it->second;
}

// one env step (or reset when force_reset) on n (1..4) consecutive environment records, as emu_main.cpp's, with the rows of p
template <bool ENVP>
static void step4(Emu* e, Envp* p, int n, float* rec, const float* action, float* obs, float* reward, uint8_t* done, float* aux, int force_reset,
                  long long env_id0) {
  float* rows = ENVP ? &p->rows[0][0] : nullptr;
  const float* mdl = e->T.mdl.data();
  const int* mdli = e->T.mdli.data();
  const float* tasks = e->T.tasks.data();
  const float* cp = e->T.cand_p.data();
  const int* cl = e->T.cand_lane.data();
  if (!force_reset) {
    for (int r = 0; r < e->P.n_sub; r++) {
      // deferred environments are packed into the solver's lane groups in list order (any order is equivalent)
      // (one list per class, as in the library: contact-free, 1, 2, 3-4, 5-8 and more contacts)
      int envs[TREX_NCLASS][4] = {}, cnt[TREX_NCLASS] = {};
      int dres[4] = {0, 0, 0, 0};
      if (e->packed && n == 4) {
        // the library's 4-warp CTA: warps are host threads, cta_sync() a pthread barrier, warp 0 runs inward_packed
        pthread_barrier_t bar;
        pthread_barrier_init(&bar, nullptr, 4);
        g_emu_cta_barrier = &bar;
        e->solves[3]++;
        std::thread th[4];
        for (int i = 0; i < 4; i++)
          th[i] = std::thread([=, &dres]() {
            dres[i] = 255 & trex::front_phase<true, ENVP>(e->P, mdl, mdli, tasks, cp, cl, e->slabs[i], rec + i * TREX_STATE_STRIDE,
                                              e->deferred ? e->work + i * TREX_WORK_STRIDE : nullptr, action + i * trex::NJ, r == 0,
                                              e->slabs, i, 0xf, e->deferred ? e->workh + i * TREX_HEAVY_STRIDE : nullptr,
                                              ENVP ? rows + i * TREX_ENVP_DIM : nullptr);
          });
        for (int i = 0; i < 4; i++) th[i].join();
        g_emu_cta_barrier = nullptr;
        pthread_barrier_destroy(&bar);
      } else {
        for (int i = 0; i < n; i++)
          dres[i] = 255 & trex::front_phase<false, ENVP>(e->P, mdl, mdli, tasks, cp, cl, e->S, rec + i * TREX_STATE_STRIDE,
                                      e->deferred ? e->work + i * TREX_WORK_STRIDE : nullptr, action + i * trex::NJ, r == 0, nullptr, 0, 0,
                                      e->deferred ? e->workh + i * TREX_HEAVY_STRIDE : nullptr, ENVP ? rows + i * TREX_ENVP_DIM : nullptr);
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
        else {  // class 5: two environments per warp (solve2), packed from the list like the kernel does
          int hv[4], nh = 0;
          for (int g = 0; g < 4; g++)
            if (pending & (1 << g)) hv[nh++] = envs[d][g];
          for (int i = 0; i < nh; i += 2) {
            const bool two = i + 1 < nh;
            int pair[2] = {hv[i], two ? hv[i + 1] : 0};
            int pend = two ? 3 : 1;
            if (e->pack_reverse && !two) { pair[1] = pair[0]; pair[0] = 0; pend = 2; }  // tests: a lone environment in the upper lane group
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
                           ENVP && p->ranges_on ? p->ranges : nullptr, p->dt);
}
extern "C" {
void emu_step4(void* h, int n, float* rec, const float* action, float* obs, float* reward, uint8_t* done, float* aux, int force_reset,
               long long env_id0) {
  if (Envp* p = envp_of(h)) step4<true>((Emu*)h, p, n, rec, action, obs, reward, done, aux, force_reset, env_id0);
  else emu_step4_uniform(h, n, rec, action, obs, reward, done, aux, force_reset, env_id0);
}
void emu_step(void* h, float* rec, const float* action, float* obs, float* reward, uint8_t* done, float* aux, int force_reset,
              long long env_id) {
  emu_step4(h, 1, rec, action, obs, reward, done, aux, force_reset, env_id);
}
void emu_destroy(void* h) {
  {
    std::lock_guard<std::mutex> g(g_envp_lock);
    auto it = g_envp.find(h);
    if (it != g_envp.end()) { delete it->second; g_envp.erase(it); }
  }
  emu_destroy_uniform(h);
}
// from now on the handle runs the ENVP instances, with rows[i] the row of environment i of emu_step4 (n rows of 32 floats;
// element 30 is recomputed from 29, as trex_set_env_params does)
void emu_set_env_params(void* h, const float* rows, int n) {
  Emu* e = (Emu*)h;
  Envp* p = envp_of(h);
  if (!p) {
    p = new Envp();
    p->dt = trex_host::substep_dt(e->T, e->P.n_sub);
    std::lock_guard<std::mutex> g(g_envp_lock);
    g_envp[h] = p;
  }
  for (int i = 0; i < n && i < 4; i++) {
    memcpy(p->rows[i], rows + i * TREX_ENVP_DIM, sizeof(p->rows[i]));
    p->rows[i][trex_host::ENVP_MAX_IMPULSE] = (float)((double)p->rows[i][trex_host::ENVP_MAX_TORQUE] * p->dt);
  }
}
// the model's default row (what trex_create puts in every row)
void emu_default_env_params(void* h, float* row) { Emu* e = (Emu*)h; trex_host::default_env_params(e->T, e->P.n_sub, row); }
void emu_get_env_params(void* h, float* rows, int n) {
  Envp* p = envp_of(h);
  for (int i = 0; p && i < n && i < 4; i++) memcpy(rows + i * TREX_ENVP_DIM, p->rows[i], sizeof(p->rows[i]));
}
// randomizer ranges (lo, hi: 32 floats each; NULL / NULL turns it off) of a handle with rows: 0, or -1 with the reason in
// emu_last_error
int emu_set_env_param_ranges(void* h, const float* lo, const float* hi) {
  Envp* p = envp_of(h);
  if (!p) { snprintf(g_err, sizeof g_err, "the handle has no parameter rows (emu_set_env_params)"); return -1; }
  if (!lo && !hi) { p->ranges_on = 0; return 0; }
  if (!lo || !hi) { snprintf(g_err, sizeof g_err, "both ranges or neither"); return -1; }
  if (const char* why = trex_host::check_env_param_ranges(lo, hi)) { snprintf(g_err, sizeof g_err, "%s", why); return -1; }
  memcpy(p->ranges, lo, TREX_ENVP_DIM * sizeof(float));
  memcpy(p->ranges + TREX_ENVP_DIM, hi, TREX_ENVP_DIM * sizeof(float));
  p->ranges_on = 1;
  return 0;
}
}
