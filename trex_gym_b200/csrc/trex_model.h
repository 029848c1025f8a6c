// trex_model.h -- host side: parse the model blob (trex_gym_b200/model_blob.py) and lay it out
// as the lane-indexed tables trex_core.h consumes.  Plain C++ (no CUDA) so that both the
// library (trex_capi.cu) and the CPU test emulator (tests/emu) build the tables identically.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <string>
#include <vector>

#include "trex_topology.h"

namespace trex_host {

enum {
  P_TIME_STEP, P_SOLVER_ITERS, P_NUM_SUBSTEPS, P_GRAVITY, P_KP, P_KD, P_MAX_TORQUE, P_LIN_DAMP, P_ANG_DAMP,
  P_MAX_COORD_VEL, P_ERP, P_CONTACT_ERP, P_SPLIT_THRESH, P_LINEAR_SLOP, P_RESIDUAL, P_WARMSTART, P_FRICTION,
  P_BREAKING, P_FLOOR, P_LIMIT_MAX_IMPULSE, P_RESET_HEIGHT, P_TARGET_HEIGHT, P_MAX_CONTACTS, P_COUNT
};

struct Blob {
  const uint8_t* base = nullptr;
  size_t bytes = 0;
  uint32_t nsec = 0;
  std::string err;

  bool open(const void* p, size_t n) {
    base = (const uint8_t*)p;
    bytes = n;
    if (n < 16 || memcmp(p, "TREXMDL1", 8) != 0) { err = "bad model blob magic"; return false; }
    uint32_t version;
    memcpy(&version, base + 8, 4);
    memcpy(&nsec, base + 12, 4);
    if (version != 3) { err = "unsupported model blob version"; return false; }
    if (16 + 40 * (size_t)nsec > n) { err = "truncated model blob"; return false; }
    return true;
  }
  bool find(const char* name, uint32_t dtype, const void** data, uint32_t* count) {
    for (uint32_t i = 0; i < nsec; i++) {
      const uint8_t* e = base + 16 + 40 * (size_t)i;
      char nm[25];
      memcpy(nm, e, 24);
      nm[24] = 0;
      if (strcmp(nm, name) != 0) continue;
      uint32_t dt, cnt;
      uint64_t off;
      memcpy(&dt, e + 24, 4); memcpy(&cnt, e + 28, 4); memcpy(&off, e + 32, 8);
      if (dt != dtype) { err = std::string("section ") + name + ": wrong dtype"; return false; }
      if (off + (size_t)cnt * (dt == 0 ? 8 : 4) > bytes) { err = std::string("section ") + name + ": out of range"; return false; }
      *data = base + off;
      *count = cnt;
      return true;
    }
    err = std::string("section ") + name + " missing";
    return false;
  }
  bool f64(const char* name, std::vector<double>& out, size_t expect = 0) {
    const void* d; uint32_t c;
    if (!find(name, 0, &d, &c)) return false;
    if (expect && c != expect) { err = std::string("section ") + name + ": unexpected size"; return false; }
    out.resize(c);
    memcpy(out.data(), d, 8 * (size_t)c);
    return true;
  }
  bool i32(const char* name, std::vector<int32_t>& out, size_t expect = 0) {
    const void* d; uint32_t c;
    if (!find(name, 1, &d, &c)) return false;
    if (expect && c != expect) { err = std::string("section ") + name + ": unexpected size"; return false; }
    out.resize(c);
    memcpy(out.data(), d, 4 * (size_t)c);
    return true;
  }
};

// Host mirror of trex::Uniform's inputs plus the lane tables.
struct ModelTables {
  std::vector<float> mdl;        // [F_COUNT][32]
  std::vector<int32_t> mdli;     // [IF_COUNT][32]
  std::vector<float> tasks;      // [rounds][4][32]  rx, ry, rz, mass
  std::vector<float> cand_p;     // [4][64]: candidate point / sphere centre x, y, z in body coordinates, sphere radius (0 = point)
  std::vector<int32_t> cand_lane;  // [64]
  std::vector<float> com;        // [3][32]: body-frame centre of mass (mc / mass in double) of each lane's body, 0 elsewhere
  int n_rounds = 0, n_cand = 0, head_lane = 0;
  float head_p[3] = {0, 0, 0};
  float r0[trex_topo::NB][3];
  double params[P_COUNT];
  float lower_sorted[trex_topo::NJ], upper_sorted[trex_topo::NJ];  // name-sorted action limits
  int obs_dof[trex_topo::NJ];
  std::string err;
};

static inline int body_lane(int b) { return b == 0 ? 25 : b - 1; }

static inline bool build_tables(const void* blob, size_t bytes, ModelTables& T, int n_float_fields, int n_int_fields) {
  using namespace trex_topo;
  Blob B;
  if (!B.open(blob, bytes)) { T.err = B.err; return false; }
  std::vector<double> pv, E0, r0, mass, mc, I, drot, lower, upper, jdamp, startq, headp, task_r, task_m, candp, candr;
  std::vector<int32_t> nbv, parent, headb, task_body, cand_body, obs_dof, order;
#define NEED(x) if (!(x)) { T.err = B.err; return false; }
  NEED(B.f64("param_values", pv, P_COUNT));
  NEED(B.i32("mb_n_bodies", nbv, 1));
  if (nbv[0] != NB) { T.err = "model blob has a different number of bodies than the compiled topology"; return false; }
  NEED(B.i32("mb_parent", parent, NB));
  for (int b = 0; b < NB; b++)
    if (parent[b] != parent_of(b)) { T.err = "model blob topology differs from the compiled topology (regenerate trex_topology.h)"; return false; }
  NEED(B.i32("noncontact_order", order, 2 * NJ));
  for (int k = 0; k < 2 * NJ; k++)
    if (order[k] != noncontact_order(k)) { T.err = "model blob constraint order differs from the compiled topology"; return false; }
  NEED(B.f64("mb_E0", E0, NB * 9)); NEED(B.f64("mb_r0", r0, NB * 3)); NEED(B.f64("mb_mass", mass, NB));
  NEED(B.f64("mb_mc", mc, NB * 3)); NEED(B.f64("mb_I", I, NB * 6)); NEED(B.f64("mb_damp_rot", drot, NB * 6));
  NEED(B.f64("mb_lower", lower, NB)); NEED(B.f64("mb_upper", upper, NB)); NEED(B.f64("mb_damping", jdamp, NB));
  NEED(B.f64("mb_start_q", startq, NB)); NEED(B.i32("mb_head_body", headb, 1)); NEED(B.f64("mb_head_p", headp, 3));
  NEED(B.i32("mb_task_body", task_body)); NEED(B.f64("mb_task_r", task_r)); NEED(B.f64("mb_task_m", task_m));
  NEED(B.i32("mb_cand_body", cand_body)); NEED(B.f64("mb_cand_p", candp));
  if (!B.f64("mb_cand_r", candr)) { candr.assign(cand_body.size(), 0.0); B.err.clear(); }  // older blobs: point candidates
  if (candr.size() != cand_body.size()) { T.err = "section mb_cand_r: unexpected size"; return false; }
  NEED(B.i32("obs_dof", obs_dof, NJ));
#undef NEED
  for (int k = 0; k < NJ; k++)
    if (obs_dof[k] != trex_topo::obs_dof(k)) { T.err = "model blob observation order differs from the compiled topology"; return false; }
  memcpy(T.params, pv.data(), sizeof(T.params));

  T.mdl.assign((size_t)n_float_fields * 32, 0.0f);
  T.mdli.assign((size_t)n_int_fields * 32, 0);
  auto F = [&](int f, int lane) -> float& { return T.mdl[(size_t)f * 32 + lane]; };
  auto IF = [&](int f, int lane) -> int32_t& { return T.mdli[(size_t)f * 32 + lane]; };
  // float fields (indices must match trex_core.h enum)
  for (int b = 0; b < NB; b++) {
    const int L = body_lane(b);
    for (int k = 0; k < 9; k++) F(0 + k, L) = (float)E0[9 * b + k];
    for (int k = 0; k < 3; k++) { F(9 + k, L) = (float)r0[3 * b + k]; T.r0[b][k] = (float)r0[3 * b + k]; }
    F(12, L) = (float)mass[b];
    for (int k = 0; k < 3; k++) F(13 + k, L) = (float)mc[3 * b + k];
    for (int k = 0; k < 6; k++) F(16 + k, L) = (float)I[6 * b + k];
    for (int k = 0; k < 6; k++) F(22 + k, L) = (float)drot[6 * b + k];
    F(28, L) = (float)lower[b]; F(29, L) = (float)upper[b]; F(30, L) = (float)jdamp[b]; F(31, L) = (float)startq[b];
  }
  T.com.assign(3 * 32, 0.0f);
  for (int b = 0; b < NB; b++)
    for (int k = 0; k < 3; k++) T.com[(size_t)k * 32 + body_lane(b)] = mass[b] > 0.0 ? (float)(mc[3 * b + k] / mass[b]) : 0.0f;
  // identity rotation for lanes without a body (harmless arithmetic)
  for (int L = 26; L < 32; L++) { F(0, L) = 1.0f; F(4, L) = 1.0f; F(8, L) = 1.0f; }
  // int fields
  int depth[NB];
  for (int b = 0; b < NB; b++) depth[b] = depth_of(b);
  for (int L = 0; L < 32; L++) {
    IF(0, L) = L;   // parent lane
    IF(1, L) = -1;  // depth
    IF(3, L) = 0x00ffffff;  // children: all "none" (63)
    IF(5, L) = L;
    IF(6, L) = 0x00ffffff;
  }
  int nchild[NB] = {0};
  for (int b = 0; b < NB; b++) {
    const int L = body_lane(b);
    IF(1, L) = depth[b];
    if (b > 0) {
      IF(0, L) = body_lane(parent[b]);
      uint32_t m = 0;
      for (int a = b; a > 0; a = parent[a]) m |= 1u << body_lane(a);
      IF(2, L) = (int32_t)m;
      const int p = parent[b];
      if (nchild[p] >= 4) { T.err = "a body has more than 4 children"; return false; }
      int32_t& ch = IF(3, body_lane(p));
      ch = (ch & ~(63 << (6 * nchild[p]))) | (L << (6 * nchild[p]));
      nchild[p]++;
    }
  }
  for (int k = 0; k < NJ; k++) {
    IF(4, obs_dof[k]) = k;  // lane (= joint dof) -> sorted slot
    T.obs_dof[k] = obs_dof[k];
    T.lower_sorted[k] = (float)lower[obs_dof[k] + 1];
    T.upper_sorted[k] = (float)upper[obs_dof[k] + 1];
  }
  // bodies of each tree depth, for the four-environments-per-warp inward pass: field 8 + (d - 1), entry i = lane of the
  // i-th body of depth d (or -1); at most 8 per depth (8 lanes serve one environment there)
  if (n_int_fields >= 8 + trex_topo::MAX_DEPTH) {
    for (int d = 1; d <= trex_topo::MAX_DEPTH; d++) {
      int cnt = 0;
      for (int i = 0; i < 32; i++) IF(8 + d - 1, i) = -1;
      for (int b = 1; b < NB; b++)
        if (depth[b] == d) {
          if (cnt >= 8) { T.err = "more than 8 bodies at one tree depth"; return false; }
          IF(8 + d - 1, cnt++) = body_lane(b);
        }
    }
  }
  // constraint order: the kernel relies on [NJ motors | NJ limit constraints]
  for (int k = 0; k < NJ; k++) {
    if (order[k] < NJ || order[NJ + k] >= NJ) { T.err = "constraint order is not [motors | limits]"; return false; }
    IF(7, k) = order[NJ + k];
  }
  // link-damping tasks: every lane evaluates the links of exactly one body; R rounds
  const int nt = (int)task_body.size();
  int per_body[NB] = {0};
  for (int t = 0; t < nt; t++) per_body[task_body[t]]++;
  int R = 1;
  for (;; R++) {
    int lanes = 0, maxc = 0;
    for (int b = 0; b < NB; b++) { int c = (per_body[b] + R - 1) / R; lanes += c; if (c > maxc) maxc = c; }
    if (lanes <= 32 && maxc <= 4) break;
    if (R > 64) { T.err = "cannot schedule link-damping tasks"; return false; }
  }
  T.n_rounds = R;
  T.tasks.assign((size_t)R * 4 * 32, 0.0f);
  {
    int next_lane = 0;
    for (int b = 0; b < NB; b++) {
      const int c = (per_body[b] + R - 1) / R;
      std::vector<int> mine;
      for (int t = 0; t < nt; t++) if (task_body[t] == b) mine.push_back(t);
      int32_t contrib = 0x00ffffff;
      for (int s = 0; s < c; s++) {
        const int L = next_lane++;
        IF(5, L) = body_lane(b);
        contrib = (contrib & ~(63 << (6 * s))) | (L << (6 * s));
        for (int rd = 0; rd < R; rd++) {
          const size_t idx = (size_t)s * R + rd;
          if (idx >= mine.size()) break;
          const int t = mine[idx];
          float* slot = &T.tasks[(size_t)rd * 4 * 32];
          slot[0 * 32 + L] = (float)task_r[3 * t + 0];
          slot[1 * 32 + L] = (float)task_r[3 * t + 1];
          slot[2 * 32 + L] = (float)task_r[3 * t + 2];
          slot[3 * 32 + L] = (float)task_m[t];
        }
      }
      IF(6, body_lane(b)) = contrib;
    }
  }
  // contact candidates
  T.n_cand = (int)cand_body.size();
  if (T.n_cand > 64) { T.err = "too many contact candidates"; return false; }
  T.cand_p.assign(4 * 64, 0.0f);
  T.cand_lane.assign(64, 25);
  for (int c = 0; c < T.n_cand; c++) {
    T.cand_lane[c] = body_lane(cand_body[c]);
    for (int k = 0; k < 3; k++) T.cand_p[(size_t)k * 64 + c] = (float)candp[3 * c + k];
    T.cand_p[(size_t)3 * 64 + c] = (float)candr[c];
  }
  T.head_lane = body_lane(headb[0]);
  for (int k = 0; k < 3; k++) T.head_p[k] = (float)headp[k];
  return true;
}


struct EnvConfig {
  int num_substeps = 5;
  float distance_weight = 1.0f, energy_weight = 0.005f, drift_weight = 0.002f;  // trex_env.py:42-44
  int max_episode_steps = 0;  // 0 = never terminate (trex_env.py:183-184)
  int enable_contacts = 1;
  int reset_mode = 0;
  unsigned seed = 0;
  long long env_offset = 0;
  float reset_z_min = 0.3f, reset_z_max = 3.0f;
  int defer_contacts = 2;  // 1: substeps with <= 8 contacts also go to the four-environments-per-warp solver; 2: and those with more to solve_heavy
};

// Fill a trex::Uniform (templated so this header stays free of the lane vocabulary).
template <class U>
static inline void fill_uniform(const ModelTables& T, const EnvConfig& C, U& P) {
  const double* p = T.params;
  const int n = C.num_substeps < 1 ? 1 : C.num_substeps;
  P.dt = (float)(p[P_TIME_STEP] / n);                 // trex_env.py:71
  P.iters = (int)(p[P_SOLVER_ITERS] / n);             // trex_env.py:72, :115
  P.n_sub = n;                                        // trex_env.py:73
  P.g = (float)p[P_GRAVITY];
  P.kp = (float)p[P_KP]; P.kd = (float)p[P_KD];
  P.max_impulse = (float)(p[P_MAX_TORQUE] * (p[P_TIME_STEP] / n));  // force * dt
  P.k_lin = (float)p[P_LIN_DAMP]; P.k_ang = (float)p[P_ANG_DAMP];
  P.maxvel = (float)p[P_MAX_COORD_VEL];
  P.erp = (float)p[P_ERP]; P.contact_erp = (float)p[P_CONTACT_ERP];
  P.split_thresh = (float)p[P_SPLIT_THRESH]; P.slop = (float)p[P_LINEAR_SLOP];
  P.resid_thresh = (float)p[P_RESIDUAL]; P.warm = (float)p[P_WARMSTART]; P.mu = (float)p[P_FRICTION];
  P.breaking = (float)p[P_BREAKING]; P.floor_z = (float)p[P_FLOOR];
  P.limit_max_impulse = (float)p[P_LIMIT_MAX_IMPULSE];
  P.reset_z = (float)p[P_RESET_HEIGHT]; P.target_h = (float)p[P_TARGET_HEIGHT];
  P.w_dist = C.distance_weight; P.w_energy = C.energy_weight; P.w_drift = C.drift_weight;
  for (int k = 0; k < 3; k++) P.head_p[k] = T.head_p[k];
  for (int b = 0; b < trex_topo::NB; b++)
    for (int k = 0; k < 3; k++) P.r0[b][k] = T.r0[b][k];
  P.max_episode_steps = C.max_episode_steps;
  P.head_lane = T.head_lane;
  P.n_cand = T.n_cand;
  P.n_rounds = T.n_rounds;
  P.contacts_on = C.enable_contacts;
  P.reset_mode = C.reset_mode;
  P.defer_contacts = C.defer_contacts;
  P.seed = C.seed;
  P.env_offset = C.env_offset;
  P.reset_z_min = C.reset_z_min; P.reset_z_max = C.reset_z_max;
  for (int k = 0; k < 2 * trex_topo::NJ; k++) P.order[k] = (unsigned char)trex_topo::noncontact_order(k);
  for (int b = 0; b < trex_topo::NB; b++) P.depth[b] = (unsigned char)trex_topo::depth_of(b);
  {
    int nch[trex_topo::NB] = {0};
    for (int b = 1; b < trex_topo::NB; b++) nch[trex_topo::parent_of(b)]++;
    for (int d = 0; d <= trex_topo::MAX_DEPTH; d++) P.max_children[d] = 0;
    for (int b = 0; b < trex_topo::NB; b++)
      if (nch[b] > P.max_children[trex_topo::depth_of(b)]) P.max_children[trex_topo::depth_of(b)] = (unsigned char)nch[b];
  }
  {  // bodies from the base's child down to the head body
    int chain[8], n = 0;
    for (int b = T.head_lane == 25 ? 0 : T.head_lane + 1; b > 0; b = trex_topo::parent_of(b)) chain[n++] = b;
    P.head_depth = n;
    for (int d = 0; d < n; d++) P.head_chain[d] = (unsigned char)body_lane(chain[n - 1 - d]);
  }
}

// ---- per-environment parameter rows (layout: trex_core.h, TREX_ENVP_DIM) ---------------------------------------------
enum { ENVP_DIM = 32, ENVP_MASS_BASE = 25, ENVP_MU = 26, ENVP_KP = 27, ENVP_KD = 28, ENVP_MAX_TORQUE = 29, ENVP_MAX_IMPULSE = 30 };

// physics substep in double: the motor impulse bound is torque * this, rounded once to float
static inline double substep_dt(const ModelTables& T, int num_substeps) {
  return T.params[P_TIME_STEP] / (num_substeps < 1 ? 1 : num_substeps);
}

// the row that reproduces the model's own constants: unit mass scales, and friction, gains and bounds as fill_uniform rounds them
static inline void default_env_params(const ModelTables& T, int num_substeps, float row[ENVP_DIM]) {
  const double* p = T.params;
  for (int k = 0; k < ENVP_DIM; k++) row[k] = k <= ENVP_MASS_BASE ? 1.0f : 0.0f;
  row[ENVP_MU] = (float)p[P_FRICTION];
  row[ENVP_KP] = (float)p[P_KP];
  row[ENVP_KD] = (float)p[P_KD];
  row[ENVP_MAX_TORQUE] = (float)p[P_MAX_TORQUE];
  row[ENVP_MAX_IMPULSE] = (float)(p[P_MAX_TORQUE] * substep_dt(T, num_substeps));
}

// randomizer ranges: lo <= hi, all finite, mass scales > 0, friction / gains / torque >= 0, elements 30-31 zero.
// Returns nullptr when valid, else what is wrong.
static inline const char* check_env_param_ranges(const float lo[ENVP_DIM], const float hi[ENVP_DIM]) {
  for (int k = 0; k < ENVP_DIM; k++) {
    if (!(lo[k] - lo[k] == 0.0f) || !(hi[k] - hi[k] == 0.0f)) return "ranges must be finite";
    if (!(lo[k] <= hi[k])) return "every low bound must be <= its high bound";
    if (k <= ENVP_MASS_BASE && !(lo[k] > 0.0f)) return "mass scales must be > 0";
    if (k > ENVP_MASS_BASE && k < ENVP_MAX_IMPULSE && !(lo[k] >= 0.0f)) return "friction, kp, kd and max torque must be >= 0";
    if (k >= ENVP_MAX_IMPULSE && (lo[k] != 0.0f || hi[k] != 0.0f)) return "elements 30 and 31 of the ranges must be zero";
  }
  return nullptr;
}

// ---- push schedule (trex_core.h: PushSchedule, push_of_step) ----------------------------------------------------------
// body 0..25 (wrench-record order: 25 = base), interval >= 1, 1 <= duration <= interval, first_step >= 0,
// 0 <= probability <= 1, 0 <= force_min <= force_max, all finite.  Returns nullptr when valid, else what is wrong.
static inline const char* check_push_schedule(int body, int interval, int duration, int first_step, float probability,
                                              float force_min, float force_max) {
  if (body < 0 || body > 25) return "body must be 0..25 (25 = base)";
  if (interval < 1) return "interval must be >= 1";
  if (duration < 1 || duration > interval) return "duration must be 1..interval";
  if (first_step < 0) return "first_step must be >= 0";
  if (!(probability >= 0.0f && probability <= 1.0f)) return "probability must be in [0, 1]";
  if (!(force_min - force_min == 0.0f) || !(force_max - force_max == 0.0f)) return "forces must be finite";
  if (!(force_min >= 0.0f && force_min <= force_max)) return "0 <= force_min <= force_max must hold";
  return nullptr;
}
// the 32 horizontal push directions (cos, sin of 2 pi k / 32), computed in double and rounded once
static inline void push_directions(float dir[32][2]) {
  for (int k = 0; k < 32; k++) {
    const double a = 6.283185307179586476925 * k / 32.0;
    dir[k][0] = (float)cos(a);
    dir[k][1] = (float)sin(a);
  }
}

}  // namespace trex_host
