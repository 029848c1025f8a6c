// trex_core.h -- the T-rex environment step, one WARP per environment.
//
// Replaces, for the 26-body merged T-rex tree, everything the reference does per
// TrexBulletEnv.step / reset:
//   /root/reference/trex_gym/trex_env.py:128-154 (step), :98-122 (reset), :186-196 (reward)
//   /root/reference/trex_gym/trex_robot.py:359-365 (observations), :377-422 (motor targets)
//   pybullet.stepSimulation (external; semantics restated in SURVEY.md Appendix A)
//
// Mapping (B200: 32-wide warps, everything in registers + a 13.7 KB per-warp shared slab):
//   lane L in [0,25)   joint L  = rigid body L+1 = generalised velocity index 6+L
//   lane 25            floating base body; lanes 25..30 own base velocity coordinates 0..5
//   lane 31            spare
// * tree passes (kinematics, bias forces, articulated inertias, accelerations) run
//   level-synchronously: a lane is a body, parents/children talk through warp shuffles or shared-memory rows;
// * the inverse joint-space inertia is built column-per-lane (31 unit-impulse passes run
//   concurrently, one per lane, reading the per-body data as shared-memory broadcasts).
//   M^-1 is symmetric, so lane d ends up holding exactly the coefficients it needs to
//   update "its" velocity coordinate in the projected Gauss-Seidel sweep;
// * the constraint solve (projected Gauss-Seidel in Bullet's row order) is deferred to kernels of its own: substeps with at
//   most 8 contacts to solve4() (four environments per warp, eight lanes each, contact rows carried in row space), substeps
//   with 9..16 contacts to solve2() (two environments per warp, sixteen lanes each, the Delassus matrix in tensor memory
//   or shared memory); only the reset step uses the one-environment sweep inside substep().
//
// Written against the lane vocabulary of lane_cuda.h (device) / tests/emu/lane_emu.h
// (host emulation for the CPU test-suite).  All control flow is warp-uniform.
#pragma once
#include "trex_topology.h"
#include <stddef.h>

#ifndef TREX_KMAX
#define TREX_KMAX 16  // contact slots per environment (model parameter max_contacts; deepest points first)
#endif
#ifndef TREX_PGS_UNROLL
#define TREX_PGS_UNROLL TREX_ROLLED
#endif
#define TREX_NCAND_MAX 64
#define TREX_MAX_ROUNDS 12
#ifdef TREX_PHASES
#define TREX_STATE_STRIDE 176  // diagnostics build: + 8 per-phase cycle counters at [160,168)
#else
#define TREX_STATE_STRIDE 160  // floats per environment record (see include/trex_b200.h)
#endif
// deferred-solve work record (floats): M^-1 columns [31][32], then per-lane rows
#define W_COL 0
#define W_RHSM 992
#define W_JDI 1024
#define W_DSELF 1056
#define W_RHSL 1088
#define W_SIGMA 1120
// ... followed, for environments with 1..TREX_KC contacts, by the contact rows in "row space" (see solve4):
#define TREX_KC 8                          // contacts per environment the four-environments-per-warp solver accepts
#define W_NC 1152                          // number of contacts (as float)
#define W_CS 1160                          // [KC][16]: rhs n,t1,t2 | jdi | J M^-1 J^T | warm-started normal impulse | candidate index
#define W_BT (W_CS + 16 * TREX_KC)         // [3*KC][32]: the row responses M^-1 J^T by lane (joints 0..24, base coordinates 25..30)
#define W_A4 (W_BT + 96 * TREX_KC)         // [3*KC][KC][4]: A4[r][c'][k'] = J_{c',k'} M^-1 J_r^T
#define TREX_WORK_STRIDE 2848
static_assert(W_A4 + 12 * TREX_KC * TREX_KC <= TREX_WORK_STRIDE && (W_BT % 4) == 0 && (W_A4 % 4) == 0 && (TREX_WORK_STRIDE % 32) == 0,
              "work record layout");
// environments with more contacts (class 5, solve2) keep their contact rows in a record of their own, so the
// main records stay dense: same fields for up to TREX_KW contacts
#define TREX_KW TREX_KMAX
#define H_NC 0
#define H_CS 8
#define H_BT (H_CS + 16 * TREX_KW)
#define H_A4 (H_BT + 96 * TREX_KW)
#define TREX_HEAVY_STRIDE (((H_A4 + 9 * TREX_KW * TREX_KW) + 31) / 32 * 32)  // A: [3*KW][3*KW], A[r][r'] = J_r' M^-1 J_r^T (symmetric)
static_assert((H_BT % 4) == 0 && (H_A4 % 4) == 0 && TREX_KC <= TREX_KW, "heavy record layout");
// deferred environments are listed by class so that the four environments of a solver warp have similar row counts
#define TREX_NCLASS 6                      // 0: contact-free; 1: 1 contact, 2: 2, 3: 3-4, 4: 5-8 (solve4); 5: 9..KW (solve2)
#define TREX_CLASS_HEAVY (TREX_NCLASS - 1)
TREX_TOPO_FN int defer_class(int n_contacts) {
  return n_contacts <= 2 ? n_contacts : (n_contacts <= 4 ? 3 : (n_contacts <= TREX_KC ? 4 : TREX_CLASS_HEAVY));
}
#ifdef TREX_PHASES
#define TREX_AUX_STRIDE 16
#define TREX_TICK(i) { const long long _t = cycle_count(); stats.phase[i] += (float)(_t - _t0); _t0 = _t; }
#else
#define TREX_AUX_STRIDE 8
#define TREX_TICK(i)
#endif

namespace trex {

using trex_topo::NB;
using trex_topo::NJ;
using trex_topo::MAX_DEPTH;

// ---- per-lane model table: float fields, layout [field][32] -----------------------------
enum {
  F_E0 = 0,        // 9: child axes in parent coordinates at q=0 (row major)
  F_R0 = 9,        // 3: child origin in parent coordinates
  F_MASS = 12,     // 1
  F_MC = 13,       // 3: first mass moment (mass * COM) in body coordinates
  F_I = 16,        // 6: rotational inertia about the body origin xx,xy,xz,yy,yz,zz
  F_DROT = 22,     // 6: sum_k R_k diag(I_k) R_k^T over the URDF links of the body (angular damping)
  F_LOWER = 28,
  F_UPPER = 29,
  F_JDAMP = 30,
  F_STARTQ = 31,
  F_COUNT = 32
};
// ---- per-lane model table: int fields, layout [field][32] -------------------------------
enum {
  IF_PARENT_LANE = 0,  // lane of the parent body (25 for children of the base; own lane for base/spare)
  IF_DEPTH = 1,        // tree depth of the body (0 base, -1 for lanes without a body)
  IF_ANC_MASK = 2,     // bit L set <=> body of lane L is this body or one of its ancestors (base excluded)
  IF_CHILDREN = 3,     // 4 x 6 bits: lanes of the children (63 = none)
  IF_OBS_SLOT = 4,     // name-sorted observation/action slot of this joint
  IF_DAMP_LANE = 5,    // lane of the body whose URDF links this lane evaluates for link damping
  IF_DAMP_CONTRIB = 6, // 4 x 6 bits: lanes whose partial damping wrench belongs to this body (63 = none)
  IF_LIMIT_ORDER = 7,  // joint whose limit constraint is solved at position `lane` of the limit block
  IF_LEVEL = 8,        // MAX_DEPTH fields: entry i (< 8) of field IF_LEVEL + d - 1 = lane of the i-th body of depth d, or -1
  IF_COUNT = 8 + MAX_DEPTH
};

struct Uniform {
  float dt, g, kp, kd, max_impulse, k_lin, k_ang, maxvel, erp, contact_erp, split_thresh, slop;
  float resid_thresh, warm, mu, breaking, floor_z, limit_max_impulse, reset_z, target_h;
  float w_dist, w_energy, w_drift;
  float head_p[3];
  float r0[NB][3];  // static-index copy of F_R0 (body index, not lane)
  int iters, n_sub, max_episode_steps, head_lane, n_cand, n_rounds, contacts_on, reset_mode;
  int defer_contacts;     // 1: substeps with 1..TREX_KC contacts are also solved four environments per warp; 2: and those with
                          // more contacts by solve2 (two environments per warp, sixteen lanes each)
  unsigned seed;
  long long env_offset;   // global id of environment 0 of this shard (keys the reset sampler)
  float reset_z_min, reset_z_max;  // reset_mode 1: base height range
  unsigned char order[2 * NJ];  // non-contact constraint order (Bullet's sorted constraint array)
  unsigned char depth[NB];      // tree depth per body
  unsigned char max_children[MAX_DEPTH + 1];  // largest child count among the bodies of each depth
  unsigned char head_chain[MAX_DEPTH];  // lanes of the bodies from the base's child down to the head body
  int head_depth;
};

// Lane-major rows read with 128-bit loads: a stride of 4 x an odd number of floats puts the eight lanes of a quarter warp
// (one 128-bit shared-memory wavefront) on eight different 16-byte bank groups (a stride of 16 would pair lane i with i + 2).
#define TREX_PACK 20  // k.pack: E (9), U (6), invD, r0 (3), parent lane (int bits)
#define TREX_XROW 28  // x.rows: articulated inertia (21) and bias force (6) in the parent's frame, 1 float of padding
static_assert(TREX_PACK % 8 == 4 && TREX_XROW % 8 == 4, "row strides must be 4 x an odd number of floats");
// 128-bit store of four consecutive floats by every lane (the predicate of st4_if is always true and folds away)
TREX_FN void st4_every_lane(float* p, vi idx, const vf v[4]) { st4_if(p, idx, v, lane_id() >= 0); }

// per-warp shared memory slab.  The kinematics-phase arrays (k) and the contact-row arrays (c) are
// never live at the same time and share storage; 13.7 KB per warp at KMAX = 16 -> 16 warps per SM (two per CTA).
struct alignas(16) WarpShared {
  float col[31][32];  // M^-1: col[g][lane] = entry g of the column owned by `lane`
  float tmp[1][32];   // staging: motor impulses / per-joint power
  float lam_cache[TREX_NCAND_MAX];
  float cpos[TREX_KMAX][4];  // active contact point (world) + pad
  int ccand[TREX_KMAX];      // candidate index of the active contact
  int clane[TREX_KMAX];      // body lane of the active contact
  union {
    struct {
      float E[9][32];     // parent -> body rotation, per body lane
      float U[6][32];     // IA * S
      float invD[32];
      float Rw[9][32];    // world -> body rotation
      float xw[3][32];    // body origin, world
      float pack[32][TREX_PACK];  // per body lane: E (9), U (6), invD, r0 (3), parent lane -- body-major, for 128-bit loads
    } k;
    struct {
      float dV[3 * TREX_KMAX][32];   // rows 3*c + {0 normal, 1 t1, 2 t2}: M^-1 J^T, indexed by lane
      float Jc[3 * TREX_KMAX][12];   // compact Jacobian rows: [0:6] base coordinates, [6:11] chain joints by depth, [11] = 0
      unsigned char slot[TREX_KMAX][32];  // which Jc entry each lane multiplies its velocity coordinate with
      unsigned char inv[TREX_KW][16];     // inverse of slot: lane (coordinate) of each Jc entry
    } c;
    struct {                  // the inward pass (both variants) and its exchange with the four-environments-per-warp pass:
      float keep[28][32];     // k.E .. k.xw stay live (k.pack is written after the pass)
      float pA[6][32];        // bias force per body lane (in), later unused
      float cc[5][32];        // Coriolis terms c0 c1 c3 c4 and the joint damping torque (in)
      float uu[32];           // tau - S^T pA per joint (out)
      float rows[32][TREX_XROW];  // per body lane: its articulated inertia and bias force in the parent's frame, handed
                                  // from the children to the parent between levels
      float base[32];         // [0:21] articulated inertia of the base, [21:27] its bias force (out)
    } x;
  };
};
static_assert(sizeof(((WarpShared*)0)->x) <= sizeof(((WarpShared*)0)->c), "exchange area must fit the union");
static_assert(sizeof(((WarpShared*)0)->x.keep) == offsetof(WarpShared, k.pack) - offsetof(WarpShared, k.E),
              "exchange area must start behind k.E .. k.xw");
static_assert(offsetof(WarpShared, x.rows) % 16 == 0 && offsetof(WarpShared, k.pack) % 16 == 0 && sizeof(WarpShared) % 16 == 0,
              "rows of 128-bit accesses");
// link-damping partial wrenches live in dV rows beyond the kinematics-phase arrays
#define TREX_PART_ROW 48  // row (of 32 floats) inside the union where the 6 damping partial rows live
static_assert(sizeof(((WarpShared*)0)->k) <= TREX_PART_ROW * 128, "partials must not overlap the kinematics arrays");
static_assert(sizeof(((WarpShared*)0)->c) >= (TREX_PART_ROW + 6) * 128, "contact-row storage too small for the damping scratch");

TREX_FN constexpr int SI(int i, int j) {  // upper-triangular index of a symmetric 6x6
  return (i <= j) ? (i * 6 - (i * (i - 1)) / 2 + (j - i)) : (j * 6 - (j * (j - 1)) / 2 + (i - j));
}
TREX_FN constexpr int body_lane(int b) { return b == 0 ? 25 : b - 1; }

struct EnvRegs {
  vf q, qd, tgt, tau;  // joint lanes
  float pos[3], quat[4], om[3], vl[3];  // floating base (uniform across lanes)
};

// Active-set signature of an env step (diagnostics for the parity tests: "did kernel and oracle solve the same
// complementarity problem?").  A 24-bit FNV-style hash folded over the substeps, per substep over
//   K  the contact candidates that got rows (two words: candidates 0..31, 32..63)        [front phase]
//   L  joints whose limit row ended with a positive impulse, M  motors that ended on their impulse bound (bit = dof)
//   NF bit c: contact slot c ended with a positive normal impulse; bit 16 + c: its friction pair ended on the cone
//   it PGS iterations executed                                                              [solver]
// kept as an exactly representable float in the environment record (ST_SIG).
TREX_FN uint32_t sig_mix_u(uint32_t h, uint32_t w) { return (h ^ w) * 16777619u; }
#define TREX_CONE_EDGE 0.9999f  // |lambda_t|^2 >= TREX_CONE_EDGE * (mu lambda_n)^2 counts as "on the cone"

struct StepStats {
  uint32_t sig;  // running active-set signature of the env step (see above)
  int iters;     // PGS iterations executed (summed over substeps)
  int contacts;  // active contact points (last substep)
  int overflow;  // contact points dropped because more than TREX_KMAX were active
#ifdef TREX_PHASES
  float phase[8];
#endif
};

#define MDL(f) ldg_ro(mdl, lane + (f) * 32)
#define MDLI(f) ldi(mdli, lane + (f) * 32)

// ---- per-environment dynamics parameters (trex_config.env_params = 1; the ENVP instances of the kernels) ----------------
// One row of 32 floats per environment, lane L reads element L (one 128-byte access per warp):
//   [0, 25)  mass scale of the body of joint L (body L + 1)    [25] mass scale of the base body
//   [26] friction coefficient   [27] motor kp   [28] motor kd   [29] motor max torque (N m)
//   [30] motor impulse bound = [29] * dt, rounded from double (written by the library only)   [31] reserved, 0
// A mass scale multiplies the body's mass, first moment, rotational inertia, angular-damping tensor and the masses of its
// link-damping tasks (uniform density scaling: the COM stays).  Lanes 26..31 hold no body and keep scale 1.
#define TREX_ENVP_DIM 32  // (trex_model.h mirrors the layout for the host: ENVP_*)
enum { EP_MASS_BASE = 25, EP_MU = 26, EP_KP = 27, EP_KD = 28, EP_MAX_TORQUE = 29, EP_MAX_IMPULSE = 30 };
// the randomizer's Philox key word (the reset sampler uses 0xfa11: the two streams stay independent)
#define TREX_ENVP_PHILOX_KEY 0xe9a5u
TREX_FN vf envp_mass_scale(const float* envp, vi lane) { return ld_if(envp, seli(lane <= EP_MASS_BASE, lane, 0), lane <= EP_MASS_BASE, 1.0f); }

// ---- external wrenches (trex_config.external_forces = 1; the EXTF instances of the front kernel) ------------------------
// Record of one environment, lane-major [6][32]: element c * 32 + L = component c of the wrench on the body of lane L (the
// lane numbering of the kernels: L < 25 the body of joint L, 25 the base; lanes 26..31 hold zeros).  Components
// fx fy fz tx ty tz in the world frame: the force acts at the body's centre of mass, the torque is a free vector.  A warp
// reads it with six coalesced 128-byte loads per substep.  com: [3][32] body-frame centre of mass of each lane's body
// (mc / mass of the model, rounded from double; a mass scale leaves it unchanged).
#define TREX_EXTF_DIM (6 * 32)
#define TREX_PUSH_DIRS 32
// the push schedule's Philox key word (0xfa11: reset sampler, 0xe9a5: parameter randomizer)
#define TREX_PUSH_PHILOX_KEY 0x9e57u
// Push schedule (a kernel argument; on == 0: off).  dir: 32 horizontal unit vectors (cos, sin of 2 pi k / 32, rounded
// from double on the host: a table keeps the device and the emulator bit-identical where sinf / cosf would not).
struct PushSchedule {
  int on, lane, interval, duration, first_step;
  float probability, force_min, force_max;
  float dir[TREX_PUSH_DIRS][2];
};
// The wrench inputs of one substep: the environment's record, the COM table, and the push of this substep (warp-uniform;
// lane < 0: none) that is added to the record's force on that lane before the rotation into the body frame.
struct ExtWrench {
  const float* rec = nullptr;
  const float* com = nullptr;
  int push_lane = -1;
  float push_fx = 0.0f, push_fy = 0.0f;
};
// The schedule of environment gid at env step t (steps completed in episode e): window w = t / interval; Philox4x32-10
// keyed by (seed, TREX_PUSH_PHILOX_KEY), counter (gid lo, gid hi, e, w) -> u0..u3.  The window holds a push iff
// u0 < probability, starting at onset o = min(floor(u1 (interval - duration + 1)), interval - duration) into the window
// and lasting `duration` steps; steps before first_step never push.  Magnitude force_min + u2 (force_max - force_min)
// (one fused multiply-add), direction dir[floor(32 u3)].  Stateless: a function of (seed, gid, e, t) only, so it
// depends neither on the number of GPUs nor on when the schedule was set.  Called warp-uniformly.
TREX_FN void push_of_step(const PushSchedule& S, unsigned seed, unsigned long long gid, float episode, float step, ExtWrench& X) {
  const int t = (int)step;
  if (!S.on || t < S.first_step) return;
  const int w = t / S.interval;
  vf u[4];
  philox4_uniform(vi((int)(unsigned)(gid & 0xffffffffull)), vi((int)(unsigned)(gid >> 32)), vi((int)episode), vi(w), seed,
                  TREX_PUSH_PHILOX_KEY, u);
  const float u0 = lane_value(u[0], 0), u1 = lane_value(u[1], 0), u2 = lane_value(u[2], 0), u3 = lane_value(u[3], 0);
  if (!(u0 < S.probability)) return;
  const int span = S.interval - S.duration;
  int o = (int)(u1 * (float)(span + 1));
  o = o < span ? o : span;
  const int r = t - w * S.interval;
  if (r < o || r >= o + S.duration) return;
  const float mag = fmaf(u2, S.force_max - S.force_min, S.force_min);
  const int d = (int)(u3 * (float)TREX_PUSH_DIRS);
  X.push_lane = S.lane;
  X.push_fx = mag * S.dir[d][0];
  X.push_fy = mag * S.dir[d][1];
}

// btClamp semantics: comparison based, so a NaN stays a NaN (fmin/fmax would launder it into a bound)
TREX_FN vf clampv(vf x, float lo, float hi) { return sel(x < lo, lo, sel(x > hi, hi, x)); }
TREX_FN float clampf(float x, float lo, float hi) { return x < lo ? lo : (x > hi ? hi : x); }
// joint torque mode: the commanded torque of a joint lane, clipped to [-bound, bound] with fmin / fmax as the targets are
// clipped; 0 elsewhere.  Unlike np.clip, a NaN command becomes -bound (a NaN target becomes the lower joint limit).  The
// front phase (applied torque) and the tail phase (reported torque) both call it, so the two agree bit for bit.
TREX_FN vf clip_torque(vf a, vb is_joint, float bound) { return sel(is_joint, vmin(vmax(a, -bound), bound), 0.0f); }

// world -> base rotation from the base -> world quaternion (x,y,z,w)
TREX_FN void quat_to_Rb(const float q[4], float Rb[9]) {
  const float x = q[0], y = q[1], z = q[2], w = q[3];
  const float s = 2.0f / (x * x + y * y + z * z + w * w);
  // base->world matrix M; Rb = M^T
  Rb[0] = 1.0f - s * (y * y + z * z); Rb[3] = s * (x * y - w * z);        Rb[6] = s * (x * z + w * y);
  Rb[1] = s * (x * y + w * z);        Rb[4] = 1.0f - s * (x * x + z * z); Rb[7] = s * (y * z - w * x);
  Rb[2] = s * (x * z - w * y);        Rb[5] = s * (y * z + w * x);        Rb[8] = 1.0f - s * (x * x + y * y);
}

// local joint rotation: E = (E0 * Rz(q))^T  (parent coordinates -> body coordinates)
TREX_FN void local_rotation(const float* mdl, vi lane, vf q, vf E[9]) {
  const vf c = vcos(q), s = vsin(q);
  vf e0[9];
  TREX_UNROLL for (int k = 0; k < 9; k++) e0[k] = MDL(F_E0 + k);
  E[0] = c * e0[0] + s * e0[1]; E[1] = c * e0[3] + s * e0[4]; E[2] = c * e0[6] + s * e0[7];
  E[3] = c * e0[1] - s * e0[0]; E[4] = c * e0[4] - s * e0[3]; E[5] = c * e0[7] - s * e0[6];
  E[6] = e0[2]; E[7] = e0[5]; E[8] = e0[8];
}

// Level-synchronous forward kinematics (+ optional spatial velocities in body coordinates).
template <bool WITH_VEL>
TREX_FN void forward_pass(const float* mdl, const int* mdli, vi lane, const EnvRegs& R, const float Rb[9],
                          const vf E[9], vf Rw[9], vf xw[3], vf v[6]) {
  const vi plane = MDLI(IF_PARENT_LANE);
  const vi depth = MDLI(IF_DEPTH);
  vf r0[3];
  TREX_UNROLL for (int k = 0; k < 3; k++) r0[k] = MDL(F_R0 + k);
  TREX_UNROLL for (int k = 0; k < 9; k++) Rw[k] = vbroadcast(Rb[k]);
  TREX_UNROLL for (int k = 0; k < 3; k++) xw[k] = vbroadcast(R.pos[k]);
  if (WITH_VEL) {
    TREX_UNROLL for (int i = 0; i < 3; i++) {
      v[i] = vbroadcast(Rb[3 * i] * R.om[0] + Rb[3 * i + 1] * R.om[1] + Rb[3 * i + 2] * R.om[2]);
      v[3 + i] = vbroadcast(Rb[3 * i] * R.vl[0] + Rb[3 * i + 1] * R.vl[1] + Rb[3 * i + 2] * R.vl[2]);
    }
  }
  TREX_ROLLED for (int d = 1; d <= MAX_DEPTH; d++) {
    const vb at = depth == d;
    vf pR[9], px[3];
    TREX_UNROLL for (int k = 0; k < 9; k++) pR[k] = shflv(Rw[k], plane);
    TREX_UNROLL for (int k = 0; k < 3; k++) px[k] = shflv(xw[k], plane);
    TREX_UNROLL for (int i = 0; i < 3; i++)
      TREX_UNROLL for (int j = 0; j < 3; j++) {
        const vf t = E[3 * i] * pR[j] + E[3 * i + 1] * pR[3 + j] + E[3 * i + 2] * pR[6 + j];
        Rw[3 * i + j] = sel(at, t, Rw[3 * i + j]);
      }
    TREX_UNROLL for (int j = 0; j < 3; j++) {
      const vf t = px[j] + pR[j] * r0[0] + pR[3 + j] * r0[1] + pR[6 + j] * r0[2];
      xw[j] = sel(at, t, xw[j]);
    }
    if (WITH_VEL) {
      vf pv[6];
      TREX_UNROLL for (int k = 0; k < 6; k++) pv[k] = shflv(v[k], plane);
      // linear velocity of the child origin in parent coordinates: v_p + w_p x r
      const vf lx = pv[3] + (pv[1] * r0[2] - pv[2] * r0[1]);
      const vf ly = pv[4] + (pv[2] * r0[0] - pv[0] * r0[2]);
      const vf lz = pv[5] + (pv[0] * r0[1] - pv[1] * r0[0]);
      TREX_UNROLL for (int i = 0; i < 3; i++) {
        vf wa = E[3 * i] * pv[0] + E[3 * i + 1] * pv[1] + E[3 * i + 2] * pv[2];
        const vf la = E[3 * i] * lx + E[3 * i + 1] * ly + E[3 * i + 2] * lz;
        if (i == 2) wa = wa + R.qd;
        v[i] = sel(at, wa, v[i]);
        v[3 + i] = sel(at, la, v[3 + i]);
      }
    }
  }
}

// Cholesky factor of a symmetric positive definite 6x6 given as SI()-packed upper triangle (uniform math):
// L (strict lower part) and the reciprocals of its diagonal.  Solving with the factor (forward + backward substitution,
// 42 operations) replaces an explicit inverse: fewer instructions (27 divisions less) and no squared condition number.
struct Chol6 {
  float L[6][6];
  float rd[6];
};
TREX_FN void spd6_factor(const float a[21], Chol6& c) {
  TREX_UNROLL for (int j = 0; j < 6; j++) {
    float s = a[SI(j, j)];
    TREX_UNROLL for (int k = 0; k < j; k++) s -= c.L[j][k] * c.L[j][k];
    const float id = 1.0f / sqrtf(s);
    c.rd[j] = id;
    TREX_UNROLL for (int i = j + 1; i < 6; i++) {
      float t = a[SI(i, j)];
      TREX_UNROLL for (int k = 0; k < j; k++) t -= c.L[i][k] * c.L[j][k];
      c.L[i][j] = t * id;
    }
  }
}
// x = -A^-1 b for the factored A; T = float (uniform) or vf (one right-hand side per lane)
template <class T>
TREX_FN void spd6_solve_neg(const Chol6& c, const T b[6], T x[6]) {
  T y[6];
  TREX_UNROLL for (int i = 0; i < 6; i++) {
    T t = b[i];
    TREX_UNROLL for (int k = 0; k < i; k++) t = t - y[k] * c.L[i][k];
    y[i] = t * c.rd[i];
  }
  TREX_UNROLL for (int i = 5; i >= 0; i--) {
    T t = y[i];
    TREX_UNROLL for (int k = i + 1; k < 6; k++) t = t - x[k] * c.L[k][i];
    x[i] = t * c.rd[i];
  }
  TREX_UNROLL for (int i = 0; i < 6; i++) x[i] = -x[i];
}

// child -> parent transform of an articulated inertia (SI packed, child coordinates) and a
// spatial force.  E: parent->child rotation, r: child origin in parent coordinates.
//   I_p = X^T I X ,  f_p = X^T f ,  X = [[E, 0], [-E [r]x, E]]
// The inertia passed in is Ia = IA - U U^T / D of a joint about the child's z axis: Ia S = 0, i.e. row and column 2
// (the angular z coordinate) vanish.  They are taken as exactly zero (not read), which shortens the congruence.
TREX_FN void to_parent(const vf E[9], const vf r[3], const vf Ia[21], const vf pa[6], vf Ip[21], vf pp[6]) {
  // rotate the blocks into parent axes: K' = E^T K E
  vf Ar[3][3], Br[3][3], Mr[3][3];
  {  // A = angular-angular block: only A00 A01 A11 are non-zero
    const vf a00 = Ia[SI(0, 0)], a01 = Ia[SI(0, 1)], a11 = Ia[SI(1, 1)];
    vf T0[3], T1[3];
    TREX_UNROLL for (int j = 0; j < 3; j++) {
      T0[j] = a00 * E[j] + a01 * E[3 + j];
      T1[j] = a01 * E[j] + a11 * E[3 + j];
    }
    TREX_UNROLL for (int i = 0; i < 3; i++)
      TREX_UNROLL for (int j = i; j < 3; j++) Ar[i][j] = E[i] * T0[j] + E[3 + i] * T1[j];
  }
  {  // B = angular-linear block: row 2 is zero
    vf T0[3], T1[3];
    TREX_UNROLL for (int j = 0; j < 3; j++) {
      T0[j] = Ia[SI(0, 3)] * E[j] + Ia[SI(0, 4)] * E[3 + j] + Ia[SI(0, 5)] * E[6 + j];
      T1[j] = Ia[SI(1, 3)] * E[j] + Ia[SI(1, 4)] * E[3 + j] + Ia[SI(1, 5)] * E[6 + j];
    }
    TREX_UNROLL for (int i = 0; i < 3; i++)
      TREX_UNROLL for (int j = 0; j < 3; j++) Br[i][j] = E[i] * T0[j] + E[3 + i] * T1[j];
  }
  {  // M = linear-linear block: full, symmetric
    vf T[3][3];
    TREX_UNROLL for (int i = 0; i < 3; i++)
      TREX_UNROLL for (int j = 0; j < 3; j++)
        T[i][j] = Ia[SI(3 + i, 3)] * E[j] + Ia[SI(3 + i, 4)] * E[3 + j] + Ia[SI(3 + i, 5)] * E[6 + j];
    TREX_UNROLL for (int i = 0; i < 3; i++)
      TREX_UNROLL for (int j = i; j < 3; j++) {
        Mr[i][j] = E[i] * T[0][j] + E[3 + i] * T[1][j] + E[6 + i] * T[2][j];
        Mr[j][i] = Mr[i][j];
      }
  }
  // K = [r]x Mr ; Bp = Br + K ; Ap = Ar + [r]x Br^T + ([r]x Bp^T)^T
  vf K[3][3], C[3][3], Dm[3][3], Bp[3][3];
  TREX_UNROLL for (int j = 0; j < 3; j++) {
    K[0][j] = r[1] * Mr[2][j] - r[2] * Mr[1][j];
    K[1][j] = r[2] * Mr[0][j] - r[0] * Mr[2][j];
    K[2][j] = r[0] * Mr[1][j] - r[1] * Mr[0][j];
  }
  TREX_UNROLL for (int i = 0; i < 3; i++)
    TREX_UNROLL for (int j = 0; j < 3; j++) Bp[i][j] = Br[i][j] + K[i][j];
  TREX_UNROLL for (int j = 0; j < 3; j++) {  // C = [r]x Br^T ; Dm = [r]x Bp^T
    C[0][j] = r[1] * Br[j][2] - r[2] * Br[j][1];
    C[1][j] = r[2] * Br[j][0] - r[0] * Br[j][2];
    C[2][j] = r[0] * Br[j][1] - r[1] * Br[j][0];
    Dm[0][j] = r[1] * Bp[j][2] - r[2] * Bp[j][1];
    Dm[1][j] = r[2] * Bp[j][0] - r[0] * Bp[j][2];
    Dm[2][j] = r[0] * Bp[j][1] - r[1] * Bp[j][0];
  }
  TREX_UNROLL for (int i = 0; i < 3; i++)
    TREX_UNROLL for (int j = i; j < 3; j++) {
      Ip[SI(i, j)] = Ar[i][j] + C[i][j] + Dm[j][i];
      Ip[SI(3 + i, 3 + j)] = Mr[i][j];
    }
  TREX_UNROLL for (int i = 0; i < 3; i++)
    TREX_UNROLL for (int j = 0; j < 3; j++) Ip[SI(i, 3 + j)] = Bp[i][j];
  // force: f' = E^T f ; n' = E^T n + r x f'
  vf fn[3], ff[3];
  TREX_UNROLL for (int i = 0; i < 3; i++) {
    fn[i] = E[i] * pa[0] + E[3 + i] * pa[1] + E[6 + i] * pa[2];
    ff[i] = E[i] * pa[3] + E[3 + i] * pa[4] + E[6 + i] * pa[5];
  }
  pp[0] = fn[0] + (r[1] * ff[2] - r[2] * ff[1]);
  pp[1] = fn[1] + (r[2] * ff[0] - r[0] * ff[2]);
  pp[2] = fn[2] + (r[0] * ff[1] - r[1] * ff[0]);
  pp[3] = ff[0]; pp[4] = ff[1]; pp[5] = ff[2];
}

// End of a physics substep: velocities += dv (each coordinate clamped, btMultiBody::applyDeltaVeeMultiDof), applied motor
// torque read-back, then positions with the NEW velocities (btMultiBody::stepPositionsMultiDof).
// dv: this lane's coordinate of the velocity change (joints on lanes 0..24, base coordinates on lanes 25..30).
TREX_FN void finish_substep(const Uniform& P, vi lane, EnvRegs& R, vf dv, vf lam_m) {
  const vb is_joint = lane < NJ;
  const float dt = P.dt;
  R.qd = sel(is_joint, clampv(R.qd + dv, -P.maxvel, P.maxvel), 0.0f);
  TREX_UNROLL for (int k = 0; k < 3; k++) {
    R.om[k] = clampf(R.om[k] + lane_value(dv, 25 + k), -P.maxvel, P.maxvel);
    R.vl[k] = clampf(R.vl[k] + lane_value(dv, 28 + k), -P.maxvel, P.maxvel);
  }
  R.tau = sel(is_joint, vdiv(lam_m, dt), 0.0f);  // appliedJointMotorTorque = impulse / dt
  TREX_UNROLL for (int k = 0; k < 3; k++) R.pos[k] += dt * R.vl[k];
  {
    float fAngle = sqrtf(R.om[0] * R.om[0] + R.om[1] * R.om[1] + R.om[2] * R.om[2]);
    if (fAngle * dt > 0.78539816339744831f) fAngle = 0.78539816339744831f / dt;
    float sc;
    if (fAngle < 0.001f) sc = 0.5f * dt - (dt * dt * dt) * 0.020833333333f * fAngle * fAngle;
    else sc = sinf(0.5f * fAngle * dt) / fAngle;
    const float ax = R.om[0] * sc, ay = R.om[1] * sc, az = R.om[2] * sc, aw = cosf(fAngle * dt * 0.5f);
    const float x = R.quat[0], y = R.quat[1], z = R.quat[2], w = R.quat[3];
    const float nx = aw * x + ax * w + ay * z - az * y;
    const float ny = aw * y - ax * z + ay * w + az * x;
    const float nz = aw * z + ax * y - ay * x + az * w;
    const float nw = aw * w - ax * x - ay * y - az * z;
    const float inv = 1.0f / sqrtf(nx * nx + ny * ny + nz * nz + nw * nw);
    R.quat[0] = nx * inv; R.quat[1] = ny * inv; R.quat[2] = nz * inv; R.quat[3] = nw * inv;
  }
  R.q = sel(is_joint, R.q + dt * R.qd, 0.0f);
}

// ------------------------------------------------------------------------------------------
// Inward pass (articulated inertias) of FOUR environments by one warp: the front kernel's 4-warp CTAs.
//
// In the one-environment pass a lane is a body and every tree level runs the whole 6x6 congruence on 32 lanes of
// which 4-7 hold a body of that depth.  Here eight lanes serve one environment and lane i of a group takes the i-th
// body of the current depth, so 16-28 of 32 lanes work on every level, for four environments at once.  Inputs (E, bias
// force, Coriolis terms) and outputs (U, 1/D, u, the base's inertia and bias force) go through the environments'
// shared slabs (WarpShared::x); children hand their transformed inertia to the parent through the slab as well.
// Same operations in the same order as the one-environment pass: bit-identical results.
// ------------------------------------------------------------------------------------------
// ENVP: envp_cta = parameter row of the CTA's first environment (the four rows are consecutive); the level constants of a
// body are scaled by its mass scale in its environment's row
template <bool ENVP = false>
TREX_FN void inward_packed(const Uniform& P, const float* mdl, const int* mdli, WarpShared* slabs, int valid_mask,
                           const float* envp_cta = nullptr) {
  const vi lane = lane_id();
  const vi e = lane >> 3, i = lane & 7;
  const vb env_ok = ((vi(valid_mask) >> e) & 1) != 0;
  float* sb = reinterpret_cast<float*>(slabs);
  const vi eo = e * (int)(sizeof(WarpShared) / sizeof(float));
  constexpr int O_E = offsetof(WarpShared, k.E) / 4, O_U = offsetof(WarpShared, k.U) / 4, O_ID = offsetof(WarpShared, k.invD) / 4;
  constexpr int O_PA = offsetof(WarpShared, x.pA) / 4, O_CC = offsetof(WarpShared, x.cc) / 4, O_UU = offsetof(WarpShared, x.uu) / 4;
  constexpr int O_ROWS = offsetof(WarpShared, x.rows) / 4, O_BASE = offsetof(WarpShared, x.base) / 4;
  // the body this lane handles at each level: the i-th of depth d (depth 0: the base, lane 0 of the group)
  vi blv[MAX_DEPTH + 1];
  blv[0] = seli(i == 0, vi(25), vi(-1));
  TREX_UNROLL for (int d = 1; d <= MAX_DEPTH; d++) blv[d] = ldi(mdli, i + (IF_LEVEL + d - 1) * 32);
  // model constants of the body, loaded one level ahead (global loads off the level-to-level dependence chain)
  vf n_mass, n_mc[3], n_I3[6], n_r0[3], n_sc = 1.0f;
  vi n_children;
  const vi ep_row = seli(env_ok, e, 0) * TREX_ENVP_DIM;
#define TREX_LOAD_LEVEL_CONSTANTS(BL)                                                       \
  {                                                                                         \
    const vi b_ = (BL);                                                                     \
    if (ENVP) n_sc = ld(envp_cta, ep_row + b_);                                             \
    n_mass = ldg_ro(mdl, b_ + F_MASS * 32);                                                 \
    TREX_UNROLL for (int k = 0; k < 3; k++) n_mc[k] = ldg_ro(mdl, b_ + (F_MC + k) * 32);    \
    TREX_UNROLL for (int k = 0; k < 6; k++) n_I3[k] = ldg_ro(mdl, b_ + (F_I + k) * 32);     \
    TREX_UNROLL for (int k = 0; k < 3; k++) n_r0[k] = ldg_ro(mdl, b_ + (F_R0 + k) * 32);    \
    n_children = ldi(mdli, b_ + IF_CHILDREN * 32);                                          \
  }
  TREX_LOAD_LEVEL_CONSTANTS(seli(env_ok && (blv[MAX_DEPTH] >= 0), blv[MAX_DEPTH], 0))
  TREX_ROLLED for (int d = MAX_DEPTH; d >= 0; d--) {
    vi bl0 = blv[0], bln = blv[0];
    TREX_UNROLL for (int dd = 1; dd <= MAX_DEPTH; dd++) {
      bl0 = seli(vi(d) == dd, blv[dd], bl0);
      bln = seli(vi(d) == dd + 1, blv[dd], bln);  // the next level's body (d - 1)
    }
    const vb has = env_ok && (bl0 >= 0);
    const vi bl = seli(has, bl0, 0);
    // own spatial inertia (model constants) and the bias force computed by the environment's own warp
    vf mc[3], I3[6], r0[3], pA[6];
    const vf mass = ENVP ? n_mass * n_sc : n_mass;
    const vi children = n_children;
    TREX_UNROLL for (int k = 0; k < 3; k++) { mc[k] = ENVP ? n_mc[k] * n_sc : n_mc[k]; r0[k] = n_r0[k]; }
    TREX_UNROLL for (int k = 0; k < 6; k++) I3[k] = ENVP ? n_I3[k] * n_sc : n_I3[k];
    if (d > 0) TREX_LOAD_LEVEL_CONSTANTS(seli(env_ok && (bln >= 0), bln, 0))
    TREX_UNROLL for (int k = 0; k < 6; k++) pA[k] = ld(sb, eo + bl + (O_PA + k * 32));
    vf IA[21];
    TREX_UNROLL for (int k = 0; k < 21; k++) IA[k] = 0.0f;
    IA[SI(0, 0)] = I3[0]; IA[SI(0, 1)] = I3[1]; IA[SI(0, 2)] = I3[2];
    IA[SI(1, 1)] = I3[3]; IA[SI(1, 2)] = I3[4]; IA[SI(2, 2)] = I3[5];
    IA[SI(0, 4)] = -mc[2]; IA[SI(0, 5)] = mc[1];
    IA[SI(1, 3)] = mc[2];  IA[SI(1, 5)] = -mc[0];
    IA[SI(2, 3)] = -mc[1]; IA[SI(2, 4)] = mc[0];
    IA[SI(3, 3)] = mass; IA[SI(4, 4)] = mass; IA[SI(5, 5)] = mass;
    // children (all one level deeper, finished in the previous round), in child-slot order
    if (d < MAX_DEPTH) {
      const int nslots = P.max_children[d];
      TREX_ROLLED for (int sidx = 0; sidx < nslots; sidx++) {
        const vi cl = (children >> (6 * sidx)) & 63;
        const vb ok = has && (cl != 63);
        const vi cls = seli(ok, cl, bl);
        // (+0 without the child, not a 0/1 factor: a row that was never written may hold anything, 0 * NaN included)
        vf row[TREX_XROW];
        TREX_UNROLL for (int j = 0; j < TREX_XROW / 4; j++) ld4_if(sb, eo + O_ROWS + cls * TREX_XROW + 4 * j, ok, row + 4 * j);
        TREX_UNROLL for (int k = 0; k < 21; k++) IA[k] = IA[k] + row[k];
        TREX_UNROLL for (int k = 0; k < 6; k++) pA[k] = pA[k] + row[21 + k];
      }
    }
    if (d == 0) {  // the base: hand its articulated inertia and bias force to the environment's warp
      TREX_UNROLL for (int k = 0; k < 21; k++) st_if(sb, eo + (O_BASE + k), IA[k], has);
      TREX_UNROLL for (int k = 0; k < 6; k++) st_if(sb, eo + (O_BASE + 21 + k), pA[k], has);
      break;
    }
    vf E[9];
    TREX_UNROLL for (int k = 0; k < 9; k++) E[k] = ld(sb, eo + bl + (O_E + k * 32));
    const vf c0 = ld(sb, eo + bl + O_CC), c1 = ld(sb, eo + bl + (O_CC + 32)), c3 = ld(sb, eo + bl + (O_CC + 64)),
             c4 = ld(sb, eo + bl + (O_CC + 96)), tau_j = ld(sb, eo + bl + (O_CC + 128));
    // U = IA S, D = S^T U, u = tau - S^T pA      (S = unit z rotation)
    vf Ut[6];
    Ut[0] = IA[SI(0, 2)]; Ut[1] = IA[SI(1, 2)]; Ut[2] = IA[SI(2, 2)];
    Ut[3] = IA[SI(2, 3)]; Ut[4] = IA[SI(2, 4)]; Ut[5] = IA[SI(2, 5)];
    const vf Dt = Ut[2];
    const vb okD = Dt >= 1.1920929e-7f;
    const vf iD = sel(okD, vdiv(1.0f, sel(okD, Dt, 1.0f)), 0.0f);
    const vf ut = tau_j - pA[2];
    TREX_UNROLL for (int k = 0; k < 6; k++) st_if(sb, eo + bl + (O_U + k * 32), Ut[k], has);
    st_if(sb, eo + bl + O_ID, iD, has);
    st_if(sb, eo + bl + O_UU, ut, has);
    vf Ia[21];
    TREX_UNROLL for (int a = 0; a < 6; a++)
      TREX_UNROLL for (int b = a; b < 6; b++) Ia[SI(a, b)] = IA[SI(a, b)] - (Ut[a] * iD) * Ut[b];
    vf pa[6];
    const vf s = ut * iD;
    TREX_UNROLL for (int a = 0; a < 6; a++)  // (row 2 of Ia is zero)
      pa[a] = a == 2 ? pA[a] + Ut[a] * s : pA[a] + (Ia[SI(a, 0)] * c0 + Ia[SI(a, 1)] * c1 + Ia[SI(a, 3)] * c3 + Ia[SI(a, 4)] * c4) + Ut[a] * s;
    vf row[TREX_XROW];  // Ip (21), pp (6), padding
    to_parent(E, r0, Ia, pa, row, row + 21);
    row[27] = 0.0f;
    TREX_UNROLL for (int j = 0; j < TREX_XROW / 4; j++) st4_if(sb, eo + O_ROWS + bl * TREX_XROW + 4 * j, row + 4 * j, has);
    warp_sync();
  }
#undef TREX_LOAD_LEVEL_CONSTANTS
  warp_sync();
}

// ------------------------------------------------------------------------------------------
// One pybullet stepSimulation (SURVEY.md Appendix A.3) for the environment owned by this warp.
// kp/kd/max_imp: motor settings of this substep (zero during the reset step).
// ------------------------------------------------------------------------------------------
// Returns 0 when the step is complete, or 1 + class when the solve was deferred (`work` != nullptr and at most TREX_KC
// contacts): the solver inputs were written to `work` and the caller finishes the step with solve4() on the
// environments of that class (0: contact-free, 1: 1-2 contacts, 2: 3-4, 3: 5-8).
// PACKED (front kernel with 4-warp CTAs): the inward pass of the CTA's four environments is done by warp 0
// (inward_packed) between two CTA barriers; cta_slabs = slab of warp 0, valid_mask = which warps hold an environment.
// ENVP: envp = this environment's parameter row (mass scales and friction; the caller passes the row's motor settings)
// EXTF: *xf = the external wrenches of this substep (record, COM table, scheduled push)
// TAU: tau_action = the step's actions [25] name-sorted, the joint torques; clipped to +-tau_bound they enter as explicit joint
// torques next to the damping (read where they are added, not held in registers across the kinematics)
template <bool PACKED = false, bool ENVP = false, bool EXTF = false, bool TAU = false>
TREX_FN int substep(const Uniform& P, const float* mdl, const int* mdli, const float* tasks, const float* cand_p,
                     const int* cand_lane, WarpShared& S, EnvRegs& R, float kp, float kd, float max_imp,
                     StepStats& stats, float* work, WarpShared* cta_slabs = nullptr, int warp_in_cta = 0, int valid_mask = 0,
                     float* workh = nullptr, const float* envp = nullptr, const ExtWrench* xf = nullptr,
                     const float* tau_action = nullptr, float tau_bound = 0.0f) {
  const vi lane = lane_id();
  const vb is_joint = lane < NJ;
  const vb is_base = lane == 25;
  const vi plane = MDLI(IF_PARENT_LANE);
  const vi depth = MDLI(IF_DEPTH);
  const vi anc = MDLI(IF_ANC_MASK);
  const float dt = P.dt;

#ifdef TREX_PHASES
  long long _t0 = cycle_count();
#endif
  float Rb[9];
  quat_to_Rb(R.quat, Rb);

  // ---- 1-2. kinematics and velocities ---------------------------------------------------
  vf E[9];
  local_rotation(mdl, lane, R.q, E);
  TREX_UNROLL for (int k = 0; k < 9; k++) E[k] = sel(is_base, vbroadcast(Rb[k]), E[k]);
  vf Rw[9], xw[3], v[6];
  forward_pass<true>(mdl, mdli, lane, R, Rb, E, Rw, xw, v);
  TREX_UNROLL for (int k = 0; k < 9; k++) st(S.k.Rw[k], lane, Rw[k]);
  TREX_UNROLL for (int k = 0; k < 3; k++) st(S.k.xw[k], lane, xw[k]);
  if (PACKED) {  // input of inward_packed
    TREX_UNROLL for (int k = 0; k < 9; k++) st(S.k.E[k], lane, E[k]);
  }

  TREX_TICK(0)
  // ---- 3. bias forces: p = v x* (I v) - gravity wrench + angular damping ------------------
  const vf msc = ENVP ? envp_mass_scale(envp, lane) : vf(1.0f);  // this lane's body's mass scale
  const vf mass = ENVP ? MDL(F_MASS) * msc : MDL(F_MASS);
  vf mc[3], I3[6];
  TREX_UNROLL for (int k = 0; k < 3; k++) mc[k] = ENVP ? MDL(F_MC + k) * msc : MDL(F_MC + k);
  TREX_UNROLL for (int k = 0; k < 6; k++) I3[k] = ENVP ? MDL(F_I + k) * msc : MDL(F_I + k);
  vf pA[6];
  {
    const vf wx = v[0], wy = v[1], wz = v[2], lx = v[3], ly = v[4], lz = v[5];
    // n = I w + mc x v ; f = m v - mc x w
    const vf nx = I3[0] * wx + I3[1] * wy + I3[2] * wz + (mc[1] * lz - mc[2] * ly);
    const vf ny = I3[1] * wx + I3[3] * wy + I3[4] * wz + (mc[2] * lx - mc[0] * lz);
    const vf nz = I3[2] * wx + I3[4] * wy + I3[5] * wz + (mc[0] * ly - mc[1] * lx);
    const vf fx = mass * lx - (mc[1] * wz - mc[2] * wy);
    const vf fy = mass * ly - (mc[2] * wx - mc[0] * wz);
    const vf fz = mass * lz - (mc[0] * wy - mc[1] * wx);
    pA[0] = (wy * nz - wz * ny) + (ly * fz - lz * fy);
    pA[1] = (wz * nx - wx * nz) + (lz * fx - lx * fz);
    pA[2] = (wx * ny - wy * nx) + (lx * fy - ly * fx);
    pA[3] = wy * fz - wz * fy;
    pA[4] = wz * fx - wx * fz;
    pA[5] = wx * fy - wy * fx;
    // gravity as an external force on every body: world (0,0,-g) in body coordinates = -g * Rw[:,2]
    const vf gx = -P.g * Rw[2], gy = -P.g * Rw[5], gz = -P.g * Rw[8];
    pA[0] -= mc[1] * gz - mc[2] * gy;
    pA[1] -= mc[2] * gx - mc[0] * gz;
    pA[2] -= mc[0] * gy - mc[1] * gx;
    pA[3] -= mass * gx; pA[4] -= mass * gy; pA[5] -= mass * gz;
    if (EXTF) {
      // external wrench (world force F at the COM c, world torque T), entering like gravity:
      // f_b = Rw F, n_b = c x f_b + Rw T (Rw: world -> body; the gravity term above reads its third column)
      vf F[3], T[3], c[3];
      TREX_UNROLL for (int k = 0; k < 3; k++) {
        F[k] = ld(xf->rec, lane + k * 32);
        T[k] = ld(xf->rec, lane + (3 + k) * 32);
        c[k] = ldg_ro(xf->com, lane + k * 32);
      }
      if (xf->push_lane >= 0) {  // the scheduled push joins the record's force before the rotation
        const vb on = lane == xf->push_lane;
        F[0] = sel(on, F[0] + xf->push_fx, F[0]);
        F[1] = sel(on, F[1] + xf->push_fy, F[1]);
      }
      vf fb[3], nb[3];
      TREX_UNROLL for (int i = 0; i < 3; i++) {
        fb[i] = Rw[3 * i] * F[0] + Rw[3 * i + 1] * F[1] + Rw[3 * i + 2] * F[2];
        nb[i] = Rw[3 * i] * T[0] + Rw[3 * i + 1] * T[1] + Rw[3 * i + 2] * T[2];
      }
      nb[0] += c[1] * fb[2] - c[2] * fb[1];
      nb[1] += c[2] * fb[0] - c[0] * fb[2];
      nb[2] += c[0] * fb[1] - c[1] * fb[0];
      TREX_UNROLL for (int k = 0; k < 3; k++) { pA[k] -= nb[k]; pA[3 + k] -= fb[k]; }
    }
    // angular damping of every URDF link of the body: (sum R I R^T) w (k + k|w|)
    vf dr[6];
    TREX_UNROLL for (int k = 0; k < 6; k++) dr[k] = ENVP ? MDL(F_DROT + k) * msc : MDL(F_DROT + k);
    const vf wn = vsqrt(wx * wx + wy * wy + wz * wz);
    const vf ka = P.k_ang + P.k_ang * wn;
    pA[0] += (dr[0] * wx + dr[1] * wy + dr[2] * wz) * ka;
    pA[1] += (dr[1] * wx + dr[3] * wy + dr[4] * wz) * ka;
    pA[2] += (dr[2] * wx + dr[4] * wy + dr[5] * wz) * ka;
  }
  // ---- 4. linear damping, evaluated at the COM of every original URDF link -----------------
  {
    const vi dl = MDLI(IF_DAMP_LANE);
    vf bv[6];
    TREX_UNROLL for (int k = 0; k < 6; k++) bv[k] = shflv(v[k], dl);
    const vf tsc = ENVP ? shflv(msc, dl) : vf(1.0f);  // mass scale of the body whose links this lane evaluates
    vf acc[6];
    TREX_UNROLL for (int k = 0; k < 6; k++) acc[k] = 0.0f;
    // (latency bound: four table loads feed ~25 dependent operations per round -- several rounds in flight)
    _Pragma("unroll 5") for (int rd = 0; rd < P.n_rounds; rd++) {
      const float* t = tasks + rd * 4 * 32;
      const vf rx = ldg_ro(t, lane), ry = ldg_ro(t, lane + 32), rz = ldg_ro(t, lane + 64), m = ENVP ? ldg_ro(t, lane + 96) * tsc : ldg_ro(t, lane + 96);
      const vf cx = bv[3] + (bv[1] * rz - bv[2] * ry);
      const vf cy = bv[4] + (bv[2] * rx - bv[0] * rz);
      const vf cz = bv[5] + (bv[0] * ry - bv[1] * rx);
      const vf sc = m * (P.k_lin + P.k_lin * vsqrt(cx * cx + cy * cy + cz * cz));
      const vf fx = cx * sc, fy = cy * sc, fz = cz * sc;
      acc[0] += ry * fz - rz * fy;
      acc[1] += rz * fx - rx * fz;
      acc[2] += rx * fy - ry * fx;
      acc[3] += fx; acc[4] += fy; acc[5] += fz;
    }
    warp_sync();
    TREX_UNROLL for (int k = 0; k < 6; k++) st(reinterpret_cast<float*>(&S.c) + (TREX_PART_ROW + k) * 32, lane, acc[k]);
    warp_sync();
    const vi contrib = MDLI(IF_DAMP_CONTRIB);
    TREX_UNROLL for (int s = 0; s < 4; s++) {
      const vi cl = (contrib >> (6 * s)) & 63;
      const vb ok = cl != 63;
      const vi cls = seli(ok, cl, lane);
      TREX_UNROLL for (int k = 0; k < 6; k++) pA[k] += sel(ok, ld(reinterpret_cast<float*>(&S.c) + (TREX_PART_ROW + k) * 32, cls), 0.0f);
    }
    warp_sync();
  }

  // Coriolis term c = v x (S qd), S = z rotation: only 4 non-zero components
  const vf c0 = R.qd * v[1], c1 = -(R.qd * v[0]), c3 = R.qd * v[4], c4 = -(R.qd * v[3]);
  // explicit joint damping torque (pybullet adds -damping*qd before each step); TAU: plus the commanded torque, written
  // -(d qd - tau) so that a zero command gives the bits of -(d qd), signed zeros included (tau - d qd would turn -0 into +0)
  const vf tau_cmd = TAU ? clip_torque(ld_if(tau_action, seli(is_joint, MDLI(IF_OBS_SLOT), 0), is_joint, 0.0f), is_joint, tau_bound) : vf(0.0f);
  const vf tau_j = TAU ? -(MDL(F_JDAMP) * R.qd - tau_cmd) : -(MDL(F_JDAMP) * R.qd);

  TREX_TICK(1)
  // ---- 5. inward pass: articulated inertias ---------------------------------------------------
  vf IA[21];
  TREX_UNROLL for (int k = 0; k < 21; k++) IA[k] = 0.0f;
  IA[SI(0, 0)] = I3[0]; IA[SI(0, 1)] = I3[1]; IA[SI(0, 2)] = I3[2];
  IA[SI(1, 1)] = I3[3]; IA[SI(1, 2)] = I3[4]; IA[SI(2, 2)] = I3[5];
  IA[SI(0, 4)] = -mc[2]; IA[SI(0, 5)] = mc[1];
  IA[SI(1, 3)] = mc[2];  IA[SI(1, 5)] = -mc[0];
  IA[SI(2, 3)] = -mc[1]; IA[SI(2, 4)] = mc[0];
  IA[SI(3, 3)] = mass; IA[SI(4, 4)] = mass; IA[SI(5, 5)] = mass;
  vf r0[3];
  TREX_UNROLL for (int k = 0; k < 3; k++) r0[k] = MDL(F_R0 + k);
  const vi children = MDLI(IF_CHILDREN);
  vf U[6], invD = 0.0f, uu = 0.0f;
  TREX_UNROLL for (int k = 0; k < 6; k++) U[k] = 0.0f;
  if (PACKED) {
    // publish this environment's inputs, let warp 0 run the pass for the CTA's four environments, fetch the results
    TREX_UNROLL for (int k = 0; k < 6; k++) st(S.x.pA[k], lane, pA[k]);
    st(S.x.cc[0], lane, c0); st(S.x.cc[1], lane, c1); st(S.x.cc[2], lane, c3); st(S.x.cc[3], lane, c4); st(S.x.cc[4], lane, tau_j);
    cta_sync();
    if (warp_in_cta == 0) inward_packed<ENVP>(P, mdl, mdli, cta_slabs, valid_mask, ENVP ? envp - TREX_ENVP_DIM * warp_in_cta : nullptr);
    cta_sync();
    TREX_UNROLL for (int k = 0; k < 6; k++) U[k] = sel(is_joint, ld(S.k.U[k], lane), 0.0f);
    invD = sel(is_joint, ld(S.k.invD, lane), 0.0f);
    uu = sel(is_joint, ld(S.x.uu, lane), 0.0f);
  }
  TREX_ROLLED for (int d = PACKED ? 0 : MAX_DEPTH; d >= 1; d--) {
    const vb at = depth == d;
    // U = IA S, D = S^T U, u = tau - S^T pA      (S = unit z rotation)
    vf Ut[6];
    Ut[0] = IA[SI(0, 2)]; Ut[1] = IA[SI(1, 2)]; Ut[2] = IA[SI(2, 2)];
    Ut[3] = IA[SI(2, 3)]; Ut[4] = IA[SI(2, 4)]; Ut[5] = IA[SI(2, 5)];
    const vf Dt = Ut[2];
    const vb okD = Dt >= 1.1920929e-7f;
    const vf iD = sel(okD, vdiv(1.0f, sel(okD, Dt, 1.0f)), 0.0f);
    const vf ut = tau_j - pA[2];
    TREX_UNROLL for (int k = 0; k < 6; k++) U[k] = sel(at, Ut[k], U[k]);
    invD = sel(at, iD, invD);
    uu = sel(at, ut, uu);
    // Ia = IA - U U^T / D
    vf Ia[21];
    TREX_UNROLL for (int i = 0; i < 6; i++)
      TREX_UNROLL for (int j = i; j < 6; j++) Ia[SI(i, j)] = IA[SI(i, j)] - (Ut[i] * iD) * Ut[j];
    // pa = pA + Ia c + U u / D
    vf pa[6];
    const vf s = ut * iD;
    TREX_UNROLL for (int i = 0; i < 6; i++)  // (row 2 of Ia is zero)
      pa[i] = i == 2 ? pA[i] + Ut[i] * s : pA[i] + (Ia[SI(i, 0)] * c0 + Ia[SI(i, 1)] * c1 + Ia[SI(i, 3)] * c3 + Ia[SI(i, 4)] * c4) + Ut[i] * s;
    vf row[TREX_XROW];  // Ip (21), pp (6), padding
    to_parent(E, r0, Ia, pa, row, row + 21);
    row[27] = 0.0f;
    // parents (depth d-1) gather from their children (all at depth d) through the lane-major rows of x.rows (seven
    // 128-bit accesses per row); only as many child slots as any body of that depth has (tree constant), accumulated
    // with a 0/1 mask through one FMA per element.  Every lane publishes its row and a lane without that child reads
    // back its own, written this level: its masked FMA adds 0 * its own value, never 0 * a stale NaN.
    float* rows = &S.x.rows[0][0];
    warp_sync();  // the previous level's gather is done with the rows
    TREX_UNROLL for (int j = 0; j < TREX_XROW / 4; j++) st4_every_lane(rows, lane * TREX_XROW + 4 * j, row + 4 * j);
    warp_sync();
    const vb parent_now = depth == (d - 1);
    const int nslots = P.max_children[d - 1];
    TREX_ROLLED for (int sidx = 0; sidx < nslots; sidx++) {
      const vi cl = (children >> (6 * sidx)) & 63;
      const vb ok = parent_now && (cl != 63);
      const vi cls = seli(ok, cl, lane);
      const vf okf = sel(ok, 1.0f, 0.0f);
      vf ch[TREX_XROW];
      TREX_UNROLL for (int j = 0; j < TREX_XROW / 4; j++) ld4(rows, cls * TREX_XROW + 4 * j, ch + 4 * j);
      TREX_UNROLL for (int k = 0; k < 21; k++) IA[k] = vfma(okf, ch[k], IA[k]);
      TREX_UNROLL for (int k = 0; k < 6; k++) pA[k] = vfma(okf, ch[21 + k], pA[k]);
    }
  }
  float ia0[21], pA0[6], a0[6];
  if (PACKED) {
    TREX_UNROLL for (int k = 0; k < 21; k++) ia0[k] = ldu(S.x.base, k);
    TREX_UNROLL for (int k = 0; k < 6; k++) pA0[k] = ldu(S.x.base, 21 + k);
  } else {
    TREX_UNROLL for (int k = 0; k < 21; k++) ia0[k] = lane_value(IA[k], 25);
    TREX_UNROLL for (int k = 0; k < 6; k++) pA0[k] = lane_value(pA[k], 25);
  }
  warp_sync();  // pack overwrites the exchange area
  {
    vf pk[TREX_PACK];
    TREX_UNROLL for (int k = 0; k < 9; k++) pk[k] = E[k];
    TREX_UNROLL for (int k = 0; k < 6; k++) pk[9 + k] = U[k];
    pk[15] = invD;
    TREX_UNROLL for (int k = 0; k < 3; k++) pk[16 + k] = r0[k];
    pk[19] = vi2f_bits(plane);
    TREX_UNROLL for (int j = 0; j < TREX_PACK / 4; j++) st4_every_lane(&S.k.pack[0][0], lane * TREX_PACK + 4 * j, pk + 4 * j);
  }

  TREX_TICK(2)
  // ---- 6. base acceleration --------------------------------------------------------------------
  Chol6 chol0;
  spd6_factor(ia0, chol0);
  spd6_solve_neg<float>(chol0, pA0, a0);

  // ---- 7. outward pass: accelerations -------------------------------------------------------------
  vf a[6];
  TREX_UNROLL for (int k = 0; k < 6; k++) a[k] = vbroadcast(a0[k]);
  vf qdd = 0.0f;
  TREX_ROLLED for (int d = 1; d <= MAX_DEPTH; d++) {
    const vb at = depth == d;
    vf ap[6];
    TREX_UNROLL for (int k = 0; k < 6; k++) ap[k] = shflv(a[k], plane);
    const vf lx = ap[3] + (ap[1] * r0[2] - ap[2] * r0[1]);
    const vf ly = ap[4] + (ap[2] * r0[0] - ap[0] * r0[2]);
    const vf lz = ap[5] + (ap[0] * r0[1] - ap[1] * r0[0]);
    vf an[6];
    TREX_UNROLL for (int i = 0; i < 3; i++) {
      an[i] = E[3 * i] * ap[0] + E[3 * i + 1] * ap[1] + E[3 * i + 2] * ap[2];
      an[3 + i] = E[3 * i] * lx + E[3 * i + 1] * ly + E[3 * i + 2] * lz;
    }
    an[0] += c0; an[1] += c1; an[3] += c3; an[4] += c4;
    const vf dd = (uu - (U[0] * an[0] + U[1] * an[1] + U[2] * an[2] + U[3] * an[3] + U[4] * an[4] + U[5] * an[5])) * invD;
    an[2] += dd;
    qdd = sel(at, dd, qdd);
    TREX_UNROLL for (int k = 0; k < 6; k++) a[k] = sel(at, an[k], a[k]);
  }

  // ---- 8. velocities += dt * acceleration, each coordinate clamped (btMultiBody::applyDeltaVeeMultiDof) ----
  R.qd = sel(is_joint, clampv(R.qd + dt * qdd, -P.maxvel, P.maxvel), 0.0f);
  {
    const float wb[3] = {Rb[0] * R.om[0] + Rb[1] * R.om[1] + Rb[2] * R.om[2], Rb[3] * R.om[0] + Rb[4] * R.om[1] + Rb[5] * R.om[2],
                         Rb[6] * R.om[0] + Rb[7] * R.om[1] + Rb[8] * R.om[2]};
    const float vb_[3] = {Rb[0] * R.vl[0] + Rb[1] * R.vl[1] + Rb[2] * R.vl[2], Rb[3] * R.vl[0] + Rb[4] * R.vl[1] + Rb[5] * R.vl[2],
                          Rb[6] * R.vl[0] + Rb[7] * R.vl[1] + Rb[8] * R.vl[2]};
    const float al[3] = {a0[3] + (wb[1] * vb_[2] - wb[2] * vb_[1]), a0[4] + (wb[2] * vb_[0] - wb[0] * vb_[2]),
                         a0[5] + (wb[0] * vb_[1] - wb[1] * vb_[0])};
    TREX_UNROLL for (int j = 0; j < 3; j++) {
      const float wd = Rb[j] * a0[0] + Rb[3 + j] * a0[1] + Rb[6 + j] * a0[2];
      const float vd = Rb[j] * al[0] + Rb[3 + j] * al[1] + Rb[6 + j] * al[2];
      R.om[j] = clampf(R.om[j] + dt * wd, -P.maxvel, P.maxvel);
      R.vl[j] = clampf(R.vl[j] + dt * vd, -P.maxvel, P.maxvel);
    }
  }
  warp_sync();

  TREX_TICK(3)
  // ---- 9. M^-1, one column per lane (btMultiBody::calcAccelerationDeltasMultiDof for unit impulses) ----
  {
    // (a) inward along this lane's own ancestor path
    vf z[6];
    TREX_UNROLL for (int k = 0; k < 6; k++) z[k] = sel(is_joint, U[k] * invD, 0.0f);
    vf Ydep[MAX_DEPTH + 1];
    TREX_UNROLL for (int dd = 0; dd <= MAX_DEPTH; dd++) Ydep[dd] = sel(is_joint && (depth == dd), 1.0f, 0.0f);
    // E, r0 and the parent lane of the body the walk has reached (while it is active): this lane's own to begin
    // with, then the parent's pack row, loaded in the step before for its U and 1/D
    vf Ec[9], rc[3];
    vi par = plane;
    TREX_UNROLL for (int k = 0; k < 9; k++) Ec[k] = E[k];
    TREX_UNROLL for (int k = 0; k < 3; k++) rc[k] = r0[k];
    TREX_ROLLED for (int s = 0; s < MAX_DEPTH; s++) {
      const vb active = is_joint && ((depth - s) >= 1);
      const vb par_joint = active && (par != 25);
      const vi ps = seli(par_joint, par, lane);
      vf pr[TREX_PACK];
      TREX_UNROLL for (int j = 0; j < TREX_PACK / 4; j++) ld4(&S.k.pack[0][0], ps * TREX_PACK + 4 * j, pr + 4 * j);
      vf fn[3], ff[3];
      TREX_UNROLL for (int i = 0; i < 3; i++) {
        fn[i] = Ec[i] * z[0] + Ec[3 + i] * z[1] + Ec[6 + i] * z[2];
        ff[i] = Ec[i] * z[3] + Ec[3 + i] * z[4] + Ec[6 + i] * z[5];
      }
      vf zn[6];
      zn[0] = fn[0] + (rc[1] * ff[2] - rc[2] * ff[1]);
      zn[1] = fn[1] + (rc[2] * ff[0] - rc[0] * ff[2]);
      zn[2] = fn[2] + (rc[0] * ff[1] - rc[1] * ff[0]);
      zn[3] = ff[0]; zn[4] = ff[1]; zn[5] = ff[2];
      // at a joint parent: Y = -S^T z ; z += U * Y / D
      const vf Yp = -zn[2];
      const vf sc = Yp * pr[15];
      TREX_UNROLL for (int k = 0; k < 6; k++) z[k] = sel(active, sel(par_joint, zn[k] + pr[9 + k] * sc, zn[k]), z[k]);
      const vi pd = depth - s - 1;
      TREX_UNROLL for (int dd = 1; dd <= MAX_DEPTH; dd++) Ydep[dd] = sel(par_joint && (pd == dd), Yp, Ydep[dd]);
      // the walk stays active only while it is below a joint parent, so the row just loaded is the next step's
      TREX_UNROLL for (int k = 0; k < 9; k++) Ec[k] = pr[k];
      TREX_UNROLL for (int k = 0; k < 3; k++) rc[k] = pr[16 + k];
      par = vf2i_bits(pr[19]);
    }
    // base-coordinate lanes: unit torque / force on the base, rotated into base coordinates
    {
      const vi kk = lane - 25;
      TREX_UNROLL for (int k = 0; k < 3; k++) {
        // column kk of Rb
        const vf rk = sel(kk == 0 || kk == 3, vbroadcast(Rb[3 * k]), sel(kk == 1 || kk == 4, vbroadcast(Rb[3 * k + 1]), vbroadcast(Rb[3 * k + 2])));
        const vb isw = (lane >= 25) && (lane < 28);
        const vb isv = (lane >= 28) && (lane < 31);
        z[k] = sel(isw, -rk, sel(is_joint, z[k], 0.0f));
        z[3 + k] = sel(isv, -rk, sel(is_joint, z[3 + k], 0.0f));
      }
    }
    // (b) base: a0 = -IA0^-1 z
    vf astk[MAX_DEPTH + 1][6];  // accelerations along the current root-to-body path, by depth
    spd6_solve_neg<vf>(chol0, z, astk[0]);
    TREX_UNROLL for (int dd = 1; dd <= MAX_DEPTH; dd++)
      TREX_UNROLL for (int k = 0; k < 6; k++) astk[dd][k] = 0.0f;
    // (c) outward over the whole tree in body order (parents first).  The loop is rolled to keep the
    // code in the instruction cache; the depth switch keeps every register index static.
    TREX_ROLLED for (int b = 1; b < NB; b++) {
      const int bl = b - 1;
      const int dep = P.depth[b];
      float pk[16];
      ldu16(&S.k.pack[0][0], bl * TREX_PACK, pk);  // four 128-bit broadcast loads
      const float* Eb = pk;
      const float* Ub = pk + 9;
      const float iDb = pk[15];
      const float rx = P.r0[b][0], ry = P.r0[b][1], rz = P.r0[b][2];
      const vb onpath = ((anc >> bl) & 1) != 0;
      vf ddq = 0.0f;
#define TREX_COL_BODY(D)                                                                              \
      {                                                                                               \
        const vf* ap = astk[(D) - 1];                                                                 \
        vf* an = astk[(D)];                                                                           \
        const vf lx = ap[3] + (ap[1] * rz - ap[2] * ry);                                              \
        const vf ly = ap[4] + (ap[2] * rx - ap[0] * rz);                                              \
        const vf lz = ap[5] + (ap[0] * ry - ap[1] * rx);                                              \
        vf t[6];                                                                                      \
        TREX_UNROLL for (int i = 0; i < 3; i++) {                                                     \
          t[i] = Eb[3 * i] * ap[0] + Eb[3 * i + 1] * ap[1] + Eb[3 * i + 2] * ap[2];                   \
          t[3 + i] = Eb[3 * i] * lx + Eb[3 * i + 1] * ly + Eb[3 * i + 2] * lz;                        \
        }                                                                                             \
        const vf Yb = sel(onpath, Ydep[(D)], 0.0f);                                                   \
        ddq = (Yb - (Ub[0] * t[0] + Ub[1] * t[1] + Ub[2] * t[2] + Ub[3] * t[3] + Ub[4] * t[4] + Ub[5] * t[5])) * iDb; \
        t[2] += ddq;                                                                                  \
        TREX_UNROLL for (int k = 0; k < 6; k++) an[k] = t[k];                                         \
      }
      switch (dep) {
        case 1: TREX_COL_BODY(1) break;
        case 2: TREX_COL_BODY(2) break;
        case 3: TREX_COL_BODY(3) break;
        case 4: TREX_COL_BODY(4) break;
        default: TREX_COL_BODY(5) break;
      }
#undef TREX_COL_BODY
      st(S.col[6 + bl], lane, ddq);
    }
    TREX_UNROLL for (int j = 0; j < 3; j++) {
      st(S.col[j], lane, Rb[j] * astk[0][0] + Rb[3 + j] * astk[0][1] + Rb[6 + j] * astk[0][2]);
      st(S.col[3 + j], lane, Rb[j] * astk[0][3] + Rb[3 + j] * astk[0][4] + Rb[6 + j] * astk[0][5]);
    }
  }
  warp_sync();

  TREX_TICK(4)
  // ---- 10. constraint rows -------------------------------------------------------------------------
  // the lane's two contact candidates (model constants): loaded here, ahead of the joint-row arithmetic, so that the two
  // dependent global loads (body lane, then its pose from shared memory) are not exposed at the contact detection
  vi c_bl[2];
  vf c_px[2], c_py[2], c_pz[2], c_pr[2];
  TREX_UNROLL for (int half = 0; half < 2; half++) {
    const vi ci = lane + 32 * half;
    const vi cis = seli(ci < P.n_cand, ci, 0);
    c_bl[half] = ldi(cand_lane, cis);
    c_px[half] = ldg_ro(cand_p, cis); c_py[half] = ldg_ro(cand_p, cis + TREX_NCAND_MAX);
    c_pz[half] = ldg_ro(cand_p, cis + 2 * TREX_NCAND_MAX); c_pr[half] = ldg_ro(cand_p, cis + 3 * TREX_NCAND_MAX);
  }
  // this lane's own velocity coordinate and diagonal of M^-1
  vf uown = R.qd;
  vf dself = 0.0f;
  TREX_UNROLL for (int k = 0; k < 3; k++) {
    uown = sel(lane == 25 + k, vbroadcast(R.om[k]), uown);
    uown = sel(lane == 28 + k, vbroadcast(R.vl[k]), uown);
  }
  uown = sel(lane == 31, 0.0f, uown);
  {
    // generalised index owned by this lane: joints 6+lane, base coordinates lane-25
    const vi gown = seli(is_joint, lane + 6, seli(lane < 31, lane - 25, 0));
    dself = sel(lane < 31, ld(&S.col[0][0], gown * 32 + lane), 0.0f);
  }
  // joint rows: J = +-e_j so the response is +-column j and J M^-1 J^T = M^-1[j][j]
  const vb okJ = is_joint && (dself > 1.1920929e-7f);
  const vf jdi = sel(okJ, vdiv(1.0f, sel(okJ, dself, 1.0f)), 0.0f);
  // motor (btMultiBodyJointMotor): target velocity kp*(target-q)/dt + qd + kd*(0-qd), impulse in [-max,max]
  const vf vt = kp * (R.tgt - R.q) / dt + R.qd + kd * (0.0f - R.qd);
  const vf rhs_m = (vt - R.qd) * jdi;
  vf lam_m = 0.0f;
  vf lamr[NJ];  // motor impulses, replicated on every lane (uniform values)
  TREX_UNROLL for (int j = 0; j < NJ; j++) lamr[j] = 0.0f;
  // joint limits (btMultiBodyJointLimitConstraint): a row only while the limit is violated
  const vf lower = MDL(F_LOWER), upper = MDL(F_UPPER);
  const vf pen_lo = R.q - lower, pen_hi = upper - R.q;
  const vb act_lo = is_joint && !(pen_lo > 0.0f);
  const vb act_hi = is_joint && !(pen_hi > 0.0f);
  // shallow violations (> split threshold, i.e. -0.04 < pen <= 0) combine the ERP push-back with the velocity term;
  // deep ones keep the velocity part only (Bullet moves their positional part to m_rhsPenetration, which the
  // multibody solver never consumes) [RECALL btMultiBodyJointLimitConstraint::createConstraintRows]
  const vf rhs_lo = sel(pen_lo > P.split_thresh, (-pen_lo * P.erp / dt + (-R.qd)) * jdi, (-R.qd) * jdi);
  const vf rhs_hi = sel(pen_hi > P.split_thresh, (-pen_hi * P.erp / dt + (R.qd)) * jdi, (R.qd) * jdi);
  vf lam_lo = 0.0f, lam_hi = 0.0f;
  const uint32_t mask_lo = vballot(act_lo), mask_hi = vballot(act_hi);
  // violated joints in the order Bullet solves their limit constraints: bit p <=> order[NJ + p] is violated
  uint32_t lim_perm;
  {
    const vi pj = ldi(mdli, lane + IF_LIMIT_ORDER * 32);
    lim_perm = vballot((lane < NJ) && ((((vi((int)(mask_lo | mask_hi))) >> pj) & 1) != 0));
  }

  // contacts: candidate points against the floor plane
  int n_act = 0;
  vf c_lam[3], c_rhs[3], c_jdi[3], c_dd[3];  // lane s holds the scalars of active contact s (normal, t1, t2)
  TREX_UNROLL for (int k = 0; k < 3; k++) { c_lam[k] = 0.0f; c_rhs[k] = 0.0f; c_jdi[k] = 0.0f; c_dd[k] = 0.0f; }
  vf dv = 0.0f;  // this lane's coordinate of the accumulated delta velocity
  if (P.contacts_on) {
    vf wpos[2][3];
    vi cbl[2];
    vb cact[2];
    uint32_t am[2];
    TREX_UNROLL for (int half = 0; half < 2; half++) {
      const vi ci = lane + 32 * half;
      const vb valid = ci < P.n_cand;
      const vi cis = seli(valid, ci, 0);
      const vi bl = c_bl[half];
      const vf px = c_px[half], py = c_py[half], pz = c_pz[half];
      // world point = xw + Rw^T p
      wpos[half][0] = ld(S.k.xw[0], bl) + ld(S.k.Rw[0], bl) * px + ld(S.k.Rw[3], bl) * py + ld(S.k.Rw[6], bl) * pz;
      wpos[half][1] = ld(S.k.xw[1], bl) + ld(S.k.Rw[1], bl) * px + ld(S.k.Rw[4], bl) * py + ld(S.k.Rw[7], bl) * pz;
      // a sphere candidate (radius > 0, contact primitives fitted to the meshes) touches the floor with its lowest point:
      // centre - r * normal, a WORLD offset (not body fixed), exactly what a sphere-plane manifold point is
      wpos[half][2] = (ld(S.k.xw[2], bl) + ld(S.k.Rw[2], bl) * px + ld(S.k.Rw[5], bl) * py + ld(S.k.Rw[8], bl) * pz) - c_pr[half];
      cbl[half] = bl;
      cact[half] = valid && ((wpos[half][2] - P.floor_z) < P.breaking);
      am[half] = vballot(cact[half]);
    }
    const int total = popc_u(am[0]) + popc_u(am[1]);
    if (total > TREX_KMAX) {
      // more candidates inside the breaking distance than contact slots: keep the TREX_KMAX deepest
      // (ties by candidate index) -- the points left out are the ones hovering highest above the floor
      stats.overflow += total - TREX_KMAX;
      TREX_UNROLL for (int half = 0; half < 2; half++) {
        vi better = 0;
        TREX_UNROLL for (int h2 = 0; h2 < 2; h2++) {
          TREX_ROLLED for (int l2 = 0; l2 < 32; l2++) {
            if (!((am[h2] >> l2) & 1u)) continue;
            const float z2 = lane_value(wpos[h2][2], l2);
            const vi idx2 = vi(l2 + 32 * h2), idx = lane + 32 * half;
            better = better + seli((z2 < wpos[half][2]) || ((z2 == wpos[half][2]) && (idx2 < idx)), vi(1), vi(0));
          }
        }
        cact[half] = cact[half] && (better < TREX_KMAX);
      }
      am[0] = vballot(cact[0]);
      am[1] = vballot(cact[1]);
    }
    TREX_UNROLL for (int half = 0; half < 2; half++) {
      const vi ci = lane + 32 * half;
      const vb valid = ci < P.n_cand;
      const vi cis = seli(valid, ci, 0);
      // slot = rank among the kept candidates, in candidate order
      const vi rank = rank_below(am[half]) + n_act;
      const vb keep = cact[half];
      const vi slot = seli(keep, rank, 0);
      st_if(&S.cpos[0][0], slot * 4 + 0, wpos[half][0], keep);
      st_if(&S.cpos[0][0], slot * 4 + 1, wpos[half][1], keep);
      st_if(&S.cpos[0][0], slot * 4 + 2, wpos[half][2], keep);
      sti_if(S.ccand, slot, ci, keep);
      sti_if(S.clane, slot, cbl[half], keep);
      // contact points that left the manifold lose their cached impulse
      st_if(S.lam_cache, cis, 0.0f, valid && !keep);
      n_act += popc_u(am[half]);
    }
    warp_sync();
    stats.sig = sig_mix_u(sig_mix_u(stats.sig, am[0]), am[1]) & 0xffffffu;  // K: the candidates with rows
  } else {
    stats.sig = sig_mix_u(sig_mix_u(stats.sig, 0u), 0u) & 0xffffffu;
  }
  // Deferred solve: solve4() finishes this substep, four environments per warp.  Always when there are no contact
  // rows (the rows are then the 25 motors and the violated joint limits, all with unit Jacobians); with up to
  // TREX_KC contacts when P.defer_contacts.  The solver inputs go to the work record: M^-1, the per-joint row
  // scalars and -- below -- the contact rows.
  // (workh: more than TREX_KC contacts go to solve2, two environments per warp)
  const bool defer_c = work != nullptr && P.defer_contacts != 0 && n_act > 0 && n_act <= ((P.defer_contacts > 1 && workh != nullptr) ? TREX_KW : TREX_KC);
  if (work != nullptr && (n_act == 0 || defer_c)) {
    _Pragma("unroll 8") for (int gq = 0; gq < trex_topo::NDOF; gq++) st(work, lane + (W_COL + gq * 32), ld(S.col[gq], lane));
    st(work, lane + W_RHSM, rhs_m);
    st(work, lane + W_JDI, jdi);
    st(work, lane + W_DSELF, sel(is_joint, dself, 0.0f));
    st(work, lane + W_RHSL, sel(act_lo, rhs_lo, sel(act_hi, rhs_hi, 0.0f)));
    st(work, lane + W_SIGMA, sel(act_lo, 1.0f, sel(act_hi, -1.0f, 0.0f)));
    stats.contacts = n_act;
    if (n_act == 0) {
      warp_sync();
      TREX_TICK(5)
      return 1;
    }
  }
  if (P.contacts_on) {
    // From here on the kinematics-phase arrays are dead: their storage becomes the contact rows.
    // axis of this lane's joint in world coordinates and its origin (registers)
    const vf ax = Rw[6], ay = Rw[7], az = Rw[8];
    const vi mydepth = seli(is_joint, depth, 0);
    TREX_ROLLED for (int c = 0; c < n_act; c++) {
      const float Px = ldu(&S.cpos[0][0], 4 * c), Py = ldu(&S.cpos[0][0], 4 * c + 1), Pz = ldu(&S.cpos[0][0], 4 * c + 2);
      const int cl = ldui(S.clane, c);
      const int cc = ldui(S.ccand, c);
      // which joints move this point: ancestors-or-self of its body
      const int ancb = cl == 25 ? 0 : lane_value_i(anc, cl);
      const vb moves = is_joint && (((vi(ancb) >> lane) & 1) != 0);
      // d(point velocity)/d(qd_lane) = axis x (P - origin)
      const vf ex = Px - xw[0], ey = Py - xw[1], ez = Pz - xw[2];
      const vf jx = sel(moves, ay * ez - az * ey, 0.0f);
      const vf jy = sel(moves, az * ex - ax * ez, 0.0f);
      const vf jz = sel(moves, ax * ey - ay * ex, 0.0f);
      // base coordinates: angular (P - x_base) x dir, linear dir
      const float bx = Px - R.pos[0], by = Py - R.pos[1], bz = Pz - R.pos[2];
      // rows: 0 normal (0,0,1) ; 1 t1 (0,-1,0) ; 2 t2 (1,0,0)      [btPlaneSpace1 of (0,0,1)]
      vf Jn = jz, J1 = -jy, J2 = jx;
      // (P-x) x (0,0,1) = (by, -bx, 0) ; (P-x) x (0,-1,0) = (bz, 0, -bx) ; (P-x) x (1,0,0) = (0, bz, -by)
      Jn = sel(lane == 25, by, sel(lane == 26, -bx, sel(lane == 30, 1.0f, Jn)));
      J1 = sel(lane == 25, bz, sel(lane == 27, -bx, sel(lane == 29, -1.0f, J1)));
      J2 = sel(lane == 26, bz, sel(lane == 27, -by, sel(lane == 28, 1.0f, J2)));
      const vf Jr[3] = {Jn, J1, J2};
      // compact storage: base lanes -> entries 0..5, chain joints -> entry 5 + depth, everyone else -> the zero entry
      const vb isb = (lane >= 25) && (lane < 31);
      const vi myslot = seli(isb, lane - 25, seli(moves, mydepth + 5, 11));
      warp_sync();
      if (defer_c) {  // the Delassus pass below walks all 11 entries of the compact rows: unused ones must read 0 * finite
        TREX_UNROLL for (int k = 0; k < 3; k++) st_if(S.c.Jc[3 * c + k], seli(lane < 12, lane, 0), 0.0f, lane < 12);
        stb(S.c.inv[c], lane & 15, vi(31));
        warp_sync();
      }
      TREX_UNROLL for (int k = 0; k < 3; k++) st_if(S.c.Jc[3 * c + k], myslot, sel(lane == 31, 0.0f, Jr[k]), isb || moves || (lane == 31));
      stb(S.c.slot[c], lane, myslot);
      if (defer_c) stb(S.c.inv[c], myslot, lane);  // entry 11 (the zero entry) ends up with an arbitrary lane
      warp_sync();
      // response dV = M^-1 J^T: this lane's coordinate = <own column, J>, over the <= 11 non-zeros of J
      vf dVr[3];
      TREX_UNROLL for (int k = 0; k < 3; k++) dVr[k] = 0.0f;
      TREX_UNROLL for (int g = 0; g < 6; g++) {
        const vf cg = ld(S.col[g], lane);
        TREX_UNROLL for (int k = 0; k < 3; k++) dVr[k] = vfma(cg, vbroadcast(ldu(S.c.Jc[3 * c + k], g)), dVr[k]);
      }
      {
        uint32_t m = (uint32_t)ancb;
        while (m) {
          const int L = ctz_u(m);
          m &= m - 1;
          const int e = 5 + P.depth[L + 1];
          const vf cg = ld(S.col[6 + L], lane);
          TREX_UNROLL for (int k = 0; k < 3; k++) dVr[k] = vfma(cg, vbroadcast(ldu(S.c.Jc[3 * c + k], e)), dVr[k]);
        }
      }
      TREX_UNROLL for (int k = 0; k < 3; k++) {
        dVr[k] = sel(lane == 31, 0.0f, dVr[k]);
        st(S.c.dV[3 * c + k], lane, dVr[k]);
      }
      // J M^-1 J^T and J u
      float dd[3], rel[3];
      TREX_UNROLL for (int k = 0; k < 3; k++) {
        dd[k] = lane_value(warp_sum(Jr[k] * dVr[k]), 0);
        rel[k] = lane_value(warp_sum(Jr[k] * uown), 0);
      }
      const float dist = Pz - P.floor_z;
      const float pen = dist + P.slop;
      float jd[3], rh[3];
      TREX_UNROLL for (int k = 0; k < 3; k++) jd[k] = dd[k] > 1.1920929e-7f ? 1.0f / dd[k] : 0.0f;
      {
        float poserr = 0.0f, velerr = -rel[0];
        if (pen > 0.0f) velerr -= pen / dt; else poserr = -pen * P.contact_erp / dt;
        rh[0] = (poserr + velerr) * jd[0];
      }
      rh[1] = -rel[1] * jd[1];
      rh[2] = -rel[2] * jd[2];
      const float warm = ldu(S.lam_cache, cc) * P.warm;
      TREX_UNROLL for (int k = 0; k < 3; k++) {
        c_rhs[k] = sel(lane == c, vbroadcast(rh[k]), c_rhs[k]);
        c_jdi[k] = sel(lane == c, vbroadcast(jd[k]), c_jdi[k]);
        c_dd[k] = sel(lane == c, vbroadcast(jd[k] != 0.0f ? dd[k] : 0.0f), c_dd[k]);
      }
      c_lam[0] = sel(lane == c, vbroadcast(warm), c_lam[0]);
      dv = vfma(dVr[0], vbroadcast(warm), dv);
    }
    if (defer_c) {
      // Contact rows for solve4, in row space: the solver tracks the velocity along every row instead of the
      // 31 coordinates, so it needs the responses at the joints (B4), at the base (for the final update) and the
      // Delassus blocks A[r'][r] = J_r' M^-1 J_r^T between contact rows.
      warp_sync();
      const bool heavy = n_act > TREX_KC;      // class 5: its own record, laid out for TREX_KW contacts
      float* cw = heavy ? workh : work;
      const int o_nc = heavy ? H_NC : W_NC, o_cs = heavy ? H_CS : W_CS, o_bt = heavy ? H_BT : W_BT, o_a4 = heavy ? H_A4 : W_A4;
      {
        const vb own = lane < n_act;
        const vi ls = seli(own, lane, 0);
        const vi sb = ls * 16 + o_cs;
        TREX_UNROLL for (int k = 0; k < 3; k++) {
          st_if(cw, sb + k, c_rhs[k], own);
          st_if(cw, sb + (3 + k), c_jdi[k], own);
          st_if(cw, sb + (6 + k), c_dd[k], own);
        }
        st_if(cw, sb + 9, c_lam[0], own);
        st_if(cw, sb + 10, vi2f(ldi(S.ccand, ls)), own);
        if (ENVP) st_if(cw, sb + 11, vbroadcast(ldu(envp, EP_MU)), own);  // the environment's friction coefficient
        st_if(cw, vi(o_nc), vbroadcast((float)n_act), lane == 0);
      }
      TREX_ROLLED for (int r = 0; r < 3 * n_act; r++) st(cw, lane + (r * 32 + o_bt), ld(S.c.dV[r], lane));
      // Delassus blocks A[r'][r] = J_r' (M^-1 J_r^T): lane <-> affected row r' (its <= 11 Jacobian entries and their
      // coordinates live in registers), uniform loop over the source row r -- every shared load of a response row is then
      // a broadcast or hits distinct banks (the transposed mapping, lanes over r, put all 32 lanes on one bank)
      const int n3 = 3 * n_act;
      TREX_ROLLED for (int t0 = 0; t0 < n3; t0 += 32) {
        const vi rp = lane + t0;                 // affected row (c', k')
        const vb valid = rp < n3;
        const vi rps = seli(valid, rp, 0);
        const vi cp = (rps * 43) >> 7, kp = rps - cp * 3;  // rp / 3, rp % 3 (rp < 48)
        vf jv[11];
        vi dl[11];
        TREX_UNROLL for (int e = 0; e < 11; e++) {
          jv[e] = ld(&S.c.Jc[0][0], rps * 12 + e);
          dl[e] = ldb(&S.c.inv[0][0], cp * 16 + e);
        }
        const vi dst = heavy ? rps + o_a4 : (cp * 4 + kp) + o_a4;
        const int rstride = heavy ? 3 * TREX_KW : 4 * TREX_KC;
        // (n3 is a multiple of 3: three source rows per trip share the eleven per-lane base addresses, the loads take immediate offsets)
        const float* dVb = &S.c.dV[0][0];
        TREX_ROLLED for (int r = 0; r < n3; r += 3) {  // source rows (c, 0..2)
          vf acc0 = 0.0f, acc1 = 0.0f, acc2 = 0.0f;
          TREX_UNROLL for (int e = 0; e < 11; e++) {
            const vi a = dl[e] + r * 32;
            acc0 = vfma(jv[e], ld(dVb, a), acc0);
            acc1 = vfma(jv[e], ld(dVb, a + 32), acc1);
            acc2 = vfma(jv[e], ld(dVb, a + 64), acc2);
          }
          st_if(cw, dst + r * rstride, acc0, valid);
          st_if(cw, dst + (r + 1) * rstride, acc1, valid);
          st_if(cw, dst + (r + 2) * rstride, acc2, valid);
        }
      }
      warp_sync();
      TREX_TICK(5)
      return 1 + defer_class(n_act);
    }
  }
  warp_sync();

  TREX_TICK(5)
  // ---- 11. projected Gauss-Seidel (btMultiBodyConstraintSolver::solveSingleIteration) --------------------
  // Velocity change dv = dvm + dvo: dvm = sum_j M^-1[:,6+j] * lambda_motor_j is rebuilt from the motor
  // impulses after every motor block (25 independent FMAs, off the critical path); dvo accumulates the
  // limit and contact rows.  Inside the motor block each lane carries only
  //     w = lambda_own + rhs_own - jdi_own * dv_own      (its own row's unclamped new impulse)
  // and updates it with the precomputed g[j] = -jdi_own * M^-1[own][6+j]  (0 for the own row, where the
  // two contributions cancel): per row FMNMX, FMNMX, SHFL, FADD, FFMA -- one shuffle is the only shared-memory
  // pipe operation.  After the block dvm is rebuilt from registers: S = sum_j g[j] lambda_j,
  // dvm_own = D_own (lambda_own - S).
  int it_done = 0;
  const float lim_hi = P.limit_max_impulse;
  const vf njdi = -jdi;
  vf g[NJ];
  TREX_UNROLL for (int j = 0; j < NJ; j++) {
    const vf cj = ld(S.col[6 + j], lane);
    g[j] = sel(is_joint, sel(lane == j, 0.0f, njdi * cj), cj);  // base-coordinate lanes keep the raw coefficient
  }
  vf dvo = dv;   // warm-started contact impulses
  vf dvm = 0.0f;
  vf w = 0.0f;
  TREX_ROLLED for (int it = 0; it < P.iters; it++) {
    vf resid = 0.0f;  // per lane: max over the rows this lane owns of (delta impulse / jacDiagABInv)^2
    const vf lam_lo0 = lam_lo, lam_hi0 = lam_hi;
    // Non-contact rows in Bullet's constraint order, direction alternating with the iteration parity.
    // Bullet's sorted constraint array for this model is [25 motors | 25 joint-limit constraints]
    // (checked in trex_model.h): the motor block is unrolled with compile-time joints; the limit block
    // visits only the violated joints, in order.
#define TREX_MOTOR_ROW(K)                                                                              \
    {                                                                                                  \
      constexpr int j = trex_topo::noncontact_order(K) - NJ;                                           \
      const vf nl = vclamp_sym(w, max_imp);              /* meaningful on lane j only */                \
      const vf t = vfma(-g[j], lamr[j], w);             /* off the critical path */                    \
      const vf nlu = vbroadcast(lane_value(nl, j));     /* new impulse of motor j, on every lane */    \
      lamr[j] = nlu;                                                                                   \
      w = vfma(g[j], nlu, t);                           /* w += g * (new - old impulse) */             \
    }
#define TREX_REBUILD_DVM()                                                                             \
    {                                                                                                  \
      /* S = sum_j g[j] * lambda_j from registers; dvm_own = D_own * (lambda_own - S) */               \
      vf a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;                                                   \
      TREX_UNROLL for (int j = 0; j + 3 < NJ; j += 4) {                                                \
        a0 = vfma(g[j], lamr[j], a0);                                                                  \
        a1 = vfma(g[j + 1], lamr[j + 1], a1);                                                          \
        a2 = vfma(g[j + 2], lamr[j + 2], a2);                                                          \
        a3 = vfma(g[j + 3], lamr[j + 3], a3);                                                          \
      }                                                                                                \
      TREX_UNROLL for (int j = NJ - (NJ % 4); j < NJ; j++) a0 = vfma(g[j], lamr[j], a0);               \
      const vf Ssum = (a0 + a1) + (a2 + a3);                                                           \
      /* this lane's own motor impulse out of the replicated registers, through shared memory */       \
      warp_sync();                                                                                     \
      TREX_UNROLL for (int j = 0; j < NJ; j++) st(S.tmp[0], vi(j), lamr[j]);                           \
      warp_sync();                                                                                     \
      const vf lam_new = sel(is_joint, ld(S.tmp[0], seli(is_joint, lane, 0)), 0.0f);                   \
      const vf dm = (lam_new - lam_m) * dself;      /* delta impulse / jacDiagABInv of the own row */  \
      lam_m = lam_new;                                                                                 \
      resid = sel(is_joint, dm * dm, 0.0f);                                                            \
      dvm = sel(is_joint, dself * (lam_m - Ssum), Ssum);  /* base lanes: g holds raw coefficients */   \
      dv = dvm + dvo;                                                                                  \
    }
#define TREX_LIMIT_BLOCK(FORWARD)                                                                      \
    {                                                                                                  \
      uint32_t m = lim_perm;                                                                           \
      while (m) {                                                                                      \
        const int pos = (FORWARD) ? ctz_u(m) : 31 - clz_u(m);                                          \
        m &= ~(1u << pos);                                                                             \
        const int j = P.order[NJ + pos];                                                               \
        const vf cj = ld(S.col[6 + j], lane);                                                          \
        TREX_UNROLL for (int pass = 0; pass < 2; pass++) {                                             \
          const bool do_lo = (pass == 0) == (FORWARD);                                                 \
          if (do_lo && ((mask_lo >> j) & 1u)) {                                                        \
            const vf sum = lam_lo + (rhs_lo - dv * jdi);                                               \
            const vf nl = vmin(vmax(sum, 0.0f), lim_hi);                                               \
            const vf dl = vbroadcast(lane_value(nl - lam_lo, j));                                      \
            lam_lo = sel(lane == j, nl, lam_lo);                                                       \
            const vf t = cj * dl;                                                                      \
            dv += t; dvo += t;                                                                         \
          }                                                                                            \
          if (!do_lo && ((mask_hi >> j) & 1u)) {                                                       \
            const vf sum = lam_hi + (rhs_hi + dv * jdi);                                               \
            const vf nl = vmin(vmax(sum, 0.0f), lim_hi);                                               \
            const vf dl = vbroadcast(lane_value(nl - lam_hi, j));                                      \
            lam_hi = sel(lane == j, nl, lam_hi);                                                       \
            const vf t = -(cj * dl);                                                                   \
            dv += t; dvo += t;                                                                         \
          }                                                                                            \
        }                                                                                              \
      }                                                                                                \
    }
#define M_(k) TREX_MOTOR_ROW(k)
#define TREX_MOTOR_BLOCK_BEGIN() w = lam_m + (rhs_m + njdi * dv);  /* exact at the start of every block */
#define TREX_MOTOR_BLOCK_END() TREX_REBUILD_DVM()
    if (it & 1) {
      TREX_MOTOR_BLOCK_BEGIN()
      M_(0) M_(1) M_(2) M_(3) M_(4) M_(5) M_(6) M_(7) M_(8) M_(9) M_(10) M_(11) M_(12) M_(13) M_(14) M_(15) M_(16)
      M_(17) M_(18) M_(19) M_(20) M_(21) M_(22) M_(23) M_(24)
      TREX_MOTOR_BLOCK_END()
      TREX_LIMIT_BLOCK(true)
    } else {
      TREX_LIMIT_BLOCK(false)
      TREX_MOTOR_BLOCK_BEGIN()
      M_(24) M_(23) M_(22) M_(21) M_(20) M_(19) M_(18) M_(17) M_(16) M_(15) M_(14) M_(13) M_(12) M_(11) M_(10) M_(9) M_(8)
      M_(7) M_(6) M_(5) M_(4) M_(3) M_(2) M_(1) M_(0)
      TREX_MOTOR_BLOCK_END()
    }
#undef TREX_MOTOR_BLOCK_BEGIN
#undef TREX_MOTOR_BLOCK_END
#undef M_
#undef TREX_MOTOR_ROW
#undef TREX_LIMIT_BLOCK
    {  // residual of the limit rows (each lane owns at most one lower / upper row)
      const vf dlo = (lam_lo - lam_lo0) * dself, dhi = (lam_hi - lam_hi0) * dself;
      resid = sel(is_joint, vmax(resid, vmax(dlo * dlo, dhi * dhi)), 0.0f);
    }
    // normal contact rows
    TREX_ROLLED for (int c = 0; c < n_act; c++) {
      const vi sl = ldb(S.c.slot[c], lane);
      const vf jdv = warp_sum(ld(S.c.Jc[3 * c], sl) * dv);
      vf dl = c_rhs[0] - jdv * c_jdi[0];
      const vf sum = c_lam[0] + dl;
      const vf nl = vmin(vmax(sum, 0.0f), 1.0e10f);
      dl = nl - c_lam[0];
      const vb own = lane == c;
      const vf dlu = vbroadcast(lane_value(dl, c));
      c_lam[0] = sel(own, nl, c_lam[0]);
      const vf dvel = dl * c_dd[0];  // delta impulse / jacDiagABInv
      resid = sel(own, vmax(resid, dvel * dvel), resid);
      const vf t = ld(S.c.dV[3 * c], lane) * dlu;
      dv += t; dvo += t;
    }
    // friction rows, implicit cone (resolveConeFrictionConstraintRows); both rows read dv before either writes
    TREX_ROLLED for (int c = 0; c < n_act; c++) {
      const vi sl = ldb(S.c.slot[c], lane);
      const vf jA = warp_sum(ld(S.c.Jc[3 * c + 1], sl) * dv);
      const vf jB = warp_sum(ld(S.c.Jc[3 * c + 2], sl) * dv);
      const vf lim = (ENVP ? ldu(envp, EP_MU) : P.mu) * c_lam[0];
      vf dB = c_rhs[2] - jB * c_jdi[2];
      const vf sumB = c_lam[2] + dB;
      vf dA = c_rhs[1] - jA * c_jdi[1];
      const vf sumA = c_lam[1] + dA;
      // |lim*sin(atan2(sumA,sumB))| , |lim*cos(atan2(sumA,sumB))| without the trigonometry
      const vf n2 = sumA * sumA + sumB * sumB;
      const vb nz = n2 > 0.0f;
      const vf rn = vrsqrt(sel(nz, n2, 1.0f));
      const vf clipA = sel(nz, vabs(lim * (sumA * rn)), 0.0f);
      const vf clipB = sel(nz, vabs(lim * (sumB * rn)), vabs(lim));
      const vf nA = vclamp_sym(sumA, clipA);
      const vf nB = vclamp_sym(sumB, clipB);
      dA = nA - c_lam[1];
      dB = nB - c_lam[2];
      const vb own = lane == c;
      const vf dAu = vbroadcast(lane_value(dA, c)), dBu = vbroadcast(lane_value(dB, c));
      c_lam[1] = sel(own, nA, c_lam[1]);
      c_lam[2] = sel(own, nB, c_lam[2]);
      const vf dvel = dA * c_dd[1] + dB * c_dd[2];
      resid = sel(own, vmax(resid, dvel * dvel), resid);
      const vf t = ld(S.c.dV[3 * c + 1], lane) * dAu + ld(S.c.dV[3 * c + 2], lane) * dBu;
      dv += t; dvo += t;
    }
    it_done = it + 1;
    const float rmax = lane_value(warp_max(resid), 0);
    if (rmax <= P.resid_thresh || it >= P.iters - 1) break;
  }
#undef TREX_REBUILD_DVM
  TREX_TICK(6)
  stats.iters += it_done;
  stats.contacts = n_act;
  {  // active-set signature of this substep's solve (see StepStats)
    const uint32_t Lm = vballot(is_joint && ((lam_lo > 0.0f) || (lam_hi > 0.0f)));
    const uint32_t Mm = vballot(is_joint && (vabs(lam_m) >= max_imp));
    const vf lim = (ENVP ? ldu(envp, EP_MU) : P.mu) * c_lam[0];
    const vb hasc = lane < n_act;
    const uint32_t Nm = vballot(hasc && (c_lam[0] > 0.0f));
    const uint32_t Fm = vballot(hasc && (c_lam[0] > 0.0f) && ((c_lam[1] * c_lam[1] + c_lam[2] * c_lam[2]) >= TREX_CONE_EDGE * (lim * lim)));
    stats.sig = sig_mix_u(sig_mix_u(sig_mix_u(sig_mix_u(stats.sig, Lm), Mm), Nm | (Fm << 16)), (uint32_t)it_done) & 0xffffffu;
  }

  // ---- 12-13. velocities += dv (clamped), motor torque, cached contact impulses, positions with the NEW velocities ----
  if (P.contacts_on) {
    const vb has = lane < n_act;
    const vi cc = ldi(S.ccand, seli(has, lane, 0));
    st_if(S.lam_cache, cc, c_lam[0], has);
  }
  warp_sync();
  finish_substep(P, lane, R, dv, lam_m);
  TREX_TICK(7)
  return 0;
}


// environment record offsets (floats), see include/trex_b200.h
enum { ST_POS = 0, ST_QUAT = 3, ST_OM = 7, ST_VL = 10, ST_Q = 13, ST_QD = 38, ST_TAU = 63, ST_LAM = 88,
       ST_STEP = 152, ST_EPISODE = 153, ST_NANRESETS = 154, ST_SIG = 158 };

TREX_FN void load_env_regs(const float* rec, vi lane, EnvRegs& R) {
  const vb is_joint = lane < NJ;
  const vi js = seli(is_joint, lane, 0);
  R.q = ld_if(rec, js + ST_Q, is_joint, 0.0f);
  R.qd = ld_if(rec, js + ST_QD, is_joint, 0.0f);
  R.tau = ld_if(rec, js + ST_TAU, is_joint, 0.0f);
  R.tgt = 0.0f;
  TREX_UNROLL for (int k = 0; k < 3; k++) { R.pos[k] = ldu(rec, ST_POS + k); R.om[k] = ldu(rec, ST_OM + k); R.vl[k] = ldu(rec, ST_VL + k); }
  TREX_UNROLL for (int k = 0; k < 4; k++) R.quat[k] = ldu(rec, ST_QUAT + k);
}
TREX_FN void load_env(const float* rec, vi lane, WarpShared& S, EnvRegs& R) {
  load_env_regs(rec, lane, R);
  st(S.lam_cache, lane, ld(rec, lane + ST_LAM));
  st(S.lam_cache, lane + 32, ld(rec, lane + (ST_LAM + 32)));
  warp_sync();
}

TREX_FN void store_env_regs(float* rec, vi lane, const EnvRegs& R) {
  const vb is_joint = lane < NJ;
  const vi js = seli(is_joint, lane, 0);
  st_if(rec, js + ST_Q, R.q, is_joint);
  st_if(rec, js + ST_QD, R.qd, is_joint);
  st_if(rec, js + ST_TAU, R.tau, is_joint);
  // base state: lanes 0..12 each write one float
  vf bs = 0.0f;
  TREX_UNROLL for (int k = 0; k < 3; k++) {
    bs = sel(lane == ST_POS + k, vbroadcast(R.pos[k]), bs);
    bs = sel(lane == ST_OM + k, vbroadcast(R.om[k]), bs);
    bs = sel(lane == ST_VL + k, vbroadcast(R.vl[k]), bs);
  }
  TREX_UNROLL for (int k = 0; k < 4; k++) bs = sel(lane == ST_QUAT + k, vbroadcast(R.quat[k]), bs);
  st_if(rec, lane, bs, lane < 13);
}
TREX_FN void store_env(float* rec, vi lane, WarpShared& S, const EnvRegs& R) {
  store_env_regs(rec, lane, R);
  warp_sync();
  st(rec, lane + ST_LAM, ld(S.lam_cache, lane));
  st(rec, lane + (ST_LAM + 32), ld(S.lam_cache, lane + 32));
}

// TrexRobot.reset / reset_configuration (trex_robot.py:39-65, 300-309).
// reset_mode 0: the reference pose (base COM frame at [0,0,reset_z], identity, crouch).
// reset_mode 1: "fallen start" sampler of BASELINE.json configs[4] (no reference counterpart): base height
//   U(reset_z_min, reset_z_max), orientation uniform on SO(3), joints U(lower, upper), zero velocity;
//   Philox4x32-10 keyed by (seed, 0xfa11) with counter (global env id, episode, block).
TREX_FN void reset_pose(const Uniform& P, const float* mdl, vi lane, WarpShared& S, EnvRegs& R, long long env_id, float episode) {
  const vb is_joint = lane < NJ;
  R.qd = 0.0f; R.tau = 0.0f; R.tgt = 0.0f;
  TREX_UNROLL for (int k = 0; k < 3; k++) { R.om[k] = 0.0f; R.vl[k] = 0.0f; }
  if (P.reset_mode == 1) {
    const unsigned long long gid = (unsigned long long)(P.env_offset + env_id);
    const vi c0 = vi((int)(unsigned)(gid & 0xffffffffull)), c1 = vi((int)(unsigned)(gid >> 32)), c2 = vi((int)episode);
    vf u[4];
    philox4_uniform(c0, c1, c2, lane >> 2, P.seed, 0xfa11u, u);  // joint lane L uses word L&3 of block L>>2
    const vi wsel = lane & 3;
    const vf uj = sel(wsel == 0, u[0], sel(wsel == 1, u[1], sel(wsel == 2, u[2], u[3])));
    const vf lo = MDL(F_LOWER), hi = MDL(F_UPPER);
    R.q = sel(is_joint, lo + (hi - lo) * uj, 0.0f);
    vf ub[4];
    philox4_uniform(c0, c1, c2, vi(8), P.seed, 0xfa11u, ub);         // block 8: base height + orientation
    const float u0 = lane_value(ub[0], 0), u1 = lane_value(ub[1], 0), u2 = lane_value(ub[2], 0), u3 = lane_value(ub[3], 0);
    R.pos[0] = 0.0f; R.pos[1] = 0.0f; R.pos[2] = P.reset_z_min + (P.reset_z_max - P.reset_z_min) * u0;
    const float a = sqrtf(1.0f - u1), b = sqrtf(u1);
    const float t2 = 6.283185307179586f * u2, t3 = 6.283185307179586f * u3;
    R.quat[0] = a * sinf(t2); R.quat[1] = a * cosf(t2); R.quat[2] = b * sinf(t3); R.quat[3] = b * cosf(t3);
  } else {
    R.q = sel(is_joint, MDL(F_STARTQ), 0.0f);
    R.pos[0] = 0.0f; R.pos[1] = 0.0f; R.pos[2] = P.reset_z;
    R.quat[0] = 0.0f; R.quat[1] = 0.0f; R.quat[2] = 0.0f; R.quat[3] = 1.0f;
  }
  st(S.lam_cache, lane, 0.0f);
  st(S.lam_cache, lane + 32, 0.0f);
  warp_sync();
}

// Randomizer of the per-environment parameters, at every reset of an environment: element L of its row is
//   lo_L + u_L (hi_L - lo_L)   (one fused multiply-add: lo == hi gives lo exactly)
// with u from Philox4x32-10 keyed by (seed, TREX_ENVP_PHILOX_KEY), counter (global env id, episode, block L >> 2), word L & 3
// -- the reset sampler's counters with a different key, so rows depend on neither the number of GPUs nor the reset-pose stream.
// Element 30 (the motor impulse bound) is then derived from the drawn torque in double, as the model's own bound is.
// ranges: lo [32] then hi [32]; dt: the physics substep in double.
TREX_FN void draw_env_params(const Uniform& P, vi lane, const float* ranges, float* envp, long long env_id, float episode, double dt) {
  const unsigned long long gid = (unsigned long long)(P.env_offset + env_id);
  const vi c0 = vi((int)(unsigned)(gid & 0xffffffffull)), c1 = vi((int)(unsigned)(gid >> 32)), c2 = vi((int)episode);
  vf u[4];
  philox4_uniform(c0, c1, c2, lane >> 2, P.seed, TREX_ENVP_PHILOX_KEY, u);
  const vi wsel = lane & 3;
  const vf ul = sel(wsel == 0, u[0], sel(wsel == 1, u[1], sel(wsel == 2, u[2], u[3])));
  const vf lo = ld(ranges, lane), hi = ld(ranges, lane + TREX_ENVP_DIM);
  vf x = vfma(ul, hi - lo, lo);
  const float imp = (float)((double)lane_value(x, EP_MAX_TORQUE) * dt);
  x = sel(lane == EP_MAX_IMPULSE, vbroadcast(imp), x);
  warp_sync();
  st(envp, lane, x);
  warp_sync();
}

// ------------------------------------------------------------------------------------------
// solve4: projected Gauss-Seidel for up to FOUR contact-free environments in one warp.
//
// Without contacts every row has a unit Jacobian (25 motors + the violated joint limits), so the solver
// only needs the joint block of M^-1.  Eight lanes serve one environment (group = lane >> 3); lane l of a
// group owns the joints at positions 4l..4l+3 of the solve order.  Each lane carries, per owned joint k,
//     w_k = lambda_m,k + rhs_m,k - jdi_k * dv_k      (the motor row's unclamped new impulse)
// and the row of coefficients g[k][j] = -jdi_k * M^-1[6+k][6+j] in registers (0 on the diagonal, where the
// impulse and velocity terms cancel).  A motor sweep goes block by block: the owner runs its four consecutive
// rows as a private register chain (clamp, difference, FMA into its later rows), then the four impulse changes
// are published with width-8 shuffles and every lane applies them -- one shuffle latency per FOUR rows on the
// dependent chain instead of one per row (measured: ~90 cycles per row with a shuffle in every row).
// Rows are visited in Bullet's order (motors in sorted-constraint order, then the violated limits; direction
// alternates with the iteration); w is rebuilt exactly from the impulses every 4th sweep.
// Ends with the velocity update, the write-back of the applied motor torque and the position integration.
// Returns the number of solver iterations each group executed (per lane of the group).
// ------------------------------------------------------------------------------------------
//
// solve4<KC> with KC > 0 also takes environments with up to KC floor contacts.  The contact rows are dense in the
// coordinates, so they are carried in ROW SPACE: lane c (< KC) of a group owns contact c and tracks the velocity
// change u along its three rows (normal, t1, t2) next to their impulses.  A joint row (motor / limit) at joint j
// adds B4[c][j][:] * d(impulse) to u, a contact row adds B4[c][j][k] * d(impulse) to the joint velocities (through w)
// and the Delassus block A4 to every owner's u: one 128-bit shared load and 3 FMAs on top of a motor row, no
// reduction over coordinates anywhere.  B4 and A4 come from front_phase through the work record.  Row order as
// in the one-environment sweep: joint rows, then the normal rows, then the friction pairs (implicit cone).
// One block of a motor sweep: rows at solve-order positions 4B..4B+3 (block 6: position 24 only), owned by lane B
// of every group.  FWD: ascending positions.  Same operations on w, in the same order, as row-by-row updates.
TREX_TOPO_FN int motor_position(int joint) {  // position of a joint's motor row in the solve order
  for (int p = 0; p < NJ; p++)
    if (trex_topo::noncontact_order(p) - NJ == joint) return p;
  return 0;
}
TREX_TOPO_FN bool limit_order_matches_motor_order() {
  for (int p = 0; p < NJ; p++)
    if (trex_topo::noncontact_order(NJ + p) != trex_topo::noncontact_order(p) - NJ) return false;
  return true;
}
// tensor-memory columns of solve4<KC, TM = true> (per lane, lane-private): the lane's own block of every Delassus row
// A4[r][own contact][0..3] at 4 r, then the responses of the lane's own contact at every solve-order position,
// B[3 own + k][pos] at S4_TM_BK + 28 k + pos
#define S4_TM_BK(KC) (12 * (KC))
#define S4_TM_COLS(KC) (S4_TM_BK(KC) + 84)
template <int B, bool FWD, int KC, bool TM>
TREX_FN void s4_motor_block(vf (&w)[4], vf (&lam_m)[4], const vf (&g)[4][NJ], vf (&cu)[3], vi glx, vi dead, vi bt_own, const float* Bs,
                            tmem_t tm, vf max_imp) {
  constexpr int n = (4 * B + 4 <= NJ) ? 4 : NJ - 4 * B;
  vf bk[3][4];  // responses of the owned contact's three rows at this block's four joints
  if (KC > 0) TREX_UNROLL for (int k = 0; k < 3; k++) {
    if (TM) tmem_ld4(tm, S4_TM_BK(KC) + k * 28 + 4 * B, bk[k]);  // (asynchronous: retired below, after the private chain)
    else ld4(Bs, bt_own + (k * 36 + 4 * B), bk[k]);
  }
  vf t[4], d[4], nl[4];
  TREX_UNROLL for (int i = 0; i < 4; i++) { t[i] = w[i]; d[i] = 0.0f; nl[i] = 0.0f; }
  // the owner's private chain (the other lanes compute on their own registers and discard): per row one symmetric clamp
  // (FMNMX.XORSIGN), the difference and one FMA into each later row of the block
  TREX_UNROLL for (int ii = 0; ii < n; ii++) {
    const int i = FWD ? ii : n - 1 - ii;
    const int j = trex_topo::noncontact_order(4 * B + i) - NJ;
    nl[i] = vclamp_sym(t[i], max_imp);
    d[i] = nl[i] - lam_m[i];
    TREX_UNROLL for (int i2 = ii + 1; i2 < n; i2++) {
      const int i3 = FWD ? i2 : n - 1 - i2;
      t[i3] = vfma(g[i3][j], d[i], t[i3]);
    }
  }
  const vb own = glx == B;  // (glx = -1 in a finished environment: it keeps its impulses ...)
  const vi src = dead | B;  // (... and publishes the zeros of its group's idle last lane: dead = 7)
  if (KC > 0 && TM) TREX_UNROLL for (int k = 0; k < 3; k++) tmem_wait4(bk[k]);
  // publish: every lane applies the four impulse changes of lane B
  TREX_UNROLL for (int ii = 0; ii < n; ii++) {
    const int i = FWD ? ii : n - 1 - ii;
    const int j = trex_topo::noncontact_order(4 * B + i) - NJ;
    lam_m[i] = sel(own, nl[i], lam_m[i]);
    const vf db = shflv_group8(d[i], src);
    vfma2s(w[0], w[1], g[0][j], g[1][j], db);  // (two FFMA2 instead of four FFMA)
    vfma2s(w[2], w[3], g[2][j], g[3][j], db);
    if (KC > 0) TREX_UNROLL for (int k = 0; k < 3; k++) cu[k] = vfma(bk[k][i], db, cu[k]);
  }
}

// warp-private shared memory of solve4<KC>, per lane group: Bp [3*KC][36] (row responses at the joints, indexed by the
// joint's POSITION in the solve order, so a motor block's four entries and a lane's four owned joints are each one
// 128-bit load; stride 36: conflict-free across the owners), A4 [3*KC][KC][4], then for all groups
// Lam [4][32 + 4*KC] (net joint impulses + contact impulses, exchanged every few sweeps)
#define TREX_BT_SIZE(KC) (108 * (KC))
#define TREX_GC_STRIDE(KC) (TREX_BT_SIZE(KC) + 12 * (KC) * (KC))
// and Lg [slots][4][32]: per lane and owned joint, the column of g of the first few joints with a violated limit
#ifndef TREX_REBUILD_MASK
#define TREX_REBUILD_MASK 3  // exact rebuild of w (and u) every 4th sweep (every 8th: the 2e-5 per-env-step parity bound is exceeded, 2.1e-5)
#endif
#ifndef TREX_REBUILD_MASK_C
#define TREX_REBUILD_MASK_C 15  // ... with contact rows (KC > 0): every 16th sweep (the parity with the oracle is set by the conditioning of
                                // the step there, as in solve2; every 4th: +3.6 % step time -- the kernel is bound by shared-memory wavefronts)
#endif
#define TREX_LIMIT_SLOTS(KC) ((KC) > 4 ? 2 : 6)
#define TREX_SOLVE_SCRATCH(KC) (4 * TREX_GC_STRIDE(KC) + 4 * (32 + 4 * (KC)) + 128 * TREX_LIMIT_SLOTS(KC))  // floats
// TM = true (tensor-memory instance of the contact solver): the Delassus blocks A4 and the responses of the lane's own contact
// along the sweep ("bk") live in TENSOR MEMORY -- both are lane-private read patterns, i.e. what tcgen05.ld 32x32b offers --
// and only the responses at the lane's own joints ("b4") stay in shared memory.  solve4<8> is bound by the shared-memory
// data pipe (69 % of the LSU wavefront peak at 48 % issue utilisation: 84 + 24 kmax wavefronts per sweep); the tensor-memory
// loads do not go through it.
#define TREX_SOLVE_SCRATCH_TM(KC) (4 * TREX_BT_SIZE(KC) + 4 * (32 + 4 * (KC)) + 128 * TREX_LIMIT_SLOTS(KC))
// envs[g] = index (relative to work0 / rec0) of the environment served by lane group g, valid when pending bit g is set.
// max_imp: motor impulse bound (per lane group).  ENVP: each contact's friction coefficient comes from word 11 of its scalars.
template <int KC, bool TM = false, bool ENVP = false>
TREX_FN vi solve4(const Uniform& P, float* scratch, const float* work0, float* rec0, const int envs[4], int pending, vf max_imp,
                  tmem_t tm = tmem_t()) {
  static_assert((KC == 0 || KC == 1 || KC == 2 || KC == 4 || KC == 8) && KC <= TREX_KC, "one contact per lane of a group");
  static_assert(!TM || KC == TREX_KC, "the tensor-memory instance serves all contact classes of solve4");
  constexpr int GC = TM ? TREX_BT_SIZE(KC) : TREX_GC_STRIDE(KC), LS = 32 + 4 * KC;
  const vi lane = lane_id();
  const vi grp = lane >> 3, gl = lane & 7;
  const vb gact = ((vi(pending) >> grp) & 1) != 0;
  const vi genv = seli(grp == 0, vi(envs[0]), seli(grp == 1, vi(envs[1]), seli(grp == 2, vi(envs[2]), vi(envs[3]))));
  const vi woff = seli(gact, genv, 0) * TREX_WORK_STRIDE, roff = seli(gact, genv, 0) * TREX_STATE_STRIDE;
  const float dt = P.dt;
  constexpr int BT = TREX_BT_SIZE(KC);
  float* Bs = scratch;                                 // [4][GC]: Bt, then A4
  float* Lam = Bs + 4 * GC;                            // [4][LS]
  float* Lg = Lam + 4 * LS;                            // [TREX_LIMIT_SLOTS][4][32]
  const vi gb = grp * GC;                              // this group's stash
  const vi glc = KC > 0 ? vmini(gl, KC - 1) : vi(0);  // contact slot of this lane (lanes >= KC shadow the last owner, unused)
  const vi bt_own = gb + glc * 108;                    // Bp rows of the owned contact

  vi kk[4];
  vb kv[4];
  vf rhs_m[4], jdi[4], dself[4], rhs_l[4], sigma[4], g[4][NJ];
  TREX_UNROLL for (int s = 0; s < 4; s++) {
    // lane l owns the joints at positions 4l .. 4l+3 of the solve order: four consecutive rows of a sweep
    kk[s] = 0;
    TREX_UNROLL for (int l = 0; l < 7; l++)
      if (4 * l + s < NJ) kk[s] = seli(gl == l, vi(trex_topo::noncontact_order(4 * l + s) - NJ), kk[s]);
    kv[s] = gact && (gl * 4 + s < NJ);
    rhs_m[s] = ld_if(work0, woff + kk[s] + W_RHSM, kv[s], 0.0f);
    jdi[s] = ld_if(work0, woff + kk[s] + W_JDI, kv[s], 0.0f);
    dself[s] = ld_if(work0, woff + kk[s] + W_DSELF, kv[s], 0.0f);
    rhs_l[s] = ld_if(work0, woff + kk[s] + W_RHSL, kv[s], 0.0f);
    sigma[s] = ld_if(work0, woff + kk[s] + W_SIGMA, kv[s], 0.0f);
    // row 6+k of M^-1 (= column 6+k: the matrix is symmetric), lanes 0..24 of the record's row: seven 128-bit loads
    TREX_UNROLL for (int j4 = 0; j4 < 7; j4++) {
      vf c4[4];
      ld4_if(work0, woff + kk[s] * 32 + (W_COL + 6 * 32 + 4 * j4), kv[s], c4);
      TREX_UNROLL for (int e = 0; e < 4; e++)
        if (4 * j4 + e < NJ) g[s][4 * j4 + e] = sel(kk[s] == 4 * j4 + e, 0.0f, -(jdi[s] * c4[e]));
    }
  }
  // contact rows: scalars of the owned contact in registers, B4 / A4 of the group's environment into the stash
  // (rows of absent contacts are zero: their updates then add exactly 0)
  vf cu[3], cl[3], crhs[3], cjdi[3], cdd[3], njdi[4];
  TREX_UNROLL for (int k = 0; k < 3; k++) { cu[k] = 0.0f; cl[k] = 0.0f; crhs[k] = 0.0f; cjdi[k] = 0.0f; cdd[k] = 0.0f; }
  TREX_UNROLL for (int s = 0; s < 4; s++) njdi[s] = -jdi[s];
  vi ccand = 0;
  vb cown = gact && !gact;
  int kmax = 0;
  vf mu_own = 0.0f;  // ENVP: friction coefficient of the owned contact's environment
  if (KC > 0) {
    const vi nc = seli(gact, vf2i(ld(work0, woff + W_NC)), 0);
    kmax = lane_value_i(warp_maxi(nc), 0);
    cown = gact && (gl < nc) && (gl < KC);
    const vi sb = woff + glc * 16 + W_CS;
    TREX_UNROLL for (int k = 0; k < 3; k++) {
      crhs[k] = ld_if(work0, sb + k, cown, 0.0f);
      cjdi[k] = ld_if(work0, sb + (3 + k), cown, 0.0f);
      cdd[k] = ld_if(work0, sb + (6 + k), cown, 0.0f);
    }
    if (ENVP) mu_own = ld_if(work0, sb + 11, cown, 0.0f);
    cl[0] = ld_if(work0, sb + 9, cown, 0.0f);  // warm start
    ccand = seli(cown, vf2i(ld_if(work0, sb + 10, cown, 0.0f)), 0);
    // Bt: rows 3c+k of the record (32 floats each) -> rows of 33; one float4 per lane and step, 8 per row
    // A4: record [r][TREX_KC][4] -> stash [r][KC][4]; lane gl takes the block of affected contact gl
    // (the three rows of one contact per step: six independent loads in flight)
    TREX_ROLLED for (int c = 0; c < kmax; c++) {
      vf b4[3][4], a4[3][4];
      TREX_UNROLL for (int k = 0; k < 3; k++) {
        TREX_UNROLL for (int s = 0; s < 4; s++)  // the lane's own four joints = positions 4 gl .. 4 gl + 3
          b4[k][s] = ld_if(work0, woff + kk[s] + ((3 * c + k) * 32 + W_BT), kv[s] && (vi(c) < nc), 0.0f);
        ld4_if(work0, woff + glc * 4 + ((3 * c + k) * (4 * TREX_KC) + W_A4), cown && (vi(c) < nc), a4[k]);
      }
      TREX_UNROLL for (int k = 0; k < 3; k++) {
        st4_if(Bs, gb + gl * 4 + (3 * c + k) * 36, b4[k], gl < 8);
        if (TM) tmem_st4(tm, 4 * (3 * c + k), a4[k][0], a4[k][1], a4[k][2], a4[k][3]);
        else st4_if(Bs, gb + glc * 4 + ((3 * c + k) * (4 * KC) + BT), a4[k], gl < KC);
      }
    }
    if (TM) {
      // the three response rows of the lane's OWN contact over all joints, in solve-order position: 7 x 128 bits per row from the
      // record (indexed by joint), permuted in registers, into the lane's tensor-memory columns
      TREX_UNROLL for (int k = 0; k < 3; k++) {
        vf row[28];
        TREX_UNROLL for (int j4 = 0; j4 < 7; j4++) {
          vf c4[4];
          ld4_if(work0, woff + glc * 96 + (W_BT + k * 32 + 4 * j4), cown, c4);
          TREX_UNROLL for (int e = 0; e < 4; e++) row[4 * j4 + e] = c4[e];
        }
        TREX_UNROLL for (int b = 0; b < 7; b++) {
          vf q[4];
          TREX_UNROLL for (int e = 0; e < 4; e++) q[e] = (4 * b + e < NJ) ? row[trex_topo::noncontact_order(4 * b + e < NJ ? 4 * b + e : 0) - NJ] : vf(0.0f);
          tmem_st4(tm, S4_TM_BK(KC) + k * 28 + 4 * b, q[0], q[1], q[2], q[3]);
        }
      }
      tmem_st_wait();
    }
  }
  warp_sync();
  // joints with a violated limit in ANY of the four environments, in Bullet's limit-constraint order
  // (bit p <=> the joint at position p; the limit block visits the joints in the same order as the motor block)
  static_assert(limit_order_matches_motor_order(), "solve4 assumes order[NJ + p] == order[p] - NJ");
  uint32_t uperm = 0;
  TREX_UNROLL for (int s = 0; s < 4; s++) {
    const uint32_t b = vballot(kv[s] && (sigma[s] != 0.0f));
    const uint32_t any = (b | (b >> 8) | (b >> 16) | (b >> 24)) & 0xffu;  // bit l: lane l of some group
    TREX_UNROLL for (int l = 0; l < 8; l++) uperm |= ((any >> l) & 1u) << (4 * l + s);
  }
  // their columns of g (joint index known only at run time) into shared memory; beyond the slots: from the record
  uint32_t cached = 0;
  {
    uint32_t m = uperm;
    TREX_ROLLED for (int slot = 0; slot < TREX_LIMIT_SLOTS(KC) && m != 0; slot++) {
      const int pos = ctz_u(m);
      m &= m - 1;
      cached |= 1u << pos;
      const int j = P.order[NJ + pos];
      TREX_UNROLL for (int s = 0; s < 4; s++)
        st(Lg, lane + (slot * 4 + s) * 32,
           sel(kk[s] == j, 0.0f, njdi[s] * ld_if(work0, woff + kk[s] * 32 + (W_COL + 6 * 32 + j), kv[s], 0.0f)));
    }
  }
  warp_sync();

  vf w[4], lam_m[4], lam_l[4];
  TREX_UNROLL for (int s = 0; s < 4; s++) { w[s] = rhs_m[s]; lam_m[s] = 0.0f; lam_l[s] = 0.0f; }
  const float lim_hi = P.limit_max_impulse;
  vb alive = gact;
  vi itd = 0;

  // one limit row of joint j (slot SJ static): sigma = +1 lower row, -1 upper row, impulse in [0, lim_hi]
#define TREX_S4_LIMIT_SLOT(SJ)                                                                         \
  {                                                                                                    \
    const vf x = (lam_m[SJ] + rhs_m[SJ]) - w[SJ];              /* jdi * dv_j */                         \
    const vf sum = lam_l[SJ] + (rhs_l[SJ] - sigma[SJ] * x);                                            \
    const vf nl = vmin(vmax(sum, 0.0f), lim_hi);                                                       \
    const vb own = alive && (gl == (pos >> 2)) && (sigma[SJ] != 0.0f);                                 \
    const vf d = sel(own, (nl - lam_l[SJ]) * sigma[SJ], 0.0f);  /* change of the net joint impulse */   \
    const vf db = shfl_group8(d, pos >> 2);                                                            \
    lam_l[SJ] = sel(own, nl, lam_l[SJ]);                                                               \
    vfma2s(w[0], w[1], gj[0], gj[1], db);                                                              \
    vfma2s(w[2], w[3], gj[2], gj[3], db);                                                              \
    w[SJ] = w[SJ] - d;                                        /* self term: dv_j += D_j * d */         \
    if (KC > 0) TREX_UNROLL for (int k = 0; k < 3; k++) cu[k] = vfma(ld(Bs, bt_own + (k * 36 + pos)), db, cu[k]); \
  }
#define TREX_S4_LIMITS(FORWARD)                                                                        \
  {                                                                                                    \
    uint32_t m = uperm;                                                                                \
    while (m) {                                                                                        \
      const int pos = (FORWARD) ? ctz_u(m) : 31 - clz_u(m);                                            \
      m &= ~(1u << pos);                                                                               \
      const int j = P.order[NJ + pos];                                                                 \
      /* column j of g from the record (limit rows are rare; their joint is only known at run time) */  \
      vf gj[4];                                                                                        \
      if ((cached >> pos) & 1u) {                                                                      \
        const int slot = popc_u(cached & ((1u << pos) - 1u));                                          \
        TREX_UNROLL for (int s = 0; s < 4; s++) gj[s] = ld(Lg, lane + (slot * 4 + s) * 32);            \
      } else {                                                                                         \
        TREX_UNROLL for (int s = 0; s < 4; s++)                                                        \
          gj[s] = sel(kk[s] == j, 0.0f, njdi[s] * ld_if(work0, woff + kk[s] * 32 + (W_COL + 6 * 32 + j), kv[s], 0.0f)); \
      }                                                                                                \
      switch (pos & 3) {  /* the limit block visits the joints in the motor block's order */            \
        case 0: TREX_S4_LIMIT_SLOT(0) break;                                                           \
        case 1: TREX_S4_LIMIT_SLOT(1) break;                                                           \
        case 2: TREX_S4_LIMIT_SLOT(2) break;                                                           \
        default: TREX_S4_LIMIT_SLOT(3) break;                                                          \
      }                                                                                                \
    }                                                                                                  \
  }
#define MB_(b, fwd) s4_motor_block<b, fwd, KC, TM>(w, lam_m, g, cu, glx, dead, bt_own, Bs, tm, max_imp);
  vf mu_l = ENVP ? mu_own : vf(P.mu);
  TREX_ROLLED for (int it = 0; it < P.iters; it++) {
    // every 4th sweep (TREX_REBUILD_MASK) rebuild w (and u) exactly from the impulses (bounds the FP32 drift of the incremental updates):
    // w_k = rhs_m,k - sigma_k lam_l,k + sum_j g[k][j] Lambda_j - jdi_k sum_r B[r][k] lambda_r
    // u_r = sum_j B[r][j] Lambda_j + sum_r' A[r][r'] lambda_r'         (also the warm-started initial state)
    if ((it & (KC > 0 ? TREX_REBUILD_MASK_C : TREX_REBUILD_MASK)) == 0 && (KC > 0 || it > 0)) {
      warp_sync();
      TREX_UNROLL for (int s = 0; s < 4; s++) st_if(Lam, grp * LS + kk[s], lam_m[s] + sigma[s] * lam_l[s], kv[s]);
      if (KC > 0) TREX_UNROLL for (int k = 0; k < 3; k++) st_if(Lam, grp * LS + glc * 4 + (32 + k), cl[k], gl < KC);
      warp_sync();
      vf acc[4], ua[3];
      TREX_UNROLL for (int s = 0; s < 4; s++) acc[s] = rhs_m[s] - sigma[s] * lam_l[s];
      TREX_UNROLL for (int k = 0; k < 3; k++) ua[k] = 0.0f;
      TREX_UNROLL for (int j = 0; j < NJ; j++) {
        const vf Lj = ld(Lam, grp * LS + j);
        vfma2s(acc[0], acc[1], g[0][j], g[1][j], Lj);
        vfma2s(acc[2], acc[3], g[2][j], g[3][j], Lj);
        if (KC > 0) TREX_UNROLL for (int k = 0; k < 3; k++) ua[k] = vfma(ld(Bs, bt_own + (k * 36 + motor_position(j))), Lj, ua[k]);
      }
      if (KC > 0) {
        vf bs[4];
        TREX_UNROLL for (int s = 0; s < 4; s++) bs[s] = 0.0f;
        TREX_ROLLED for (int c = 0; c < kmax; c++) {
          TREX_UNROLL for (int k = 0; k < 3; k++) {
            const vf Lr = ld(Lam, grp * LS + (32 + c * 4 + k));
            vf b4[4];
            ld4(Bs, gb + gl * 4 + (3 * c + k) * 36, b4);
            TREX_UNROLL for (int s = 0; s < 4; s++) bs[s] = vfma(b4[s], Lr, bs[s]);
            vf a4[4];
            if (TM) { tmem_ld4(tm, 4 * (3 * c + k), a4); tmem_wait4(a4); }
            else ld4(Bs, gb + glc * 4 + ((3 * c + k) * (4 * KC) + BT), a4);
            TREX_UNROLL for (int k2 = 0; k2 < 3; k2++) ua[k2] = vfma(a4[k2], Lr, ua[k2]);
          }
        }
        TREX_UNROLL for (int s = 0; s < 4; s++) acc[s] = vfma(njdi[s], bs[s], acc[s]);
        TREX_UNROLL for (int k = 0; k < 3; k++) cu[k] = ua[k];
      }
      TREX_UNROLL for (int s = 0; s < 4; s++) w[s] = sel(alive, acc[s], w[s]);
    }
    vf lam_m0[4], lam_l0[4];
    vf cres = 0.0f;
    TREX_UNROLL for (int s = 0; s < 4; s++) { lam_m0[s] = lam_m[s]; lam_l0[s] = lam_l[s]; }
    // an environment that has finished (converged) is frozen without a select on the dependent chain: it owns no motor row
    // (glx = -1) and publishes the zeros of its group's idle lane 7 (dead = 7); its contact rows have jdi = rhs = 0 and an
    // unbounded cone (below), so they reproduce their impulses exactly
    const vi glx = seli(alive, gl, vi(-1)), dead = seli(alive, vi(0), vi(7));
    if (it & 1) {
      MB_(0, true) MB_(1, true) MB_(2, true) MB_(3, true) MB_(4, true) MB_(5, true) MB_(6, true)
      TREX_S4_LIMITS(true)
    } else {
      TREX_S4_LIMITS(false)
      MB_(6, false) MB_(5, false) MB_(4, false) MB_(3, false) MB_(2, false) MB_(1, false) MB_(0, false)
    }
    if (KC > 0) {
      // normal rows: every lane evaluates its own contact, the owner of contact c publishes.  Dependent chain per row:
      // FFMA, FMNMX, FADD, SHFL, FFMA (the impulse + rhs sum is taken before the loop; Bullet's upper bound 1e10 cannot bind
      // on a state that passes the NaN / overflow guard; no select: rows of absent contacts and of finished environments
      // have jdi = rhs = 0 and reproduce their impulse)
      // (most warps of this kernel hold environments with 1-2 contacts: fetching the A4 / Bp rows one iteration ahead, as
      // solve2 does for its 9-16 contacts, only adds loads here -- measured +30 % on the benchmark batch)
      const vf cl0_0 = cl[0], cl1_0 = cl[1], cl2_0 = cl[2];
      const vf pre0 = cl[0] + crhs[0];
      TREX_ROLLED for (int c = 0; c < kmax; c++) {
        vf a4[4];
        if (TM) tmem_ld4(tm, 4 * (3 * c), a4);  // (in flight under the clamp chain and the shuffle)
        else ld4(Bs, gb + glc * 4 + ((3 * c) * (4 * KC) + BT), a4);
        const vf nl = vmax(vfma(-cu[0], cjdi[0], pre0), 0.0f);
        const vf d = shfl_group8(nl - cl[0], c);
        cl[0] = sel(gl == c, nl, cl[0]);
        if (TM) tmem_wait4(a4);
        TREX_UNROLL for (int k = 0; k < 3; k++) cu[k] = vfma(a4[k], d, cu[k]);
        vf b4[4];
        ld4(Bs, gb + gl * 4 + (3 * c) * 36, b4);
        vf nd[4];
        vmul2s(nd[0], nd[1], njdi[0], njdi[1], d);
        vmul2s(nd[2], nd[3], njdi[2], njdi[3], d);
        vfma2v(w[0], w[1], b4[0], b4[1], nd[0], nd[1]);
        vfma2v(w[2], w[3], b4[2], b4[3], nd[2], nd[3]);
      }
      // friction pairs, implicit cone; both rows read the velocities before either writes.  |lim sin|, |lim cos| of
      // atan2(sumA, sumB) = lim |sum| / sqrt(sumA^2 + sumB^2); at sumA = sumB = 0 both clips multiply a zero, which is
      // what the reference's clamp of a zero sum gives
      const vf lim = mu_l * cl[0];
      const vf preA = cl[1] + crhs[1], preB = cl[2] + crhs[2];
      TREX_ROLLED for (int c = 0; c < kmax; c++) {
        vf aA[4], aB[4];
        if (TM) {
          tmem_ld4(tm, 4 * (3 * c + 1), aA);
          tmem_ld4(tm, 4 * (3 * c + 2), aB);
        } else {
          ld4(Bs, gb + glc * 4 + ((3 * c + 1) * (4 * KC) + BT), aA);
          ld4(Bs, gb + glc * 4 + ((3 * c + 2) * (4 * KC) + BT), aB);
        }
        const vf sumB = vfma(-cu[2], cjdi[2], preB);
        const vf sumA = vfma(-cu[1], cjdi[1], preA);
        const vf rn = vrsqrt(vmax(sumA * sumA + sumB * sumB, 1.0e-30f));
        const vf nA = vclamp_sym(sumA, lim * vabs(sumA * rn));
        const vf nB = vclamp_sym(sumB, lim * vabs(sumB * rn));
        const vf dAu = shfl_group8(nA - cl[1], c), dBu = shfl_group8(nB - cl[2], c);
        const vb mine = gl == c;
        cl[1] = sel(mine, nA, cl[1]);
        cl[2] = sel(mine, nB, cl[2]);
        if (TM) { tmem_wait4(aA); tmem_wait4(aB); }
        TREX_UNROLL for (int k = 0; k < 3; k++) cu[k] = vfma(aA[k], dAu, vfma(aB[k], dBu, cu[k]));
        vf bA[4], bB[4];
        ld4(Bs, gb + gl * 4 + (3 * c + 1) * 36, bA);
        ld4(Bs, gb + gl * 4 + (3 * c + 2) * 36, bB);
        vf tb[4];
        vmul2s(tb[0], tb[1], bB[0], bB[1], dBu);
        vmul2s(tb[2], tb[3], bB[2], bB[3], dBu);
        vfma2s(tb[0], tb[1], bA[0], bA[1], dAu);
        vfma2s(tb[2], tb[3], bA[2], bA[3], dAu);
        vfma2v(w[0], w[1], njdi[0], njdi[1], tb[0], tb[1]);
        vfma2v(w[2], w[3], njdi[2], njdi[3], tb[2], tb[3]);
      }
      {  // residual of the contact rows: every row is visited once per sweep, so its impulse change is end - start
        const vf dn = (cl[0] - cl0_0) * cdd[0];
        const vf dt2 = (cl[1] - cl1_0) * cdd[1] + (cl[2] - cl2_0) * cdd[2];
        cres = vmax(dn * dn, dt2 * dt2);
      }
    }
    // residual per environment: max over its rows of (delta impulse / jacDiagABInv)^2
    vf r = cres;
    TREX_UNROLL for (int s = 0; s < 4; s++) {
      const vf dm = (lam_m[s] - lam_m0[s]) * dself[s];
      r = vmax(r, dm * dm);
    }
    if (uperm != 0u) {  // limit rows exist in this warp (uniform; otherwise their impulses never leave 0)
      TREX_UNROLL for (int s = 0; s < 4; s++) {
        const vf dl = (lam_l[s] - lam_l0[s]) * dself[s];
        r = vmax(r, dl * dl);
      }
    }
    // (leastSquaresResidual <= threshold stops the environment: true iff no lane of the group exceeds it)
    const uint32_t over = vballot(alive && !(r <= P.resid_thresh));
    itd = itd + seli(alive, vi(1), vi(0));
    const vi ob = seli(grp == 0, vi((int)(over & 0xffu)), seli(grp == 1, vi((int)((over >> 8) & 0xffu)),
                       seli(grp == 2, vi((int)((over >> 16) & 0xffu)), vi((int)(over >> 24)))));
    alive = alive && (ob != 0) && (it < P.iters - 1);
    if (over == 0u || it >= P.iters - 1) break;
    if (KC > 0) {  // freeze the contact rows of an environment that has just finished
      TREX_UNROLL for (int k = 0; k < 3; k++) { crhs[k] = sel(alive, crhs[k], 0.0f); cjdi[k] = sel(alive, cjdi[k], 0.0f); }
      mu_l = sel(alive, mu_l, 1.0e30f);
    }
  }
#undef MB_
#undef TREX_S4_LIMIT_SLOT
#undef TREX_S4_LIMITS

  // ---- velocity change of every coordinate from the final impulses ------------------------------------
  warp_sync();
  TREX_UNROLL for (int s = 0; s < 4; s++) st_if(Lam, grp * LS + kk[s], lam_m[s] + sigma[s] * lam_l[s], kv[s]);
  if (KC > 0) TREX_UNROLL for (int k = 0; k < 3; k++) st_if(Lam, grp * LS + glc * 4 + (32 + k), cl[k], gl < KC);
  warp_sync();
  vf Ssum[4], bsum[4];
  TREX_UNROLL for (int s = 0; s < 4; s++) { Ssum[s] = 0.0f; bsum[s] = 0.0f; }
  TREX_UNROLL for (int j = 0; j < NJ; j++) {
    const vf Lj = ld(Lam, grp * LS + j);
    vfma2s(Ssum[0], Ssum[1], g[0][j], g[1][j], Lj);
    vfma2s(Ssum[2], Ssum[3], g[2][j], g[3][j], Lj);
  }
  vf dvb[6];
  TREX_UNROLL for (int b = 0; b < 6; b++) dvb[b] = 0.0f;
  TREX_UNROLL for (int s = 0; s < 4; s++) {
    const vf Lk = lam_m[s] + sigma[s] * lam_l[s];
    TREX_UNROLL for (int b = 0; b < 6; b++) dvb[b] = vfma(ld_if(work0, woff + kk[s] + (W_COL + b * 32), kv[s], 0.0f), Lk, dvb[b]);
  }
  if (KC > 0) {
    // contact impulses: joint coordinates through B4, base coordinates through the owner's rows of M^-1 J^T
    TREX_ROLLED for (int c = 0; c < kmax; c++)
      TREX_UNROLL for (int k = 0; k < 3; k++) {
        const vf Lr = ld(Lam, grp * LS + (32 + c * 4 + k));
        vf b4[4];
        ld4(Bs, gb + gl * 4 + (3 * c + k) * 36, b4);
        TREX_UNROLL for (int s = 0; s < 4; s++) bsum[s] = vfma(b4[s], Lr, bsum[s]);
      }
    TREX_UNROLL for (int k = 0; k < 3; k++)
      TREX_UNROLL for (int b = 0; b < 6; b++)
        dvb[b] = vfma(ld_if(work0, woff + glc * 96 + (W_BT + k * 32 + 25 + b), cown, 0.0f), cl[k], dvb[b]);
    st_if(rec0, roff + ccand + ST_LAM, cl[0], cown);  // cached normal impulse of the candidate (next substep's warm start)
  }
  TREX_UNROLL for (int b = 0; b < 6; b++) dvb[b] = group8_sum(dvb[b]);

  // ---- velocities += dv (clamped), applied motor torque, positions with the NEW velocities ----------------
  TREX_UNROLL for (int s = 0; s < 4; s++) {
    const vf Lk = lam_m[s] + sigma[s] * lam_l[s];
    const vf dvk = dself[s] * (Lk - Ssum[s]) + bsum[s];  // M^-1 row k times the joint impulses = D_k Lambda_k - S_k / jdi_k, + contacts
    const vf qd0 = ld_if(rec0, roff + kk[s] + ST_QD, kv[s], 0.0f);
    const vf q0 = ld_if(rec0, roff + kk[s] + ST_Q, kv[s], 0.0f);
    const vf qd1 = clampv(qd0 + dvk, -P.maxvel, P.maxvel);
    st_if(rec0, roff + kk[s] + ST_QD, qd1, kv[s]);
    st_if(rec0, roff + kk[s] + ST_Q, q0 + dt * qd1, kv[s]);
    st_if(rec0, roff + kk[s] + ST_TAU, vdiv(lam_m[s], dt), kv[s]);
  }
  {
    const vi rb = roff;
    vf om[3], vl[3], pos[3], qt[4];
    TREX_UNROLL for (int k = 0; k < 3; k++) {
      om[k] = clampv(ld(rec0, rb + (ST_OM + k)) + dvb[k], -P.maxvel, P.maxvel);
      vl[k] = clampv(ld(rec0, rb + (ST_VL + k)) + dvb[3 + k], -P.maxvel, P.maxvel);
      pos[k] = ld(rec0, rb + (ST_POS + k)) + dt * vl[k];
    }
    TREX_UNROLL for (int k = 0; k < 4; k++) qt[k] = ld(rec0, rb + (ST_QUAT + k));
    // btMultiBody::stepPositionsMultiDof: exponential map of the world angular velocity, q <- dq * q
    vf fa = vsqrt(om[0] * om[0] + om[1] * om[1] + om[2] * om[2]);
    fa = sel(fa * dt > 0.78539816339744831f, vbroadcast(0.78539816339744831f / dt), fa);
    const vb small = fa < 0.001f;
    const vf sc = sel(small, 0.5f * dt - (dt * dt * dt) * 0.020833333333f * fa * fa, vdiv(vsin(0.5f * fa * dt), sel(small, 1.0f, fa)));
    const vf ax = om[0] * sc, ay = om[1] * sc, az = om[2] * sc, aw = vcos(fa * dt * 0.5f);
    const vf nx = aw * qt[0] + ax * qt[3] + ay * qt[2] - az * qt[1];
    const vf ny = aw * qt[1] - ax * qt[2] + ay * qt[3] + az * qt[0];
    const vf nz = aw * qt[2] + ax * qt[1] - ay * qt[0] + az * qt[3];
    const vf nw = aw * qt[3] - ax * qt[0] - ay * qt[1] - az * qt[2];
    const vf inv = vdiv(1.0f, vsqrt(nx * nx + ny * ny + nz * nz + nw * nw));
    warp_sync();
    // lanes 0..12 of the group's first 13... one lane per field: lane gl + 8*t covers fields gl, gl+8
    TREX_UNROLL for (int t = 0; t < 2; t++) {
      const vi f = gl + 8 * t;  // field index 0..15 of the base block [pos3 quat4 om3 vl3]
      vf val = 0.0f;
      TREX_UNROLL for (int k = 0; k < 3; k++) {
        val = sel(f == ST_POS + k, pos[k], val);
        val = sel(f == ST_OM + k, om[k], val);
        val = sel(f == ST_VL + k, vl[k], val);
      }
      val = sel(f == ST_QUAT, nx * inv, sel(f == ST_QUAT + 1, ny * inv, sel(f == ST_QUAT + 2, nz * inv, sel(f == ST_QUAT + 3, nw * inv, val))));
      st_if(rec0, rb + f, val, gact && (f < 13));
    }
  }
  {  // active-set signature of this substep's solve (StepStats), per environment: OR over the group's lanes, lane 0 folds
    vi Lm = 0, Mm = 0;
    TREX_UNROLL for (int s = 0; s < 4; s++) {
      Lm = Lm | seli(kv[s] && (lam_l[s] > 0.0f), vi(1) << kk[s], vi(0));
      Mm = Mm | seli(kv[s] && (vabs(lam_m[s]) >= max_imp), vi(1) << kk[s], vi(0));
    }
    vi NF = 0;
    if (KC > 0) {
      const vf lim = (ENVP ? mu_own : vf(P.mu)) * cl[0];
      const vb pos = cown && (cl[0] > 0.0f);
      NF = seli(pos, vi(1) << gl, vi(0)) |
           seli(pos && ((cl[1] * cl[1] + cl[2] * cl[2]) >= TREX_CONE_EDGE * (lim * lim)), vi(65536) << gl, vi(0));
    }
    TREX_UNROLL for (int m = 4; m > 0; m >>= 1) { Lm = Lm | shfl_xor_i(Lm, m); Mm = Mm | shfl_xor_i(Mm, m); NF = NF | shfl_xor_i(NF, m); }
    const vb wr = gact && (gl == 0);
    const vi si = seli(wr, roff + ST_SIG, 0);
    const vi h = sig_mix_v(sig_mix_v(sig_mix_v(sig_mix_v(vf2i(ld(rec0, si)), Lm), Mm), NF), itd) & 0xffffff;
    st_if(rec0, si, vi2f(h), wr);
  }
  warp_sync();
  return itd;
}

// ------------------------------------------------------------------------------------------
// solve2: projected Gauss-Seidel for up to TWO environments with many contacts (class 5: more than TREX_KC and up to
// TREX_KW = 16, e.g. a T-rex standing on both feet: 14-16 points) in one warp, SIXTEEN lanes per environment.
//
// The same row-space sweep as solve4<KC> with the lane group twice as wide: lane l of a group owns the joints at
// positions 2l, 2l+1 of the solve order (g[2][25] = 50 registers instead of 100) and contact l (one contact per lane).
// A motor sweep goes in 13 blocks of two private rows (one width-16 shuffle latency per two rows); the contact rows
// read the Delassus matrix A (48 x 48, row r = the velocity change along every row per unit impulse of row r) and the
// joint responses Bp (48 x 26, indexed by solve-order position) from the warp's shared scratch: 14.2 KB per
// environment, which is what bounds the number of environments in flight per SM (14).
// Row order, clamps, residual, rebuild period and integration are those of solve4.
// ------------------------------------------------------------------------------------------
#define TREX_S2_NR (3 * TREX_KW)                    // contact rows per environment (48)
#define TREX_S2_BS 26                               // Bp row stride: 25 positions + 1, even (64-bit loads); 3 * 26 * c mod 32 is conflict-free over the 16 owners
#define TREX_S2_ENV (TREX_S2_NR * TREX_S2_NR + TREX_S2_NR * TREX_S2_BS + 16)  // floats per environment: A, then Bp; + 16: the two groups' stashes are
                                                                           // 16 banks apart, so their stride-3 reads of A never share a bank
#define TREX_S2_LS (32 + 4 * TREX_KW)               // Lam per environment: net joint impulses by joint, then [KW][4] contact impulses
#define TREX_S2_LIMIT_SLOTS 2
#define TREX_SOLVE2_SCRATCH (2 * TREX_S2_ENV + 2 * TREX_S2_LS + 64 * TREX_S2_LIMIT_SLOTS)  // floats per warp
// solve2<true>: the Delassus matrix lives in TENSOR MEMORY (lane c' holds its own three entries of row r in TMEM columns
// 4 r .. 4 r + 2 of its lane: 192 of the 256 columns a 4-warp CTA allocates), the shared scratch shrinks to Bp + the small parts
#define TREX_S2_ENV_TM (TREX_S2_NR * TREX_S2_BS + 16)
#define TREX_SOLVE2_SCRATCH_TM (2 * TREX_S2_ENV_TM + 2 * TREX_S2_LS + 64 * TREX_S2_LIMIT_SLOTS)
#define TREX_S2_TMEM_COLS 256
#ifndef TREX_S2_REBUILD_MASK
#define TREX_S2_REBUILD_MASK 15  // exact rebuild of w and u every 16th sweep: with 9-16 contacts the parity with the oracle is set by the
                                 // conditioning of the step, not by the drift of the incremental updates (per substep on the standing T-rex,
                                 // median / max error: every 4th 1.6e-4 / 2.0e-3, every 8th 1.3e-4 / 2.1e-3, every 16th 1.3e-4 / 1.5e-3)
#endif
// rows of the Delassus matrix for the lane's own contact: from the shared stash (three 32-bit loads, a[3] unused) or from TMEM
template <bool TM>
TREX_FN void s2_fetch_a(const float* Sc, vi a_own, tmem_t tm, int row, vf (&a)[4]) {
  if (TM) {
    tmem_ld4(tm, 4 * row, a);
  } else {
    TREX_UNROLL for (int k = 0; k < 3; k++) a[k] = ld(Sc, a_own + (row * TREX_S2_NR + k));
  }
}
template <bool TM>
TREX_FN void s2_ready_a(vf (&a)[4]) { if (TM) tmem_wait4(a); }

template <int B, bool FWD>
TREX_FN void s2_motor_block(vf (&w)[2], vf (&lam_m)[2], const vf (&g)[2][NJ], vf (&cu)[3], vi glx, vi dead, vi bp_own, const float* Sc, vf max_imp) {
  constexpr int n = (2 * B + 2 <= NJ) ? 2 : NJ - 2 * B;
  vf bk[3][2];  // responses of the owned contact's three rows at this block's joints
  TREX_UNROLL for (int k = 0; k < 3; k++) ld2(Sc, bp_own + (k * TREX_S2_BS + 2 * B), bk[k]);
  constexpr int i0 = FWD ? 0 : n - 1, i1 = FWD ? 1 : 0;  // first / second row of the block in visiting order
  constexpr int j0 = trex_topo::noncontact_order(2 * B + i0) - NJ;
  vf nl[2];
  nl[0] = 0.0f; nl[1] = 0.0f;
  // the owner's private chain: clamp (one FMNMX.XORSIGN), difference, FMA, clamp
  nl[i0] = vclamp_sym(w[i0], max_imp);
  if (n == 2) nl[i1] = vclamp_sym(vfma(g[i1][j0], nl[i0] - lam_m[i0], w[i1]), max_imp);
  const vb own = glx == B;  // (a finished environment owns nothing and publishes the zeros of its idle lane 15)
  const vi src = dead | B;
  TREX_UNROLL for (int ii = 0; ii < n; ii++) {  // publish: every lane applies the impulse changes of lane B
    const int i = FWD ? ii : n - 1 - ii;
    const int j = trex_topo::noncontact_order(2 * B + i) - NJ;
    const vf db = shflv_group16(nl[i] - lam_m[i], src);
    lam_m[i] = sel(own, nl[i], lam_m[i]);
    vfma2s(w[0], w[1], g[0][j], g[1][j], db);
    TREX_UNROLL for (int k = 0; k < 3; k++) cu[k] = vfma(bk[k][i], db, cu[k]);
  }
}

// envs[g] = index (relative to work0 / workh0 / rec0) of the environment served by lane group g, valid when pending bit g is set.
template <bool TM, bool ENVP = false>
TREX_FN vi solve2(const Uniform& P, float* scratch, tmem_t tm, const float* work0, const float* workh0, float* rec0, const int envs[2],
                  int pending, vf max_imp) {
  constexpr int NR = TREX_S2_NR, BS = TREX_S2_BS, LS = TREX_S2_LS, AOFF = 0, BOFF = TM ? 0 : NR * NR;
  constexpr int ENV = TM ? TREX_S2_ENV_TM : TREX_S2_ENV;
  const vi lane = lane_id();
  const vi grp = lane >> 4, gl = lane & 15;
  const vb gact = ((vi(pending) >> grp) & 1) != 0;
  const vi genv = seli(grp == 0, vi(envs[0]), vi(envs[1]));
  const vi es = seli(gact, genv, 0);
  const vi woff = es * TREX_WORK_STRIDE, hoff = es * TREX_HEAVY_STRIDE, roff = es * TREX_STATE_STRIDE;
  const float dt = P.dt;
  float* Sc = scratch;                                 // [2][ENV]: A (unless in TMEM), then Bp
  float* Lam = Sc + 2 * ENV;                           // [2][LS]
  float* Lg = Lam + 2 * LS;                            // [TREX_S2_LIMIT_SLOTS][2][32]
  const vi gb = grp * ENV;                             // this group's stash
  const vi a_own = gb + (AOFF + 3 * gl);               // column block of the owned contact in every row of A
  const vi bp_own = gb + (BOFF + 3 * BS * gl);         // Bp rows of the owned contact
  const vi bp_mine = gb + (BOFF + 2 * gl);             // the lane's two joints in every row of Bp

  vi kk[2];
  vb kv[2];
  vf rhs_m[2], jdi[2], dself[2], rhs_l[2], sigma[2], njdi[2], g[2][NJ];
  TREX_UNROLL for (int s = 0; s < 2; s++) {
    kk[s] = 0;
    TREX_UNROLL for (int l = 0; l < 13; l++)
      if (2 * l + s < NJ) kk[s] = seli(gl == l, vi(trex_topo::noncontact_order(2 * l + s) - NJ), kk[s]);
    kv[s] = gact && (gl * 2 + s < NJ);
    rhs_m[s] = ld_if(work0, woff + kk[s] + W_RHSM, kv[s], 0.0f);
    jdi[s] = ld_if(work0, woff + kk[s] + W_JDI, kv[s], 0.0f);
    dself[s] = ld_if(work0, woff + kk[s] + W_DSELF, kv[s], 0.0f);
    rhs_l[s] = ld_if(work0, woff + kk[s] + W_RHSL, kv[s], 0.0f);
    sigma[s] = ld_if(work0, woff + kk[s] + W_SIGMA, kv[s], 0.0f);
    njdi[s] = -jdi[s];
    TREX_UNROLL for (int j4 = 0; j4 < 7; j4++) {  // row 6+k of the symmetric M^-1: seven 128-bit loads
      vf c4[4];
      ld4_if(work0, woff + kk[s] * 32 + (W_COL + 6 * 32 + 4 * j4), kv[s], c4);
      TREX_UNROLL for (int e = 0; e < 4; e++)
        if (4 * j4 + e < NJ) g[s][4 * j4 + e] = sel(kk[s] == 4 * j4 + e, 0.0f, -(jdi[s] * c4[e]));
    }
  }
  // contact rows: scalars of the owned contact in registers, A / Bp of the group's environment into the stash
  // (rows of absent contacts are zero: their updates then add exactly 0)
  vf cu[3], cl[3], crhs[3], cjdi[3], cdd[3];
  const vi nc = seli(gact, vf2i(ld(workh0, hoff + H_NC)), 0);
  const int kmax = lane_value_i(warp_maxi(nc), 0);
  const vb cown = gact && (gl < nc);
  {
    const vi sb = hoff + gl * 16 + H_CS;
    TREX_UNROLL for (int k = 0; k < 3; k++) {
      crhs[k] = ld_if(workh0, sb + k, cown, 0.0f);
      cjdi[k] = ld_if(workh0, sb + (3 + k), cown, 0.0f);
      cdd[k] = ld_if(workh0, sb + (6 + k), cown, 0.0f);
      cu[k] = 0.0f; cl[k] = 0.0f;
    }
    cl[0] = ld_if(workh0, sb + 9, cown, 0.0f);  // warm start
  }
  const vf mu_own = ENVP ? ld_if(workh0, hoff + gl * 16 + (H_CS + 11), cown, 0.0f) : vf(P.mu);  // ENVP: the environment's friction
  const vi ccand = seli(cown, vf2i(ld_if(workh0, hoff + gl * 16 + (H_CS + 10), cown, 0.0f)), 0);
  {
    const vi nr = nc * 3;
    _Pragma("unroll 4") for (int r = 0; r < 3 * kmax; r++) {  // (several rows in flight: the copy is latency bound)
      const vb rok = gact && (vi(r) < nr);
      if (TM) {
        // A row r -> tensor memory: every lane stores its own three entries A[r][3 gl .. 3 gl + 2] (zero for absent contacts)
        vf a3[3];
        TREX_UNROLL for (int k = 0; k < 3; k++) a3[k] = ld_if(workh0, hoff + gl * 3 + (r * NR + H_A4 + k), rok && ((gl * 3 + k) < nr), 0.0f);
        tmem_st4(tm, 4 * r, a3[0], a3[1], a3[2], vf(0.0f));
      } else {
        // A row r: 48 floats = 12 float4, lanes 0..11 of the group; columns of absent contacts read as zero
        vf a4[4];
        const vb al = gl < (NR / 4);
        const vi gls = seli(al, gl, 0);
        ld4_if(workh0, hoff + gls * 4 + (r * NR + H_A4), rok && al, a4);
        TREX_UNROLL for (int e = 0; e < 4; e++) a4[e] = sel((gls * 4 + e) < nr, a4[e], 0.0f);
        st4_if(Sc, gb + gls * 4 + (AOFF + r * NR), a4, al);
      }
      // Bp row r: the lane's own two joints (positions 2 gl, 2 gl + 1; the pad position 25 gets 0)
      vf b2[2];
      TREX_UNROLL for (int s = 0; s < 2; s++) b2[s] = ld_if(workh0, hoff + kk[s] + (r * 32 + H_BT), rok && kv[s], 0.0f);
      st2_if(Sc, bp_mine + r * BS, b2, gl < 13);
    }
    if (TM) tmem_st_wait();
  }
  warp_sync();
  // joints with a violated limit in either environment, in Bullet's limit-constraint order (bit p <=> position p)
  static_assert(limit_order_matches_motor_order(), "solve2 assumes order[NJ + p] == order[p] - NJ");
  uint32_t uperm = 0;
  TREX_UNROLL for (int s = 0; s < 2; s++) {
    const uint32_t b = vballot(kv[s] && (sigma[s] != 0.0f));
    const uint32_t any = (b | (b >> 16)) & 0xffffu;  // bit l: lane l of either group
    TREX_UNROLL for (int l = 0; l < 13; l++) uperm |= ((any >> l) & 1u) << (2 * l + s);
  }
  uint32_t cached = 0;
  {
    uint32_t m = uperm;
    TREX_ROLLED for (int slot = 0; slot < TREX_S2_LIMIT_SLOTS && m != 0; slot++) {
      const int pos = ctz_u(m);
      m &= m - 1;
      cached |= 1u << pos;
      const int j = P.order[NJ + pos];
      TREX_UNROLL for (int s = 0; s < 2; s++)
        st(Lg, lane + (slot * 2 + s) * 32,
           sel(kk[s] == j, 0.0f, njdi[s] * ld_if(work0, woff + kk[s] * 32 + (W_COL + 6 * 32 + j), kv[s], 0.0f)));
    }
  }
  warp_sync();

  vf w[2], lam_m[2], lam_l[2];
  TREX_UNROLL for (int s = 0; s < 2; s++) { w[s] = rhs_m[s]; lam_m[s] = 0.0f; lam_l[s] = 0.0f; }
  const float lim_hi = P.limit_max_impulse;
  vb alive = gact;
  vi itd = 0;

#define TREX_S2_LIMIT_SLOT(SJ)                                                                         \
  {                                                                                                    \
    const vf x = (lam_m[SJ] + rhs_m[SJ]) - w[SJ];              /* jdi * dv_j */                         \
    const vf sum = lam_l[SJ] + (rhs_l[SJ] - sigma[SJ] * x);                                            \
    const vf nl = vmin(vmax(sum, 0.0f), lim_hi);                                                       \
    const vb own = alive && (gl == (pos >> 1)) && (sigma[SJ] != 0.0f);                                 \
    const vf d = sel(own, (nl - lam_l[SJ]) * sigma[SJ], 0.0f);  /* change of the net joint impulse */   \
    const vf db = shfl_group16(d, pos >> 1);                                                           \
    lam_l[SJ] = sel(own, nl, lam_l[SJ]);                                                               \
    vfma2s(w[0], w[1], gj[0], gj[1], db);                                                              \
    w[SJ] = w[SJ] - d;                                        /* self term: dv_j += D_j * d */         \
    TREX_UNROLL for (int k = 0; k < 3; k++) cu[k] = vfma(ld(Sc, bp_own + (k * BS + pos)), db, cu[k]);  \
  }
#define TREX_S2_LIMITS(FORWARD)                                                                        \
  {                                                                                                    \
    uint32_t m = uperm;                                                                                \
    while (m) {                                                                                        \
      const int pos = (FORWARD) ? ctz_u(m) : 31 - clz_u(m);                                            \
      m &= ~(1u << pos);                                                                               \
      const int j = P.order[NJ + pos];                                                                 \
      vf gj[2];                                                                                        \
      if ((cached >> pos) & 1u) {                                                                      \
        const int slot = popc_u(cached & ((1u << pos) - 1u));                                          \
        TREX_UNROLL for (int s = 0; s < 2; s++) gj[s] = ld(Lg, lane + (slot * 2 + s) * 32);            \
      } else {                                                                                         \
        TREX_UNROLL for (int s = 0; s < 2; s++)                                                        \
          gj[s] = sel(kk[s] == j, 0.0f, njdi[s] * ld_if(work0, woff + kk[s] * 32 + (W_COL + 6 * 32 + j), kv[s], 0.0f)); \
      }                                                                                                \
      if (pos & 1) TREX_S2_LIMIT_SLOT(1) else TREX_S2_LIMIT_SLOT(0)                                    \
    }                                                                                                  \
  }
#define MB_(b, fwd) s2_motor_block<b, fwd>(w, lam_m, g, cu, glx, dead, bp_own, Sc, max_imp);
  vf mu_l = ENVP ? mu_own : vf(P.mu);
  TREX_ROLLED for (int it = 0; it < P.iters; it++) {
    // every 16th sweep (TREX_S2_REBUILD_MASK) rebuild w and u exactly from the impulses (also the warm-started initial state):
    // w_k = rhs_m,k - sigma_k lam_l,k + sum_j g[k][j] Lambda_j - jdi_k sum_r B[r][k] lambda_r
    // u_r = sum_j B[r][j] Lambda_j + sum_r' A[r'][r] lambda_r'
    if ((it & TREX_S2_REBUILD_MASK) == 0) {
      warp_sync();
      TREX_UNROLL for (int s = 0; s < 2; s++) st_if(Lam, grp * LS + kk[s], lam_m[s] + sigma[s] * lam_l[s], kv[s]);
      TREX_UNROLL for (int k = 0; k < 3; k++) st(Lam, grp * LS + gl * 4 + (32 + k), cl[k]);
      warp_sync();
      vf acc[2], ua[3], bs[2];
      TREX_UNROLL for (int s = 0; s < 2; s++) { acc[s] = rhs_m[s] - sigma[s] * lam_l[s]; bs[s] = 0.0f; }
      TREX_UNROLL for (int k = 0; k < 3; k++) ua[k] = 0.0f;
      TREX_UNROLL for (int j = 0; j < NJ; j++) {
        const vf Lj = ld(Lam, grp * LS + j);
        vfma2s(acc[0], acc[1], g[0][j], g[1][j], Lj);
        TREX_UNROLL for (int k = 0; k < 3; k++) ua[k] = vfma(ld(Sc, bp_own + (k * BS + motor_position(j))), Lj, ua[k]);
      }
      TREX_ROLLED for (int c = 0; c < kmax; c++) {
        vf ar[3][4];
        TREX_UNROLL for (int k = 0; k < 3; k++) s2_fetch_a<TM>(Sc, a_own, tm, 3 * c + k, ar[k]);
        TREX_UNROLL for (int k = 0; k < 3; k++) s2_ready_a<TM>(ar[k]);
        TREX_UNROLL for (int k = 0; k < 3; k++) {
          const vf Lr = ld(Lam, grp * LS + (32 + c * 4 + k));
          vf b2[2];
          ld2(Sc, bp_mine + (3 * c + k) * BS, b2);
          TREX_UNROLL for (int s = 0; s < 2; s++) bs[s] = vfma(b2[s], Lr, bs[s]);
          TREX_UNROLL for (int k2 = 0; k2 < 3; k2++) ua[k2] = vfma(ar[k][k2], Lr, ua[k2]);
        }
      }
      TREX_UNROLL for (int s = 0; s < 2; s++) acc[s] = vfma(njdi[s], bs[s], acc[s]);
      TREX_UNROLL for (int k = 0; k < 3; k++) cu[k] = ua[k];
      TREX_UNROLL for (int s = 0; s < 2; s++) w[s] = sel(alive, acc[s], w[s]);
    }
    vf lam_m0[2], lam_l0[2];
    vf cres = 0.0f;
    TREX_UNROLL for (int s = 0; s < 2; s++) { lam_m0[s] = lam_m[s]; lam_l0[s] = lam_l[s]; }
    // a finished environment is frozen without a select on the dependent chain (see solve4): no motor row of its own, the
    // zeros of its idle lane 15 published, contact rows with jdi = rhs = 0 and an unbounded cone
    const vi glx = seli(alive, gl, vi(-1)), dead = seli(alive, vi(0), vi(15));
    if (it & 1) {
      MB_(0, true) MB_(1, true) MB_(2, true) MB_(3, true) MB_(4, true) MB_(5, true) MB_(6, true) MB_(7, true) MB_(8, true) MB_(9, true)
      MB_(10, true) MB_(11, true) MB_(12, true)
      TREX_S2_LIMITS(true)
    } else {
      TREX_S2_LIMITS(false)
      MB_(12, false) MB_(11, false) MB_(10, false) MB_(9, false) MB_(8, false) MB_(7, false) MB_(6, false) MB_(5, false) MB_(4, false)
      MB_(3, false) MB_(2, false) MB_(1, false) MB_(0, false)
    }
    // normal rows: every lane evaluates its own contact, the owner of contact c publishes.  The rows of A and Bp a
    // publication needs do not depend on the sweep's data: they are fetched one iteration ahead (software pipeline), so
    // the shared-memory latency sits under the owner's clamp chain instead of behind the shuffle.
    const vf cl0_0 = cl[0], cl1_0 = cl[1], cl2_0 = cl[2];
    // (two register sets alternate -- the loop is unrolled by two -- so the pipeline costs no register moves)
#define TREX_S2_NORMAL(C, A3, B2, AN, BN)                                                                 \
    {                                                                                                      \
      const int cn = (C) + 1 < kmax ? (C) + 1 : (C);                                                       \
      s2_ready_a<TM>(A3);                                                                                  \
      s2_fetch_a<TM>(Sc, a_own, tm, 3 * cn, AN);                                                           \
      ld2(Sc, bp_mine + (3 * cn) * BS, BN);                                                                \
      const vf nl = vmax(vfma(-cu[0], cjdi[0], pre0), 0.0f);  /* chain: FFMA, FMNMX, FADD, SHFL, FFMA */  \
      const vf d = shfl_group16(nl - cl[0], (C));                                                          \
      cl[0] = sel(gl == (C), nl, cl[0]);                                                                   \
      TREX_UNROLL for (int k = 0; k < 3; k++) cu[k] = vfma(A3[k], d, cu[k]);                               \
      vf nd[2];                                                                                            \
      vmul2s(nd[0], nd[1], njdi[0], njdi[1], d);                                                           \
      vfma2v(w[0], w[1], B2[0], B2[1], nd[0], nd[1]);                                                      \
    }
    const vf pre0 = cl[0] + crhs[0];
    {
      vf a0[4], b0[2], a1[4], b1[2];
      s2_fetch_a<TM>(Sc, a_own, tm, 0, a0);
      ld2(Sc, bp_mine, b0);
      TREX_ROLLED for (int c = 0; c < kmax; c += 2) {
        TREX_S2_NORMAL(c, a0, b0, a1, b1)
        if (c + 1 < kmax) TREX_S2_NORMAL(c + 1, a1, b1, a0, b0) else s2_ready_a<TM>(a1);
      }
      if ((kmax & 1) == 0) s2_ready_a<TM>(a0);  /* (the last prefetch is never used: retire it) */
    }
#undef TREX_S2_NORMAL
    // friction pairs, implicit cone; both rows read the velocities before either writes
#define TREX_S2_FRICTION(C, AA, AB, BA, BB, AAN, ABN, BAN, BBN)                                            \
    {                                                                                                      \
      const int cn = (C) + 1 < kmax ? (C) + 1 : (C);                                                       \
      s2_ready_a<TM>(AA);                                                                                  \
      s2_ready_a<TM>(AB);                                                                                  \
      s2_fetch_a<TM>(Sc, a_own, tm, 3 * cn + 1, AAN);                                                      \
      s2_fetch_a<TM>(Sc, a_own, tm, 3 * cn + 2, ABN);                                                      \
      ld2(Sc, bp_mine + (3 * cn + 1) * BS, BAN);                                                           \
      ld2(Sc, bp_mine + (3 * cn + 2) * BS, BBN);                                                           \
      const vf sumB = vfma(-cu[2], cjdi[2], preB);                                                         \
      const vf sumA = vfma(-cu[1], cjdi[1], preA);                                                         \
      const vf rn = vrsqrt(vmax(sumA * sumA + sumB * sumB, 1.0e-30f));                                     \
      const vf nA = vclamp_sym(sumA, lim * vabs(sumA * rn));                                               \
      const vf nB = vclamp_sym(sumB, lim * vabs(sumB * rn));                                               \
      const vf dAu = shfl_group16(nA - cl[1], (C)), dBu = shfl_group16(nB - cl[2], (C));                   \
      const vb mine = gl == (C);                                                                           \
      cl[1] = sel(mine, nA, cl[1]);                                                                        \
      cl[2] = sel(mine, nB, cl[2]);                                                                        \
      TREX_UNROLL for (int k = 0; k < 3; k++) cu[k] = vfma(AA[k], dAu, vfma(AB[k], dBu, cu[k]));           \
      vf tb[2];                                                                                            \
      vmul2s(tb[0], tb[1], BB[0], BB[1], dBu);                                                             \
      vfma2s(tb[0], tb[1], BA[0], BA[1], dAu);                                                             \
      vfma2v(w[0], w[1], njdi[0], njdi[1], tb[0], tb[1]);                                                  \
    }
    const vf lim = mu_l * cl[0];
    const vf preA = cl[1] + crhs[1], preB = cl[2] + crhs[2];
    {
      vf aA0[4], aB0[4], bA0[2], bB0[2], aA1[4], aB1[4], bA1[2], bB1[2];
      s2_fetch_a<TM>(Sc, a_own, tm, 1, aA0);
      s2_fetch_a<TM>(Sc, a_own, tm, 2, aB0);
      ld2(Sc, bp_mine + BS, bA0);
      ld2(Sc, bp_mine + 2 * BS, bB0);
      TREX_ROLLED for (int c = 0; c < kmax; c += 2) {
        TREX_S2_FRICTION(c, aA0, aB0, bA0, bB0, aA1, aB1, bA1, bB1)
        if (c + 1 < kmax) TREX_S2_FRICTION(c + 1, aA1, aB1, bA1, bB1, aA0, aB0, bA0, bB0) else { s2_ready_a<TM>(aA1); s2_ready_a<TM>(aB1); }
      }
      if ((kmax & 1) == 0) { s2_ready_a<TM>(aA0); s2_ready_a<TM>(aB0); }
    }
#undef TREX_S2_FRICTION
    {  // residual of the contact rows: every row is visited once per sweep, so its impulse change is end - start
      const vf dn = (cl[0] - cl0_0) * cdd[0];
      const vf dt2 = (cl[1] - cl1_0) * cdd[1] + (cl[2] - cl2_0) * cdd[2];
      cres = vmax(dn * dn, dt2 * dt2);
    }
    // residual per environment: max over its rows of (delta impulse / jacDiagABInv)^2
    vf r = cres;
    TREX_UNROLL for (int s = 0; s < 2; s++) {
      const vf dm = (lam_m[s] - lam_m0[s]) * dself[s];
      r = vmax(r, dm * dm);
    }
    if (uperm != 0u) {
      TREX_UNROLL for (int s = 0; s < 2; s++) {
        const vf dlm = (lam_l[s] - lam_l0[s]) * dself[s];
        r = vmax(r, dlm * dlm);
      }
    }
    const uint32_t over = vballot(alive && !(r <= P.resid_thresh));
    itd = itd + seli(alive, vi(1), vi(0));
    const vi ob = seli(grp == 0, vi((int)(over & 0xffffu)), vi((int)(over >> 16)));
    alive = alive && (ob != 0) && (it < P.iters - 1);
    if (over == 0u || it >= P.iters - 1) break;
    // freeze the contact rows of an environment that has just finished
    TREX_UNROLL for (int k = 0; k < 3; k++) { crhs[k] = sel(alive, crhs[k], 0.0f); cjdi[k] = sel(alive, cjdi[k], 0.0f); }
    mu_l = sel(alive, mu_l, 1.0e30f);
  }
#undef MB_
#undef TREX_S2_LIMIT_SLOT
#undef TREX_S2_LIMITS

  // ---- velocity change of every coordinate from the final impulses ------------------------------------
  warp_sync();
  TREX_UNROLL for (int s = 0; s < 2; s++) st_if(Lam, grp * LS + kk[s], lam_m[s] + sigma[s] * lam_l[s], kv[s]);
  TREX_UNROLL for (int k = 0; k < 3; k++) st(Lam, grp * LS + gl * 4 + (32 + k), cl[k]);
  warp_sync();
  vf Ssum[2], bsum[2];
  TREX_UNROLL for (int s = 0; s < 2; s++) { Ssum[s] = 0.0f; bsum[s] = 0.0f; }
  TREX_UNROLL for (int j = 0; j < NJ; j++) {
    const vf Lj = ld(Lam, grp * LS + j);
    vfma2s(Ssum[0], Ssum[1], g[0][j], g[1][j], Lj);
  }
  vf dvb[6];
  TREX_UNROLL for (int b = 0; b < 6; b++) dvb[b] = 0.0f;
  TREX_UNROLL for (int s = 0; s < 2; s++) {
    const vf Lk = lam_m[s] + sigma[s] * lam_l[s];
    TREX_UNROLL for (int b = 0; b < 6; b++) dvb[b] = vfma(ld_if(work0, woff + kk[s] + (W_COL + b * 32), kv[s], 0.0f), Lk, dvb[b]);
  }
  TREX_ROLLED for (int c = 0; c < kmax; c++)
    TREX_UNROLL for (int k = 0; k < 3; k++) {
      const vf Lr = ld(Lam, grp * LS + (32 + c * 4 + k));
      vf b2[2];
      ld2(Sc, bp_mine + (3 * c + k) * BS, b2);
      TREX_UNROLL for (int s = 0; s < 2; s++) bsum[s] = vfma(b2[s], Lr, bsum[s]);
    }
  TREX_UNROLL for (int k = 0; k < 3; k++)
    TREX_UNROLL for (int b = 0; b < 6; b++)
      dvb[b] = vfma(ld_if(workh0, hoff + gl * 96 + (H_BT + k * 32 + 25 + b), cown, 0.0f), cl[k], dvb[b]);
  st_if(rec0, roff + ccand + ST_LAM, cl[0], cown);  // cached normal impulse of the candidate (next substep's warm start)
  TREX_UNROLL for (int b = 0; b < 6; b++) dvb[b] = group16_sum(dvb[b]);

  // ---- velocities += dv (clamped), applied motor torque, positions with the NEW velocities ----------------
  TREX_UNROLL for (int s = 0; s < 2; s++) {
    const vf Lk = lam_m[s] + sigma[s] * lam_l[s];
    const vf dvk = dself[s] * (Lk - Ssum[s]) + bsum[s];
    const vf qd0 = ld_if(rec0, roff + kk[s] + ST_QD, kv[s], 0.0f);
    const vf q0 = ld_if(rec0, roff + kk[s] + ST_Q, kv[s], 0.0f);
    const vf qd1 = clampv(qd0 + dvk, -P.maxvel, P.maxvel);
    st_if(rec0, roff + kk[s] + ST_QD, qd1, kv[s]);
    st_if(rec0, roff + kk[s] + ST_Q, q0 + dt * qd1, kv[s]);
    st_if(rec0, roff + kk[s] + ST_TAU, vdiv(lam_m[s], dt), kv[s]);
  }
  {
    vf om[3], vl[3], pos[3], qt[4];
    TREX_UNROLL for (int k = 0; k < 3; k++) {
      om[k] = clampv(ld(rec0, roff + (ST_OM + k)) + dvb[k], -P.maxvel, P.maxvel);
      vl[k] = clampv(ld(rec0, roff + (ST_VL + k)) + dvb[3 + k], -P.maxvel, P.maxvel);
      pos[k] = ld(rec0, roff + (ST_POS + k)) + dt * vl[k];
    }
    TREX_UNROLL for (int k = 0; k < 4; k++) qt[k] = ld(rec0, roff + (ST_QUAT + k));
    // btMultiBody::stepPositionsMultiDof: exponential map of the world angular velocity, q <- dq * q
    vf fa = vsqrt(om[0] * om[0] + om[1] * om[1] + om[2] * om[2]);
    fa = sel(fa * dt > 0.78539816339744831f, vbroadcast(0.78539816339744831f / dt), fa);
    const vb small = fa < 0.001f;
    const vf sc = sel(small, 0.5f * dt - (dt * dt * dt) * 0.020833333333f * fa * fa, vdiv(vsin(0.5f * fa * dt), sel(small, 1.0f, fa)));
    const vf ax = om[0] * sc, ay = om[1] * sc, az = om[2] * sc, aw = vcos(fa * dt * 0.5f);
    const vf nx = aw * qt[0] + ax * qt[3] + ay * qt[2] - az * qt[1];
    const vf ny = aw * qt[1] - ax * qt[2] + ay * qt[3] + az * qt[0];
    const vf nz = aw * qt[2] + ax * qt[1] - ay * qt[0] + az * qt[3];
    const vf nw = aw * qt[3] - ax * qt[0] - ay * qt[1] - az * qt[2];
    const vf inv = vdiv(1.0f, vsqrt(nx * nx + ny * ny + nz * nz + nw * nw));
    warp_sync();
    // one lane per field of the base block [pos3 quat4 om3 vl3]
    vf val = 0.0f;
    TREX_UNROLL for (int k = 0; k < 3; k++) {
      val = sel(gl == ST_POS + k, pos[k], val);
      val = sel(gl == ST_OM + k, om[k], val);
      val = sel(gl == ST_VL + k, vl[k], val);
    }
    val = sel(gl == ST_QUAT, nx * inv, sel(gl == ST_QUAT + 1, ny * inv, sel(gl == ST_QUAT + 2, nz * inv, sel(gl == ST_QUAT + 3, nw * inv, val))));
    st_if(rec0, roff + gl, val, gact && (gl < 13));
  }
  {  // active-set signature of this substep's solve (StepStats), per environment: OR over the group's lanes, lane 0 folds
    vi Lm = 0, Mm = 0;
    TREX_UNROLL for (int s = 0; s < 2; s++) {
      Lm = Lm | seli(kv[s] && (lam_l[s] > 0.0f), vi(1) << kk[s], vi(0));
      Mm = Mm | seli(kv[s] && (vabs(lam_m[s]) >= max_imp), vi(1) << kk[s], vi(0));
    }
    vi NF = 0;
    {
      const vf lim = (ENVP ? mu_own : vf(P.mu)) * cl[0];
      const vb pos = cown && (cl[0] > 0.0f);
      NF = seli(pos, vi(1) << gl, vi(0)) |
           seli(pos && ((cl[1] * cl[1] + cl[2] * cl[2]) >= TREX_CONE_EDGE * (lim * lim)), vi(65536) << gl, vi(0));
    }
    TREX_UNROLL for (int m = 8; m > 0; m >>= 1) { Lm = Lm | shfl_xor_i(Lm, m); Mm = Mm | shfl_xor_i(Mm, m); NF = NF | shfl_xor_i(NF, m); }
    const vb wr = gact && (gl == 0);
    const vi si = seli(wr, roff + ST_SIG, 0);
    const vi h = sig_mix_v(sig_mix_v(sig_mix_v(sig_mix_v(vf2i(ld(rec0, si)), Lm), Mm), NF), itd) & 0xffffff;
    st_if(rec0, si, vi2f(h), wr);
  }
  warp_sync();
  return itd;
}

// reward (trex_env.py:186-196), termination (trex_env.py:183-184 + optional horizon / NaN guard) of one environment
TREX_FN void reward_and_done(const Uniform& P, const float* mdl, vi lane, WarpShared& S, const EnvRegs& R, vi slot,
                             float step_count, float head[3], float terms[3], float& rew, bool& bad, bool& is_done) {
  const vb is_joint = lane < NJ;
  // head-link COM in world: forward kinematics along the base -> head chain only (uniform arithmetic)
  float Rh[9], xh[3] = {R.pos[0], R.pos[1], R.pos[2]};
  quat_to_Rb(R.quat, Rh);
  TREX_ROLLED for (int d = 0; d < P.head_depth; d++) {
    const int L = P.head_chain[d];
    const float qj = lane_value(R.q, L);
    const float c = cosf(qj), sn = sinf(qj);
    float e0[9], r0h[3], El[9], Rn[9];
    TREX_UNROLL for (int k = 0; k < 9; k++) e0[k] = ldu(mdl, (F_E0 + k) * 32 + L);
    TREX_UNROLL for (int k = 0; k < 3; k++) r0h[k] = ldu(mdl, (F_R0 + k) * 32 + L);
    TREX_UNROLL for (int j = 0; j < 3; j++) xh[j] += Rh[j] * r0h[0] + Rh[3 + j] * r0h[1] + Rh[6 + j] * r0h[2];
    El[0] = c * e0[0] + sn * e0[1]; El[1] = c * e0[3] + sn * e0[4]; El[2] = c * e0[6] + sn * e0[7];
    El[3] = c * e0[1] - sn * e0[0]; El[4] = c * e0[4] - sn * e0[3]; El[5] = c * e0[7] - sn * e0[6];
    El[6] = e0[2]; El[7] = e0[5]; El[8] = e0[8];
    TREX_UNROLL for (int i = 0; i < 3; i++)
      TREX_UNROLL for (int j = 0; j < 3; j++) Rn[3 * i + j] = El[3 * i] * Rh[j] + El[3 * i + 1] * Rh[3 + j] + El[3 * i + 2] * Rh[6 + j];
    TREX_UNROLL for (int k = 0; k < 9; k++) Rh[k] = Rn[k];
  }
  TREX_UNROLL for (int j = 0; j < 3; j++) head[j] = xh[j] + Rh[j] * P.head_p[0] + Rh[3 + j] * P.head_p[1] + Rh[6 + j] * P.head_p[2];
  // total |qd * tau| in sorted-joint order, sequential non-fused sum (reproducible from the outputs)
  warp_sync();
  st_if(S.tmp[0], slot, vabs(vmul_rn(R.qd, R.tau)), is_joint);
  warp_sync();
  float power = 0.0f;
  TREX_ROLLED for (int k = 0; k < NJ; k++) power = fadd_rn(power, ldu(S.tmp[0], k));
  const float dz = fadd_rn(P.target_h, -head[2]);
  terms[0] = fmul_rn(P.w_dist, fmul_rn(dz, dz));                                                 // lifting
  terms[1] = fmul_rn(P.w_drift, fadd_rn(fmul_rn(head[0], head[0]), fmul_rn(head[1], head[1])));  // station keeping
  terms[2] = fmul_rn(P.w_energy, power);                                                         // energy
  rew = fadd_rn(fadd_rn(-terms[0], -terms[1]), -terms[2]);
  warp_sync();
  bad = vany(visnan(R.q) || visnan(R.qd)) || !(fabsf(R.pos[0]) + fabsf(R.pos[1]) + fabsf(R.pos[2]) <= 3.0e38f) ||
        !(fabsf(R.quat[0]) + fabsf(R.quat[3]) <= 3.0e38f) || !(fabsf(R.om[0]) + fabsf(R.om[1]) + fabsf(R.om[2]) <= 3.0e38f);
  is_done = bad || (P.max_episode_steps > 0 && step_count >= (float)P.max_episode_steps);
}

// ------------------------------------------------------------------------------------------
// One TrexBulletEnv.step (trex_env.py:128-154) = n_sub x [front_phase ; solve_phase] ; tail_phase, each phase
// a kernel of its own (trex_capi.cu).  Splitting keeps every kernel's hot loop resident in the instruction
// cache (a fused kernel mixing the two solvers measured 7.6 no-instruction stalls per issue) and lets the
// 4-environments-per-warp solver run at its own occupancy.
// ------------------------------------------------------------------------------------------
enum { ST_ACC_ITERS = 155, ST_ACC_CONTACTS = 156, ST_ACC_OVERFLOW = 157 };  // per-step accumulators in the record (ST_SIG = 158 follows)
static_assert(ST_SIG == ST_ACC_ITERS + 3, "front_phase stores the four accumulators as one block");

// front_phase: one physics substep of ONE environment by one warp up to the solve: kinematics, bias forces,
// articulated inertias, accelerations, velocity update, M^-1, row setup, contact detection.  With more than TREX_KC
// contacts the substep is finished here (one-environment solver + integration); otherwise the solver inputs go to
// `work` and the function returns 1 + class (solve_phase finishes the substep).   action: [25] name-sorted (trex_robot.py:311-314)
// ENVP: envp = the environment's parameter row (mass scales, friction, motor gains and impulse bound)
// EXTF: extf = the environment's wrench record [6][32], com = the COM table [3][32], push = the push schedule,
// env_id = index of the environment in this launch (P.env_offset + env_id keys the schedule)
// TAU (trex_config.actuation = TREX_ACTUATION_TORQUE): the action is the joint torque, clipped to +-tau_max (ENVP: +-the row's
// element EP_MAX_TORQUE) and applied in this substep; the motors run with kp = kd = 0 and impulse bound 0
template <bool PACKED = false, bool ENVP = false, bool EXTF = false, bool TAU = false>
TREX_FN int front_phase(const Uniform& P, const float* mdl, const int* mdli, const float* tasks, const float* cand_p,
                         const int* cand_lane, WarpShared& S, float* rec, float* work, const float* action, bool first_round,
                         WarpShared* cta_slabs = nullptr, int warp_in_cta = 0, int valid_mask = 0, float* workh = nullptr,
                         const float* envp = nullptr, const float* extf = nullptr, const float* com = nullptr,
                         const PushSchedule* push = nullptr, long long env_id = 0, float tau_max = 0.0f) {
  const vi lane = lane_id();
  const vb is_joint = lane < NJ;
  const vi slot = seli(is_joint, MDLI(IF_OBS_SLOT), 0);
  EnvRegs R;
  load_env(rec, lane, S, R);
  // np.clip(action, low, high)  (trex_env.py:147); the targets are re-applied every substep (:148-150)
  const vf a = ld_if(action, slot, is_joint, 0.0f);
  if (!TAU) R.tgt = vmin(vmax(a, MDL(F_LOWER)), MDL(F_UPPER));  // (TAU: R.tgt stays 0, the motors have no gain)
  StepStats st;
  st.iters = 0; st.contacts = 0; st.overflow = 0;
  st.sig = first_round ? 0u : (uint32_t)ldu(rec, ST_SIG);
#ifdef TREX_PHASES
  for (int i = 0; i < 8; i++) st.phase[i] = 0.0f;
#endif
  const float kp = TAU ? 0.0f : (ENVP ? ldu(envp, EP_KP) : P.kp), kd = TAU ? 0.0f : (ENVP ? ldu(envp, EP_KD) : P.kd);
  const float max_imp = TAU ? 0.0f : (ENVP ? ldu(envp, EP_MAX_IMPULSE) : P.max_impulse);
  ExtWrench xf;
  if (EXTF) {
    xf.rec = extf;
    xf.com = com;
    // the step count as the tail kernel left it: steps completed in this episode
    push_of_step(*push, P.seed, (unsigned long long)(P.env_offset + env_id), ldu(rec, ST_EPISODE), ldu(rec, ST_STEP), xf);
  }
  const int deferred = substep<PACKED, ENVP, EXTF, TAU>(P, mdl, mdli, tasks, cand_p, cand_lane, S, R, kp, kd, max_imp, st, work,
                                                        cta_slabs, warp_in_cta, valid_mask, workh, envp, EXTF ? &xf : nullptr, action,
                                                        TAU ? (ENVP ? ldu(envp, EP_MAX_TORQUE) : tau_max) : 0.0f);
  store_env(rec, lane, S, R);  // deferred: positions unchanged, velocities after the unconstrained update
  const float it0 = first_round ? 0.0f : ldu(rec, ST_ACC_ITERS), ov0 = first_round ? 0.0f : ldu(rec, ST_ACC_OVERFLOW);
  vf acc = 0.0f;
  acc = sel(lane == 0, vbroadcast(it0 + (float)st.iters), acc);
  acc = sel(lane == 1, vbroadcast((float)st.contacts), acc);
  acc = sel(lane == 2, vbroadcast(ov0 + (float)st.overflow), acc);
  acc = sel(lane == 3, vbroadcast((float)(st.sig & 0xffffffu)), acc);
  warp_sync();
  st_if(rec, lane + ST_ACC_ITERS, acc, lane < 4);  // ST_ACC_ITERS, ST_ACC_CONTACTS, ST_ACC_OVERFLOW, ST_SIG
#ifdef TREX_PHASES
  {  // cycles per phase of this environment's front kernel work, summed over the substeps of the env step
    vf ph = 0.0f;
    for (int i = 0; i < 8; i++) ph = sel(lane == i, vbroadcast(st.phase[i] + (first_round ? 0.0f : ldu(rec, 160 + i))), ph);
    st_if(rec, lane + 160, ph, lane < 8);
  }
#endif
  return deferred + 256 * st.contacts;  // low byte: 0 = substep complete, 1 + class = solve deferred; above: active contacts
}

// solve_phase: the deferred solves of up to four environments (any four: the groups are independent)
// ENVP: envp0 = parameter rows indexed like rec0 (the motor impulse bound of each group's environment)
template <int KC, bool TM = false, bool ENVP = false>
TREX_FN void solve_phase(const Uniform& P, float* scratch, const float* work0, float* rec0, const int envs[4], int pending,
                         tmem_t tm = tmem_t(), const float* envp0 = nullptr) {
  const vi lane = lane_id();
  vf max_imp = P.max_impulse;
  if (ENVP) {
    const vi g = lane >> 3;
    const vi ge = seli(g == 0, vi(envs[0]), seli(g == 1, vi(envs[1]), seli(g == 2, vi(envs[2]), vi(envs[3]))));
    const vb gp = ((vi(pending) >> g) & 1) != 0;
    max_imp = ld_if(envp0, seli(gp, ge, 0) * TREX_ENVP_DIM + EP_MAX_IMPULSE, gp, 0.0f);
  }
  const vi itd = solve4<KC, TM, ENVP>(P, scratch, work0, rec0, envs, pending, max_imp, tm);
  // iterations executed per environment -> its accumulator (lane 8e holds group e's count)
  const vi grp = lane >> 3;
  const vb wr = ((lane & 7) == 0) && ((((vi(pending)) >> grp) & 1) != 0);
  const vi genv = seli(grp == 0, vi(envs[0]), seli(grp == 1, vi(envs[1]), seli(grp == 2, vi(envs[2]), vi(envs[3]))));
  const vi idx = seli(wr, genv * TREX_STATE_STRIDE + ST_ACC_ITERS, 0);
  st_if(rec0, idx, ld(rec0, idx) + vi2f(itd), wr);
}

// heavy_phase: the deferred solves of up to two environments with more than TREX_KC contacts (any two)
template <bool TM = false, bool ENVP = false>
TREX_FN void heavy_phase(const Uniform& P, float* scratch, tmem_t tm, const float* work0, const float* workh0, float* rec0, const int envs[2],
                         int pending, const float* envp0 = nullptr) {
  const vi lane = lane_id();
  vf max_imp = P.max_impulse;
  if (ENVP) {
    const vi g = lane >> 4;
    const vi ge = seli(g == 0, vi(envs[0]), vi(envs[1]));
    const vb gp = ((vi(pending) >> g) & 1) != 0;
    max_imp = ld_if(envp0, seli(gp, ge, 0) * TREX_ENVP_DIM + EP_MAX_IMPULSE, gp, 0.0f);
  }
  const vi itd = solve2<TM, ENVP>(P, scratch, tm, work0, workh0, rec0, envs, pending, max_imp);
  const vi grp = lane >> 4;
  const vb wr = ((lane & 15) == 0) && ((((vi(pending)) >> grp) & 1) != 0);
  const vi genv = seli(grp == 0, vi(envs[0]), vi(envs[1]));
  const vi idx = seli(wr, genv * TREX_STATE_STRIDE + ST_ACC_ITERS, 0);
  st_if(rec0, idx, ld(rec0, idx) + vi2f(itd), wr);
}

// tail_phase: end of the env step for ONE environment: reward (trex_env.py:186-196), done (trex_env.py:183-184 +
// optional horizon / NaN guard), VecEnv auto-reset = TrexBulletEnv.reset (trex_env.py:98-122: reset pose, zero-gain
// zero-force motors, ONE physics step), observations (trex_robot.py:359-365), diagnostics.
// force_reset: only the reset (trex_reset).
//   obs : [75] q | qd | motor torque   aux : [TREX_AUX_STRIDE] head xyz, lifting/station/energy, PGS iterations, contacts
// ENVP: envp = the environment's parameter row (mass scales and friction apply to the reset step; its motor gains stay zero).
// ranges != nullptr: the randomizer is on -- every reset first draws a new row (draw_env_params).
// TAU: action = the step's actions [25] name-sorted, tau_max = the torque bound without ENVP: the applied torque the reward and
// the observation report (and record [63:88] keeps) is the clipped command, not the motors' impulse / dt.  A reset reports
// the reset step's own value.
template <bool ENVP = false, bool TAU = false>
TREX_FN void tail_phase(const Uniform& P, const float* mdl, const int* mdli, const float* tasks, const float* cand_p,
                        const int* cand_lane, WarpShared& S, float* rec, float* obs, float* reward, uint8_t* done,
                        float* aux, bool force_reset, long long env_id, float* envp = nullptr, const float* ranges = nullptr,
                        double dt = 0.0, const float* action = nullptr, float tau_max = 0.0f) {
  const vi lane = lane_id();
  const vb is_joint = lane < NJ;
  const vi slot = seli(is_joint, MDLI(IF_OBS_SLOT), 0);
  EnvRegs R;
  load_env(rec, lane, S, R);
  bool is_done = false;
  if (!force_reset) {
    if (TAU) {
      R.tau = clip_torque(ld_if(action, slot, is_joint, 0.0f), is_joint, ENVP ? ldu(envp, EP_MAX_TORQUE) : tau_max);
      st_if(rec, seli(is_joint, lane, 0) + ST_TAU, R.tau, is_joint);
    }
    const float step_count = ldu(rec, ST_STEP) + 1.0f;
    float head[3], terms[3], rew;
    bool bad;
    reward_and_done(P, mdl, lane, S, R, slot, step_count, head, terms, rew, bad, is_done);
    vf meta = 0.0f;
    meta = sel(lane == 0, vbroadcast(step_count), meta);
    meta = sel(lane == 2, vbroadcast(ldu(rec, ST_NANRESETS) + (bad ? 1.0f : 0.0f)), meta);
    st_if(rec, lane + ST_STEP, meta, (lane == 0) || (lane == 2));
    if (reward) st_if(reward, vi(0), vbroadcast(rew), lane == 0);
    if (done) st_u8_if(done, vi(0), vi(is_done ? 1 : 0), lane == 0);
    if (aux) {
      vf ax = 0.0f;
      TREX_UNROLL for (int k = 0; k < 3; k++) {
        ax = sel(lane == k, vbroadcast(head[k]), ax);
        ax = sel(lane == 3 + k, vbroadcast(terms[k]), ax);
      }
      ax = sel(lane == 6, vbroadcast(ldu(rec, ST_ACC_ITERS)), ax);
      ax = sel(lane == 7, vbroadcast(ldu(rec, ST_ACC_CONTACTS) + 1000.0f * ldu(rec, ST_ACC_OVERFLOW)), ax);
      st_if(aux, lane, ax, lane < 8);
#ifdef TREX_PHASES
      st_if(aux, lane, ld(rec, seli(lane >= 8 && lane < 16, lane + 152, 0)), lane >= 8 && lane < 16);
#endif
    }
    warp_sync();
  }
  if (force_reset || is_done) {
    const float episode = ldu(rec, ST_EPISODE);
    reset_pose(P, mdl, lane, S, R, env_id, episode);
    if (ENVP && ranges != nullptr) draw_env_params(P, lane, ranges, envp, env_id, episode, dt);
    StepStats rs;
    rs.iters = 0; rs.contacts = 0; rs.overflow = 0; rs.sig = 0u;
#ifdef TREX_PHASES
    for (int i = 0; i < 8; i++) rs.phase[i] = 0.0f;
#endif
    substep<false, ENVP>(P, mdl, mdli, tasks, cand_p, cand_lane, S, R, 0.0f, 0.0f, 0.0f, rs, nullptr, nullptr, 0, 0, nullptr, envp);
    store_env(rec, lane, S, R);
    vf meta = 0.0f;
    meta = sel(lane == 1, vbroadcast(episode + 1.0f), meta);
    warp_sync();
    st_if(rec, lane + ST_STEP, meta, lane < 2);  // step count 0, episode + 1
  }
  if (obs) {
    st_if(obs, slot, R.q, is_joint);
    st_if(obs, slot + NJ, R.qd, is_joint);
    st_if(obs, slot + 2 * NJ, R.tau, is_joint);
  }
}

// ------------------------------------------------------------------------------------------
// Per-body world states and floor contact forces of ONE environment (trex_get_body_states), one warp, lane L = the body of
// lane L (L < 25: the body of joint L, 25: the base) -- the user order of the query.  Reads the record, writes nothing to it.
//   states [NB][13]: p (COM, world) | q (body -> world, x y z w) | v (COM velocity, world) | w (angular velocity, world).
//     The body frame is the kernels' frame (joint axis +z); the base row's q and w are the record's [3:7] and [7:10].
//   forces [NB]: the floor's normal force in the last physics substep, sum over the body's candidates in ascending candidate
//     index of the cached normal impulse / dt (sequential, unfused); 0 without contacts.
// com: the [3][32] body-frame COM table; stage: TREX_BODY_STAGE floats of the warp's shared memory (the rows are staged there
// and leave as coalesced stores).  Either output may be nullptr.
// ------------------------------------------------------------------------------------------
#define TREX_BODY_DIM 13
#define TREX_BODY_STAGE (trex_topo::NB * TREX_BODY_DIM)
TREX_FN void body_states_phase(const Uniform& P, const float* mdl, const int* mdli, const int* cand_lane, const float* com,
                               const float* rec, float* stage, float* states, float* forces) {
  const vi lane = lane_id();
  const vb is_body = lane < NB;
  if (states) {
    EnvRegs R;
    load_env_regs(rec, lane, R);
    float Rb[9];
    quat_to_Rb(R.quat, Rb);
    vf E[9], Rw[9], xw[3], v[6], c[3];
    local_rotation(mdl, lane, R.q, E);  // (the base keeps Rw = Rb: forward_pass starts at depth 1)
    forward_pass<true>(mdl, mdli, lane, R, Rb, E, Rw, xw, v);
    TREX_UNROLL for (int k = 0; k < 3; k++) c[k] = ldg_ro(com, lane + k * 32);
    // COM velocity in body coordinates: v_origin + w x c
    const vf bx = v[3] + (v[1] * c[2] - v[2] * c[1]);
    const vf by = v[4] + (v[2] * c[0] - v[0] * c[2]);
    const vf bz = v[5] + (v[0] * c[1] - v[1] * c[0]);
    vf o[TREX_BODY_DIM];
    TREX_UNROLL for (int j = 0; j < 3; j++) {  // world = Rw^T body
      o[j] = xw[j] + (Rw[j] * c[0] + Rw[3 + j] * c[1] + Rw[6 + j] * c[2]);
      o[7 + j] = Rw[j] * bx + Rw[3 + j] * by + Rw[6 + j] * bz;
      o[10 + j] = Rw[j] * v[0] + Rw[3 + j] * v[1] + Rw[6 + j] * v[2];
    }
    {  // body -> world quaternion from M = Rw^T (M[i][j] = Rw[3 j + i]), Shepperd's method: the largest of 4 w^2, 4 x^2,
       // 4 y^2, 4 z^2 is taken from the diagonal, the other three from off-diagonal sums / differences; sign: w >= 0
      const vf m00 = Rw[0], m11 = Rw[4], m22 = Rw[8];
      const vf a = Rw[5] - Rw[7], b = Rw[6] - Rw[2], d = Rw[1] - Rw[3];  // M21 - M12, M02 - M20, M10 - M01
      const vf e = Rw[1] + Rw[3], f = Rw[2] + Rw[6], g = Rw[5] + Rw[7];  // M01 + M10, M02 + M20, M12 + M21
      const vf tr = m00 + m11 + m22;
      const vb kx = (m00 > tr) && (m00 >= m11) && (m00 >= m22);
      const vb ky = !kx && (m11 > tr) && (m11 >= m22);
      const vb kz = !kx && !ky && (m22 > tr);
      const vb kw = !kx && !ky && !kz;
      const vf t = sel(kw, 1.0f + tr, sel(kx, 1.0f + m00 - m11 - m22, sel(ky, 1.0f - m00 + m11 - m22, 1.0f - m00 - m11 + m22)));
      const vf r = 0.5f * vsqrt(t);
      const vf s = vdiv(vf(0.25f), r);
      const vf qx = sel(kx, r, sel(kw, a * s, sel(ky, e * s, f * s)));
      const vf qy = sel(ky, r, sel(kw, b * s, sel(kx, e * s, g * s)));
      const vf qz = sel(kz, r, sel(kw, d * s, sel(kx, f * s, g * s)));
      const vf qw = sel(kw, r, sel(kx, a * s, sel(ky, b * s, d * s)));
      const vb neg = qw < 0.0f;
      o[3] = sel(neg, -qx, qx); o[4] = sel(neg, -qy, qy); o[5] = sel(neg, -qz, qz); o[6] = sel(neg, -qw, qw);
    }
    const vb is_base = lane == 25;  // the base's orientation and angular velocity as the record holds them
    TREX_UNROLL for (int k = 0; k < 4; k++) o[3 + k] = sel(is_base, vbroadcast(R.quat[k]), o[3 + k]);
    TREX_UNROLL for (int k = 0; k < 3; k++) o[10 + k] = sel(is_base, vbroadcast(R.om[k]), o[10 + k]);
    // stage the [NB][13] rows (stride 13 is odd: no bank conflicts) and store them as 11 coalesced rows of 32 floats
    const vi row = seli(is_body, lane, 0) * TREX_BODY_DIM;
    TREX_UNROLL for (int k = 0; k < TREX_BODY_DIM; k++) st_if(stage, row + k, o[k], is_body);
    warp_sync();
    TREX_UNROLL for (int i = 0; i < (TREX_BODY_STAGE + 31) / 32; i++) {
      const vi idx = lane + 32 * i;
      const vb in = idx < TREX_BODY_STAGE;
      st_if(states, idx, ld_if(stage, seli(in, idx, 0), in, 0.0f), in);
    }
  }
  if (forces) {
    vf fsum = 0.0f;
    if (P.contacts_on) {
      // lane l holds candidates l and l + 32: impulse / dt and body lane (-1 beyond the model's candidates)
      vf fc[2];
      vi lc[2];
      TREX_UNROLL for (int h = 0; h < 2; h++) {
        const vi ci = lane + 32 * h;
        const vb ok = ci < P.n_cand;
        const vi cs = seli(ok, ci, 0);
        fc[h] = vdiv(ld_if(rec, cs + ST_LAM, ok, 0.0f), vf(P.dt));
        lc[h] = seli(ok, ldi(cand_lane, cs), vi(-1));
      }
      TREX_ROLLED for (int ci = 0; ci < P.n_cand; ci++) {
        const float fk = lane_value(ci < 32 ? fc[0] : fc[1], ci & 31);
        const int lk = lane_value_i(ci < 32 ? lc[0] : lc[1], ci & 31);
        fsum = sel(lane == lk, fsum + fk, fsum);
      }
    }
    st_if(forces, lane, fsum, is_body);
  }
}

// ------------------------------------------------------------------------------------------
// Joint-space mass matrix, bias forces and body Jacobians of ONE environment (trex_get_dynamics), one warp.  Reads the
// record, writes nothing to it.  Generalized velocity u (31): [0:3] base angular velocity (world, record [7:10]), [3:6]
// velocity of the base frame's origin p0 (world, record [10:13]), [6:31] joint rates in lane order (record [38:63]); lane
// L < 25 owns coordinate 6 + L, lanes 25..30 own coordinates 0..5.
//   M [31][31]: kinetic energy = u^T M u / 2; full, each entry below the diagonal a copy of its mirror image
//   b [31]: M du/dt + b = tau: gravity, Coriolis and centrifugal terms only (no damping, motors, limits, contacts, wrenches)
//   J [NB][6][31]: J_k u = [velocity of body k's COM; its angular velocity], world frame
// All vectors are in world axes, positions relative to p0 (the values stay small where the base is far from the world
// origin).  M and b come from subtree sums (dyn_composite, dyn_force_sum) that each lane takes about its own joint's origin:
// the entries of a light distal joint are then not the small difference of large moments about p0.  envp: this
// environment's parameter row (nullptr: the model's masses; a scale multiplies mass and inertia first, as in the step; the
// COM stays).  com: the [3][32] COM table.  stage: TREX_DYN_STAGE floats of the warp's shared memory.  Any output may be
// nullptr and is then not computed.
// ------------------------------------------------------------------------------------------
#define TREX_DYN_NDOF 31
#define TREX_DYN_JROWS 6
#define TREX_DYN_MSIZE (TREX_DYN_NDOF * TREX_DYN_NDOF)
#define TREX_DYN_JSIZE (trex_topo::NB * TREX_DYN_JROWS * TREX_DYN_NDOF)
#define TREX_DYN_SUMS 10                                            // rows of 32 floats for the subtree sums
#define TREX_DYN_STAGE (TREX_DYN_SUMS * 32 + TREX_DYN_MSIZE + 3)  // + M staged row-major; + 3: a multiple of 16 bytes

// whether body j (lane j) lies in the subtree of the lane's body (the base's lane: every body)
TREX_FN vb dyn_in_subtree(const int* mdli, vi lane, int j) {
  return lane == 25 || (((vi(ldui(mdli, IF_ANC_MASK * 32 + j)) >> lane) & 1) != 0);
}

// Composite inertia of the lane's subtree about the point r (from p0): B = the lane's body's COM inertia (xx xy xz yy yz zz,
// world axes) | COM (from p0) | mass; C = inertia about r | first moment about r | mass, summed in ascending lane order.
TREX_FN void dyn_composite(const int* mdli, vi lane, float* rows, const vf B[10], const vf r[3], vf C[10]) {
  TREX_UNROLL for (int k = 0; k < 10; k++) { st(rows, lane + 32 * k, B[k]); C[k] = 0.0f; }
  warp_sync();
  TREX_ROLLED for (int j = 0; j < NB; j++) {
    const vb in = dyn_in_subtree(mdli, lane, j);
    vf x[10];
    TREX_UNROLL for (int k = 0; k < 10; k++) x[k] = ld(rows, vi(32 * k + j));
    const vf d0 = x[6] - r[0], d1 = x[7] - r[1], d2 = x[8] - r[2], m = x[9];
    const vf t[10] = {x[0] + m * (d1 * d1 + d2 * d2), x[1] - m * (d0 * d1), x[2] - m * (d0 * d2), x[3] + m * (d0 * d0 + d2 * d2),
                      x[4] - m * (d1 * d2), x[5] + m * (d0 * d0 + d1 * d1), m * d0, m * d1, m * d2, m};
    TREX_UNROLL for (int k = 0; k < 10; k++) C[k] = sel(in, C[k] + t[k], C[k]);
  }
  warp_sync();
}

// Force of the lane's subtree about the point r: B = the lane's body's [n (about its COM); f] | COM (from p0); F = sum of
// [n + (c - r) x f; f] in ascending lane order.
TREX_FN void dyn_force_sum(const int* mdli, vi lane, float* rows, const vf B[9], const vf r[3], vf F[6]) {
  TREX_UNROLL for (int k = 0; k < 9; k++) st(rows, lane + 32 * k, B[k]);
  TREX_UNROLL for (int k = 0; k < 6; k++) F[k] = 0.0f;
  warp_sync();
  TREX_ROLLED for (int j = 0; j < NB; j++) {
    const vb in = dyn_in_subtree(mdli, lane, j);
    vf x[9];
    TREX_UNROLL for (int k = 0; k < 9; k++) x[k] = ld(rows, vi(32 * k + j));
    const vf d0 = x[6] - r[0], d1 = x[7] - r[1], d2 = x[8] - r[2];
    const vf t[6] = {x[0] + (d1 * x[5] - d2 * x[4]), x[1] + (d2 * x[3] - d0 * x[5]), x[2] + (d0 * x[4] - d1 * x[3]), x[3], x[4], x[5]};
    TREX_UNROLL for (int k = 0; k < 6; k++) F[k] = sel(in, F[k] + t[k], F[k]);
  }
  warp_sync();
}

TREX_FN void dynamics_phase(const Uniform& P, const float* mdl, const int* mdli, const float* com, const float* envp,
                            const float* rec, float* stage, float* Mout, float* bout, float* Jout) {
  const vi lane = lane_id();
  const vb is_joint = lane < NJ;
  const vb owns = lane < TREX_DYN_NDOF;
  const vi col = seli(is_joint, lane + 6, lane - 25);  // the coordinate of u this lane owns
  EnvRegs R;
  load_env_regs(rec, lane, R);
  float Rb[9];
  quat_to_Rb(R.quat, Rb);
  vf E[9], Rw[9], xw[3], v[6];
  local_rotation(mdl, lane, R.q, E);
  forward_pass<false>(mdl, mdli, lane, R, Rb, E, Rw, xw, v);
  // joint axis a (world: the body's z axis) through the body origin r (from p0; the base's lane: r = 0), and the body's COM
  // cw (from p0): c of the COM table in world axes
  vf r[3], a[3], c[3], cw[3];
  TREX_UNROLL for (int k = 0; k < 3; k++) { r[k] = xw[k] - R.pos[k]; a[k] = Rw[6 + k]; c[k] = ldg_ro(com, lane + k * 32); }
  TREX_UNROLL for (int i = 0; i < 3; i++) cw[i] = r[i] + (Rw[i] * c[0] + Rw[3 + i] * c[1] + Rw[6 + i] * c[2]);

  // the body's mass and COM inertia in world axes, Ic = Rw^T (I - m (|c|^2 1 - c c^T)) Rw (I: about the body origin)
  vf m, Ic[6];
  if (Mout || bout) {
    const vf msc = envp ? envp_mass_scale(envp, lane) : vf(1.0f);
    m = MDL(F_MASS) * msc;
    vf I6[6];
    TREX_UNROLL for (int k = 0; k < 6; k++) I6[k] = MDL(F_I + k) * msc;
    const vf cc = c[0] * c[0] + c[1] * c[1] + c[2] * c[2];
    const vf Ib[3][3] = {{I6[0] - m * (cc - c[0] * c[0]), I6[1] + m * (c[0] * c[1]), I6[2] + m * (c[0] * c[2])},
                         {I6[1] + m * (c[0] * c[1]), I6[3] - m * (cc - c[1] * c[1]), I6[4] + m * (c[1] * c[2])},
                         {I6[2] + m * (c[0] * c[2]), I6[4] + m * (c[1] * c[2]), I6[5] - m * (cc - c[2] * c[2])}};
    vf T[3][3];
    TREX_UNROLL for (int i = 0; i < 3; i++)
      TREX_UNROLL for (int j = 0; j < 3; j++) T[i][j] = Ib[i][0] * Rw[j] + Ib[i][1] * Rw[3 + j] + Ib[i][2] * Rw[6 + j];
    int n = 0;
    TREX_UNROLL for (int i = 0; i < 3; i++)
      TREX_UNROLL for (int j = i; j < 3; j++) Ic[n++] = Rw[i] * T[0][j] + Rw[3 + i] * T[1][j] + Rw[6 + i] * T[2][j];
  }

  if (Mout) {  // composite-rigid-body algorithm
    vf C[10];
    {
      const vf B[10] = {Ic[0], Ic[1], Ic[2], Ic[3], Ic[4], Ic[5], cw[0], cw[1], cw[2], m};
      dyn_composite(mdli, lane, stage, B, r, C);
    }
    float* Ms = stage + TREX_DYN_SUMS * 32;
    TREX_UNROLL for (int i = 0; i < (TREX_DYN_MSIZE + 31) / 32; i++) {
      const vi idx = lane + 32 * i;
      st_if(Ms, seli(idx < TREX_DYN_MSIZE, idx, 0), 0.0f, idx < TREX_DYN_MSIZE);
    }
    warp_sync();
    // joint lanes: F = [I a; a x h], the force about the joint's origin that moves the subtree with a unit joint rate.
    // Row 6 + lane of M: F about p0 in the base columns, S_j . F for j the joint or one of its ancestors, 0 elsewhere.
    vf F[6];
    F[0] = C[0] * a[0] + C[1] * a[1] + C[2] * a[2];
    F[1] = C[1] * a[0] + C[3] * a[1] + C[4] * a[2];
    F[2] = C[2] * a[0] + C[4] * a[1] + C[5] * a[2];
    F[3] = a[1] * C[8] - a[2] * C[7];
    F[4] = a[2] * C[6] - a[0] * C[8];
    F[5] = a[0] * C[7] - a[1] * C[6];
    const vf Fb[6] = {F[0] + (r[1] * F[5] - r[2] * F[4]), F[1] + (r[2] * F[3] - r[0] * F[5]), F[2] + (r[0] * F[4] - r[1] * F[3]),
                      F[3], F[4], F[5]};
    const vi row = seli(is_joint, lane + 6, 0);
    TREX_UNROLL for (int q = 0; q < 6; q++) {
      st_if(Ms, row * TREX_DYN_NDOF + q, Fb[q], is_joint);
      st_if(Ms, q * TREX_DYN_NDOF + row, Fb[q], is_joint);
    }
    vi anc = lane;
    TREX_ROLLED for (int d = 0; d < MAX_DEPTH; d++) {
      // joint j = anc moves the point r with a x (r - r_j)
      const vb ok = is_joint && anc < NJ;
      vf sa[3], e3[3];
      TREX_UNROLL for (int k = 0; k < 3; k++) { sa[k] = shflv(a[k], anc); e3[k] = r[k] - shflv(r[k], anc); }
      const vf l0 = sa[1] * e3[2] - sa[2] * e3[1], l1 = sa[2] * e3[0] - sa[0] * e3[2], l2 = sa[0] * e3[1] - sa[1] * e3[0];
      const vf e = sa[0] * F[0] + sa[1] * F[1] + sa[2] * F[2] + (l0 * F[3] + l1 * F[4] + l2 * F[5]);
      const vi other = seli(ok, anc + 6, 0);
      st_if(Ms, row * TREX_DYN_NDOF + other, e, ok);
      st_if(Ms, other * TREX_DYN_NDOF + row, e, ok);
      anc = ldi(mdli, anc + IF_PARENT_LANE * 32);
    }
    // the base block: the whole tree's inertia about p0 [[I, [h]x], [[h]x^T, m 1]] (lane 25)
    const vb is_base = lane == 25;
    const vf hx[3][3] = {{0.0f, -C[8], C[7]}, {C[8], 0.0f, -C[6]}, {-C[7], C[6], 0.0f}};
    const int si[3][3] = {{0, 1, 2}, {1, 3, 4}, {2, 4, 5}};
    TREX_UNROLL for (int i = 0; i < 3; i++) {
      TREX_UNROLL for (int j = 0; j < 3; j++) {
        st_if(Ms, vi(i * TREX_DYN_NDOF + j), C[si[i][j]], is_base);
        st_if(Ms, vi(i * TREX_DYN_NDOF + 3 + j), hx[i][j], is_base);
        st_if(Ms, vi((3 + j) * TREX_DYN_NDOF + i), hx[i][j], is_base);
      }
      st_if(Ms, vi((3 + i) * TREX_DYN_NDOF + 3 + i), C[9], is_base);
    }
    warp_sync();
    TREX_UNROLL for (int i = 0; i < (TREX_DYN_MSIZE + 31) / 32; i++) {  // coalesced, in flat-index order
      const vi idx = lane + 32 * i;
      const vb in = idx < TREX_DYN_MSIZE;
      st_if(Mout, idx, ld_if(Ms, seli(in, idx, 0), in, 0.0f), in);
    }
    warp_sync();
  }

  if (bout) {  // Newton-Euler with du/dt = 0
    // Motion V = [w; v at p0] and spatial acceleration A (at p0) of every body, gravity entering as an upward acceleration
    // of the base.  The base's A is [0; -w x v] when its classical acceleration du/dt is 0; a joint adds (V x S) qd, with
    // S = [a; r x a] its motion at p0 (the axis moves with the body).
    vf s[3];
    s[0] = r[1] * a[2] - r[2] * a[1];
    s[1] = r[2] * a[0] - r[0] * a[2];
    s[2] = r[0] * a[1] - r[1] * a[0];
    vf V[6], A[6];
    TREX_UNROLL for (int k = 0; k < 3; k++) { V[k] = vbroadcast(R.om[k]); V[3 + k] = vbroadcast(R.vl[k]); A[k] = 0.0f; }
    A[3] = vbroadcast(-(R.om[1] * R.vl[2] - R.om[2] * R.vl[1]));
    A[4] = vbroadcast(-(R.om[2] * R.vl[0] - R.om[0] * R.vl[2]));
    A[5] = vbroadcast(P.g - (R.om[0] * R.vl[1] - R.om[1] * R.vl[0]));
    const vi plane = MDLI(IF_PARENT_LANE);
    const vi depth = MDLI(IF_DEPTH);
    TREX_ROLLED for (int d = 1; d <= MAX_DEPTH; d++) {
      const vb at = depth == d;
      vf pV[6], pA[6];
      TREX_UNROLL for (int k = 0; k < 6; k++) { pV[k] = shflv(V[k], plane); pA[k] = shflv(A[k], plane); }
      vf cr[6];  // (pV x S) qd
      cr[0] = (pV[1] * a[2] - pV[2] * a[1]) * R.qd;
      cr[1] = (pV[2] * a[0] - pV[0] * a[2]) * R.qd;
      cr[2] = (pV[0] * a[1] - pV[1] * a[0]) * R.qd;
      cr[3] = ((pV[1] * s[2] - pV[2] * s[1]) + (pV[4] * a[2] - pV[5] * a[1])) * R.qd;
      cr[4] = ((pV[2] * s[0] - pV[0] * s[2]) + (pV[5] * a[0] - pV[3] * a[2])) * R.qd;
      cr[5] = ((pV[0] * s[1] - pV[1] * s[0]) + (pV[3] * a[1] - pV[4] * a[0])) * R.qd;
      TREX_UNROLL for (int k = 0; k < 3; k++) {
        V[k] = sel(at, pV[k] + a[k] * R.qd, V[k]);
        V[3 + k] = sel(at, pV[3 + k] + s[k] * R.qd, V[3 + k]);
      }
      TREX_UNROLL for (int k = 0; k < 6; k++) A[k] = sel(at, pA[k] + cr[k], A[k]);
    }
    // at the COM: v_c = v + w x c, classical acceleration a_c = A_lin + alpha x c + w x v_c; f = m a_c, n = Ic alpha + w x Ic w
    const vf vc[3] = {V[3] + (V[1] * cw[2] - V[2] * cw[1]), V[4] + (V[2] * cw[0] - V[0] * cw[2]), V[5] + (V[0] * cw[1] - V[1] * cw[0])};
    const vf ac[3] = {A[3] + (A[1] * cw[2] - A[2] * cw[1]) + (V[1] * vc[2] - V[2] * vc[1]),
                      A[4] + (A[2] * cw[0] - A[0] * cw[2]) + (V[2] * vc[0] - V[0] * vc[2]),
                      A[5] + (A[0] * cw[1] - A[1] * cw[0]) + (V[0] * vc[1] - V[1] * vc[0])};
    const vf L[3] = {Ic[0] * V[0] + Ic[1] * V[1] + Ic[2] * V[2], Ic[1] * V[0] + Ic[3] * V[1] + Ic[4] * V[2],
                     Ic[2] * V[0] + Ic[4] * V[1] + Ic[5] * V[2]};
    const vf B[9] = {Ic[0] * A[0] + Ic[1] * A[1] + Ic[2] * A[2] + (V[1] * L[2] - V[2] * L[1]),
                     Ic[1] * A[0] + Ic[3] * A[1] + Ic[4] * A[2] + (V[2] * L[0] - V[0] * L[2]),
                     Ic[2] * A[0] + Ic[4] * A[1] + Ic[5] * A[2] + (V[0] * L[1] - V[1] * L[0]),
                     m * ac[0], m * ac[1], m * ac[2], cw[0], cw[1], cw[2]};
    vf F[6];
    dyn_force_sum(mdli, lane, stage, B, r, F);
    // joint lanes: a . n of their subtree about the joint's origin; base lanes 25..30: component lane - 25 of the whole
    // tree's [n about p0; f] (lane 25)
    vf out = a[0] * F[0] + a[1] * F[1] + a[2] * F[2];
    TREX_UNROLL for (int k = 0; k < 6; k++) out = sel(lane == 25 + k, shfl(F[k], 25), out);
    st_if(bout, col, out, owns);
  }

  if (Jout) {
    // lane L < 25: column 6 + L, the joint's [a x (c_k - r); a] where it moves body k; lanes 25..27: the base angular
    // coordinate e = unit L - 25, [e x c_k; e]; lanes 28..30: the base linear coordinate, [e; 0]
    vf u[3];
    const vb wcol = lane >= 25 && lane < 28, vcol = lane >= 28 && lane < 31;
    TREX_UNROLL for (int k = 0; k < 3; k++) u[k] = sel((wcol && lane == 25 + k) || (vcol && lane == 28 + k), 1.0f, 0.0f);
    TREX_ROLLED for (int k = 0; k < NB; k++) {
      vf ck[3], d[3], jr[6];
      TREX_UNROLL for (int i = 0; i < 3; i++) { ck[i] = shfl(cw[i], k); d[i] = ck[i] - r[i]; }
      const vb in = is_joint && dyn_in_subtree(mdli, lane, k);
      const vf bv[3] = {u[1] * ck[2] - u[2] * ck[1], u[2] * ck[0] - u[0] * ck[2], u[0] * ck[1] - u[1] * ck[0]};
      jr[0] = sel(in, a[1] * d[2] - a[2] * d[1], sel(wcol, bv[0], u[0]));
      jr[1] = sel(in, a[2] * d[0] - a[0] * d[2], sel(wcol, bv[1], u[1]));
      jr[2] = sel(in, a[0] * d[1] - a[1] * d[0], sel(wcol, bv[2], u[2]));
      TREX_UNROLL for (int i = 0; i < 3; i++) jr[3 + i] = sel(in, a[i], sel(wcol, u[i], 0.0f));
      float* Jk = Jout + k * (TREX_DYN_JROWS * TREX_DYN_NDOF);
      TREX_UNROLL for (int i = 0; i < 6; i++) st_if(Jk, col + i * TREX_DYN_NDOF, jr[i], owns);
    }
  }
}

}  // namespace trex
