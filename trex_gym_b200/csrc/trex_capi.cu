// trex_capi.cu -- sm_100a kernels + the C ABI declared in include/trex_b200.h.
//
// One warp per environment; see trex_core.h for the algorithm and the lane mapping.
// There is no CPU path in this library: every entry point launches CUDA kernels.
#include "lane_cuda.h"
#include "trex_core.h"
#include "trex_model.h"
#include "trex_policy.h"

#include "../../include/trex_b200.h"

#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <new>

#ifndef TREX_MIN_BLOCKS
#define TREX_MIN_BLOCKS 16        // resident warps per SM targeted by the front / tail kernels (128 registers)
#endif
#ifndef TREX_SOLVE_MIN_BLOCKS
#define TREX_SOLVE_MIN_BLOCKS 12  // ... by the 4-environments-per-warp solve kernel (168 registers)
#endif
#ifndef TREX_SOLVEC_MIN_BLOCKS
#define TREX_SOLVEC_MIN_BLOCKS 8  // ... by its contact variant (<= 255 registers: 2 warps per scheduler; 3 would cap it at 168 and spill)
#endif
#define TREX_STR2(x) #x
#define TREX_STR(x) TREX_STR2(x)

#ifndef TREX_PHASES
#define TREX_S4_TMEM_COLS 256
static_assert(S4_TM_COLS(TREX_KC) <= TREX_S4_TMEM_COLS, "tensor-memory columns of solve4");
static_assert(TREX_STATE_DIM == TREX_STATE_STRIDE, "state record size");
static_assert(TREX_AUX_DIM == TREX_AUX_STRIDE, "aux record size");
#endif
static_assert(trex::F_COUNT == 32, "float field table");
static_assert(TREX_ENV_PARAM_DIM == TREX_ENVP_DIM && TREX_ENVP_DIM == (int)trex_host::ENVP_DIM &&
              (int)trex::EP_MAX_IMPULSE == (int)trex_host::ENVP_MAX_IMPULSE && (int)trex::EP_MU == (int)trex_host::ENVP_MU &&
              (int)trex::EP_MAX_TORQUE == (int)trex_host::ENVP_MAX_TORQUE, "parameter row layout");
static_assert(TREX_EXT_BODIES == trex_topo::NB && TREX_EXTF_DIM == 6 * 32, "wrench record layout");
static_assert(sizeof(trex_push_schedule) == 16 * 4, "trex_push_schedule layout");
static_assert(TREX_BODY_STATE_DIM == TREX_BODY_DIM && TREX_BODY_STAGE == TREX_EXT_BODIES * TREX_BODY_STATE_DIM, "body state layout");
static_assert(TREX_NUM_DOFS == TREX_DYN_NDOF && TREX_NUM_DOFS == trex_topo::NDOF && TREX_JACOBIAN_ROWS == TREX_DYN_JROWS &&
              (TREX_DYN_STAGE % 4) == 0, "dynamics layout");

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, const char* detail = "") {
  snprintf(g_err, sizeof g_err, fmt, detail);
  return code;
}
#define CUDA_TRY(expr)                                                                 \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) return fail(TREX_ERR_CUDA, #expr ": %s", cudaGetErrorString(_e)); \
  } while (0)

// ------------------------------------------------------------------------------------------------
// One env step = n_sub x [trex_front_kernel ; trex_solve_kernel] ; trex_tail_kernel   (trex_core.h).
// Warp-private shared slabs; the only block-level synchronisation is the pair of barriers around the packed inward pass.
// ------------------------------------------------------------------------------------------------
// one warp per environment: dynamics front end of one physics substep (+ the whole substep when the solve is not deferred).
// PACKED (4 warps per CTA): the inward pass of the CTA's four environments is done by warp 0, four environments at a time.
// ENVP (trex_config.env_params): every environment's mass scales, friction and motor settings come from its row of envp
// (indexed like state); without it envp is unused and the instance is the one the library had before the record existed.
// EXTF (trex_config.external_forces): every environment's wrench record (extf, [6][32] per environment, indexed like state),
// the COM table com [3][32] and the push schedule enter the bias forces; without it the three are unused.
// TAU (trex_config.actuation = TREX_ACTUATION_TORQUE): the actions are joint torques, clipped to +-tau_max (ENVP: the row's
// bound) and applied as explicit joint torques; the motors have no gain and no strength.  Without it tau_max is unused.
template <int WARPS, bool PACKED, bool ENVP, bool EXTF, bool TAU>
__global__ void __launch_bounds__(32 * WARPS, TREX_MIN_BLOCKS / WARPS)
trex_front_kernel(const trex::Uniform P, const float* __restrict__ mdl, const int* __restrict__ mdli,
                  const float* __restrict__ tasks, const float* __restrict__ cand_p, const int* __restrict__ cand_lane,
                  float* __restrict__ state, float* __restrict__ work, float* __restrict__ workh, const float* __restrict__ action,
                  int* __restrict__ list, int* __restrict__ list_count, const int* __restrict__ heavy_hint, int heavy_div, int n_envs,
                  int first_round, const float* __restrict__ envp, const float* __restrict__ extf, const float* __restrict__ com,
                  const __grid_constant__ trex::PushSchedule push, float tau_max) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  trex::WarpShared* slabs = reinterpret_cast<trex::WarpShared*>(smem_raw);
  const int warp = threadIdx.x >> 5;
  static_assert(!PACKED || WARPS == 4, "the packed inward pass serves four environments");
  const int env = blockIdx.x * WARPS + warp;
  int valid_mask = 0;
  if (PACKED) {
    for (int w = 0; w < WARPS; w++) valid_mask |= (blockIdx.x * WARPS + w < n_envs) ? (1 << w) : 0;
    if (env >= n_envs) {  // keep the CTA's two barriers balanced; warp 0 always holds an environment
      __syncthreads();
      __syncthreads();
      return;
    }
  } else if (env >= n_envs) {
    return;
  }
#ifdef TREX_PHASES
  const long long t_entry = clock64();
#endif
  const int front_result = trex::front_phase<PACKED, ENVP, EXTF, TAU>(P, mdl, mdli, tasks, cand_p, cand_lane, slabs[warp], state + (size_t)env * TREX_STATE_STRIDE,
                                                  work ? work + (size_t)env * TREX_WORK_STRIDE : nullptr, action + (size_t)env * trex::NJ,
                                                  first_round != 0, slabs, warp, valid_mask,
                                                  // class 5 (more than TREX_KC contacts) always goes to its own solver unless heavy_share_div asks for the batch-dependent rule
                                                  (workh != nullptr && (heavy_div <= 0 || (long long)(*heavy_hint) * heavy_div <= (long long)n_envs)) ? workh + (size_t)env * TREX_HEAVY_STRIDE : nullptr,
                                                  ENVP ? envp + (size_t)env * TREX_ENVP_DIM : nullptr,
                                                  EXTF ? extf + (size_t)env * TREX_EXTF_DIM : nullptr, com, &push, (long long)env, tau_max);
  const int deferred = front_result & 255, n_contacts = front_result >> 8;
  // append to the list of its class of deferred environments (any order: the solver's lane groups are independent):
  // class 0 = contact-free substeps, classes 1..4 = 1 / 2 / 3-4 / 5-8 contacts, 5 = more; list c at list + c * n_envs, counters + 64 * c
  if (deferred && (threadIdx.x & 31) == 0) {
    const int which = deferred - 1;
    list[(size_t)which * n_envs + atomicAdd(list_count + 64 * which, 1)] = env;
  }
  // environments with more than TREX_KC contacts in this round, whichever solver takes them (steers the next round)
  if ((threadIdx.x & 31) == 0 && n_contacts > TREX_KC) atomicAdd(list_count + 64 * TREX_NCLASS, 1);
#ifdef TREX_PHASES
  __syncwarp();
  if ((threadIdx.x & 31) == 0) state[(size_t)env * TREX_STATE_STRIDE + 167] += (float)(clock64() - t_entry);  // warp lifetime
#endif
}

// one warp per FOUR deferred environments of one class, eight lanes per environment; KC = 0: the contact-free list,
// KC > 0: the lists of the contact classes CLO..CHI (rows in row space, see solve4), warps assigned class by class.
// (A second instance with KC = 2 for the environments with 1-2 contacts -- 168 registers, 12 warps per SM -- was measured:
// 70 spilled registers in the sweep, 9.3 instead of 8.1 ms per env step on the benchmark batch.  One instance serves 1-8.)
// (Round 2 also measured both instances with the coefficient rows g in a lane-private shared-memory copy instead of 100
// registers per thread -- 16 instead of 12 warps per SM contact-free, 12 instead of 8 for a 1-2-contact instance: +11 % and
// +30 % step time.  And the contact instance held to 6 / 4 warps per SM by extra shared memory: +1 % / +10 %.  These kernels
// are not bound by the number of resident warps.)
template <int WARPS, int KC, int CLO, int CHI, bool ENVP>
__global__ void __launch_bounds__(32 * WARPS, (KC ? TREX_SOLVEC_MIN_BLOCKS : TREX_SOLVE_MIN_BLOCKS) / WARPS)
trex_solve_kernel(const trex::Uniform P, float* __restrict__ state, const float* __restrict__ work,
                  const int* __restrict__ list, const int* __restrict__ list_count, int n_envs, const float* __restrict__ envp) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* scratch = reinterpret_cast<float*>(smem_raw) + (threadIdx.x >> 5) * TREX_SOLVE_SCRATCH(KC);
  const int warp = threadIdx.x >> 5;
  int first = (blockIdx.x * WARPS + warp) * 4;
  int count = *list_count;
  if (KC > 0) {
    // list / list_count point at class 0.  Warps are handed out heaviest class first (CHI, then down to CLO):
    // the longest-running warps start first instead of forming the tail of the launch.
    list += (size_t)CHI * n_envs;
    list_count += 64 * CHI;
    count = *list_count;
    for (int c = CHI; c > CLO && first >= ((count + 3) & ~3); c--) {
      first -= (count + 3) & ~3;
      list -= n_envs;
      list_count -= 64;
      count = *list_count;
    }
  }
  if (first >= count) return;
  int envs[4] = {0, 0, 0, 0}, pending = 0;
  for (int e = 0; e < 4 && first + e < count; e++) { envs[e] = list[first + e]; pending |= 1 << e; }
  trex::solve_phase<KC, false, ENVP>(P, scratch, work, state, envs, pending, tmem_t(), envp);
}

// The contact solver with its Delassus blocks and sweep responses in TENSOR MEMORY (solve4<TREX_KC, true>): persistent 4-warp
// CTAs (the four warps of a CTA reach the four 32-lane quarters of its tensor-memory columns), 256 columns per CTA, two CTAs =
// 8 warps per SM.  Warps pull tasks (four environments of one class, heaviest class first) from a counter.
template <int CLO, int CHI, bool ENVP>
__global__ void __launch_bounds__(128, 2)
trex_solve_tm_kernel(const trex::Uniform P, float* __restrict__ state, const float* __restrict__ work,
                     const int* __restrict__ list, const int* __restrict__ list_count, int* __restrict__ next_task, int n_envs,
                     const float* __restrict__ envp) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5;
  float* scratch = reinterpret_cast<float*>(smem_raw) + warp * TREX_SOLVE_SCRATCH_TM(TREX_KC);
  int tasks_of[CHI + 1], total = 0;
#pragma unroll
  for (int c = CHI; c >= CLO; c--) { tasks_of[c] = (list_count[64 * c] + 3) >> 2; total += tasks_of[c]; }
  if (total == 0) return;  // (uniform over the CTA: nobody allocates)
  __shared__ uint32_t tmem_slot;
  tmem_t tm;
  tm.base = tmem_alloc_cta<TREX_S4_TMEM_COLS>(&tmem_slot) + ((uint32_t)(warp & 3) << 21);  // lane 32 * (warp % 4) in bits 31:16
  for (;;) {
    int t = 0;
    if ((threadIdx.x & 31) == 0) t = atomicAdd(next_task, 1);
    t = __shfl_sync(0xffffffffu, t, 0);
    if (t >= total) break;
    int c = CHI;
#pragma unroll
    for (int cc = CHI; cc > CLO; cc--)
      if (c == cc && t >= tasks_of[cc]) { t -= tasks_of[cc]; c = cc - 1; }
    const int* lst = list + (size_t)c * n_envs;
    const int count = list_count[64 * c], first = 4 * t;
    int envs[4] = {0, 0, 0, 0}, pending = 0;
    for (int e = 0; e < 4 && first + e < count; e++) { envs[e] = lst[first + e]; pending |= 1 << e; }
    trex::solve_phase<TREX_KC, true, ENVP>(P, scratch, work, state, envs, pending, tm, envp);
    __syncwarp();
  }
  tmem_free_cta<TREX_S4_TMEM_COLS>(tm.base - ((uint32_t)(warp & 3) << 21));
}

// one warp per TWO environments of class 5 (more than TREX_KC contacts; sixteen lanes each, see solve2).  Persistent warps pull
// pairs of environments from a shared task counter.  Two instances run CONCURRENTLY on the same list, because the number of
// environments in flight per SM is what bounds this solver and each instance is bounded by a different memory:
//   TM = true : 4-warp CTAs, the Delassus matrices in TENSOR MEMORY (256 columns per CTA: 2 CTAs = 8 warps per SM),
//               11.4 KB of shared memory per warp
//   TM = false: 1-warp CTAs, the Delassus matrices in shared memory (29.8 KB per warp): they fill the shared memory left
template <int WARPS, bool TM, bool ENVP>
__global__ void __launch_bounds__(32 * WARPS)
trex_heavy_kernel(const trex::Uniform P, float* __restrict__ state, const float* __restrict__ work, const float* __restrict__ workh,
                  const int* __restrict__ list, const int* __restrict__ list_count, const int* __restrict__ seen, int* __restrict__ hint,
                  int* __restrict__ next_task, const float* __restrict__ envp) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5;
  float* scratch = reinterpret_cast<float*>(smem_raw) + warp * (TM ? TREX_SOLVE2_SCRATCH_TM : TREX_SOLVE2_SCRATCH);
  const int count = *list_count;
  if (blockIdx.x == 0 && threadIdx.x == 0 && hint != nullptr) *hint = *seen;  // environments with > TREX_KC contacts in this round
  tmem_t tm = {0u};
  __shared__ uint32_t tmem_slot;
  if (TM) {
    if (count == 0) return;  // (uniform over the CTA: nobody allocates)
    tm.base = tmem_alloc_cta<TREX_S2_TMEM_COLS>(&tmem_slot) + ((uint32_t)(warp & 3) << 21);  // lane 32 * (warp % 4) in bits 31:16
  }
  for (;;) {
    int i = 0;
    if ((threadIdx.x & 31) == 0) i = atomicAdd(next_task, 2);
    i = __shfl_sync(0xffffffffu, i, 0);
    if (i >= count) break;
    const bool two = i + 1 < count;
    const int envs[2] = {list[i], two ? list[i + 1] : 0};
    trex::heavy_phase<TM, ENVP>(P, scratch, tm, work, workh, state, envs, two ? 3 : 1, envp);
    __syncwarp();
  }
  if (TM) tmem_free_cta<TREX_S2_TMEM_COLS>(tm.base - ((uint32_t)(warp & 3) << 21));
}

// one warp per environment: reward / done / auto-reset / observations (mode 0), or reset only (mode 1, optional mask)
// ENVP: mass scales and friction of each environment's row apply to its reset step; ranges != nullptr: every reset first draws
// the environment's row (the randomizer; dt = physics substep in double, for the impulse bound)
// TAU: the applied joint torque the step reports is the clipped action (action, tau_max); without it both are unused.
template <int WARPS, bool ENVP, bool TAU>
__global__ void __launch_bounds__(32 * WARPS, TREX_MIN_BLOCKS / WARPS)
trex_tail_kernel(const trex::Uniform P, const float* __restrict__ mdl, const int* __restrict__ mdli,
                 const float* __restrict__ tasks, const float* __restrict__ cand_p, const int* __restrict__ cand_lane,
                 float* __restrict__ state, float* __restrict__ obs, float* __restrict__ reward, uint8_t* __restrict__ done,
                 float* __restrict__ aux, const uint8_t* __restrict__ mask, int n_envs, int mode, float* envp,
                 const float* __restrict__ ranges, double dt, const float* __restrict__ action, float tau_max) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  trex::WarpShared* slabs = reinterpret_cast<trex::WarpShared*>(smem_raw);
  const int warp = threadIdx.x >> 5;
  const int env = blockIdx.x * WARPS + warp;
  if (env >= n_envs) return;
  if (mode == 1 && mask != nullptr && mask[env] == 0) return;
  trex::tail_phase<ENVP, TAU>(P, mdl, mdli, tasks, cand_p, cand_lane, slabs[warp], state + (size_t)env * TREX_STATE_STRIDE,
                   obs ? obs + (size_t)env * (3 * trex::NJ) : nullptr, (mode == 0 && reward) ? reward + env : nullptr,
                   (mode == 0 && done) ? done + env : nullptr, (mode == 0 && aux) ? aux + (size_t)env * TREX_AUX_STRIDE : nullptr,
                   mode == 1, (long long)env, ENVP ? envp + (size_t)env * TREX_ENVP_DIM : nullptr, ranges, dt,
                   TAU && mode == 0 ? action + (size_t)env * trex::NJ : nullptr, tau_max);
}

// trex_set_env_params: rows (all, or those with mask != 0) from the caller's buffer, the impulse bound recomputed in double
__global__ void __launch_bounds__(256)
trex_set_env_params_kernel(float* __restrict__ envp, const float* __restrict__ src, const uint8_t* __restrict__ mask, double dt, int n_envs) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int env = i / TREX_ENVP_DIM, k = i % TREX_ENVP_DIM;
  if (env >= n_envs || (mask != nullptr && mask[env] == 0)) return;
  const float* row = src + (size_t)env * TREX_ENVP_DIM;
  envp[i] = k == trex::EP_MAX_IMPULSE ? (float)((double)row[trex::EP_MAX_TORQUE] * dt) : row[k];
}

// trex_set_external_forces / trex_get_external_forces: user layout [N][26][6] <-> the record [N][6][32] (lanes 26..31 zero).
// One thread per record element; to_record: all environments, or those with mask != 0.
__global__ void __launch_bounds__(256)
trex_external_forces_kernel(float* __restrict__ rec, float* __restrict__ user, const uint8_t* __restrict__ mask, int n_envs,
                            int to_record) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long env = i / TREX_EXTF_DIM;
  const int c = (int)(i % TREX_EXTF_DIM) / 32, lane = (int)(i % 32);
  if (env >= n_envs) return;
  float* u = user + (size_t)env * (TREX_EXT_BODIES * 6) + lane * 6 + c;
  if (to_record) {
    if (mask == nullptr || mask[env] != 0) rec[i] = lane < TREX_EXT_BODIES ? *u : 0.0f;
  } else if (lane < TREX_EXT_BODIES) {
    *u = rec[i];
  }
}

// trex_get_body_states: one warp per environment (trex_core.h: body_states_phase); reads the records and the model tables,
// writes only the outputs.  The warp's rows are staged in a 1,352-byte slice of static shared memory.
#define TREX_BODY_WARPS 8
__global__ void __launch_bounds__(32 * TREX_BODY_WARPS)
trex_body_states_kernel(const trex::Uniform P, const float* __restrict__ mdl, const int* __restrict__ mdli,
                        const int* __restrict__ cand_lane, const float* __restrict__ com, const float* __restrict__ state,
                        float* __restrict__ states, float* __restrict__ forces, int n_envs) {
  __shared__ __align__(16) float stage[TREX_BODY_WARPS][TREX_BODY_STAGE];
  const int warp = threadIdx.x >> 5;
  const int env = blockIdx.x * TREX_BODY_WARPS + warp;
  if (env >= n_envs) return;
  trex::body_states_phase(P, mdl, mdli, cand_lane, com, state + (size_t)env * TREX_STATE_STRIDE, stage[warp],
                          states ? states + (size_t)env * TREX_BODY_STAGE : nullptr, forces ? forces + (size_t)env * trex::NB : nullptr);
}

// trex_get_dynamics: one warp per environment (trex_core.h: dynamics_phase); reads the records, the model tables and (with
// env_params) the parameter rows, writes only the outputs.  The warp's subtree sums and its M are staged in a 5,136-byte
// slice of static shared memory.
#define TREX_DYN_WARPS 8
__global__ void __launch_bounds__(32 * TREX_DYN_WARPS)
trex_dynamics_kernel(const trex::Uniform P, const float* __restrict__ mdl, const int* __restrict__ mdli,
                     const float* __restrict__ com, const float* __restrict__ envp, const float* __restrict__ state,
                     float* __restrict__ M, float* __restrict__ b, float* __restrict__ J, int n_envs) {
  __shared__ __align__(16) float stage[TREX_DYN_WARPS][TREX_DYN_STAGE];
  const int warp = threadIdx.x >> 5;
  const int env = blockIdx.x * TREX_DYN_WARPS + warp;
  if (env >= n_envs) return;
  trex::dynamics_phase(P, mdl, mdli, com, envp ? envp + (size_t)env * TREX_ENVP_DIM : nullptr,
                       state + (size_t)env * TREX_STATE_STRIDE, stage[warp], M ? M + (size_t)env * TREX_DYN_MSIZE : nullptr,
                       b ? b + (size_t)env * TREX_DYN_NDOF : nullptr, J ? J + (size_t)env * TREX_DYN_JSIZE : nullptr);
}

// ------------------------------------------------------------------------------------------------
// synthetic actions: Philox4x32-10, key (seed, 0x5eed), counter (env lo, env hi, step lo, step hi ^ block)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}

__global__ void __launch_bounds__(256)
trex_random_action_kernel(float* __restrict__ action, const float* __restrict__ lower, const float* __restrict__ upper,
                          uint32_t seed, uint64_t step, int64_t env_offset, int n_envs) {
  // one thread per (env, block of 4 joints): 7 blocks cover 25 joints
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int env = idx / 7, blk = idx % 7;
  if (env >= n_envs) return;
  const uint64_t genv = (uint64_t)(env_offset + env);
  uint32_t c[4] = {(uint32_t)genv, (uint32_t)(genv >> 32), (uint32_t)step, (uint32_t)(step >> 32) ^ ((uint32_t)blk << 24)};
  philox4x32_10(c, seed, 0x5eedu);
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const int j = blk * 4 + k;
    if (j < trex::NJ) {
      const float u = (float)(c[k] >> 8) * (1.0f / 16777216.0f);  // [0,1)
      action[(size_t)env * trex::NJ + j] = lower[j] + (upper[j] - lower[j]) * u;
    }
  }
}

// FP32 FFMA peak microbenchmark (register resident, 8 independent chains per thread): the
// roofline denominator for this path (SURVEY.md section 8d: MEASURED_PEAKS.json has no FP32 figure).
__global__ void __launch_bounds__(256)
trex_ffma_peak_kernel(float* out, int iters, float a, float b) {
  float x0 = threadIdx.x * 1e-3f, x1 = x0 + 1.0f, x2 = x0 + 2.0f, x3 = x0 + 3.0f, x4 = x0 + 4.0f, x5 = x0 + 5.0f, x6 = x0 + 6.0f,
        x7 = x0 + 7.0f;
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int u = 0; u < 16; u++) {
      x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
      x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}

// ------------------------------------------------------------------------------------------------
// Rollout post-processing (SURVEY.md section 8f row 1; caller of the path: trex_train.py:49-61, baselines ppo2 Runner):
// generalised advantage estimation over a [T][N] rollout, one thread per environment, reverse scan over time
// (loads/stores coalesced across environments).
//   delta_t = r_t + gamma * V_{t+1} * (1 - done_{t+1}) - V_t ;  A_t = delta_t + gamma * lam * (1 - done_{t+1}) * A_{t+1}
// done_in[t] is the flag of the state the action of step t was taken in (baselines convention: mb_dones[t] =
// dones BEFORE step t; last_done closes the rollout), returns = A + V.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
trex_gae_kernel(const float* __restrict__ rew, const float* __restrict__ val, const uint8_t* __restrict__ done_in,
                const float* __restrict__ last_val, const uint8_t* __restrict__ last_done, float gamma, float lam,
                float* __restrict__ adv, float* __restrict__ ret, int T, int N) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  float next_val = last_val[e];
  float next_nonterminal = 1.0f - (float)(last_done[e] != 0);
  float a = 0.0f;
  for (int t = T - 1; t >= 0; t--) {
    const size_t i = (size_t)t * N + e;
    const float v = val[i];
    const float delta = __fadd_rn(__fadd_rn(rew[i], __fmul_rn(__fmul_rn(gamma, next_val), next_nonterminal)), -v);
    a = __fadd_rn(delta, __fmul_rn(__fmul_rn(__fmul_rn(gamma, lam), next_nonterminal), a));
    adv[i] = a;
    ret[i] = __fadd_rn(a, v);
    next_val = v;
    next_nonterminal = 1.0f - (float)(done_in[i] != 0);
  }
}

// VecNormalize-style observation normalisation (baselines VecNormalize: clip((obs - mean) / sqrt(var + eps), -clip, clip))
__global__ void __launch_bounds__(256)
trex_normalize_kernel(const float* __restrict__ x, const float* __restrict__ mean, const float* __restrict__ var, float eps,
                      float clip, float* __restrict__ out, int64_t n_rows, int dim) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_rows * dim) return;
  const int d = (int)(i % dim);
  const float z = (x[i] - mean[d]) / sqrtf(var[d] + eps);
  out[i] = fminf(fmaxf(z, -clip), clip);
}

struct DevStats {
  double steps, episodes, nan_resets, iters, contacts, overflow;
};

__global__ void __launch_bounds__(256)
trex_stats_kernel(const float* __restrict__ state, const float* __restrict__ aux, int n_envs, DevStats* out) {
  double ep = 0, nn = 0, it = 0, ct = 0, ov = 0;
  for (int env = blockIdx.x * blockDim.x + threadIdx.x; env < n_envs; env += gridDim.x * blockDim.x) {
    const float* rec = state + (size_t)env * TREX_STATE_STRIDE;
    ep += rec[trex::ST_EPISODE];
    nn += rec[trex::ST_NANRESETS];
    it += aux[(size_t)env * TREX_AUX_STRIDE + 6];
    const float cv = aux[(size_t)env * TREX_AUX_STRIDE + 7];
    const float o = floorf(cv / 1000.0f);
    ov += o;
    ct += cv - 1000.0f * o;
  }
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) {
    ep += __shfl_xor_sync(0xffffffffu, ep, m); nn += __shfl_xor_sync(0xffffffffu, nn, m);
    it += __shfl_xor_sync(0xffffffffu, it, m); ct += __shfl_xor_sync(0xffffffffu, ct, m);
    ov += __shfl_xor_sync(0xffffffffu, ov, m);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&out->episodes, ep); atomicAdd(&out->nan_resets, nn); atomicAdd(&out->iters, it);
    atomicAdd(&out->contacts, ct); atomicAdd(&out->overflow, ov);
  }
}

}  // namespace

#ifndef TREX_DEFAULT_CHUNK_PIPES
#define TREX_DEFAULT_CHUNK_PIPES 2
#endif

struct trex_handle {
  int device = 0;
  int n_envs = 0;
  int warps_per_block = 2;  // front / tail kernels; the solve kernels then use 1 (see dispatch_step)
  bool deferred_solve = true;  // substeps with <= TREX_KC contacts solved four environments per warp (solve4)
  trex_host::ModelTables T;
  trex_host::EnvConfig C;
  trex::Uniform P;
  float *d_mdl = nullptr, *d_tasks = nullptr, *d_cand_p = nullptr, *d_state = nullptr, *d_aux = nullptr, *d_work = nullptr;
  float* d_workh = nullptr;     // contact rows of the environments with more than TREX_KC contacts (class 5)
  float *d_lower = nullptr, *d_upper = nullptr;
  int *d_mdli = nullptr, *d_cand_lane = nullptr;
  // staging for the host-buffer entry points: two sets of output buffers, so the device->host copy of one step (on the
  // copy stream, behind an event) can run under the next step's host->device copy and kernels (trex_step_host_async)
  float *d_action[2] = {nullptr, nullptr}, *d_obs[2] = {nullptr, nullptr}, *d_reward[2] = {nullptr, nullptr};
  uint8_t* d_done[2] = {nullptr, nullptr};
  cudaStream_t host_main = nullptr, host_copy = nullptr, host_in = nullptr;
  cudaEvent_t ev_step_done[2] = {nullptr, nullptr}, ev_copy_done[2] = {nullptr, nullptr}, ev_in_done[2] = {nullptr, nullptr};
  int host_slot = 0;
  DevStats* d_stats = nullptr;
  // Environments are independent, so the batch is stepped as `n_pipes` groups, each with its own chain
  // front -> solves -> front -> ... -> tail on its own stream.  The groups' kernels overlap freely: while one group's
  // solvers (latency bound, few warps per SM) drain, another group's front kernel (issue bound) fills the issue slots --
  // the hardware block scheduler interleaves their CTAs.  Within a group the three solve kernels of a round also run
  // concurrently (caller-side stream + two side streams).  Fork / join by events only: no host synchronisation, and the
  // whole step stays capturable into a CUDA graph from the caller's stream.
  //
  // L2-resident work records (trex_config.chunk_envs): every group walks its share of the batch CHUNK by chunk -- all
  // substeps of a chunk (front -> solves -> ... -> tail) before the next chunk starts -- and all chunks of a group use the
  // same work-record slots.  The records written by the front kernel (M^-1, row scalars, contact rows: 4.6 .. 11.4 KB per
  // environment and substep) are then read back by the solvers out of the 126 MB L2 and overwritten in place by the next
  // substep / chunk: they never travel to HBM, and the state record of an environment crosses HBM once per env step
  // instead of once per substep.  Footprint in flight: groups x chunk x ~6 KB.
  static constexpr int MAX_PIPES = 8;
  int chunk = 0;                // environments per chunk (multiple of 4); 0: one chunk per group (records in HBM)
  int n_chunks = 0;             // chunk c = environments [c * chunk, ...) goes to group c % n_pipes
  struct Pipe {
    int first = 0, count = 0;     // environments [first, first + count) (unchunked: the group's whole share)
    size_t work_slot = 0;         // first work-record slot of this group (chunked: p * chunk; else == first)
    cudaStream_t main = nullptr;  // pipe 0 runs on the caller's stream instead
    cudaStream_t side = nullptr, side2 = nullptr, side3 = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_join2 = nullptr, ev_join3 = nullptr, ev_done = nullptr;
    int* d_list = nullptr;        // [TREX_NCLASS][count] environments whose solve was deferred in the current substep round, by class
    int* d_list_count = nullptr;  // [TREX_NCLASS + 4][64] one counter per class and substep round, + heavy seen, solve2 task counters, hint, solve4-TM task counters
  } pipe[MAX_PIPES];
  int n_pipes = 0;              // 0 until trex_create decides (config / default)
  cudaEvent_t ev_start = nullptr, ev_stagger = nullptr;
  bool concurrent_solves = true;  // the contact-free solve kernel on a second side stream, under the contact solver
  int heavy_div = 0;            // > 0: class 5 goes to trex_heavy_kernel only while at most n_envs / heavy_div environments are in it (0: always)
  int heavy_grid = 148 * 7;     // CTAs of trex_heavy_kernel<1, false> alone (one warp each): every SM full
  int heavy_grid_tm = 148 * 2;  // CTAs of trex_heavy_kernel<4, true> (tensor-memory instance: 256 of the 512 columns each)
  int heavy_grid_mixed = 148 * 4;  // CTAs of the shared-memory instance next to the tensor-memory one
  bool solve_tm = true;         // contact solver (1-8 contacts) with its Delassus blocks / sweep responses in tensor memory (trex_config.contact_memory)
  int solve_tm_grid = 148 * 2;
  int heavy_mode = 0;           // 0: both instances concurrently; 1: shared memory only; 2: tensor memory only (TREX_HEAVY_MODE, measurement aid)
  int64_t launches = 0;
  int64_t env_steps = 0;
  // per-environment dynamics parameters (trex_config.env_params = 1): d_envp [n_envs][TREX_ENVP_DIM]; the randomizer's ranges
  // d_envp_ranges (lo [32] | hi [32]) are used while ranges_on
  bool envp_on = false, ranges_on = false;
  float *d_envp = nullptr, *d_envp_ranges = nullptr;
  double dt = 0.0;              // physics substep in double (the motor impulse bound = torque * dt)
  // external wrenches (trex_config.external_forces = 1): d_extf [n_envs][6][32] and the push schedule passed to every front
  // kernel launch (push.on = 0: off); the COM table d_com [3][32] (every handle: trex_get_body_states and
  // trex_get_dynamics read it too)
  bool extf_on = false;
  float *d_extf = nullptr, *d_com = nullptr;
  trex::PushSchedule push = {};
  // joint torque control (trex_config.actuation = TREX_ACTUATION_TORQUE): the model's torque bound (the action limits +-tau_max,
  // passed to the TAU kernel instances) and the action limits of trex_fill_random_actions (d_act_lo / d_act_hi, 25 floats each:
  // the joint limits in position mode, +-tau_max in torque mode)
  bool tau_on = false;
  float tau_max = 0.0f;
  float *d_act_lo = nullptr, *d_act_hi = nullptr;
  // the impulse bound an env-param row derives from its torque: dt in position mode, 0 in torque mode (the motors have no
  // strength there, so the shared solver instances read a zero bound from the row)
  double imp_dt() const { return tau_on ? 0.0 : dt; }
};

namespace {

template <class K>
int configure_kernel(K kernel, size_t smem) {
  CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  return TREX_OK;
}

// mode 0: one env step (n_sub front/solve rounds + tail); mode 1: reset (tail only).
// WF: warps per CTA of the front / tail kernels (one environment per warp; 2 gives 16 resident warps per SM),
// WS: warps per CTA of the solve kernels (four environments per warp; 1 with the default WF = 2: finest scheduling grain).
// host buffers of a group-staged step (trex_step_host): every group's action rows are copied in on the group's own stream right
// before its kernels and its observation / reward / done rows copied out right behind its tail kernel; the second group
// starts behind the first group's first dynamics kernel, so it also ends later and the first group's copy out runs under its
// last solve (measured without the stagger: the groups finish together and nothing overlaps)
struct HostIO {
  const float* action;
  float* obs;
  float* reward;
  uint8_t* done;
};

template <int WF, int WS, bool ENVP, bool EXTF, bool TAU>
int launch_step(trex_handle* h, const float* action, float* obs, float* reward, uint8_t* done, const uint8_t* mask,
                int mode, cudaStream_t st, const HostIO* io = nullptr) {
  static const size_t extra_c = getenv("TREX_SOLVEC_EXTRA_SMEM") ? (size_t)atoi(getenv("TREX_SOLVEC_EXTRA_SMEM")) : 0;  // measurement aid: fewer resident warps
  static const size_t extra_s = getenv("TREX_SOLVE_EXTRA_SMEM") ? (size_t)atoi(getenv("TREX_SOLVE_EXTRA_SMEM")) : 0;
  const size_t smem_f = sizeof(trex::WarpShared) * WF, smem_s = sizeof(float) * TREX_SOLVE_SCRATCH(0) * WS + extra_s,
               smem_c = sizeof(float) * TREX_SOLVE_SCRATCH(TREX_KC) * WS + extra_c, smem_h = sizeof(float) * TREX_SOLVE2_SCRATCH, smem_ht = sizeof(float) * TREX_SOLVE2_SCRATCH_TM * 4,
               smem_ct = sizeof(float) * TREX_SOLVE_SCRATCH_TM(TREX_KC) * 4;
  // per template instance and device; handles may be created and stepped from different host threads
  static bool configured[16] = {false};
  static std::mutex configure_lock;
  std::lock_guard<std::mutex> guard(configure_lock);
  if (!configured[h->device & 15]) {
    int rc;
    if ((rc = configure_kernel(trex_front_kernel<WF, WF == 4, ENVP, EXTF, TAU>, smem_f)) != TREX_OK) return rc;
    if ((rc = configure_kernel(trex_solve_kernel<WS, 0, 0, 0, ENVP>, smem_s)) != TREX_OK) return rc;
    if ((rc = configure_kernel(trex_solve_kernel<WS, TREX_KC, 1, TREX_CLASS_HEAVY - 1, ENVP>, smem_c)) != TREX_OK) return rc;
    if ((rc = configure_kernel(trex_solve_tm_kernel<1, TREX_CLASS_HEAVY - 1, ENVP>, smem_ct)) != TREX_OK) return rc;
    if ((rc = configure_kernel(trex_heavy_kernel<1, false, ENVP>, smem_h)) != TREX_OK) return rc;
    if ((rc = configure_kernel(trex_heavy_kernel<4, true, ENVP>, smem_ht)) != TREX_OK) return rc;
    if ((rc = configure_kernel(trex_tail_kernel<WF, ENVP, TAU>, smem_f)) != TREX_OK) return rc;
    configured[h->device & 15] = true;
  }
  if (h->n_pipes > 1) CUDA_TRY(cudaEventRecord(h->ev_start, st));
  cudaStream_t sp[trex_handle::MAX_PIPES];
  for (int p = 0; p < h->n_pipes; p++) {
    sp[p] = p == 0 ? st : h->pipe[p].main;
    if (p > 0) CUDA_TRY(cudaStreamWaitEvent(sp[p], h->ev_start, 0));
  }
  const int n_rounds = mode == 0 ? h->P.n_sub : 0;
  // chunk c of the batch belongs to group c % n_pipes; the host issues the chains of the groups' k-th chunks one after
  // the other (the streams run them concurrently)
  for (int c = 0; c < h->n_chunks; c++) {
    const int p = c % h->n_pipes;
    trex_handle::Pipe& q = h->pipe[p];
    cudaStream_t s = sp[p];
    const int first = h->chunk > 0 ? c * h->chunk : q.first;
    const int count = h->chunk > 0 ? (first + h->chunk <= h->n_envs ? h->chunk : h->n_envs - first) : q.count;
    if (count <= 0) continue;
    const bool stagger = io != nullptr && h->n_chunks == 2 && h->n_pipes == 2;
    if (io) CUDA_TRY(cudaMemcpyAsync(const_cast<float*>(action) + (size_t)first * trex::NJ, io->action + (size_t)first * trex::NJ,
                                     (size_t)count * trex::NJ * sizeof(float), cudaMemcpyHostToDevice, s));
    if (stagger && c == 1) CUDA_TRY(cudaStreamWaitEvent(s, h->ev_stagger, 0));
    trex::Uniform Pc = h->P;
    Pc.env_offset = h->P.env_offset + first;  // the reset sampler is keyed by the global environment id
    if (mode == 0 && h->d_work) {
      CUDA_TRY(cudaMemsetAsync(q.d_list_count, 0, 64 * (TREX_NCLASS + 2) * sizeof(int), s));  // class counters, heavy seen, solve2 task counters (not the hint behind them)
      if (h->solve_tm) CUDA_TRY(cudaMemsetAsync(q.d_list_count + 64 * (TREX_NCLASS + 3), 0, 64 * sizeof(int), s));  // task counters of the tensor-memory contact solver
    }
    const size_t e0 = (size_t)first;
    const int grid1 = (count + WF - 1) / WF;            // one warp per environment
    const int grid4 = (count + 4 * WS - 1) / (4 * WS);  // one warp per four environments
    float* state = h->d_state + e0 * TREX_STATE_STRIDE;
    float* work = h->d_work ? h->d_work + q.work_slot * TREX_WORK_STRIDE : nullptr;
    float* workh = h->d_workh ? h->d_workh + q.work_slot * TREX_HEAVY_STRIDE : nullptr;
    float* envp = ENVP ? h->d_envp + e0 * TREX_ENVP_DIM : nullptr;  // rows indexed like state
    const float* extf = EXTF ? h->d_extf + e0 * TREX_EXTF_DIM : nullptr;  // wrench records indexed like state
    for (int r = 0; r < n_rounds; r++) {
      trex_front_kernel<WF, WF == 4, ENVP, EXTF, TAU><<<grid1, 32 * WF, smem_f, s>>>(Pc, h->d_mdl, h->d_mdli, h->d_tasks, h->d_cand_p, h->d_cand_lane,
                                                          state, work, workh, action + e0 * trex::NJ, q.d_list, q.d_list_count + r,
                                                          q.d_list_count + 64 * (TREX_NCLASS + 2), h->heavy_div, count, r == 0, envp,
                                                          extf, h->d_com, h->push, h->tau_max);
      CUDA_TRY(cudaGetLastError());
      h->launches++;
      if (stagger && c == 0 && r == 0) CUDA_TRY(cudaEventRecord(h->ev_stagger, s));
      if (!h->d_work) continue;
      // The three solve kernels of a round work on disjoint lists of environments.  The two latency-bound ones go first:
      // the contact solver on the group's stream, the many-contact solver on a side stream; the contact-free solver
      // (issue bound) runs on a second side stream and fills the issue slots they leave.
      const bool contacts = h->P.defer_contacts && h->P.contacts_on;
      const bool heavy = h->P.defer_contacts > 1 && h->P.contacts_on && workh != nullptr;
      const bool split = contacts && h->concurrent_solves && q.side2 != nullptr;
      if (heavy || split) CUDA_TRY(cudaEventRecord(q.ev_fork, s));
      // launch order: the many-contact solver first (few environments, the longest latency: its CTAs must not queue behind the
      // persistent contact solver, whose two CTAs per SM take the whole register file), then the contact solver, then the
      // contact-free one (measured: 7.47 vs 7.49-7.59 ms per step with the contact solver first)
      if (heavy) {  // class 5: more than TREX_KC contacts, two environments per warp; two instances share the task counter
        int* next_task = q.d_list_count + 64 * (TREX_NCLASS + 1) + r;
        const int* cnt = q.d_list_count + 64 * TREX_CLASS_HEAVY + r;
        const int* lst = q.d_list + (size_t)TREX_CLASS_HEAVY * count;
        int* hint = q.d_list_count + 64 * (TREX_NCLASS + 2);
        CUDA_TRY(cudaStreamWaitEvent(q.side, q.ev_fork, 0));
        if (h->heavy_mode != 1) {  // the tensor-memory instance first: its CTAs take their two slots per SM ...
          trex_heavy_kernel<4, true, ENVP><<<h->heavy_grid_tm, 128, smem_ht, q.side>>>(Pc, state, work, workh, lst, cnt, q.d_list_count + 64 * TREX_NCLASS + r, hint, next_task, envp);
          CUDA_TRY(cudaGetLastError());
          h->launches++;
        }
        if (h->heavy_mode != 2) {  // ... and the shared-memory instance fills what is left of the shared memory
          cudaStream_t sh = h->heavy_mode == 0 ? q.side3 : q.side;
          if (h->heavy_mode == 0) CUDA_TRY(cudaStreamWaitEvent(q.side3, q.ev_fork, 0));
          trex_heavy_kernel<1, false, ENVP><<<h->heavy_mode == 0 ? h->heavy_grid_mixed : h->heavy_grid, 32, smem_h, sh>>>(
              Pc, state, work, workh, lst, cnt, q.d_list_count + 64 * TREX_NCLASS + r, h->heavy_mode == 0 ? nullptr : hint, next_task, envp);
          CUDA_TRY(cudaGetLastError());
          h->launches++;
          if (h->heavy_mode == 0) {
            CUDA_TRY(cudaEventRecord(q.ev_join3, q.side3));
            CUDA_TRY(cudaStreamWaitEvent(q.side, q.ev_join3, 0));
          }
        }
        CUDA_TRY(cudaEventRecord(q.ev_join, q.side));
      }
      if (contacts && h->solve_tm) {
        trex_solve_tm_kernel<1, TREX_CLASS_HEAVY - 1, ENVP><<<h->solve_tm_grid, 128, smem_ct, s>>>(Pc, state, work, q.d_list, q.d_list_count + r,
                                                                                         q.d_list_count + 64 * (TREX_NCLASS + 3) + r, count, envp);
        CUDA_TRY(cudaGetLastError());
        h->launches++;
      } else if (contacts) {
        trex_solve_kernel<WS, TREX_KC, 1, TREX_CLASS_HEAVY - 1, ENVP><<<grid4 + 4, 32 * WS, smem_c, s>>>(Pc, state, work, q.d_list, q.d_list_count + r, count, envp);
        CUDA_TRY(cudaGetLastError());
        h->launches++;
      }
      cudaStream_t s0 = split ? q.side2 : s;
      if (split) CUDA_TRY(cudaStreamWaitEvent(q.side2, q.ev_fork, 0));
      trex_solve_kernel<WS, 0, 0, 0, ENVP><<<grid4, 32 * WS, smem_s, s0>>>(Pc, state, work, q.d_list, q.d_list_count + r, count, envp);
      CUDA_TRY(cudaGetLastError());
      h->launches++;
      if (split) {
        CUDA_TRY(cudaEventRecord(q.ev_join2, q.side2));
        CUDA_TRY(cudaStreamWaitEvent(s, q.ev_join2, 0));
      }
      if (heavy) CUDA_TRY(cudaStreamWaitEvent(s, q.ev_join, 0));
    }
    trex_tail_kernel<WF, ENVP, TAU><<<grid1, 32 * WF, smem_f, s>>>(Pc, h->d_mdl, h->d_mdli, h->d_tasks, h->d_cand_p, h->d_cand_lane,
                                                        h->d_state + e0 * TREX_STATE_STRIDE, obs ? obs + e0 * 3 * trex::NJ : nullptr,
                                                        reward ? reward + e0 : nullptr, done ? done + e0 : nullptr,
                                                        h->d_aux + e0 * TREX_AUX_STRIDE, mask ? mask + e0 : nullptr, count, mode, envp,
                                                        ENVP && h->ranges_on ? h->d_envp_ranges : nullptr, h->imp_dt(),
                                                        action ? action + e0 * trex::NJ : nullptr, h->tau_max);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    if (io) {
      if (io->obs) CUDA_TRY(cudaMemcpyAsync(io->obs + e0 * 3 * trex::NJ, obs + e0 * 3 * trex::NJ, (size_t)count * 3 * trex::NJ * sizeof(float), cudaMemcpyDeviceToHost, s));
      if (io->reward) CUDA_TRY(cudaMemcpyAsync(io->reward + e0, reward + e0, (size_t)count * sizeof(float), cudaMemcpyDeviceToHost, s));
      if (io->done) CUDA_TRY(cudaMemcpyAsync(io->done + e0, done + e0, (size_t)count, cudaMemcpyDeviceToHost, s));
    }
  }
  for (int p = 1; p < h->n_pipes; p++) {
    CUDA_TRY(cudaEventRecord(h->pipe[p].ev_done, sp[p]));
    CUDA_TRY(cudaStreamWaitEvent(st, h->pipe[p].ev_done, 0));
  }
  return TREX_OK;
}

// warps per CTA (1, 2, 4) x ENVP x EXTF x TAU: 24 instances of the step
template <bool TAU>
int dispatch_actuation(trex_handle* h, const float* action, float* obs, float* reward, uint8_t* done, const uint8_t* mask,
                       int mode, cudaStream_t st, const HostIO* io) {
  switch (h->warps_per_block * 4 + (h->envp_on ? 1 : 0) + (h->extf_on ? 2 : 0)) {
    case 4: return launch_step<1, 2, false, false, TAU>(h, action, obs, reward, done, mask, mode, st, io);
    case 8: return launch_step<2, 1, false, false, TAU>(h, action, obs, reward, done, mask, mode, st, io);
    case 16: return launch_step<4, 4, false, false, TAU>(h, action, obs, reward, done, mask, mode, st, io);
    case 5: return launch_step<1, 2, true, false, TAU>(h, action, obs, reward, done, mask, mode, st, io);
    case 9: return launch_step<2, 1, true, false, TAU>(h, action, obs, reward, done, mask, mode, st, io);
    case 17: return launch_step<4, 4, true, false, TAU>(h, action, obs, reward, done, mask, mode, st, io);
    case 6: return launch_step<1, 2, false, true, TAU>(h, action, obs, reward, done, mask, mode, st, io);
    case 10: return launch_step<2, 1, false, true, TAU>(h, action, obs, reward, done, mask, mode, st, io);
    case 18: return launch_step<4, 4, false, true, TAU>(h, action, obs, reward, done, mask, mode, st, io);
    case 7: return launch_step<1, 2, true, true, TAU>(h, action, obs, reward, done, mask, mode, st, io);
    case 11: return launch_step<2, 1, true, true, TAU>(h, action, obs, reward, done, mask, mode, st, io);
    case 19: return launch_step<4, 4, true, true, TAU>(h, action, obs, reward, done, mask, mode, st, io);
    default: return fail(TREX_ERR_INVALID, "warps_per_block must be 1, 2 or 4%s");
  }
}

int dispatch_step(trex_handle* h, const float* action, float* obs, float* reward, uint8_t* done, const uint8_t* mask,
                  int mode, cudaStream_t st, const HostIO* io = nullptr) {
  return h->tau_on ? dispatch_actuation<true>(h, action, obs, reward, done, mask, mode, st, io)
                   : dispatch_actuation<false>(h, action, obs, reward, done, mask, mode, st, io);
}

template <class Tp>
int upload(Tp** dst, const std::vector<Tp>& src) {
  CUDA_TRY(cudaMalloc((void**)dst, src.size() * sizeof(Tp)));
  CUDA_TRY(cudaMemcpy(*dst, src.data(), src.size() * sizeof(Tp), cudaMemcpyHostToDevice));
  return TREX_OK;
}

}  // namespace

extern "C" {

const char* trex_last_error(void) { return g_err; }
const char* trex_version(void) { return "trex_b200 0.1 (sm_100a, warp-per-environment, KMAX=" TREX_STR(TREX_KMAX) ")"; }

int trex_create(const void* model_blob, size_t bytes, int32_t n_envs, int32_t device, const trex_config* cfg,
                trex_handle** out) {
  if (!out) return fail(TREX_ERR_INVALID, "out is NULL%s");
  *out = nullptr;
  if (!model_blob || n_envs <= 0) return fail(TREX_ERR_INVALID, "model_blob is NULL or n_envs <= 0%s");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(TREX_ERR_CUDA, "no CUDA device available (%s); libtrex_b200 has no CPU path", cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(TREX_ERR_INVALID, "device index out of range%s");
  CUDA_TRY(cudaSetDevice(device));
  trex_handle* h = new (std::nothrow) trex_handle();
  if (!h) return fail(TREX_ERR_INVALID, "out of host memory%s");
  h->device = device;
  h->n_envs = n_envs;
  if (!trex_host::build_tables(model_blob, bytes, h->T, trex::F_COUNT, trex::IF_COUNT)) {
    int rc = fail(TREX_ERR_MODEL, "model blob rejected: %s", h->T.err.c_str());
    delete h;
    return rc;
  }
  if (cfg) {
    h->C.num_substeps = cfg->num_substeps > 0 ? (cfg->num_substeps > 64 ? 64 : cfg->num_substeps) : 5;
    h->C.distance_weight = cfg->distance_weight; h->C.energy_weight = cfg->energy_weight; h->C.drift_weight = cfg->drift_weight;
    h->C.max_episode_steps = cfg->max_episode_steps; h->C.enable_contacts = cfg->enable_contacts;
    h->C.reset_mode = cfg->reset_mode; h->C.seed = cfg->seed;
    h->C.env_offset = (long long)cfg->env_offset;
    if (cfg->warps_per_block != 0 && cfg->warps_per_block != 1 && cfg->warps_per_block != 2 && cfg->warps_per_block != 4) {
      delete h;
      return fail(TREX_ERR_INVALID, "trex_config.warps_per_block must be 0 (default), 1, 2 or 4%s");
    }
    if (cfg->warps_per_block) h->warps_per_block = cfg->warps_per_block;
    if (cfg->solver_placement < TREX_SOLVE_DEFAULT || cfg->solver_placement > TREX_SOLVE_NO_HEAVY) {
      delete h;
      return fail(TREX_ERR_INVALID, "trex_config.solver_placement must be one of TREX_SOLVE_*%s");
    }
    h->deferred_solve = cfg->solver_placement != TREX_SOLVE_FRONT;
    h->C.defer_contacts = cfg->solver_placement == TREX_SOLVE_DEFAULT ? 2 : (cfg->solver_placement == TREX_SOLVE_NO_HEAVY ? 1 : 0);
    if (cfg->heavy_share_div < 0) {
      delete h;
      return fail(TREX_ERR_INVALID, "trex_config.heavy_share_div must be >= 0%s");
    }
    h->heavy_div = cfg->heavy_share_div;
    if (cfg->pipelines < 0 || cfg->pipelines > trex_handle::MAX_PIPES) {
      delete h;
      return fail(TREX_ERR_INVALID, "trex_config.pipelines must be 0 (default) .. 8%s");
    }
    h->n_pipes = cfg->pipelines;
    if (cfg->chunk_envs < -1 || (cfg->chunk_envs > 0 && (cfg->chunk_envs & 3))) {
      delete h;
      return fail(TREX_ERR_INVALID, "trex_config.chunk_envs must be -1 (off), 0 (default) or a positive multiple of 4%s");
    }
    h->chunk = cfg->chunk_envs;
    if (cfg->contact_memory < TREX_CONTACT_TENSOR || cfg->contact_memory > TREX_CONTACT_SHARED) {
      delete h;
      return fail(TREX_ERR_INVALID, "trex_config.contact_memory must be one of TREX_CONTACT_*%s");
    }
    h->solve_tm = cfg->contact_memory == TREX_CONTACT_TENSOR;
    if (cfg->heavy_memory < TREX_HEAVY_BOTH || cfg->heavy_memory > TREX_HEAVY_TENSOR) {
      delete h;
      return fail(TREX_ERR_INVALID, "trex_config.heavy_memory must be one of TREX_HEAVY_*%s");
    }
    h->heavy_mode = cfg->heavy_memory;
    if (cfg->env_params != 0 && cfg->env_params != 1) {
      delete h;
      return fail(TREX_ERR_INVALID, "trex_config.env_params must be 0 or 1%s");
    }
    h->envp_on = cfg->env_params == 1;
    if (cfg->external_forces != 0 && cfg->external_forces != 1) {
      delete h;
      return fail(TREX_ERR_INVALID, "trex_config.external_forces must be 0 or 1%s");
    }
    h->extf_on = cfg->external_forces == 1;
    if (cfg->actuation != TREX_ACTUATION_POSITION && cfg->actuation != TREX_ACTUATION_TORQUE) {
      delete h;
      return fail(TREX_ERR_INVALID, "trex_config.actuation must be TREX_ACTUATION_POSITION or TREX_ACTUATION_TORQUE%s");
    }
    h->tau_on = cfg->actuation == TREX_ACTUATION_TORQUE;
    for (int i = 0; i < 4; i++)
      if (cfg->reserved[i] != 0) {
        delete h;
        return fail(TREX_ERR_INVALID, "trex_config.reserved must be zero%s");
      }
  }
  if ((int)h->T.params[trex_host::P_MAX_CONTACTS] != TREX_KMAX) {
    int rc_ = fail(TREX_ERR_MODEL, "model blob max_contacts differs from the compiled contact capacity (TREX_KMAX)%s");
    delete h;
    return rc_;
  }
  if (const char* e = getenv("TREX_CHUNK")) { const int v = atoi(e); if (v == -1 || (v > 0 && !(v & 3))) h->chunk = v; }  // measurement aids
  if (const char* e = getenv("TREX_PIPES")) { const int v = atoi(e); if (v >= 1 && v <= trex_handle::MAX_PIPES) h->n_pipes = v; }
  // default: off.  Measured on the benchmark batch (65,536 environments, one B200): chunks of 8,192 on 2 streams cost 6 % of
  // step time (8.37 vs 7.89 ms), 4,096 on 4 streams 8 % -- the small launches pay their tails and launch gaps, and HBM is at 7 %
  // of its bandwidth without them -- while the DRAM traffic per env step falls from 3.5 GB to the figure in DESIGN.md.
  if (h->chunk > 0 && h->chunk >= n_envs) h->chunk = -1;
  if (h->chunk < 0) h->chunk = 0;
  if (h->n_pipes <= 0) h->n_pipes = h->chunk > 0 ? TREX_DEFAULT_CHUNK_PIPES : (n_envs >= 8192 ? 2 : 1);  // small batches: one group fills the machine no better split
  if (h->n_pipes > n_envs) h->n_pipes = 1;
  if (h->chunk > 0) {
    h->n_chunks = (n_envs + h->chunk - 1) / h->chunk;
    if (h->n_pipes > h->n_chunks) h->n_pipes = h->n_chunks;
  }
  trex_host::fill_uniform(h->T, h->C, h->P);
  h->dt = trex_host::substep_dt(h->T, h->C.num_substeps);
  h->tau_max = (float)h->T.params[trex_host::P_MAX_TORQUE];
  if (h->tau_on) {  // the motors of every kernel that reads the uniform settings: no gain, no strength
    h->P.kp = 0.0f; h->P.kd = 0.0f; h->P.max_impulse = 0.0f;
  }
  {
    // trex_heavy_kernel strides over its list with a fixed grid: exactly the CTAs that are resident at once (a larger
    // grid would run its surplus CTAs as a second wave after the first has walked the whole list)
    int sms = 148, per_sm = 7;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    cudaFuncSetAttribute(trex_heavy_kernel<1, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(float) * TREX_SOLVE2_SCRATCH));
    cudaFuncSetAttribute(trex_heavy_kernel<1, false, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, trex_heavy_kernel<1, false, false>, 32, sizeof(float) * TREX_SOLVE2_SCRATCH) != cudaSuccess || per_sm < 1)
      per_sm = 7;
    if (sms > 0) {
      h->heavy_grid = sms * per_sm;
      const int np = h->n_pipes > 0 ? h->n_pipes : 1;  // the groups' solvers run concurrently and share the SM's tensor memory
      int tm_per_sm = (512 / TREX_S2_TMEM_COLS) / np;
      if (tm_per_sm < 1) tm_per_sm = 1;
      h->heavy_grid_tm = sms * tm_per_sm;
      // shared memory left next to the tensor-memory CTAs (4 warps x 11.4 KB + 1 KB each), in one-warp CTAs of 29.8 + 1 KB
      const int left = 227 * 1024 - (512 / TREX_S2_TMEM_COLS) * ((int)(sizeof(float) * TREX_SOLVE2_SCRATCH_TM * 4) + 1024);
      const int fit = left / ((int)(sizeof(float) * TREX_SOLVE2_SCRATCH) + 1024);
      h->heavy_grid_mixed = sms * ((fit / np) > 0 ? fit / np : 1);
    }
    if (const char* e = getenv("TREX_HEAVY_MODE")) { const int v = atoi(e); if (v >= 0 && v <= 2) h->heavy_mode = v; }
    if (const char* e = getenv("TREX_SOLVE_TM")) h->solve_tm = e[0] == '1';  // measurement aid
    if (sms > 0) h->solve_tm_grid = sms * 2;  // persistent CTAs, two per SM (255 registers); measured best also with two groups in flight
    if (const char* e = getenv("TREX_SOLVE_TM_GRID")) { const int v = atoi(e); if (v > 0) h->solve_tm_grid = v; }
  }
  int rc;
#define TRY(x) if ((rc = (x)) != TREX_OK) { trex_destroy(h); return rc; }
  TRY(upload(&h->d_mdl, h->T.mdl)); TRY(upload(&h->d_mdli, h->T.mdli)); TRY(upload(&h->d_tasks, h->T.tasks));
  TRY(upload(&h->d_cand_p, h->T.cand_p)); TRY(upload(&h->d_cand_lane, h->T.cand_lane));
  {
    std::vector<float> lo(h->T.lower_sorted, h->T.lower_sorted + trex::NJ), hi(h->T.upper_sorted, h->T.upper_sorted + trex::NJ);
    TRY(upload(&h->d_lower, lo)); TRY(upload(&h->d_upper, hi));
    float alo[trex::NJ], ahi[trex::NJ];
    trex_get_action_limits(h, alo, ahi);
    TRY(upload(&h->d_act_lo, std::vector<float>(alo, alo + trex::NJ))); TRY(upload(&h->d_act_hi, std::vector<float>(ahi, ahi + trex::NJ)));
  }
#undef TRY
#define CTRY(expr) { cudaError_t _e = (expr); if (_e != cudaSuccess) { int r_ = fail(TREX_ERR_CUDA, #expr ": %s", cudaGetErrorString(_e)); trex_destroy(h); return r_; } }
  const size_t N = (size_t)n_envs;
  CTRY(cudaMalloc((void**)&h->d_state, N * TREX_STATE_STRIDE * sizeof(float)));
  CTRY(cudaMemset(h->d_state, 0, N * TREX_STATE_STRIDE * sizeof(float)));
  // work records: one slot per environment, or (chunked) one slot per environment of the chunks in flight
  const size_t work_slots = h->chunk > 0 ? (size_t)h->n_pipes * (size_t)h->chunk : N;
  if (h->deferred_solve) CTRY(cudaMalloc((void**)&h->d_work, work_slots * TREX_WORK_STRIDE * sizeof(float)));
  const bool with_heavy = h->deferred_solve && h->C.defer_contacts > 1 && h->C.enable_contacts;
  if (with_heavy) CTRY(cudaMalloc((void**)&h->d_workh, work_slots * TREX_HEAVY_STRIDE * sizeof(float)));
  if (const char* e = getenv("TREX_SERIAL_SOLVES")) h->concurrent_solves = !(e[0] == '1');  // measurement aids
  CTRY(cudaEventCreateWithFlags(&h->ev_start, cudaEventDisableTiming));
  CTRY(cudaEventCreateWithFlags(&h->ev_stagger, cudaEventDisableTiming));
  for (int p = 0; p < h->n_pipes; p++) {
    trex_handle::Pipe& q = h->pipe[p];
    // groups of (almost) equal size, boundaries on multiples of four environments (the solvers' work unit)
    const int per = ((n_envs + h->n_pipes - 1) / h->n_pipes + 3) & ~3;
    q.first = p * per < n_envs ? p * per : n_envs;
    q.count = (q.first + per <= n_envs) ? per : n_envs - q.first;
    q.work_slot = h->chunk > 0 ? (size_t)p * (size_t)h->chunk : (size_t)q.first;
    const int list_cap = h->chunk > 0 ? h->chunk : (q.count > 0 ? q.count : 1);
    if (p > 0) CTRY(cudaStreamCreateWithFlags(&q.main, cudaStreamNonBlocking));
    if (with_heavy) {
      CTRY(cudaStreamCreateWithFlags(&q.side, cudaStreamNonBlocking));
      CTRY(cudaStreamCreateWithFlags(&q.side2, cudaStreamNonBlocking));
      CTRY(cudaStreamCreateWithFlags(&q.side3, cudaStreamNonBlocking));
      CTRY(cudaEventCreateWithFlags(&q.ev_join3, cudaEventDisableTiming));
      CTRY(cudaEventCreateWithFlags(&q.ev_fork, cudaEventDisableTiming));
      CTRY(cudaEventCreateWithFlags(&q.ev_join, cudaEventDisableTiming));
      CTRY(cudaEventCreateWithFlags(&q.ev_join2, cudaEventDisableTiming));
    }
    CTRY(cudaEventCreateWithFlags(&q.ev_done, cudaEventDisableTiming));
    CTRY(cudaMalloc((void**)&q.d_list, (size_t)TREX_NCLASS * list_cap * sizeof(int)));
    CTRY(cudaMalloc((void**)&q.d_list_count, 64 * (TREX_NCLASS + 4) * sizeof(int)));
    CTRY(cudaMemset(q.d_list_count, 0, 64 * (TREX_NCLASS + 4) * sizeof(int)));
  }
  while (h->chunk == 0 && h->n_pipes > 1 && h->pipe[h->n_pipes - 1].count <= 0) h->n_pipes--;
  if (h->chunk == 0) h->n_chunks = h->n_pipes;
  CTRY(cudaMalloc((void**)&h->d_aux, N * TREX_AUX_STRIDE * sizeof(float)));
  CTRY(cudaMemset(h->d_aux, 0, N * TREX_AUX_STRIDE * sizeof(float)));
  // (the staging buffers of the host-buffer entry points are allocated on first use: ensure_host_path)
  CTRY(cudaMalloc((void**)&h->d_stats, sizeof(DevStats)));
  if (h->envp_on) {  // every row starts as the model's own constants
    float row[TREX_ENVP_DIM];
    trex_host::default_env_params(h->T, h->C.num_substeps, row);
    if (h->tau_on) row[trex_host::ENVP_MAX_IMPULSE] = 0.0f;
    std::vector<float> rows(N * TREX_ENVP_DIM);
    for (size_t i = 0; i < rows.size(); i++) rows[i] = row[i % TREX_ENVP_DIM];
    CTRY(cudaMalloc((void**)&h->d_envp, rows.size() * sizeof(float)));
    CTRY(cudaMemcpy(h->d_envp, rows.data(), rows.size() * sizeof(float), cudaMemcpyHostToDevice));
    CTRY(cudaMalloc((void**)&h->d_envp_ranges, 2 * TREX_ENVP_DIM * sizeof(float)));
  }
  if (h->extf_on) {  // the record starts at zero
    CTRY(cudaMalloc((void**)&h->d_extf, N * TREX_EXTF_DIM * sizeof(float)));
    CTRY(cudaMemset(h->d_extf, 0, N * TREX_EXTF_DIM * sizeof(float)));
  }
  // the COM table: where an external force acts, and the point trex_get_body_states reports (every handle, 384 bytes)
  CTRY(cudaMalloc((void**)&h->d_com, h->T.com.size() * sizeof(float)));
  CTRY(cudaMemcpy(h->d_com, h->T.com.data(), h->T.com.size() * sizeof(float), cudaMemcpyHostToDevice));
#undef CTRY
  // all environments start from the reference reset (TrexBulletEnv.__init__ calls reset(), trex_env.py:92)
  rc = trex_reset(h, nullptr, nullptr, nullptr);
  if (rc != TREX_OK) { trex_destroy(h); return rc; }
  {
    cudaError_t e2 = cudaDeviceSynchronize();
    if (e2 != cudaSuccess) { int r_ = fail(TREX_ERR_CUDA, "initial reset failed: %s", cudaGetErrorString(e2)); trex_destroy(h); return r_; }
  }
  *out = h;
  return TREX_OK;
}

void trex_destroy(trex_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaFree(h->d_mdl); cudaFree(h->d_mdli); cudaFree(h->d_tasks); cudaFree(h->d_cand_p); cudaFree(h->d_cand_lane);
  cudaFree(h->d_work); cudaFree(h->d_workh);
  cudaFree(h->d_lower); cudaFree(h->d_upper); cudaFree(h->d_state); cudaFree(h->d_aux); cudaFree(h->d_stats);
  cudaFree(h->d_envp); cudaFree(h->d_envp_ranges);
  cudaFree(h->d_extf); cudaFree(h->d_com);
  cudaFree(h->d_act_lo); cudaFree(h->d_act_hi);
  for (int b = 0; b < 2; b++) {
    cudaFree(h->d_action[b]); cudaFree(h->d_obs[b]); cudaFree(h->d_reward[b]); cudaFree(h->d_done[b]);
    if (h->ev_step_done[b]) cudaEventDestroy(h->ev_step_done[b]);
    if (h->ev_copy_done[b]) cudaEventDestroy(h->ev_copy_done[b]);
    if (h->ev_in_done[b]) cudaEventDestroy(h->ev_in_done[b]);
  }
  if (h->host_main) cudaStreamDestroy(h->host_main);
  if (h->host_copy) cudaStreamDestroy(h->host_copy);
  if (h->host_in) cudaStreamDestroy(h->host_in);
  for (int p = 0; p < trex_handle::MAX_PIPES; p++) {
    trex_handle::Pipe& q = h->pipe[p];
    cudaFree(q.d_list); cudaFree(q.d_list_count);
    if (q.main) cudaStreamDestroy(q.main);
    if (q.side) cudaStreamDestroy(q.side);
    if (q.side2) cudaStreamDestroy(q.side2);
    if (q.side3) cudaStreamDestroy(q.side3);
    if (q.ev_join3) cudaEventDestroy(q.ev_join3);
    if (q.ev_fork) cudaEventDestroy(q.ev_fork);
    if (q.ev_join) cudaEventDestroy(q.ev_join);
    if (q.ev_join2) cudaEventDestroy(q.ev_join2);
    if (q.ev_done) cudaEventDestroy(q.ev_done);
  }
  if (h->ev_start) cudaEventDestroy(h->ev_start);
  if (h->ev_stagger) cudaEventDestroy(h->ev_stagger);
  delete h;
}

int trex_reset(trex_handle* h, const uint8_t* mask_dev, float* obs_dev, void* stream) {
  if (!h) return fail(TREX_ERR_INVALID, "handle is NULL%s");
  CUDA_TRY(cudaSetDevice(h->device));
  return dispatch_step(h, nullptr, obs_dev, nullptr, nullptr, mask_dev, 1, (cudaStream_t)stream);
}

int trex_step(trex_handle* h, const float* action_dev, float* obs_dev, float* reward_dev, uint8_t* done_dev, void* stream) {
  if (!h) return fail(TREX_ERR_INVALID, "handle is NULL%s");
  if (!action_dev) return fail(TREX_ERR_INVALID, "action is NULL%s");
  CUDA_TRY(cudaSetDevice(h->device));
  int rc = dispatch_step(h, action_dev, obs_dev, reward_dev, done_dev, nullptr, 0, (cudaStream_t)stream);
  if (rc == TREX_OK) h->env_steps += h->n_envs;
  return rc;
}

// staging buffers, streams and events of the host-buffer entry points (first use)
static int ensure_host_path(trex_handle* h) {
  if (h->host_main) return TREX_OK;
  const size_t N = (size_t)h->n_envs;
  for (int b = 0; b < 2; b++) {
    CUDA_TRY(cudaMalloc((void**)&h->d_action[b], N * trex::NJ * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h->d_obs[b], N * 3 * trex::NJ * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h->d_reward[b], N * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h->d_done[b], N));
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_step_done[b], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_copy_done[b], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_in_done[b], cudaEventDisableTiming));
  }
  CUDA_TRY(cudaStreamCreateWithFlags(&h->host_copy, cudaStreamNonBlocking));
  CUDA_TRY(cudaStreamCreateWithFlags(&h->host_in, cudaStreamNonBlocking));
  CUDA_TRY(cudaStreamCreateWithFlags(&h->host_main, cudaStreamNonBlocking));
  return TREX_OK;
}

int trex_step_host_async(trex_handle* h, const float* action_host, float* obs_host, float* reward_host, uint8_t* done_host) {
  if (!h) return fail(TREX_ERR_INVALID, "handle is NULL%s");
  if (!action_host) return fail(TREX_ERR_INVALID, "action is NULL%s");
  CUDA_TRY(cudaSetDevice(h->device));
  int rc = ensure_host_path(h);
  if (rc != TREX_OK) return rc;
  const size_t N = (size_t)h->n_envs;
  const int b = h->host_slot;
  h->host_slot ^= 1;
  // host->device copy on its own stream: it may run under the previous step's kernels (which read the other action buffer);
  // the kernels that read THIS buffer two calls ago are complete once ev_step_done[b] has fired
  CUDA_TRY(cudaStreamWaitEvent(h->host_in, h->ev_step_done[b], 0));
  CUDA_TRY(cudaMemcpyAsync(h->d_action[b], action_host, N * trex::NJ * sizeof(float), cudaMemcpyHostToDevice, h->host_in));
  CUDA_TRY(cudaEventRecord(h->ev_in_done[b], h->host_in));
  CUDA_TRY(cudaStreamWaitEvent(h->host_main, h->ev_in_done[b], 0));
  // the copy-out that last used this output buffer set (two calls ago) must have drained before the kernels overwrite it
  CUDA_TRY(cudaStreamWaitEvent(h->host_main, h->ev_copy_done[b], 0));
  rc = dispatch_step(h, h->d_action[b], h->d_obs[b], h->d_reward[b], h->d_done[b], nullptr, 0, h->host_main);
  if (rc != TREX_OK) return rc;
  h->env_steps += h->n_envs;
  CUDA_TRY(cudaEventRecord(h->ev_step_done[b], h->host_main));
  CUDA_TRY(cudaStreamWaitEvent(h->host_copy, h->ev_step_done[b], 0));
  if (obs_host) CUDA_TRY(cudaMemcpyAsync(obs_host, h->d_obs[b], N * 3 * trex::NJ * sizeof(float), cudaMemcpyDeviceToHost, h->host_copy));
  if (reward_host) CUDA_TRY(cudaMemcpyAsync(reward_host, h->d_reward[b], N * sizeof(float), cudaMemcpyDeviceToHost, h->host_copy));
  if (done_host) CUDA_TRY(cudaMemcpyAsync(done_host, h->d_done[b], N, cudaMemcpyDeviceToHost, h->host_copy));
  CUDA_TRY(cudaEventRecord(h->ev_copy_done[b], h->host_copy));
  // contract: on return the PREVIOUS call's outputs are in host memory (this call's follow with the next call / trex_host_wait)
  CUDA_TRY(cudaEventSynchronize(h->ev_copy_done[b ^ 1]));
  return TREX_OK;
}

int trex_host_wait(trex_handle* h) {
  if (!h) return fail(TREX_ERR_INVALID, "handle is NULL%s");
  CUDA_TRY(cudaSetDevice(h->device));
  if (h->host_main) {
    CUDA_TRY(cudaStreamSynchronize(h->host_in));
    CUDA_TRY(cudaStreamSynchronize(h->host_main));
    CUDA_TRY(cudaStreamSynchronize(h->host_copy));
  }
  return TREX_OK;
}

int trex_step_host(trex_handle* h, const float* action_host, float* obs_host, float* reward_host, uint8_t* done_host) {
  if (!h) return fail(TREX_ERR_INVALID, "handle is NULL%s");
  if (!action_host) return fail(TREX_ERR_INVALID, "action is NULL%s");
  static const bool staged_off = getenv("TREX_HOST_STAGED") && getenv("TREX_HOST_STAGED")[0] == '0';  // measurement aid
  if (h->n_pipes < 2 || staged_off) {  // one group: one copy in, the step, one copy out
    const int rc = trex_step_host_async(h, action_host, obs_host, reward_host, done_host);
    return rc != TREX_OK ? rc : trex_host_wait(h);
  }
  // group-staged (see HostIO): the copies ride on the groups' own streams
  CUDA_TRY(cudaSetDevice(h->device));
  int rc = ensure_host_path(h);
  if (rc != TREX_OK) return rc;
  rc = trex_host_wait(h);  // (a pipelined step may still be in flight)
  if (rc != TREX_OK) return rc;
  const HostIO io = {action_host, obs_host, reward_host, done_host};
  rc = dispatch_step(h, h->d_action[0], h->d_obs[0], h->d_reward[0], h->d_done[0], nullptr, 0, h->host_main, &io);
  if (rc != TREX_OK) return rc;
  h->env_steps += h->n_envs;
  CUDA_TRY(cudaStreamSynchronize(h->host_main));
  return TREX_OK;
}

int trex_reset_host(trex_handle* h, float* obs_host) {
  if (!h) return fail(TREX_ERR_INVALID, "handle is NULL%s");
  CUDA_TRY(cudaSetDevice(h->device));
  int rc = ensure_host_path(h);
  if (rc != TREX_OK) return rc;
  rc = trex_host_wait(h);
  if (rc != TREX_OK) return rc;
  rc = dispatch_step(h, nullptr, h->d_obs[0], nullptr, nullptr, nullptr, 1, h->host_main);
  if (rc != TREX_OK) return rc;
  if (obs_host) CUDA_TRY(cudaMemcpyAsync(obs_host, h->d_obs[0], (size_t)h->n_envs * 3 * trex::NJ * sizeof(float), cudaMemcpyDeviceToHost, h->host_main));
  CUDA_TRY(cudaStreamSynchronize(h->host_main));
  return TREX_OK;
}

int trex_get_state(trex_handle* h, float* state_dev, void* stream) {
  if (!h || !state_dev) return fail(TREX_ERR_INVALID, "NULL argument%s");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMemcpyAsync(state_dev, h->d_state, (size_t)h->n_envs * TREX_STATE_STRIDE * sizeof(float), cudaMemcpyDeviceToDevice,
                           (cudaStream_t)stream));
  return TREX_OK;
}

int trex_set_state(trex_handle* h, const float* state_dev, void* stream) {
  if (!h || !state_dev) return fail(TREX_ERR_INVALID, "NULL argument%s");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMemcpyAsync(h->d_state, state_dev, (size_t)h->n_envs * TREX_STATE_STRIDE * sizeof(float), cudaMemcpyDeviceToDevice,
                           (cudaStream_t)stream));
  return TREX_OK;
}

int trex_set_env_params(trex_handle* h, const float* params_dev, const uint8_t* mask_dev, void* stream) {
  if (!h || !params_dev) return fail(TREX_ERR_INVALID, "NULL argument%s");
  if (!h->envp_on) return fail(TREX_ERR_INVALID, "trex_set_env_params: the handle was created with env_params = 0%s");
  CUDA_TRY(cudaSetDevice(h->device));
  const int total = h->n_envs * TREX_ENVP_DIM;
  trex_set_env_params_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(h->d_envp, params_dev, mask_dev, h->imp_dt(), h->n_envs);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return TREX_OK;
}

int trex_get_env_params(trex_handle* h, float* params_dev, void* stream) {
  if (!h || !params_dev) return fail(TREX_ERR_INVALID, "NULL argument%s");
  if (!h->envp_on) return fail(TREX_ERR_INVALID, "trex_get_env_params: the handle was created with env_params = 0%s");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMemcpyAsync(params_dev, h->d_envp, (size_t)h->n_envs * TREX_ENVP_DIM * sizeof(float), cudaMemcpyDeviceToDevice,
                           (cudaStream_t)stream));
  return TREX_OK;
}

int trex_set_env_param_ranges(trex_handle* h, const float* lo32_host, const float* hi32_host) {
  if (!h) return fail(TREX_ERR_INVALID, "handle is NULL%s");
  if (!h->envp_on) return fail(TREX_ERR_INVALID, "trex_set_env_param_ranges: the handle was created with env_params = 0%s");
  if (!lo32_host && !hi32_host) {
    h->ranges_on = false;
    return TREX_OK;
  }
  if (!lo32_host || !hi32_host) return fail(TREX_ERR_INVALID, "trex_set_env_param_ranges: pass both ranges or neither%s");
  if (const char* why = trex_host::check_env_param_ranges(lo32_host, hi32_host)) return fail(TREX_ERR_INVALID, "trex_set_env_param_ranges: %s", why);
  CUDA_TRY(cudaSetDevice(h->device));
  float both[2 * TREX_ENVP_DIM];
  memcpy(both, lo32_host, TREX_ENVP_DIM * sizeof(float));
  memcpy(both + TREX_ENVP_DIM, hi32_host, TREX_ENVP_DIM * sizeof(float));
  // resets already enqueued (on any stream) finish with the old ranges before the new ones land
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy(h->d_envp_ranges, both, sizeof both, cudaMemcpyHostToDevice));
  h->ranges_on = true;
  return TREX_OK;
}

int trex_set_external_forces(trex_handle* h, const float* wrench_dev, const uint8_t* mask_dev, void* stream) {
  if (!h || !wrench_dev) return fail(TREX_ERR_INVALID, "NULL argument%s");
  if (!h->extf_on) return fail(TREX_ERR_INVALID, "trex_set_external_forces: the handle was created with external_forces = 0%s");
  CUDA_TRY(cudaSetDevice(h->device));
  const long long total = (long long)h->n_envs * TREX_EXTF_DIM;
  trex_external_forces_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      h->d_extf, const_cast<float*>(wrench_dev), mask_dev, h->n_envs, 1);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return TREX_OK;
}

int trex_get_external_forces(trex_handle* h, float* wrench_dev, void* stream) {
  if (!h || !wrench_dev) return fail(TREX_ERR_INVALID, "NULL argument%s");
  if (!h->extf_on) return fail(TREX_ERR_INVALID, "trex_get_external_forces: the handle was created with external_forces = 0%s");
  CUDA_TRY(cudaSetDevice(h->device));
  const long long total = (long long)h->n_envs * TREX_EXTF_DIM;
  trex_external_forces_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->d_extf, wrench_dev, nullptr,
                                                                                                   h->n_envs, 0);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return TREX_OK;
}

int trex_set_push_schedule(trex_handle* h, const trex_push_schedule* s) {
  if (!h) return fail(TREX_ERR_INVALID, "handle is NULL%s");
  if (!h->extf_on) return fail(TREX_ERR_INVALID, "trex_set_push_schedule: the handle was created with external_forces = 0%s");
  if (!s) {
    h->push.on = 0;
    return TREX_OK;
  }
  if (const char* why = trex_host::check_push_schedule(s->body, s->interval, s->duration, s->first_step, s->probability,
                                                       s->force_min, s->force_max))
    return fail(TREX_ERR_INVALID, "trex_set_push_schedule: %s", why);
  for (int i = 0; i < 9; i++)
    if (s->reserved[i] != 0) return fail(TREX_ERR_INVALID, "trex_set_push_schedule: reserved must be zero%s");
  trex::PushSchedule p = {};
  p.on = 1;
  p.lane = s->body;  // record order = lane order
  p.interval = s->interval; p.duration = s->duration; p.first_step = s->first_step;
  p.probability = s->probability; p.force_min = s->force_min; p.force_max = s->force_max;
  trex_host::push_directions(p.dir);
  h->push = p;
  return TREX_OK;
}

int trex_get_body_states(trex_handle* h, float* states_dev, float* contact_force_dev, void* stream) {
  if (!h) return fail(TREX_ERR_INVALID, "handle is NULL%s");
  if (!states_dev && !contact_force_dev) return fail(TREX_ERR_INVALID, "trex_get_body_states: both outputs are NULL%s");
  CUDA_TRY(cudaSetDevice(h->device));
  trex_body_states_kernel<<<(unsigned)((h->n_envs + TREX_BODY_WARPS - 1) / TREX_BODY_WARPS), 32 * TREX_BODY_WARPS, 0,
                            (cudaStream_t)stream>>>(h->P, h->d_mdl, h->d_mdli, h->d_cand_lane, h->d_com, h->d_state, states_dev,
                                                    contact_force_dev, h->n_envs);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return TREX_OK;
}

int trex_get_dynamics(trex_handle* h, float* mass_matrix_dev, float* bias_dev, float* jacobian_dev, void* stream) {
  if (!h) return fail(TREX_ERR_INVALID, "handle is NULL%s");
  if (!mass_matrix_dev && !bias_dev && !jacobian_dev) return fail(TREX_ERR_INVALID, "trex_get_dynamics: all outputs are NULL%s");
  CUDA_TRY(cudaSetDevice(h->device));
  trex_dynamics_kernel<<<(unsigned)((h->n_envs + TREX_DYN_WARPS - 1) / TREX_DYN_WARPS), 32 * TREX_DYN_WARPS, 0, (cudaStream_t)stream>>>(
      h->P, h->d_mdl, h->d_mdli, h->d_com, h->envp_on ? h->d_envp : nullptr, h->d_state, mass_matrix_dev, bias_dev, jacobian_dev,
      h->n_envs);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return TREX_OK;
}

int trex_get_aux(trex_handle* h, float* aux_dev, void* stream) {
  if (!h || !aux_dev) return fail(TREX_ERR_INVALID, "NULL argument%s");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMemcpyAsync(aux_dev, h->d_aux, (size_t)h->n_envs * TREX_AUX_STRIDE * sizeof(float), cudaMemcpyDeviceToDevice,
                           (cudaStream_t)stream));
  return TREX_OK;
}

int trex_get_joint_limits(trex_handle* h, float* lower25_host, float* upper25_host) {
  if (!h || !lower25_host || !upper25_host) return fail(TREX_ERR_INVALID, "NULL argument%s");
  memcpy(lower25_host, h->T.lower_sorted, sizeof(float) * trex::NJ);
  memcpy(upper25_host, h->T.upper_sorted, sizeof(float) * trex::NJ);
  return TREX_OK;
}

int trex_get_action_limits(trex_handle* h, float* lo25_host, float* hi25_host) {
  if (!h || !lo25_host || !hi25_host) return fail(TREX_ERR_INVALID, "NULL argument%s");
  if (!h->tau_on) return trex_get_joint_limits(h, lo25_host, hi25_host);
  for (int i = 0; i < trex::NJ; i++) { lo25_host[i] = -h->tau_max; hi25_host[i] = h->tau_max; }
  return TREX_OK;
}

int trex_fill_random_actions(trex_handle* h, float* action_dev, uint32_t seed, uint64_t step, int64_t env_offset, void* stream) {
  if (!h || !action_dev) return fail(TREX_ERR_INVALID, "NULL argument%s");
  CUDA_TRY(cudaSetDevice(h->device));
  const int total = h->n_envs * 7;
  trex_random_action_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(action_dev, h->d_act_lo, h->d_act_hi, seed, step,
                                                                                     env_offset, h->n_envs);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  return TREX_OK;
}

int trex_get_stats(trex_handle* h, trex_stats* out) {
  if (!h || !out) return fail(TREX_ERR_INVALID, "NULL argument%s");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMemsetAsync(h->d_stats, 0, sizeof(DevStats), 0));
  trex_stats_kernel<<<296, 256>>>(h->d_state, h->d_aux, h->n_envs, h->d_stats);
  CUDA_TRY(cudaGetLastError());
  h->launches++;
  DevStats s;
  CUDA_TRY(cudaMemcpy(&s, h->d_stats, sizeof s, cudaMemcpyDeviceToHost));
  out->env_steps = h->env_steps;
  out->episodes = (int64_t)s.episodes;
  out->nan_resets = (int64_t)s.nan_resets;
  out->mean_solver_iterations = s.iters / ((double)h->n_envs * h->P.n_sub);
  out->mean_contacts = s.contacts / (double)h->n_envs;
  out->contact_overflow = (int64_t)s.overflow;
  return TREX_OK;
}

int trex_gae(int32_t device, const float* reward_dev, const float* value_dev, const uint8_t* done_dev, const float* last_value_dev,
             const uint8_t* last_done_dev, float gamma, float lam, float* adv_dev, float* ret_dev, int32_t T, int32_t N, void* stream) {
  if (!reward_dev || !value_dev || !done_dev || !last_value_dev || !last_done_dev || !adv_dev || !ret_dev || T <= 0 || N <= 0)
    return fail(TREX_ERR_INVALID, "trex_gae: NULL buffer or empty rollout%s");
  CUDA_TRY(cudaSetDevice(device));
  trex_gae_kernel<<<(N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(reward_dev, value_dev, done_dev, last_value_dev, last_done_dev, gamma,
                                                                    lam, adv_dev, ret_dev, T, N);
  CUDA_TRY(cudaGetLastError());
  return TREX_OK;
}

int trex_normalize(int32_t device, const float* x_dev, const float* mean_dev, const float* var_dev, float eps, float clip,
                   float* out_dev, int64_t n_rows, int32_t dim, void* stream) {
  if (!x_dev || !mean_dev || !var_dev || !out_dev || n_rows <= 0 || dim <= 0) return fail(TREX_ERR_INVALID, "trex_normalize: bad argument%s");
  CUDA_TRY(cudaSetDevice(device));
  const int64_t n = n_rows * dim;
  trex_normalize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x_dev, mean_dev, var_dev, eps, clip, out_dev, n_rows, dim);
  CUDA_TRY(cudaGetLastError());
  return TREX_OK;
}

int trex_policy_param_count(void) { return trex_policy::PARAM_COUNT; }

int trex_policy_forward(int32_t device, const float* obs_dev, const float* ob_mean_dev, const float* ob_var_dev, float eps, float clip,
                        const float* params_dev, uint32_t seed, uint64_t step, int64_t env_offset, int32_t deterministic,
                        float* action_dev, float* neglogp_dev, float* value_dev, float* mean_dev, int64_t n_rows, void* stream) {
  if (!obs_dev || !params_dev || !action_dev || n_rows <= 0 || ((ob_mean_dev == nullptr) != (ob_var_dev == nullptr)))
    return fail(TREX_ERR_INVALID, "trex_policy_forward: bad argument%s");
  CUDA_TRY(cudaSetDevice(device));
  static bool configured[16] = {false};
  if (!configured[device & 15]) {
    CUDA_TRY(cudaFuncSetAttribute(trex_policy::forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)trex_policy::SMEM_BYTES));
    configured[device & 15] = true;
  }
  const unsigned grid = (unsigned)((n_rows + trex_policy::ROWS - 1) / trex_policy::ROWS);
  trex_policy::forward_kernel<<<grid, trex_policy::ROWS, trex_policy::SMEM_BYTES, (cudaStream_t)stream>>>(
      obs_dev, ob_mean_dev, ob_var_dev, eps, clip, params_dev, seed, step, env_offset, deterministic, action_dev, neglogp_dev, value_dev,
      mean_dev, n_rows);
  CUDA_TRY(cudaGetLastError());
  return TREX_OK;
}

int trex_measure_fp32_peak(int32_t device, double* tflops_out) {
  if (!tflops_out) return fail(TREX_ERR_INVALID, "NULL argument%s");
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
  float* buf = nullptr;
  CUDA_TRY(cudaMalloc((void**)&buf, (size_t)blocks * threads * sizeof(float)));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 6; rep++) {
    CUDA_TRY(cudaEventRecord(e0, 0));
    trex_ffma_peak_kernel<<<blocks, threads>>>(buf, iters, 0.999f, 0.001f);
    CUDA_TRY(cudaEventRecord(e1, 0));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0.0f;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 8 * 16 * (double)iters * blocks * threads;
    const double tf = flops / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(buf);
  *tflops_out = best;
  return TREX_OK;
}

int64_t trex_kernel_launches(const trex_handle* h) { return h ? h->launches : 0; }
int32_t trex_num_envs(const trex_handle* h) { return h ? h->n_envs : 0; }

}  // extern "C"
