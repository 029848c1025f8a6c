// emu_dyn_main.cpp -- builds libtrex_emu_dyn.so: the emulator of emu_main.cpp plus the dynamics query (trex_get_dynamics:
// trex_core.h, dynamics_phase) over records the caller passes in.  TEST INFRASTRUCTURE ONLY.
//
// The emulator is included as it is; the query runs one emulated warp per record, with a stage poisoned like the emulator's
// shared memory (all-ones: NaN), so that a read of a stage location the warp did not write shows up in the results.
#include "emu_main.cpp"

extern "C" {
// n records rec [n][TREX_STATE_STRIDE] (and their parameter rows envp [n][TREX_ENVP_DIM], or NULL: the model's masses) ->
// M [n][31][31], b [n][31], J [n][26][6][31] (any may be NULL)
void emu_dynamics(void* h, int n, const float* rec, const float* envp, float* M, float* b, float* J) {
  Emu* e = (Emu*)h;
  alignas(16) float stage[TREX_DYN_STAGE];
  for (int i = 0; i < n; i++) {
    memset(stage, 0xff, sizeof stage);
    trex::dynamics_phase(e->P, e->T.mdl.data(), e->T.mdli.data(), e->T.com.data(), envp ? envp + (size_t)i * TREX_ENVP_DIM : nullptr,
                         rec + (size_t)i * TREX_STATE_STRIDE, stage, M ? M + (size_t)i * TREX_DYN_MSIZE : nullptr,
                         b ? b + (size_t)i * TREX_DYN_NDOF : nullptr, J ? J + (size_t)i * TREX_DYN_JSIZE : nullptr);
  }
}
}
