// Version and error strings of the C ABI (include/fragnet_b200.h).
#include <cstdlib>

#include "common.cuh"

unsigned long long g_fnb_launches = 0;

extern "C" int fnb_version(void) { return FNB_ABI_VERSION; }

extern "C" uint64_t fnb_launch_count(void) { return __atomic_load_n(&g_fnb_launches, __ATOMIC_RELAXED); }

extern "C" const char *fnb_error_string(int code) {
  switch (code) {
    case 0: return "ok";
    case FNB_ERR_NULL: return "required pointer is NULL";
    case FNB_ERR_SIZE: return "invalid size (negative, zero where positive is required, or >= 2^31 for an int32 index space)";
    case FNB_ERR_MODE: return "unknown mode or unsupported width";
    case FNB_ERR_WORKSPACE: return "workspace too small";
    case FNB_ERR_ALIGN: return "pointer or stride not 16-byte aligned";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
  }
}

// Library-owned auxiliary stream + fork/join events per device (created on first use, never destroyed): the
// whole-encoder programs run the fragment-connection chain, which is independent of the bond/atom chain until the
// fragment block of the last layer, on it.  FNB_STREAMS=1 in the environment keeps everything on the caller's stream.
int fnb_aux_streams(FnbAux *out) {
  static FnbAux aux[64];
  static bool ready[64] = {};
  static const bool single = [] { const char *e = getenv("FNB_STREAMS"); return e && e[0] == '1'; }();
  if (single) return 1;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 1;
  if (!ready[dev]) {
    FnbAux a{};
    if (cudaStreamCreateWithFlags(&a.stream, cudaStreamNonBlocking) != cudaSuccess) return 1;
    if (cudaEventCreateWithFlags(&a.fork, cudaEventDisableTiming) != cudaSuccess) return 1;
    if (cudaEventCreateWithFlags(&a.join, cudaEventDisableTiming) != cudaSuccess) return 1;
    if (cudaStreamCreateWithFlags(&a.wstream, cudaStreamNonBlocking) != cudaSuccess) return 1;
    if (cudaStreamCreateWithFlags(&a.astream, cudaStreamNonBlocking) != cudaSuccess) return 1;
    if (cudaStreamCreateWithFlags(&a.estream, cudaStreamNonBlocking) != cudaSuccess) return 1;
    if (cudaStreamCreateWithFlags(&a.hstream, cudaStreamNonBlocking) != cudaSuccess) return 1;
    if (cudaEventCreateWithFlags(&a.h_done, cudaEventDisableTiming) != cudaSuccess) return 1;
    if (cudaStreamCreateWithFlags(&a.pstream, cudaStreamNonBlocking) != cudaSuccess) return 1;
    if (cudaStreamCreateWithFlags(&a.wstream2, cudaStreamNonBlocking) != cudaSuccess) return 1;
    for (cudaEvent_t *e : {&a.p_fwd, &a.p_done, &a.step_begin})
      if (cudaEventCreateWithFlags(e, cudaEventDisableTiming) != cudaSuccess) return 1;
    cudaEvent_t *evs[16] = {&a.ready[0], &a.ready[1], &a.done[0], &a.done[1], &a.done2[0], &a.done2[1], &a.wjoin,
                            &a.a_fork, &a.a_dz, &a.a_table, &a.a_join, &a.plan_fwd, &a.e_ready, &a.e_done[0],
                            &a.e_done[1], &a.e_join};
    for (cudaEvent_t *e : evs)
      if (cudaEventCreateWithFlags(e, cudaEventDisableTiming) != cudaSuccess) return 1;
    aux[dev] = a;
    ready[dev] = true;
  }
  *out = aux[dev];
  return 0;
}

bool fnb_pdl_enabled() {
  static const bool on = [] { const char *e = getenv("FNB_PDL"); return !(e && e[0] == '0'); }();
  return on;
}
