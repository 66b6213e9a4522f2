// Internal: the batch object behind the opaque ox_batch handle, shared by ox_batch.cu and ox_env.cu.
#pragma once
#include <cuda_runtime.h>

#include <cstdlib>
#include <map>
#include <string>

#include "ox_internal.h"
#include "ox_model.h"
#include "ox_arena.h"
#include "ox_spec.cuh"

struct ox_batch {
  const ox_model* model = nullptr;
  ox_batch_config cfg{};
  int nenv = 0, stride = 0, block = 32, grid = 0, lanes = 32;
  bool f64 = false;
  cudaStream_t stream = nullptr;
  unsigned char* arena = nullptr;
  size_t arena_bytes = 0;
  unsigned char* d_blob = nullptr;
  int blob_bytes = 0;
  ox::DevBatch<float> bf{};
  ox::DevBatch<double> bd{};
  std::map<int, ox::FieldInfo> fields;
  long long launches = 0;
  int philox = 0;
  uint64_t seed = 0;
  long long h_step = 0;          // Philox step index of the next step (passed to the kernels by value)
  long long* d_step = nullptr;   // device copy, read only by a captured CUDA graph (staged mode)
  long long d_step_val = 0;      // what *d_step holds (host's view)
  bool derived_stale = false;    // see field_live() below
  float ctrl_scale = 1.0f;       // amplitude of the Philox control stream
  int applied = 0;               // a user wrote qfrc_applied / xfrc_applied since the last full reset
  void* d_tmp = nullptr;  // staging for bulk I/O
  size_t d_tmp_bytes = 0;
  void* h_tmp = nullptr;  // pinned staging for per-env I/O
  size_t h_tmp_bytes = 0;
  uint8_t* d_mask = nullptr;
  cudaGraphExec_t graph_exec = nullptr;
  cudaGraph_t graph = nullptr;
  bool split = false;  // fused mode: specialised PRE/POST kernels around the warp-cooperative solver
  bool coop = false;  // staged mode: warp-cooperative Newton solver (ox_solve_coop.cu) instead of the thread-per-env solve stage
  const ox::SpecEntry* spec = nullptr;  // model-specialised step kernel, when one was compiled in for this model
  ox::SpecRuntime spec_rt{};
  std::string jit_note;  // why a batch that wanted a specialised kernel fell back to the generic one
  // transient: set by ox_batch_step_io around one do_step (device-addressable env-major buffers, see StepArgs)
  const void* io_ctrl = nullptr;
  void* io_qpos = nullptr;
  void* io_qvel = nullptr;
  int io_f64 = 0;
  int* d_coop_ctr = nullptr;   // {next env ticket, warps done} of the persistent cooperative solver
  int coop_resident = 0;       // CTAs the device keeps resident for it (its grid size)
};


// Which fields hold current values. The generic kernels keep every mjData field in the batch; the model-specialised step
// kernel keeps intermediates on-chip and writes back only the state, qacc, qacc_warmstart, sensordata and the counters
// (the split pipeline for large models also exchanges qM, the smooth forces / accelerations and the constraint rows).
// After such a step every other field still holds what the last ox_batch_forward / generic step left there, so reading
// it is refused (loudly) until ox_batch_forward has refreshed the batch.
inline bool field_live(bool stale, bool split, int field) {
  if (!stale) return true;
  switch (field) {
    case OX_F_QPOS: case OX_F_QVEL: case OX_F_CTRL: case OX_F_QFRC_APPLIED: case OX_F_XFRC_APPLIED: case OX_F_QACC_WARMSTART:
    case OX_F_TIME: case OX_F_ACT: case OX_F_ACT_DOT: case OX_F_QACC: case OX_F_SENSORDATA: case OX_F_NCON: case OX_F_NEFC: case OX_F_SOLVER_NITER:
    case OX_F_DIVERGED: case OX_F_MOCAP_POS: case OX_F_MOCAP_QUAT: case OX_F_EQ_ACTIVE:
    case OX_F_QFRC_INVERSE:   // no step writes it: it holds what the last ox_batch_inverse wrote
      return true;
    case OX_F_QM: case OX_F_QFRC_SMOOTH: case OX_F_QACC_SMOOTH: case OX_F_QFRC_CONSTRAINT: case OX_F_EFC_J: case OX_F_EFC_POS:
    case OX_F_EFC_MARGIN: case OX_F_EFC_D: case OX_F_EFC_AREF: case OX_F_EFC_FORCE:
      return split;
    default:
      return false;
  }
}
inline bool field_live(const ox_batch* b, int field) { return field_live(b->derived_stale, b->split, field); }
#define OX_STALE_MSG(field)                                                                                              \
  ("field " + std::to_string(field) + " is not maintained by the model-specialised step kernel (it writes back qpos, qvel, " \
   "time, qacc, qacc_warmstart, sensordata and the counters only): call ox_batch_forward() first, or create the batch with " \
   "specialize = 0")

#define CU_TRY(expr)                                                                                   \
  do {                                                                                                 \
    cudaError_t err__ = (expr);                                                                        \
    if (err__ != cudaSuccess) {                                                                        \
      ox::set_error(std::string("CUDA error: ") + cudaGetErrorString(err__) + " at " #expr);           \
      return OX_ERR_CUDA;                                                                              \
    }                                                                                                  \
  } while (0)


namespace ox {
// Pinned (page-locked, mapped) host memory is addressable from the device: the pack kernels then read / write the
// caller's buffer directly over PCIe instead of staging through a device buffer plus a cudaMemcpyAsync. Returns the
// device-side alias, or nullptr for pageable memory (staged path). OX_ZERO_COPY=0 in the environment disables it.
inline void* host_mapped(const void* p) {
  static const bool enabled = [] { const char* v = getenv("OX_ZERO_COPY"); return !(v && v[0] == '0'); }();
  if (!enabled || !p) return nullptr;
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}

}  // namespace ox
