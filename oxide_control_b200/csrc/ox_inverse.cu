// Batched inverse dynamics (ox_batch_inverse, mj_inverse): one thread per environment, on every kind of batch. The kernel
// reads and writes the batch's SoA arena like k_forward_fused, so after a coop-mode step (rows stored env-contiguously) or a
// model-specialised step (intermediates kept on chip) it rewrites every derived field in the arena's own layout.
#include <cuda_runtime.h>

#include "ox_internal.h"
#include "ox_kernels.cuh"
#include "ox_inverse.cuh"
#include "ox_batch_internal.cuh"

namespace ox {

template <typename T>
__global__ void k_inverse(const unsigned char* __restrict__ gblob, int bytes, DevBatch<T> b, T* __restrict__ qfrc_inverse) {
  DevModel<T> m{stage_model(gblob, bytes)};
  const int e = env_index(b);
  if (e < 0) return;
  Env<T> env(m, b, e);
  env_inverse(env, qfrc_inverse);
}

template <typename T>
static cudaError_t launch_inverse(ox_batch* b, const DevBatch<T>& db) {
  // the model tables are staged into dynamic shared memory; above 48 KB the kernel must opt in (per device, so per call)
  if (b->blob_bytes > 48 * 1024) {
    const cudaError_t err = cudaFuncSetAttribute(k_inverse<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, b->blob_bytes);
    if (err != cudaSuccess) return err;
  }
  T* out = static_cast<T*>(b->fields.at(OX_F_QFRC_INVERSE).ptr);
  k_inverse<T><<<b->grid, b->block, b->blob_bytes, b->stream>>>(b->d_blob, b->blob_bytes, db, out);
  return cudaGetLastError();
}

}  // namespace ox

extern "C" ox_status ox_batch_inverse(ox_batch* b) {
  if (!b) { ox::set_error("ox_batch_inverse: null batch"); return OX_ERR_INVALID; }
  CU_TRY(cudaSetDevice(b->cfg.device));
  b->launches++;
  CU_TRY(b->f64 ? ox::launch_inverse<double>(b, b->bd) : ox::launch_inverse<float>(b, b->bf));
  b->derived_stale = false;
  return OX_OK;
}
