// Warp-cooperative primal Newton solver (mj_fwdConstraint / mj_solNewton; SURVEY.md A.11): ONE WARP PER ENVIRONMENT,
// lane = dof. It replaces the thread-per-env solve stage for models whose constraint problem is too large to sit in
// one thread's registers (humanoid class: nv = 27, H = 27x27): there the serial solve is >90 % of the step and the GPU
// holds only nenv/32 warps. The solve itself is group_newton (ox_group_solve.cuh) with G = 32; this kernel gives each
// warp shared-memory scratch for it, including per-row scalar arrays for envs with at most COOP_RCAP rows.
// Eligibility (checked on the host): Newton solver, nv <= 32.
#include "ox_kernels.cuh"
#include "ox_group_solve.cuh"

namespace ox {

constexpr int COOP_WARPS = 8;      // warps (= consecutive envs) per CTA: their gathers from the [element][env] arena share 32-byte sectors
constexpr int COOP_RCAP = 96;      // rows whose per-row scalars live in shared memory; envs with more rows use the arena's row arrays

// per-warp shared memory: five row arrays of RCAP, J staging (SROWS x 33), the Cholesky factor (32 x 33) for the back substitution
__host__ __device__ inline size_t coop_warp_words() { return 5 * (size_t)COOP_RCAP + COOP_SROWS * 33 + 32 * 33; }

// PERSISTENT launch: the grid holds as many CTAs as the device keeps resident; every warp draws its next environment from a
// global ticket counter. Solve times vary several-fold between envs (0 .. 8 Newton iterations, 0 .. 90 rows), and with the
// static env -> warp map a CTA's slot stayed occupied until its slowest warp finished (ncu: 10 of 16 resident warps active,
// 1.7 waves of CTAs); drawing tickets keeps every resident warp busy until the batch is done and stages the model tables once
// per CTA instead of once per 8 envs. The last warp to leave resets both counters for the next launch (stream-ordered).
template <typename T>
__global__ void __launch_bounds__(32 * COOP_WARPS) k_solve_coop(const unsigned char* __restrict__ gblob, int bytes, DevBatch<T> b, int* __restrict__ ctr) {
  DevModel<T> m{stage_model(gblob, bytes)};
  extern __shared__ __align__(128) unsigned char ox_smem[];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  T* srow = reinterpret_cast<T*>(ox_smem + ((bytes + 127) / 128) * 128) + (size_t)wib * coop_warp_words();
  T* sJ = srow + 5 * COOP_RCAP;
  T* sL = sJ + COOP_SROWS * 33;
  const LaneGroup<32> g{lane, 0xffffffffu};
  for (;;) {
    int env = 0;
    if (lane == 0) env = atomicAdd(&ctr[0], 1);
    env = __shfl_sync(0xffffffffu, env, 0);
    if (env >= b.nenv) break;
    // ends with a warp sync: the warp's shared-memory scratch is then free for its next environment
    group_newton<T, 32, COOP_RCAP>(g, m, b, ElemAt{(uint32_t)b.stride, (uint32_t)env}, sJ, sL, srow);
  }
  if (lane == 0) {
    const int done = atomicAdd(&ctr[1], 1);
    if (done == (int)gridDim.x * COOP_WARPS - 1) { ctr[0] = 0; ctr[1] = 0; __threadfence(); }
  }
}

constexpr size_t COOP_SMEM_LIMIT = 200 * 1024;  // opt-in dynamic shared memory per CTA this kernel asks for (the SM has 227 KB)

size_t solve_coop_smem(int blob_bytes, bool f64) {
  return (size_t)((blob_bytes + 127) / 128) * 128 + (size_t)COOP_WARPS * coop_warp_words() * (f64 ? sizeof(double) : sizeof(float));
}

// cudaFuncSetAttribute is per DEVICE: called from ox_batch_create (after cudaSetDevice) for every batch that will use the
// cooperative solver, so that a second batch on another GPU of the same process gets the opt-in too.
cudaError_t solve_coop_prepare(int blob_bytes, bool f64) {
  if (solve_coop_smem(blob_bytes, f64) > COOP_SMEM_LIMIT) return cudaErrorInvalidValue;
  return f64 ? cudaFuncSetAttribute(k_solve_coop<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)COOP_SMEM_LIMIT)
             : cudaFuncSetAttribute(k_solve_coop<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)COOP_SMEM_LIMIT);
}

// CTAs the current device keeps resident for this kernel (0 on error): the size of the persistent grid
int solve_coop_resident_ctas(int blob_bytes, bool f64) {
  int dev = 0, sms = 0, per_sm = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  const size_t smem = solve_coop_smem(blob_bytes, f64);
  const cudaError_t e = f64 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_solve_coop<double>, 32 * COOP_WARPS, smem)
                            : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_solve_coop<float>, 32 * COOP_WARPS, smem);
  if (e != cudaSuccess || per_sm < 1) return 0;
  return sms * per_sm;
}

template <typename T>
static cudaError_t launch_coop(cudaStream_t stream, const unsigned char* blob, int bytes, const DevBatch<T>& b, int resident_ctas, int* ctr) {
  const size_t smem = solve_coop_smem(bytes, sizeof(T) == 8);
  int grid = (b.nenv + COOP_WARPS - 1) / COOP_WARPS;
  if (resident_ctas > 0 && grid > resident_ctas) grid = resident_ctas;
  k_solve_coop<T><<<grid, 32 * COOP_WARPS, smem, stream>>>(blob, bytes, b, ctr);
  return cudaPeekAtLastError();  // the caller propagates it (CU_TRY); peek so that the sticky state is not silently cleared
}

cudaError_t launch_solve_coop_f32(cudaStream_t s, const unsigned char* blob, int bytes, const DevBatch<float>& b, int resident_ctas, int* ctr) { return launch_coop<float>(s, blob, bytes, b, resident_ctas, ctr); }
cudaError_t launch_solve_coop_f64(cudaStream_t s, const unsigned char* blob, int bytes, const DevBatch<double>& b, int resident_ctas, int* ctr) { return launch_coop<double>(s, blob, bytes, b, resident_ctas, ctr); }
bool solve_coop_eligible(const ox_model_tables& t) {
  return t.solver == OX_SOL_NEWTON && t.noslip_iterations == 0 && t.nfloss == 0 && t.cone == OX_CONE_PYRAMIDAL && t.nv >= 1 && t.nv <= 32;
}

}  // namespace ox
