// TEST-ONLY: the inverse kernel's per-env body (csrc/ox_inverse.cuh) run on the host. This translation unit compiles the host
// instantiation (ox_hostcheck.cu, which stays as it is) and adds hc_inverse, writing the arena's qfrc_inverse region. Built
// with ox_inverse_oracle.cpp into libox_inverse_check.so by tests/inverse_support.py; never linked into the product.
#include "ox_hostcheck.cu"
#include "../../oxide_control_b200/csrc/ox_inverse.cuh"

extern "C" HC_API void hc_inverse(hc_batch* b) {
  void* out = b->fields.at(OX_F_QFRC_INVERSE).ptr;
  DISPATCH(env_inverse(env, (decltype(env.b.qacc))out))
}
