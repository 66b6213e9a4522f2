// Inverse dynamics of one environment (mj_inverse, continuous time), composed from the public stage functions of Env.
// Included by the inverse kernel (ox_inverse.cu) and by the test-only host instantiation, so both run the same arithmetic.
// It lives outside ox_stages.cuh, whose text the run-time specialisation embeds: the specialised kernels' sources stay as
// they are.
#pragma once
#include "ox_stages.cuh"

namespace ox {

// qfrc_inverse[i] (field layout of the batch, element i at Env::at) = M qacc + qfrc_bias - qfrc_passive - qfrc_constraint,
// with efc_force / qfrc_constraint the soft-constraint force at J qacc - aref (mj_invConstraint is mj_constraintUpdate at the
// given qacc). The forward stages up to the smooth acceleration refresh every derived field the way mj_forward does, so the
// actuation fields and qfrc_smooth / qacc_smooth are current too; sensors then read the given qacc and the inverse forces.
template <typename T, typename M, bool LOCAL>
OX_HDN void env_inverse(const Env<T, M, LOCAL>& env, T* qfrc_inverse) {
  const DevBatch<T>& b = env.b;
  const int nv = env.m.h().nv;
  env.fwd_position();
  env.fwd_velocity();
  env.make_constraint();
  env.actuation();
  env.fwd_acceleration();
  const int nefc = env.ati(b.nefc, 0);
  for (int r = 0; r < nefc; r++) env.at(b.s_Jaref, r) = env.row_dot(r, b.qacc, nv) - env.at(b.efc_aref, r);
  env.mul_m(b.s_Ma, b.qacc);   // qM carries dof_armature: s_Ma includes armature * qacc
  T gauss;
  env.update_constraint(nv, nefc, &gauss);
  for (int i = 0; i < nv; i++)
    env.at(qfrc_inverse, i) = env.at(b.s_Ma, i) + env.at(b.qfrc_bias, i) - env.at(b.qfrc_passive, i) - env.at(b.qfrc_constraint, i);
  env.sensors();
}

}  // namespace ox
