// TEST-ONLY: the oracle's inverse dynamics (mj_inverse, continuous time). This translation unit compiles the oracle's source
// (oracle/ox_oracle.cpp, which stays as it is) and adds oxo_inverse on top of its stage functions. Built together with
// ox_inverse_hostcheck.cpp into libox_inverse_check.so by tests/inverse_support.py; never linked into the product.
#include "../../oracle/ox_oracle.cpp"

namespace {

// MuJoCo's route: position and velocity stages, the inverse constraint (mj_invConstraint = the solver's constraint update at
// the given qacc), then RNE with the acceleration term (flg_acc = 1: cacc includes cdof qacc), plus armature qacc, minus the
// passive and constraint forces. The product takes M qacc + qfrc_bias instead; the two routes must agree. The actuation and
// smooth-acceleration stages run too (the product refreshes those fields), and sensors read the given qacc.
void inverseDynamics(const Model* m, Data* d, double* qfrc_inverse) {
  const int nb = m->nbody, nv = m->nv;
  kinematics(m, d);
  comPos(m, d);
  crb(m, d);
  factorM(m, d);
  collision(m, d);
  comVel(m, d);
  makeConstraint(m, d);
  passive(m, d);
  rne(m, d);
  actuation(m, d);
  fwdAcceleration(m, d);
  Solver s(m, d);
  mulM(m, d->qM.data(), s.Ma.data(), d->qacc.data());
  for (int r = 0; r < d->nefc; r++) {
    double v = -d->efc_aref[r];
    for (int i = 0; i < nv; i++) v += d->efc_J[(size_t)r * nv + i] * d->qacc[i];
    s.Jaref[r] = v;
  }
  s.updateConstraint();
  std::vector<double> cacc, cfrc(6 * nb, 0.0);
  bodyAcc(m, d, cacc);
  for (int b = 1; b < nb; b++) {
    double tmp[6], tmp1[6];
    mulInertVec(&cfrc[6 * b], &d->cinert[10 * b], &cacc[6 * b]);
    mulInertVec(tmp, &d->cinert[10 * b], &d->cvel[6 * b]);
    crossForce(tmp1, &d->cvel[6 * b], tmp);
    for (int c = 0; c < 6; c++) cfrc[6 * b + c] += tmp1[c];
  }
  for (int b = nb - 1; b > 0; b--) {
    const int p = m->body_parentid[b];
    if (p) for (int c = 0; c < 6; c++) cfrc[6 * p + c] += cfrc[6 * b + c];
  }
  for (int i = 0; i < nv; i++)
    qfrc_inverse[i] = dot6(&d->cdof[6 * i], &cfrc[6 * m->dof_bodyid[i]]) + m->dof_armature[i] * d->qacc[i] - d->qfrc_passive[i] - d->qfrc_constraint[i];
  sensors(m, d);
}

}  // namespace

// qfrc_inverse: nv doubles written by the call
extern "C" __attribute__((visibility("default"))) void oxo_inverse(const Model* m, oxo_data* d, double* qfrc_inverse) {
  inverseDynamics(m, d, qfrc_inverse);
}
