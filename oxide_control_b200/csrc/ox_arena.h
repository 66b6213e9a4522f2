// Arena layout of the SoA batch + the field-id registry of the C ABI (shared with tests/native).
#pragma once
#include <algorithm>
#include <map>

#include "ox_blob.h"

namespace ox {

struct FieldInfo {
  void* ptr;
  int count;
  bool is_int;
};

template <typename T>
size_t layout_arena(const ox_model_tables& t, int stride, unsigned char* base, DevBatch<T>* out, std::map<int, FieldInfo>* fields) {
  const long nq = t.nq, nv = t.nv, nu = t.nu, na = t.na, nb = t.nbody, nj = t.njnt, ng = t.ngeom, ns = t.nsite, nM = t.nM;
  const long ncm = std::max(1, t.nconmax), nem = std::max(1, t.nefcmax), nsd = t.nsensordata, nmc = t.nmocap, neq = t.neq, nten = t.ntendon;
  size_t off = 0;
  auto take = [&](size_t elems, size_t esz) {
    size_t o = off;
    off += (std::max<size_t>(elems, 1) * (size_t)stride * esz + 255) / 256 * 256;
    return o;
  };
#define OX_X(name, cnt)                                                       \
  {                                                                           \
    size_t o = take((size_t)(cnt), sizeof(T));                                \
    if (out) out->name = reinterpret_cast<T*>(base + o);                      \
  }
  OX_BATCH_REAL_FIELDS(OX_X)
#undef OX_X
#define OX_X(name, cnt)                                                       \
  {                                                                           \
    size_t o = take((size_t)(cnt), sizeof(int32_t));                          \
    if (out) out->name = reinterpret_cast<int32_t*>(base + o);                \
  }
  OX_BATCH_INT_FIELDS(OX_X)
#undef OX_X
  // qfrc_inverse (ox_batch_inverse): appended after every DevBatch field and kept out of DevBatch, whose size and field
  // lists fix the shared-memory and per-thread layouts of the step kernels; k_inverse receives the pointer as an argument
  const size_t off_inverse = take((size_t)nv, sizeof(T));
  if (out && fields) {
    auto& f = *fields;
#define R(id, name, cnt) f[id] = FieldInfo{out->name, (int)(cnt), false};
    R(OX_F_QPOS, qpos, nq) R(OX_F_QVEL, qvel, nv) R(OX_F_CTRL, ctrl, nu) R(OX_F_QFRC_APPLIED, qfrc_applied, nv)
    R(OX_F_XFRC_APPLIED, xfrc_applied, 6 * nb) R(OX_F_QACC_WARMSTART, qacc_warmstart, nv) R(OX_F_TIME, time, 1)
    R(OX_F_QACC, qacc, nv) R(OX_F_SENSORDATA, sensordata, nsd) R(OX_F_XPOS, xpos, 3 * nb) R(OX_F_XQUAT, xquat, 4 * nb)
    R(OX_F_XMAT, xmat, 9 * nb) R(OX_F_XIPOS, xipos, 3 * nb) R(OX_F_XIMAT, ximat, 9 * nb) R(OX_F_XANCHOR, xanchor, 3 * nj)
    R(OX_F_XAXIS, xaxis, 3 * nj) R(OX_F_GEOM_XPOS, geom_xpos, 3 * ng) R(OX_F_GEOM_XMAT, geom_xmat, 9 * ng)
    R(OX_F_SITE_XPOS, site_xpos, 3 * ns) R(OX_F_SITE_XMAT, site_xmat, 9 * ns) R(OX_F_SUBTREE_COM, subtree_com, 3 * nb)
    R(OX_F_CINERT, cinert, 10 * nb) R(OX_F_CDOF, cdof, 6 * nv) R(OX_F_QM, qM, nM) R(OX_F_QLD, qLD, nM)
    R(OX_F_QLDIAGINV, qLDiagInv, nv) R(OX_F_CVEL, cvel, 6 * nb) R(OX_F_CDOF_DOT, cdof_dot, 6 * nv)
    R(OX_F_QFRC_BIAS, qfrc_bias, nv) R(OX_F_QFRC_PASSIVE, qfrc_passive, nv) R(OX_F_ACTUATOR_FORCE, actuator_force, nu)
    R(OX_F_QFRC_ACTUATOR, qfrc_actuator, nv) R(OX_F_QFRC_SMOOTH, qfrc_smooth, nv) R(OX_F_QACC_SMOOTH, qacc_smooth, nv)
    R(OX_F_QFRC_CONSTRAINT, qfrc_constraint, nv) R(OX_F_CON_DIST, con_dist, ncm) R(OX_F_CON_POS, con_pos, 3 * ncm)
    R(OX_F_CON_FRAME, con_frame, 9 * ncm) R(OX_F_EFC_J, efc_J, nem * nv) R(OX_F_EFC_POS, efc_pos, nem)
    R(OX_F_EFC_MARGIN, efc_margin, nem) R(OX_F_EFC_D, efc_D, nem) R(OX_F_EFC_AREF, efc_aref, nem) R(OX_F_EFC_FORCE, efc_force, nem)
    R(OX_F_ACT, act, na) R(OX_F_ACT_DOT, act_dot, na) R(OX_F_MOCAP_POS, mocap_pos, 3 * nmc) R(OX_F_MOCAP_QUAT, mocap_quat, 4 * nmc)
    R(OX_F_EQ_ACTIVE, eq_active, neq) R(OX_F_TEN_LENGTH, ten_length, nten) R(OX_F_TEN_J, ten_J, nten * nv)
#undef R
    f[OX_F_QFRC_INVERSE] = FieldInfo{base + off_inverse, (int)nv, false};
#define I(id, name, cnt) f[id] = FieldInfo{out->name, (int)(cnt), true};
    I(OX_F_NCON, ncon, 1) I(OX_F_NEFC, nefc, 1) I(OX_F_SOLVER_NITER, solver_niter, 1) I(OX_F_DIVERGED, diverged, 1)
    I(OX_F_CON_PAIR, con_pair, ncm)
#undef I
  }
  return off;
}


}  // namespace ox
