// ox_b200.hpp — header-only C++17 mirror of oxide_control's `Physics` over the C ABI (ox_b200.h).
//
// The reference's host language is Rust; no Rust toolchain exists in this image, so this header (compiled and
// exercised by tests/native/test_cpp_api.cpp) and rust/ox_b200 (sources only) both sit where the reference's
// `src/physics.rs` sits. Method names, argument meaning and error behaviour follow src/physics.rs:6-171 and
// src/error.rs:3-82; std::optional stands for Option, ox::Error for `enum Error`.
#pragma once
#include <array>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "ox_b200.h"

namespace ox_b200 {

struct Error : std::runtime_error {           // src/error.rs:3-15
  enum class Kind { Mujoco, Mjs, NameNotFound, PhysicsDiverged, JointTypeNotMatch, Cuda, Invalid };
  Kind kind;
  Error(Kind k, const std::string& msg) : std::runtime_error(msg), kind(k) {}
};

inline void check(ox_status s) {
  if (s == OX_OK) return;
  const std::string msg = ox_last_error_message();
  switch (s) {
    case OX_ERR_PARSE: case OX_ERR_IO: throw Error(Error::Kind::Mujoco, msg);   // From<MjError>, src/error.rs:17-21
    case OX_ERR_COMPILE: throw Error(Error::Kind::Mjs, msg);                    // src/physics.rs:21
    case OX_ERR_CUDA: throw Error(Error::Kind::Cuda, msg);
    default: throw Error(Error::Kind::Invalid, msg);
  }
}

template <int ObjType> struct ObjectId { int index; };   // rusty_mujoco::ObjectId<O>
namespace obj {
using Body = ObjectId<OX_OBJ_BODY>; using Joint = ObjectId<OX_OBJ_JOINT>; using Dof = ObjectId<OX_OBJ_DOF>;
using Actuator = ObjectId<OX_OBJ_ACTUATOR>; using Equality = ObjectId<OX_OBJ_EQUALITY>; using Plugin = ObjectId<OX_OBJ_PLUGIN>;
}  // namespace obj
namespace joint {  // rusty_mujoco::joint: Qpos / Qvel widths
struct Free { static constexpr int type = OX_JNT_FREE, nq = 7, nv = 6; };
struct Ball { static constexpr int type = OX_JNT_BALL, nq = 4, nv = 3; };
struct Slide { static constexpr int type = OX_JNT_SLIDE, nq = 1, nv = 1; };
struct Hinge { static constexpr int type = OX_JNT_HINGE, nq = 1, nv = 1; };
}  // namespace joint

class Model {
 public:
  static Model from_xml_string(const std::string& xml) { ox_model* m = nullptr; check(ox_model_from_xml_string(xml.c_str(), &m)); return Model(m); }
  static Model from_xml(const std::string& path) { ox_model* m = nullptr; check(ox_model_from_xml_path(path.c_str(), &m)); return Model(m); }
  // binary model format (MuJoCo: mj_saveModel / mj_loadModel)
  static Model load(const std::string& path) { ox_model* m = nullptr; check(ox_model_load(path.c_str(), &m)); return Model(m); }
  void save(const std::string& path) const { check(ox_model_save(m_, path.c_str())); }
  Model(Model&& o) noexcept : m_(o.m_) { o.m_ = nullptr; }
  Model(const Model&) = delete;
  ~Model() { ox_model_free(m_); }
  const ox_model* handle() const { return m_; }
  const ox_model_tables& tables() const { return *ox_model_get_tables(m_); }
  template <int O> std::optional<ObjectId<O>> object_id(const std::string& name) const {   // src/physics.rs:56-58
    int i = ox_model_name2id(m_, O, name.c_str());
    if (i < 0) return std::nullopt;
    return ObjectId<O>{i};
  }
  template <int O> std::string object_name(ObjectId<O> id) const {                          // src/physics.rs:60-62
    const char* s = ox_model_id2name(m_, O, id.index);
    if (!s) throw Error(Error::Kind::Invalid, "object id out of range");
    return s;
  }
 private:
  explicit Model(ox_model* m) : m_(m) {}
  ox_model* m_;
};

// nenv copies of mjData on one GPU
class BatchedPhysics {
 public:
  BatchedPhysics(const Model& model, ox_batch_config cfg) : model_(&model) { check(ox_batch_create(model.handle(), &cfg, &b_)); }
  BatchedPhysics(const BatchedPhysics&) = delete;
  ~BatchedPhysics() { ox_batch_free(b_); }
  static ox_batch_config default_config(int nenv, int precision = OX_F32) {
    ox_batch_config c; ox_batch_config_default(&c); c.nenv = nenv; c.precision = precision; return c;
  }
  void step(int nsteps = 1) { check(ox_batch_step(b_, nsteps)); }
  void forward() { check(ox_batch_forward(b_)); }
  void inverse() { check(ox_batch_inverse(b_)); }   // extension: mj_inverse for every env, result in OX_F_QFRC_INVERSE
  // ctrl in, one step, qpos / qvel out in one call (Action::apply + step + Observation::generate, src/lib.rs:63-66)
  void step_io(const void* ctrl, void* qpos, void* qvel, int dtype, int mem = OX_MEM_HOST) { check(ox_batch_step_io(b_, ctrl, qpos, qvel, dtype, mem)); }
  void reset(const uint8_t* mask = nullptr) { check(ox_batch_reset(b_, mask)); }
  void sync() { check(ox_batch_sync(b_)); }
  void set(int field, const void* buf, int dtype, int mem = OX_MEM_HOST, int layout = OX_LAYOUT_ENV_MAJOR) { check(ox_batch_set(b_, field, buf, dtype, mem, layout)); }
  void get(int field, void* buf, int dtype, int mem = OX_MEM_HOST, int layout = OX_LAYOUT_ENV_MAJOR) { check(ox_batch_get(b_, field, buf, dtype, mem, layout)); }
  std::vector<double> get1(int field, int env, int offset, int count) { std::vector<double> v(count); check(ox_batch_get1(b_, field, env, offset, count, v.data())); return v; }
  void set1(int field, int env, int offset, const double* v, int count) { check(ox_batch_set1(b_, field, env, offset, count, v)); }
  ox_batch* handle() { return b_; }
  const Model& model() const { return *model_; }
 private:
  const Model* model_;
  ox_batch* b_ = nullptr;
};

// N1: Environment<T: Task> over a BatchedPhysics (src/lib.rs:28-88), evaluated on device from a declarative task.
struct BatchedTimeStep {                               // enum TimeStep<O> for every env (src/lib.rs:50-60)
  std::vector<double> observation, reward, discount;   // [nenv*obs_dim], [nenv], [nenv] (discount 0 = Finish)
  std::vector<uint8_t> finished;                       // [nenv]
};
class BatchedEnvironment {
 public:
  BatchedEnvironment(BatchedPhysics& physics, const ox_task_spec& task) : physics_(physics) { check(ox_env_create(physics.handle(), &task, &e_)); }
  BatchedEnvironment(const BatchedEnvironment&) = delete;
  ~BatchedEnvironment() { ox_env_free(e_); }
  static ox_task_spec default_task() { ox_task_spec t; ox_task_spec_default(&t); return t; }
  int obs_dim() const { return ox_env_obs_dim(e_); }
  BatchedPhysics& physics_mut() { return physics_; }                                                              // :45-47
  std::vector<double> reset() {                                                                                  // :62-65
    std::vector<double> obs((size_t)nenv() * obs_dim());
    check(ox_env_reset(e_, obs.data(), OX_F64, OX_MEM_HOST));
    return obs;
  }
  BatchedTimeStep step(const double* action) {                                                                   // :67-87
    BatchedTimeStep ts;
    ts.observation.resize((size_t)nenv() * obs_dim()); ts.reward.resize(nenv()); ts.discount.resize(nenv()); ts.finished.resize(nenv());
    check(ox_env_step(e_, action, ts.observation.data(), ts.reward.data(), ts.discount.data(), ts.finished.data(), OX_F64, OX_MEM_HOST));
    return ts;
  }
  ox_env* handle() { return e_; }
 private:
  int nenv() const { return ox_batch_nenv(physics_.handle()); }
  BatchedPhysics& physics_;
  ox_env* e_ = nullptr;
};

class Physics;
class Actuators {                                  // src/physics.rs:65-79
 public:
  explicit Actuators(Physics& p) : p_(p) {}
  void set(obj::Actuator id, double control);
 private:
  Physics& p_;
};

// One environment: method-for-method mirror of src/physics.rs (a BatchedPhysics of size 1 in fp64).
class Physics {
 public:
  static Physics from_xml(const std::string& path) { return Physics(Model::from_xml(path)); }                    // :12-16
  static Physics from_xml_string(const std::string& xml) { return Physics(Model::from_xml_string(xml)); }       // :18-24
  const Model& model() const { return model_; }                                                                  // :26-28
  BatchedPhysics& data_mut() { return batch_; }                                                                  // :33-35
  void step() { batch_.step(1); batch_.sync(); }                                                                 // :44-46
  void forward() { batch_.forward(); batch_.sync(); }                                                            // :48-50
  void inverse() { batch_.inverse(); batch_.sync(); }                                                            // extension: mj_inverse
  void reset() { batch_.reset(); batch_.sync(); }                                                                // :52-54
  template <int O> std::optional<ObjectId<O>> object_id(const std::string& n) const { return model_.object_id<O>(n); }
  template <int O> std::string object_name(ObjectId<O> id) const { return model_.object_name(id); }
  Actuators actuators() { return Actuators(*this); }                                                             // :73-79
  double time() { return batch_.get1(OX_F_TIME, 0, 0, 1)[0]; }                                                   // :82-87
  void set_time(double t) { batch_.set1(OX_F_TIME, 0, 0, &t, 1); }
  double ctrl(obj::Actuator id) { return batch_.get1(OX_F_CTRL, 0, id.index, 1)[0]; }                            // :89-94
  void set_ctrl(obj::Actuator id, double v) { batch_.set1(OX_F_CTRL, 0, id.index, &v, 1); }
  // :96-102: Some(activation) for stateful actuators (dyntype integrator / filter / filterexact), None for stateless ones
  int actadr(obj::Actuator id) const { return model_.tables().na > 0 ? model_.tables().actuator_actadr[id.index] : -1; }
  std::optional<double> act(obj::Actuator id) {
    const int adr = actadr(id);
    if (adr < 0) return std::nullopt;
    return batch_.get1(OX_F_ACT, 0, adr, 1)[0];
  }
  std::optional<std::monostate> set_act(obj::Actuator id, double value) {
    const int adr = actadr(id);
    if (adr < 0) return std::nullopt;
    batch_.set1(OX_F_ACT, 0, adr, &value, 1); return std::monostate{};
  }
  template <class J> std::array<double, J::nq> qpos(obj::Joint id) {                                             // :104-109
    check_joint<J>(id);
    auto v = batch_.get1(OX_F_QPOS, 0, model_.tables().jnt_qposadr[id.index], J::nq);
    std::array<double, J::nq> a; for (int i = 0; i < J::nq; i++) a[i] = v[i]; return a;
  }
  template <class J> void set_qpos(obj::Joint id, const std::array<double, J::nq>& q) {
    check_joint<J>(id); batch_.set1(OX_F_QPOS, 0, model_.tables().jnt_qposadr[id.index], q.data(), J::nq);
  }
  template <class J> std::array<double, J::nv> qvel(obj::Joint id) {                                             // :111-116
    check_joint<J>(id);
    auto v = batch_.get1(OX_F_QVEL, 0, model_.tables().jnt_dofadr[id.index], J::nv);
    std::array<double, J::nv> a; for (int i = 0; i < J::nv; i++) a[i] = v[i]; return a;
  }
  template <class J> void set_qvel(obj::Joint id, const std::array<double, J::nv>& q) {
    check_joint<J>(id); batch_.set1(OX_F_QVEL, 0, model_.tables().jnt_dofadr[id.index], q.data(), J::nv);
  }
  double qacc_warmstart(obj::Dof id) { return batch_.get1(OX_F_QACC_WARMSTART, 0, id.index, 1)[0]; }             // :118-123
  void set_qacc_warmstart(obj::Dof id, double v) { batch_.set1(OX_F_QACC_WARMSTART, 0, id.index, &v, 1); }
  std::optional<double> plugin_state(obj::Plugin) { return std::nullopt; }                                       // :125-131
  double qfrc_applied(obj::Dof id) { return batch_.get1(OX_F_QFRC_APPLIED, 0, id.index, 1)[0]; }                 // :133-138
  void set_qfrc_applied(obj::Dof id, double v) { batch_.set1(OX_F_QFRC_APPLIED, 0, id.index, &v, 1); }
  std::array<double, 6> xfrc_applied(obj::Body id) {                                                             // :140-145
    auto v = batch_.get1(OX_F_XFRC_APPLIED, 0, 6 * id.index, 6); std::array<double, 6> a; for (int i = 0; i < 6; i++) a[i] = v[i]; return a;
  }
  void set_xfrc_applied(obj::Body id, const std::array<double, 6>& f) { batch_.set1(OX_F_XFRC_APPLIED, 0, 6 * id.index, f.data(), 6); }
  bool eq_active(obj::Equality id) { return batch_.get1(OX_F_EQ_ACTIVE, 0, id.index, 1)[0] != 0; }                // :147-152
  void set_eq_active(obj::Equality id, bool on) { const double v = on ? 1 : 0; batch_.set1(OX_F_EQ_ACTIVE, 0, id.index, &v, 1); }
  // :154-170: None when the body is not a mocap body
  int mocapid(obj::Body id) const { return model_.tables().nmocap > 0 ? model_.tables().body_mocapid[id.index] : -1; }
  std::optional<std::array<double, 3>> mocap_pos(obj::Body id) {
    const int m = mocapid(id);
    if (m < 0) return std::nullopt;
    auto v = batch_.get1(OX_F_MOCAP_POS, 0, 3 * m, 3); return std::array<double, 3>{v[0], v[1], v[2]};
  }
  std::optional<std::monostate> set_mocap_pos(obj::Body id, const std::array<double, 3>& p) {
    const int m = mocapid(id);
    if (m < 0) return std::nullopt;
    batch_.set1(OX_F_MOCAP_POS, 0, 3 * m, p.data(), 3); return std::monostate{};
  }
  std::optional<std::array<double, 4>> mocap_quat(obj::Body id) {
    const int m = mocapid(id);
    if (m < 0) return std::nullopt;
    auto v = batch_.get1(OX_F_MOCAP_QUAT, 0, 4 * m, 4); return std::array<double, 4>{v[0], v[1], v[2], v[3]};
  }
  std::optional<std::monostate> set_mocap_quat(obj::Body id, const std::array<double, 4>& q) {
    const int m = mocapid(id);
    if (m < 0) return std::nullopt;
    batch_.set1(OX_F_MOCAP_QUAT, 0, 4 * m, q.data(), 4); return std::monostate{};
  }
  // data(): derived arrays the reference reaches through Physics::data() (src/physics.rs:30-32)
  std::vector<double> qacc() { return batch_.get1(OX_F_QACC, 0, 0, model_.tables().nv); }
  std::vector<double> sensordata() { return batch_.get1(OX_F_SENSORDATA, 0, 0, model_.tables().nsensordata); }
 private:
  // one env, fp64, generic kernels: data() stands for &mjData, so every derived field must be current after step()
  static ox_batch_config single_config() { ox_batch_config c = BatchedPhysics::default_config(1, OX_F64); c.specialize = 0; return c; }
  explicit Physics(Model&& m) : model_(std::move(m)), batch_(model_, single_config()) {}
  template <class J> void check_joint(obj::Joint id) const {
    if (model_.tables().jnt_type[id.index] != J::type) throw Error(Error::Kind::JointTypeNotMatch, "joint type does not match");
  }
  Model model_;
  BatchedPhysics batch_;
};
inline void Actuators::set(obj::Actuator id, double control) { p_.set_ctrl(id, control); }

}  // namespace ox_b200
