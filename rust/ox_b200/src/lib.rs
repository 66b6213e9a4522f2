//! Safe wrapper over libox_b200.so with the surface of `oxide_control::physics::Physics` (reference src/physics.rs:6-171),
//! plus what the reference does not have: `BatchedPhysics` (nenv copies of mjData on one GPU), `PhysicsGroup` (one batch
//! per GPU of the box, one host process) and `BatchedEnvironment` (reference src/lib.rs:28-88 for a whole batch, on device).
//!
//! NOT COMPILED in the build environment (the image has no cargo / rustc). The executable mirrors of the same C ABI are
//! include/ox_b200.hpp (C++) and oxide_control_b200/physics.py (Python); tests/test_rust_sources.py checks that this file
//! declares every method of the reference's `Physics` with the reference's receiver (`&self` / `&mut self`).
//!
//! Getters take `&self` as in the reference: the raw handle is a pointer, and every call is serialised on the batch's
//! stream by the library. The types are `Send` but not `Sync` (one stream per batch, SURVEY 8b).
#![allow(non_upper_case_globals)]
use ox_b200_sys as sys;
use std::ffi::{CStr, CString};
use std::marker::PhantomData;

pub const mjMAXVAL: f64 = sys::OX_MAXVAL; // re-exported by the reference at src/physics.rs:2
pub const mjMINVAL: f64 = sys::OX_MINVAL;

// ------------------------------------------------------------------------------------------------ errors (src/error.rs)
/// `oxide_control::error::Error` (src/error.rs:3-15) with a CUDA variant for the device side.
pub enum Error {
    Mujoco(String),
    Mjs(String),
    NameNotFound(&'static str),
    PhysicsDiverged,
    JointTypeNotMatch { expected: i32, found: i32 },
    ActuatorStateless(ObjectId<obj::Actuator>),
    PluginStateless(ObjectId<obj::Plugin>),
    BodyNotMocap(ObjectId<obj::Body>),
    Cuda(String),
    Invalid(String),
}
impl std::fmt::Debug for Error {
    fn fmt(&self, f: &mut std::fmt::Formatter<'_>) -> std::fmt::Result {
        match self {
            Error::Mujoco(e) => write!(f, "Error::MuJoCo({e:?})"),
            Error::Mjs(msg) => write!(f, "Error::Mjs({msg})"),
            Error::NameNotFound(name) => write!(f, "Error::NameNotFound({name})"),
            Error::PhysicsDiverged => write!(f, "Error::PhysicsDiverged"),
            Error::JointTypeNotMatch { expected, found } => write!(f, "Error::JointTypeNotMatch(expected: {expected:?}, found: {found:?})"),
            Error::ActuatorStateless(id) => write!(f, "Error::ActuatorStateless({:?})", id.index),
            Error::PluginStateless(id) => write!(f, "Error::PluginStateless({:?})", id.index),
            Error::BodyNotMocap(id) => write!(f, "Error::BodyNotMocap({:?})", id.index),
            Error::Cuda(msg) => write!(f, "Error::Cuda({msg})"),
            Error::Invalid(msg) => write!(f, "Error::Invalid({msg})"),
        }
    }
}
impl std::fmt::Display for Error {
    fn fmt(&self, f: &mut std::fmt::Formatter<'_>) -> std::fmt::Result { std::fmt::Debug::fmt(self, f) }
}
impl std::error::Error for Error {}

fn last_error() -> String { unsafe { CStr::from_ptr(sys::ox_last_error_message()).to_string_lossy().into_owned() } }
fn check(s: sys::ox_status) -> Result<(), Error> {
    match s {
        sys::OX_OK => Ok(()),
        sys::OX_ERR_PARSE | sys::OX_ERR_IO => Err(Error::Mujoco(last_error())),   // From<MjError>, src/error.rs:17-21
        sys::OX_ERR_COMPILE => Err(Error::Mjs(last_error())),                      // src/physics.rs:21
        sys::OX_ERR_CUDA => Err(Error::Cuda(last_error())),
        _ => Err(Error::Invalid(last_error())),
    }
}

// ------------------------------------------------------------------------------------------------ typed ids (rusty_mujoco::{ObjectId, obj, Joint, joint})
pub trait Obj { const TYPE: i32; }
pub mod obj {
    use super::{sys, Obj};
    macro_rules! objs { ($($n:ident = $t:expr),*) => { $( #[derive(Clone, Copy, Debug)] pub struct $n; impl Obj for $n { const TYPE: i32 = $t; } )* } }
    objs!(Body = sys::OX_OBJ_BODY, Joint = sys::OX_OBJ_JOINT, Dof = sys::OX_OBJ_DOF, Geom = sys::OX_OBJ_GEOM, Site = sys::OX_OBJ_SITE,
          Equality = sys::OX_OBJ_EQUALITY, Actuator = sys::OX_OBJ_ACTUATOR, Sensor = sys::OX_OBJ_SENSOR, Plugin = sys::OX_OBJ_PLUGIN);
}
pub struct ObjectId<O> { pub index: usize, _o: PhantomData<O> }
impl<O> ObjectId<O> { pub fn new(index: usize) -> Self { Self { index, _o: PhantomData } } }
impl<O> Clone for ObjectId<O> { fn clone(&self) -> Self { *self } }
impl<O> Copy for ObjectId<O> {}

/// `rusty_mujoco::Joint`: a joint type with its qpos / qvel widths (src/physics.rs:104-116 are generic over it).
pub trait Joint: Obj {
    const MJT: i32;
    type Qpos: AsRef<[f64]> + AsMut<[f64]> + Default;
    type Qvel: AsRef<[f64]> + AsMut<[f64]> + Default;
}
pub mod joint {
    use super::{sys, Joint, Obj};
    macro_rules! joints { ($($n:ident = $t:expr, $q:expr, $v:expr);*) => { $(
        #[derive(Clone, Copy, Debug)] pub struct $n;
        impl Obj for $n { const TYPE: i32 = sys::OX_OBJ_JOINT; }
        impl Joint for $n { const MJT: i32 = $t; type Qpos = [f64; $q]; type Qvel = [f64; $v]; }
    )* } }
    joints!(Free = sys::OX_JNT_FREE, 7, 6; Ball = sys::OX_JNT_BALL, 4, 3; Slide = sys::OX_JNT_SLIDE, 1, 1; Hinge = sys::OX_JNT_HINGE, 1, 1);
}

// ------------------------------------------------------------------------------------------------ model
/// Compiled model: stands where the reference holds `mjModel` (src/physics.rs:7). Immutable, shareable.
pub struct Model { raw: *mut sys::ox_model }
impl Model {
    pub fn from_xml_string(xml: impl Into<String>) -> Result<Self, Error> {
        let c = CString::new(xml.into()).map_err(|e| Error::Mujoco(e.to_string()))?;
        let mut raw = std::ptr::null_mut();
        check(unsafe { sys::ox_model_from_xml_string(c.as_ptr(), &mut raw) })?;
        Ok(Self { raw })
    }
    pub fn from_xml(path: impl AsRef<std::path::Path>) -> Result<Self, Error> {
        let c = CString::new(path.as_ref().to_str().unwrap()).unwrap();            // same unwrap as src/physics.rs:13
        let mut raw = std::ptr::null_mut();
        check(unsafe { sys::ox_model_from_xml_path(c.as_ptr(), &mut raw) })?;
        Ok(Self { raw })
    }
    /// binary model format (MuJoCo: mj_loadModel / mj_saveModel)
    pub fn load(path: impl AsRef<std::path::Path>) -> Result<Self, Error> {
        let c = CString::new(path.as_ref().to_str().unwrap()).unwrap();
        let mut raw = std::ptr::null_mut();
        check(unsafe { sys::ox_model_load(c.as_ptr(), &mut raw) })?;
        Ok(Self { raw })
    }
    pub fn save(&self, path: impl AsRef<std::path::Path>) -> Result<(), Error> {
        let c = CString::new(path.as_ref().to_str().unwrap()).unwrap();
        check(unsafe { sys::ox_model_save(self.raw, c.as_ptr()) })
    }
    pub fn size(&self, name: &str) -> i32 { let c = CString::new(name).unwrap(); unsafe { sys::ox_model_size(self.raw, c.as_ptr()) } }
    /// a compiled integer table by mjModel field name ("jnt_type", "jnt_qposadr", "actuator_actadr", ...)
    pub fn int_table(&self, name: &str) -> &[i32] {
        let (c, mut p, mut n) = (CString::new(name).unwrap(), std::ptr::null(), 0);
        if unsafe { sys::ox_model_int_table(self.raw, c.as_ptr(), &mut p, &mut n) } != sys::OX_OK || n <= 0 { return &[]; }
        unsafe { std::slice::from_raw_parts(p, n as usize) }
    }
    pub fn real_table(&self, name: &str) -> &[f64] {
        let (c, mut p, mut n) = (CString::new(name).unwrap(), std::ptr::null(), 0);
        if unsafe { sys::ox_model_real_table(self.raw, c.as_ptr(), &mut p, &mut n) } != sys::OX_OK || n <= 0 { return &[]; }
        unsafe { std::slice::from_raw_parts(p, n as usize) }
    }
    pub fn object_id<O: Obj>(&self, name: &str) -> Option<ObjectId<O>> {
        let c = CString::new(name).ok()?;
        let i = unsafe { sys::ox_model_name2id(self.raw, O::TYPE, c.as_ptr()) };
        if i < 0 { None } else { Some(ObjectId::new(i as usize)) }
    }
    pub fn object_name<O: Obj>(&self, id: ObjectId<O>) -> String {
        let p = unsafe { sys::ox_model_id2name(self.raw, O::TYPE, id.index as i32) };
        if p.is_null() { String::new() } else { unsafe { CStr::from_ptr(p).to_string_lossy().into_owned() } }
    }
    /// run-time specialisation ahead of time (needs nvcc, not a GPU): compiles the model's step kernel into the on-disk cache
    pub fn jit_compile(&self, f64_validation: bool) -> Result<String, Error> {
        let mut buf = vec![0 as std::os::raw::c_char; 4096];
        check(unsafe { sys::ox_jit_compile(self.raw, if f64_validation { sys::OX_F64 } else { sys::OX_F32 }, buf.as_mut_ptr(), 4096) })?;
        Ok(unsafe { CStr::from_ptr(buf.as_ptr()).to_string_lossy().into_owned() })
    }
}
impl Drop for Model { fn drop(&mut self) { unsafe { sys::ox_model_free(self.raw) } } }
unsafe impl Send for Model {}
unsafe impl Sync for Model {}   // immutable after construction

// ------------------------------------------------------------------------------------------------ batch
/// Options of `BatchedPhysics::new` (ox_batch_config).
#[derive(Clone, Copy)]
pub struct BatchOptions { pub f64_validation: bool, pub device: i32, pub env_id_offset: i64, pub specialize: i32, pub staged: bool }
impl Default for BatchOptions { fn default() -> Self { Self { f64_validation: false, device: 0, env_id_offset: 0, specialize: 1, staged: false } } }

/// nenv copies of mjData on one GPU (SURVEY 8b). Stands where the reference holds `mjData`.
pub struct BatchedPhysics { raw: *mut sys::ox_batch, nenv: usize, owned: bool }
impl BatchedPhysics {
    pub fn new(model: &Model, nenv: usize, opt: BatchOptions) -> Result<Self, Error> {
        let mut cfg = unsafe { std::mem::zeroed::<sys::ox_batch_config>() };
        unsafe { sys::ox_batch_config_default(&mut cfg) };
        cfg.nenv = nenv as i32; cfg.device = opt.device; cfg.env_id_offset = opt.env_id_offset; cfg.specialize = opt.specialize;
        cfg.precision = if opt.f64_validation { sys::OX_F64 } else { sys::OX_F32 };
        cfg.mode = if opt.staged { sys::OX_MODE_STAGED } else { sys::OX_MODE_FUSED };
        let mut raw = std::ptr::null_mut();
        check(unsafe { sys::ox_batch_create(model.raw, &cfg, &mut raw) })?;
        Ok(Self { raw, nenv, owned: true })
    }
    pub fn nenv(&self) -> usize { self.nenv }
    pub fn kernel_name(&self) -> String { unsafe { CStr::from_ptr(sys::ox_batch_kernel_name(self.raw)).to_string_lossy().into_owned() } }
    pub fn step(&mut self, nsteps: i32) { let _ = unsafe { sys::ox_batch_step(self.raw, nsteps) }; }     // infallible like src/physics.rs:44
    pub fn forward(&mut self) { let _ = unsafe { sys::ox_batch_forward(self.raw) }; }
    /// extension: mj_inverse for every env; the result is the field `OX_F_QFRC_INVERSE` (infallible like `forward`)
    pub fn inverse(&mut self) { let _ = unsafe { sys::ox_batch_inverse(self.raw) }; }
    pub fn reset(&mut self, mask: Option<&[u8]>) { let _ = unsafe { sys::ox_batch_reset(self.raw, mask.map_or(std::ptr::null(), |m| m.as_ptr())) }; }
    pub fn sync(&self) -> Result<(), Error> { check(unsafe { sys::ox_batch_sync(self.raw) }) }
    /// controls in, one step, qpos / qvel out in one call (Action::apply + step + Observation::generate, src/lib.rs:63-66)
    pub fn step_io(&mut self, ctrl: &[f32], qpos: &mut [f32], qvel: &mut [f32]) -> Result<(), Error> {
        check(unsafe { sys::ox_batch_step_io(self.raw, ctrl.as_ptr() as *const _, qpos.as_mut_ptr() as *mut _, qvel.as_mut_ptr() as *mut _, sys::OX_F32, sys::OX_MEM_HOST) })
    }
    pub fn ctrl_philox(&mut self, enable: bool, seed: u64) -> Result<(), Error> { check(unsafe { sys::ox_batch_ctrl_philox(self.raw, enable as i32, seed) }) }
    pub fn field_size(&self, field: i32) -> usize { unsafe { sys::ox_batch_field_size(self.raw, field) }.max(0) as usize }
    /// bulk `[nenv][field_size]` read / write in f64 from host memory
    pub fn get(&self, field: i32, out: &mut [f64]) -> Result<(), Error> {
        check(unsafe { sys::ox_batch_get(self.raw, field, out.as_mut_ptr() as *mut _, sys::OX_F64, sys::OX_MEM_HOST, sys::OX_LAYOUT_ENV_MAJOR) })
    }
    pub fn set(&mut self, field: i32, v: &[f64]) -> Result<(), Error> {
        check(unsafe { sys::ox_batch_set(self.raw, field, v.as_ptr() as *const _, sys::OX_F64, sys::OX_MEM_HOST, sys::OX_LAYOUT_ENV_MAJOR) })
    }
    /// per-env slice; `Ok(None)` = optional feature absent (OX_ABSENT), the reference's `Option::None`
    pub fn get1(&self, field: i32, env: usize, offset: usize, out: &mut [f64]) -> Result<Option<()>, Error> {
        match unsafe { sys::ox_batch_get1(self.raw, field, env as i32, offset as i32, out.len() as i32, out.as_mut_ptr()) } {
            sys::OX_ABSENT => Ok(None), s => check(s).map(Some),
        }
    }
    pub fn set1(&mut self, field: i32, env: usize, offset: usize, v: &[f64]) -> Result<Option<()>, Error> {
        match unsafe { sys::ox_batch_set1(self.raw, field, env as i32, offset as i32, v.len() as i32, v.as_ptr()) } {
            sys::OX_ABSENT => Ok(None), s => check(s).map(Some),
        }
    }
    /// checkpoint / resume: `[nenv][state_size]` records (time, qpos, qvel, act, ctrl, qfrc_applied, xfrc_applied, qacc_warmstart)
    pub fn state_size(&self) -> usize { unsafe { sys::ox_batch_state_size(self.raw) }.max(0) as usize }
    pub fn get_state(&self) -> Result<Vec<f64>, Error> {
        let mut v = vec![0.0; self.nenv * self.state_size()];
        check(unsafe { sys::ox_batch_get_state(self.raw, v.as_mut_ptr() as *mut _, sys::OX_F64, sys::OX_MEM_HOST) })?;
        Ok(v)
    }
    pub fn set_state(&mut self, state: &[f64]) -> Result<(), Error> {
        if state.len() != self.nenv * self.state_size() { return Err(Error::Invalid("set_state: wrong length".into())); }
        check(unsafe { sys::ox_batch_set_state(self.raw, state.as_ptr() as *const _, sys::OX_F64, sys::OX_MEM_HOST) })
    }
    /// number of mj_check* auto-resets per env (the home of `Error::PhysicsDiverged`, src/error.rs:7)
    pub fn check_diverged(&self) -> Result<(), Error> {
        let mut s = [0.0f64; 4];
        check(unsafe { sys::ox_batch_stats(self.raw, s.as_mut_ptr()) })?;
        if s[3] > 0.0 { Err(Error::PhysicsDiverged) } else { Ok(()) }
    }
}
impl Drop for BatchedPhysics { fn drop(&mut self) { if self.owned { unsafe { sys::ox_batch_free(self.raw) } } } }
unsafe impl Send for BatchedPhysics {}

/// One batch per GPU of the box, driven from this process (ox_group_*): envs shard by global env id, one host thread per
/// device issues its launches, and the only exchange is the NCCL all-reduce of the statistics vector (SURVEY 8e).
pub struct PhysicsGroup { raw: *mut sys::ox_group, batches: Vec<BatchedPhysics> }
impl PhysicsGroup {
    pub fn new(model: &Model, nenv_per_device: usize, ndevices: usize, opt: BatchOptions) -> Result<Self, Error> {
        let mut cfg = unsafe { std::mem::zeroed::<sys::ox_batch_config>() };
        unsafe { sys::ox_batch_config_default(&mut cfg) };
        cfg.nenv = nenv_per_device as i32; cfg.env_id_offset = opt.env_id_offset; cfg.specialize = opt.specialize;
        cfg.precision = if opt.f64_validation { sys::OX_F64 } else { sys::OX_F32 };
        let mut raw = std::ptr::null_mut();
        check(unsafe { sys::ox_group_create(model.raw, &cfg, ndevices as i32, std::ptr::null(), &mut raw) })?;
        let batches = (0..ndevices).map(|r| BatchedPhysics { raw: unsafe { sys::ox_group_batch(raw, r as i32) }, nenv: nenv_per_device, owned: false }).collect();
        Ok(Self { raw, batches })
    }
    pub fn size(&self) -> usize { self.batches.len() }
    pub fn batch(&mut self, rank: usize) -> &mut BatchedPhysics { &mut self.batches[rank] }
    pub fn step(&mut self, nsteps: i32) { let _ = unsafe { sys::ox_group_step(self.raw, nsteps) }; }
    pub fn sync(&self) -> Result<(), Error> { check(unsafe { sys::ox_group_sync(self.raw) }) }
    pub fn reset(&mut self) { let _ = unsafe { sys::ox_group_reset(self.raw) }; }
    pub fn ctrl_philox(&mut self, enable: bool, seed: u64) -> Result<(), Error> { check(unsafe { sys::ox_group_ctrl_philox(self.raw, enable as i32, seed) }) }
    /// [sum ncon, sum nefc, sum solver iterations, divergence resets] over every env of every GPU
    pub fn stats(&mut self) -> Result<[f64; 4], Error> { let mut s = [0.0; 4]; check(unsafe { sys::ox_group_stats(self.raw, s.as_mut_ptr()) })?; Ok(s) }
}
impl Drop for PhysicsGroup { fn drop(&mut self) { self.batches.clear(); unsafe { sys::ox_group_free(self.raw) } } }
unsafe impl Send for PhysicsGroup {}

// ------------------------------------------------------------------------------------------------ Physics (src/physics.rs)
/// One environment: the method set, receivers and return types of `oxide_control::physics::Physics`.
/// fp64, generic kernels (every mjData field stays current, which `data()` promises).
pub struct Physics { model: Model, data: BatchedPhysics }

impl Physics {
    fn with_model(model: Model) -> Result<Self, Error> {
        let data = BatchedPhysics::new(&model, 1, BatchOptions { f64_validation: true, specialize: 0, ..Default::default() })?;
        Ok(Self { model, data })
    }
    pub fn from_xml(xml_path: impl AsRef<std::path::Path>) -> Result<Self, Error> { Self::with_model(Model::from_xml(xml_path)?) }       // :12-16
    pub fn from_xml_string(xml_string: impl Into<String>) -> Result<Self, Error> { Self::with_model(Model::from_xml_string(xml_string)?) } // :18-24

    pub fn model(&self) -> &Model { &self.model }                                   // :26-28
    pub fn data(&self) -> &BatchedPhysics { &self.data }                            // :30-32
    pub fn data_mut(&mut self) -> &mut BatchedPhysics { &mut self.data }            // :33-35
    pub fn model_data(&self) -> (&Model, &BatchedPhysics) { (&self.model, &self.data) }                  // :37-39
    pub fn model_datamut(&mut self) -> (&Model, &mut BatchedPhysics) { (&self.model, &mut self.data) }   // :40-42

    pub fn step(&mut self) { self.data.step(1); let _ = self.data.sync(); }         // :44-46  mj_step
    pub fn forward(&mut self) { self.data.forward(); let _ = self.data.sync(); }    // :48-50  mj_forward
    /// extension (no counterpart in the reference): mj_inverse; read `OX_F_QFRC_INVERSE` through `data()`
    pub fn inverse(&mut self) { self.data.inverse(); let _ = self.data.sync(); }
    pub fn reset(&mut self) { self.data.reset(None); let _ = self.data.sync(); }    // :52-54  mj_resetData

    pub fn object_id<O: Obj>(&self, name: &str) -> Option<ObjectId<O>> { self.model.object_id(name) }    // :56-58
    pub fn object_name<O: Obj>(&self, id: ObjectId<O>) -> String { self.model.object_name(id) }          // :60-62
}

pub struct Actuators<'a> { physics: &'a mut Physics }                                // :65-67
impl<'a> Actuators<'a> {
    pub fn set(&mut self, id: ObjectId<obj::Actuator>, control: f64) { self.physics.set_ctrl(id, control); }   // :69-71
}
impl Physics {
    pub fn actuators(&mut self) -> Actuators<'_> { Actuators { physics: self } }    // :74-78
}

impl Physics {
    fn scalar(&self, field: i32, off: usize) -> f64 { let mut v = [0.0]; let _ = self.data.get1(field, 0, off, &mut v); v[0] }
    fn put(&mut self, field: i32, off: usize, v: &[f64]) { let _ = self.data.set1(field, 0, off, v); }
    fn joint_adr<J: Joint>(&self, id: ObjectId<J>) -> (usize, usize) {
        let found = self.model.int_table("jnt_type")[id.index];
        assert!(found == J::MJT, "{:?}", Error::JointTypeNotMatch { expected: J::MJT, found });       // rusty_mujoco panics on a mismatched typed id
        (self.model.int_table("jnt_qposadr")[id.index] as usize, self.model.int_table("jnt_dofadr")[id.index] as usize)
    }
    fn act_adr(&self, id: ObjectId<obj::Actuator>) -> Option<usize> {
        let t = self.model.int_table("actuator_actadr");
        if id.index < t.len() && t[id.index] >= 0 { Some(t[id.index] as usize) } else { None }
    }

    pub fn time(&self) -> f64 { self.scalar(sys::OX_F_TIME, 0) }                                        // :82-84
    pub fn set_time(&mut self, time: f64) { self.put(sys::OX_F_TIME, 0, &[time]); }                      // :85-87

    pub fn ctrl(&self, id: ObjectId<obj::Actuator>) -> f64 { self.scalar(sys::OX_F_CTRL, id.index) }     // :89-91
    pub fn set_ctrl(&mut self, id: ObjectId<obj::Actuator>, value: f64) { self.put(sys::OX_F_CTRL, id.index, &[value]); }   // :92-94

    /// `None` when the actuator is stateless (dyntype none).                                          // :96-98
    pub fn act(&self, id: ObjectId<obj::Actuator>) -> Option<f64> { self.act_adr(id).map(|a| self.scalar(sys::OX_F_ACT, a)) }
    /// Set the actuator activation value. `None` when the actuator is stateless.                      // :99-102
    pub fn set_act(&mut self, id: ObjectId<obj::Actuator>, value: f64) -> Option<()> { let a = self.act_adr(id)?; self.put(sys::OX_F_ACT, a, &[value]); Some(()) }

    pub fn qpos<J: Joint>(&self, id: ObjectId<J>) -> J::Qpos {                                          // :104-106
        let (qa, _) = self.joint_adr(id);
        let mut q = J::Qpos::default();
        let _ = self.data.get1(sys::OX_F_QPOS, 0, qa, q.as_mut());
        q
    }
    pub fn set_qpos<J: Joint>(&mut self, id: ObjectId<J>, qpos: J::Qpos) { let (qa, _) = self.joint_adr(id); self.put(sys::OX_F_QPOS, qa, qpos.as_ref()); }   // :107-109
    pub fn qvel<J: Joint>(&self, id: ObjectId<J>) -> J::Qvel {                                          // :111-113
        let (_, da) = self.joint_adr(id);
        let mut v = J::Qvel::default();
        let _ = self.data.get1(sys::OX_F_QVEL, 0, da, v.as_mut());
        v
    }
    pub fn set_qvel<J: Joint>(&mut self, id: ObjectId<J>, qvel: J::Qvel) { let (_, da) = self.joint_adr(id); self.put(sys::OX_F_QVEL, da, qvel.as_ref()); }   // :114-116

    pub fn qacc_warmstart(&self, id: ObjectId<obj::Dof>) -> f64 { self.scalar(sys::OX_F_QACC_WARMSTART, id.index) }                   // :118-120
    pub fn set_qacc_warmstart(&mut self, id: ObjectId<obj::Dof>, value: f64) { self.put(sys::OX_F_QACC_WARMSTART, id.index, &[value]); } // :121-123

    /// Plugins are outside the supported MJCF subset: no plugin has a state.                          // :125-127
    pub fn plugin_state(&self, _id: ObjectId<obj::Plugin>) -> Option<f64> { None }
    /// Set the plugin state. Returns `None` if the plugin does not have a state.                      // :128-131
    pub fn set_plugin_state(&mut self, _id: ObjectId<obj::Plugin>, _value: f64) -> Option<()> { None }

    pub fn qfrc_applied(&self, id: ObjectId<obj::Dof>) -> f64 { self.scalar(sys::OX_F_QFRC_APPLIED, id.index) }                       // :133-135
    pub fn set_qfrc_applied(&mut self, id: ObjectId<obj::Dof>, value: f64) { self.put(sys::OX_F_QFRC_APPLIED, id.index, &[value]); }  // :136-138

    pub fn xfrc_applied(&self, id: ObjectId<obj::Body>) -> [f64; 6] {                                   // :140-142
        let mut v = [0.0; 6];
        let _ = self.data.get1(sys::OX_F_XFRC_APPLIED, 0, 6 * id.index, &mut v);
        v
    }
    pub fn set_xfrc_applied(&mut self, id: ObjectId<obj::Body>, value: [f64; 6]) { self.put(sys::OX_F_XFRC_APPLIED, 6 * id.index, &value); }   // :143-145

    /// Whether equality constraint `id` (connect / joint) is currently enforced.                                     // :147-149
    pub fn eq_active(&self, id: ObjectId<obj::Equality>) -> bool { self.scalar(sys::OX_F_EQ_ACTIVE, id.index) != 0.0 }
    pub fn set_eq_active(&mut self, id: ObjectId<obj::Equality>, value: bool) { self.put(sys::OX_F_EQ_ACTIVE, id.index, &[if value { 1.0 } else { 0.0 }]); }   // :150-152

    fn mocap_id(&self, id: ObjectId<obj::Body>) -> Option<usize> {
        let t = self.model.int_table("body_mocapid");
        if id.index < t.len() && t[id.index] >= 0 { Some(t[id.index] as usize) } else { None }
    }
    /// `None` when the body is not a mocap body.                                                      // :154-157
    pub fn mocap_pos(&self, id: ObjectId<obj::Body>) -> Option<[f64; 3]> {
        let m = self.mocap_id(id)?;
        let mut v = [0.0; 3];
        let _ = self.data.get1(sys::OX_F_MOCAP_POS, 0, 3 * m, &mut v);
        Some(v)
    }
    /// Set the mocap position. Returns `None` if the body is not a mocap body.                        // :158-161
    pub fn set_mocap_pos(&mut self, id: ObjectId<obj::Body>, pos: [f64; 3]) -> Option<()> { let m = self.mocap_id(id)?; self.put(sys::OX_F_MOCAP_POS, 3 * m, &pos); Some(()) }
    /// `None` when the body is not a mocap body.                                                      // :163-166
    pub fn mocap_quat(&self, id: ObjectId<obj::Body>) -> Option<[f64; 4]> {
        let m = self.mocap_id(id)?;
        let mut v = [0.0; 4];
        let _ = self.data.get1(sys::OX_F_MOCAP_QUAT, 0, 4 * m, &mut v);
        Some(v)
    }
    /// Set the mocap quaternion. Returns `None` if the body is not a mocap body.                      // :167-170
    pub fn set_mocap_quat(&mut self, id: ObjectId<obj::Body>, quat: [f64; 4]) -> Option<()> { let m = self.mocap_id(id)?; self.put(sys::OX_F_MOCAP_QUAT, 4 * m, &quat); Some(()) }
}

// ------------------------------------------------------------------------------------------------ Environment (src/lib.rs)
/// `enum TimeStep<O>` (src/lib.rs:50-60) for every env: `finished[e]` selects `Finish` (no discount) or `Step`.
pub struct BatchedTimeStep<'a> { pub observation: &'a [f32], pub reward: &'a [f32], pub discount: &'a [f32], pub finished: &'a [u8] }
pub struct BatchedEnvironment<'p> {
    raw: *mut sys::ox_env, physics: &'p mut BatchedPhysics, obs_dim: usize,
    obs: Vec<f32>, reward: Vec<f32>, discount: Vec<f32>, finished: Vec<u8>,
}
impl<'p> BatchedEnvironment<'p> {
    /// `Environment::new(physics, task)` (src/lib.rs:33-36); the task is declarative because it runs inside a kernel.
    pub fn new(physics: &'p mut BatchedPhysics, task: &sys::ox_task_spec) -> Result<Self, Error> {
        let mut raw = std::ptr::null_mut();
        check(unsafe { sys::ox_env_create(physics.raw, task, &mut raw) })?;
        let (n, d) = (physics.nenv(), unsafe { sys::ox_env_obs_dim(raw) } as usize);
        Ok(Self { raw, physics, obs_dim: d, obs: vec![0.0; n * d], reward: vec![0.0; n], discount: vec![0.0; n], finished: vec![0; n] })
    }
    pub fn physics(&self) -> &BatchedPhysics { self.physics }                                            // src/lib.rs:42-44
    pub fn physics_mut(&mut self) -> &mut BatchedPhysics { self.physics }                               // src/lib.rs:45-47
    pub fn obs_dim(&self) -> usize { self.obs_dim }
    /// `Environment::reset` (src/lib.rs:63-66)
    pub fn reset(&mut self) -> Result<&[f32], Error> {
        check(unsafe { sys::ox_env_reset(self.raw, self.obs.as_mut_ptr() as *mut _, sys::OX_F32, sys::OX_MEM_HOST) })?;
        Ok(&self.obs)
    }
    /// `Environment::step` (src/lib.rs:68-87): `action` is `[nenv][nu]`.
    pub fn step(&mut self, action: &[f32]) -> Result<BatchedTimeStep<'_>, Error> {
        check(unsafe { sys::ox_env_step(self.raw, action.as_ptr() as *const _, self.obs.as_mut_ptr() as *mut _, self.reward.as_mut_ptr() as *mut _,
                                        self.discount.as_mut_ptr() as *mut _, self.finished.as_mut_ptr(), sys::OX_F32, sys::OX_MEM_HOST) })?;
        Ok(BatchedTimeStep { observation: &self.obs, reward: &self.reward, discount: &self.discount, finished: &self.finished })
    }
}
impl Drop for BatchedEnvironment<'_> { fn drop(&mut self) { unsafe { sys::ox_env_free(self.raw) } } }
