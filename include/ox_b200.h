/*
 * ox_b200.h — C ABI of libox_b200.so: the B200-native batched `mj_step` path
 * behind oxide_control's `Physics` API.
 *
 * Every entry point below replaces one call the reference makes into
 * `rusty_mujoco` (reference = /root/reference, cited as src/...:line):
 *
 *   ox_model_from_xml_path      <- Physics::from_xml        src/physics.rs:12-16  (mj_loadXML + mj_makeData)
 *   ox_model_from_xml_string    <- Physics::from_xml_string src/physics.rs:18-24  (mj_parseXMLString + mj_compile + mjs_getError)
 *   ox_batch_create             <- mj_makeData              src/physics.rs:14,22  (batched: nenv copies of mjData, SoA on device)
 *   ox_batch_step               <- Physics::step            src/physics.rs:44-46  (mj_step)      ** the hot path **
 *   ox_batch_forward            <- Physics::forward         src/physics.rs:48-50  (mj_forward)
 *   ox_batch_inverse            <- (extension)              mj_inverse, batched
 *   ox_batch_reset              <- Physics::reset           src/physics.rs:52-54  (mj_resetData, masked)
 *   ox_model_name2id/id2name    <- object_id / object_name  src/physics.rs:56-62
 *   ox_batch_set1/get1, set/get <- Actuators::set, time/ctrl/act/qpos/qvel/qacc_warmstart/qfrc_applied/
 *                                  xfrc_applied getters+setters src/physics.rs:65-171, and data() src/physics.rs:30
 *
 * Conventions (SURVEY.md §8b):
 *   - every function returns ox_status (0 = OK) unless it returns a size or a pointer;
 *     ox_last_error_message() returns a thread-local NUL-terminated string owned by the library.
 *   - "feature absent" (stateless actuator, non-mocap body, no plugin) is OX_ABSENT, which the
 *     Rust wrapper maps to Option::None exactly as src/physics.rs:96-102,125-131,154-170 do.
 *   - parse errors map to Error::Mujoco, compile errors to Error::Mjs(msg) (src/error.rs:4-6).
 *   - divergence (NaN / |x| > mjMAXVAL) is not an error: reference step() is infallible
 *     (src/physics.rs:44); the env is auto-reset like mj_step does and a per-env flag is raised
 *     (home of Error::PhysicsDiverged, src/error.rs:7).
 *   - nothing throws or aborts across this boundary; no torch/STL types in any signature.
 *   - there is NO CPU fallback: without a CUDA device ox_batch_create fails with OX_ERR_CUDA.
 */
#ifndef OX_B200_H
#define OX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define OX_API
#else
#define OX_API __attribute__((visibility("default")))
#endif

typedef int32_t ox_status;
enum {
  OX_OK = 0,
  OX_ERR_PARSE = 1,     /* malformed XML / unknown element or attribute  -> Error::Mujoco */
  OX_ERR_COMPILE = 2,   /* well-formed but un-compilable model           -> Error::Mjs    */
  OX_ERR_CUDA = 3,      /* no device / allocation / launch failure                         */
  OX_ERR_INVALID = 4,   /* bad argument (null handle, index out of range, wrong field)     */
  OX_ABSENT = 5,        /* optional feature absent                       -> Option::None   */
  OX_ERR_IO = 6         /* file could not be read                        -> Error::Mujoco */
};

/* mjtJoint / mjtGeom / mjtObj numeric values of MuJoCo 3.3.2 (rusty_mujoco::bindgen). */
enum { OX_JNT_FREE = 0, OX_JNT_BALL = 1, OX_JNT_SLIDE = 2, OX_JNT_HINGE = 3 };
enum { OX_GEOM_PLANE = 0, OX_GEOM_HFIELD = 1, OX_GEOM_SPHERE = 2, OX_GEOM_CAPSULE = 3,
       OX_GEOM_ELLIPSOID = 4, OX_GEOM_CYLINDER = 5, OX_GEOM_BOX = 6, OX_GEOM_MESH = 7 };
enum { OX_OBJ_UNKNOWN = 0, OX_OBJ_BODY = 1, OX_OBJ_XBODY = 2, OX_OBJ_JOINT = 3, OX_OBJ_TENDON = 18, OX_OBJ_DOF = 4,
       OX_OBJ_GEOM = 5, OX_OBJ_SITE = 6, OX_OBJ_EQUALITY = 17, OX_OBJ_ACTUATOR = 19,
       OX_OBJ_SENSOR = 20, OX_OBJ_PLUGIN = 25 };
enum { OX_INT_EULER = 0, OX_INT_RK4 = 1, OX_INT_IMPLICIT = 2 /* refused by the compiler */, OX_INT_IMPLICITFAST = 3 };
/* mjtDyn subset: activation dynamics of stateful actuators (act, src/physics.rs:96-102) */
enum { OX_DYN_NONE = 0, OX_DYN_INTEGRATOR = 1, OX_DYN_FILTER = 2, OX_DYN_FILTEREXACT = 3 };
/* mjtEq subset: equality constraints */
enum { OX_EQ_CONNECT = 0, OX_EQ_WELD = 1, OX_EQ_JOINT = 2 };
enum { OX_SOL_PGS = 0, OX_SOL_CG = 1, OX_SOL_NEWTON = 2 };
enum { OX_CONE_PYRAMIDAL = 0, OX_CONE_ELLIPTIC = 1 };
enum { OX_GAIN_FIXED = 0, OX_GAIN_AFFINE = 1 };
/* mjtTrn subset: what an actuator pulls on (actuator_trnid is a joint id or a tendon id) */
enum { OX_TRN_JOINT = 0, OX_TRN_TENDON = 3 };
/* tendon kinds: fixed = linear combination of joint coordinates (wrap_objid = joints, wrap_prm = coefficients);
 * spatial = straight segments through sites (wrap_objid = sites; wrapping geoms and pulleys are refused) */
enum { OX_TEN_FIXED = 0, OX_TEN_SPATIAL = 1 };
enum { OX_BIAS_NONE = 0, OX_BIAS_AFFINE = 1 };
/* mjtDisableBit subset */
enum { OX_DSBL_CONSTRAINT = 1 << 0, OX_DSBL_LIMIT = 1 << 3, OX_DSBL_CONTACT = 1 << 4,
       OX_DSBL_PASSIVE = 1 << 5, OX_DSBL_GRAVITY = 1 << 6, OX_DSBL_CLAMPCTRL = 1 << 7,
       OX_DSBL_WARMSTART = 1 << 8, OX_DSBL_FILTERPARENT = 1 << 9, OX_DSBL_ACTUATION = 1 << 10,
       OX_DSBL_REFSAFE = 1 << 11, OX_DSBL_EULERDAMP = 1 << 13, OX_DSBL_EQUALITY = 1 << 1, OX_DSBL_FRICTIONLOSS = 1 << 2 };
/* mjtSensor subset */
enum { OX_SENS_TOUCH = 0, OX_SENS_ACCELEROMETER = 1, OX_SENS_VELOCIMETER = 2, OX_SENS_GYRO = 3, OX_SENS_FORCE = 4, OX_SENS_TORQUE = 5,
       OX_SENS_JOINTPOS = 8, OX_SENS_JOINTVEL = 9, OX_SENS_TENDONPOS = 11, OX_SENS_TENDONVEL = 12, OX_SENS_ACTUATORPOS = 13, OX_SENS_ACTUATORVEL = 14,
       OX_SENS_ACTUATORFRC = 15, OX_SENS_JOINTACTFRC = 16, OX_SENS_BALLQUAT = 17, OX_SENS_BALLANGVEL = 18,
       OX_SENS_FRAMEPOS = 25, OX_SENS_FRAMEQUAT = 26, OX_SENS_FRAMEXAXIS = 27, OX_SENS_FRAMEYAXIS = 28, OX_SENS_FRAMEZAXIS = 29,
       OX_SENS_FRAMELINVEL = 30, OX_SENS_FRAMEANGVEL = 31, OX_SENS_FRAMELINACC = 32, OX_SENS_FRAMEANGACC = 33, OX_SENS_SUBTREECOM = 34,
       OX_SENS_SUBTREELINVEL = 35, OX_SENS_CLOCK = 45 };

#define OX_MAXVAL 1e10  /* mjMAXVAL re-exported at src/physics.rs:2 */
#define OX_MINVAL 1e-15 /* mjMINVAL re-exported at src/physics.rs:2 */
#define OX_MINIMP 0.0001
#define OX_MAXIMP 0.9999

/* ---- compiled-model constant tables (host, fp64; mirror of the mjModel fields the path reads) ----
 * X(name, count_field, width): array of count_field*width entries.                                  */
#define OX_MODEL_INT_TABLES(X)                                                                      \
  X(body_parentid, nbody, 1) X(body_rootid, nbody, 1) X(body_weldid, nbody, 1)                     \
  X(body_jntadr, nbody, 1) X(body_jntnum, nbody, 1) X(body_dofadr, nbody, 1) X(body_dofnum, nbody, 1) \
  X(body_mocapid, nbody, 1)                                                                         \
  X(eq_type, neq, 1) X(eq_obj1id, neq, 1) X(eq_obj2id, neq, 1) X(eq_active0, neq, 1)                \
  X(tendon_adr, ntendon, 1) X(tendon_num, ntendon, 1) X(tendon_limited, ntendon, 1) X(tendon_type, ntendon, 1) X(wrap_objid, nwrap, 1) \
  X(jnt_type, njnt, 1) X(jnt_qposadr, njnt, 1) X(jnt_dofadr, njnt, 1) X(jnt_bodyid, njnt, 1)       \
  X(jnt_limited, njnt, 1)                                                                           \
  X(dof_bodyid, nv, 1) X(dof_jntid, nv, 1) X(dof_parentid, nv, 1) X(dof_Madr, nv, 1) X(dof_depth, nv, 1) X(dof_Mdense, nvv, 1)               \
  X(geom_type, ngeom, 1) X(geom_bodyid, ngeom, 1) X(geom_contype, ngeom, 1)                        \
  X(geom_conaffinity, ngeom, 1) X(geom_condim, ngeom, 1) X(geom_priority, ngeom, 1)                \
  X(site_bodyid, nsite, 1) X(site_type, nsite, 1)                                                   \
  X(pair_geom1, npair, 1) X(pair_geom2, npair, 1) X(pair_dim, npair, 1) X(pair_maxcon, npair, 1) X(pair_conadr, npair, 1)   \
  X(actuator_trnid, nu, 1) X(actuator_trntype, nu, 1) X(actuator_gaintype, nu, 1) X(actuator_biastype, nu, 1)                 \
  X(actuator_ctrllimited, nu, 1) X(actuator_forcelimited, nu, 1)                                    \
  X(actuator_dyntype, nu, 1) X(actuator_actadr, nu, 1) X(actuator_actlimited, nu, 1)                \
  X(sensor_type, nsensor, 1) X(sensor_objtype, nsensor, 1) X(sensor_objid, nsensor, 1)             \
  X(sensor_adr, nsensor, 1) X(sensor_dim, nsensor, 1)

#define OX_MODEL_REAL_TABLES(X)                                                                     \
  X(qpos0, nq, 1) X(qpos_spring, nq, 1)                                                             \
  X(body_pos, nbody, 3) X(body_quat, nbody, 4) X(body_ipos, nbody, 3) X(body_iquat, nbody, 4)      \
  X(body_mass, nbody, 1) X(body_inertia, nbody, 3) X(body_subtreemass, nbody, 1)                   \
  X(body_invweight0, nbody, 2) X(body_fluid, nfluid, 11) X(body_gravcomp, ngravcomp, 1)                                          \
  X(jnt_pos, njnt, 3) X(jnt_axis, njnt, 3) X(jnt_stiffness, njnt, 1) X(jnt_range, njnt, 2)         \
  X(jnt_margin, njnt, 1) X(jnt_solref, njnt, 2) X(jnt_solimp, njnt, 5)                             \
  X(dof_armature, nv, 1) X(dof_damping, nv, 1) X(dof_invweight0, nv, 1)                            \
  X(dof_frictionloss, nv, 1) X(dof_solref_fri, nv, 2) X(dof_solimp_fri, nv, 5)                     \
  X(geom_size, ngeom, 3) X(geom_pos, ngeom, 3) X(geom_quat, ngeom, 4) X(geom_friction, ngeom, 3)   \
  X(geom_solmix, ngeom, 1) X(geom_solref, ngeom, 2) X(geom_solimp, ngeom, 5)                       \
  X(geom_margin, ngeom, 1) X(geom_gap, ngeom, 1)                                                    \
  X(site_pos, nsite, 3) X(site_quat, nsite, 4) X(site_size, nsite, 3)                               \
  X(pair_friction, npair, 5) X(pair_solref, npair, 2) X(pair_solimp, npair, 5)                     \
  X(pair_margin, npair, 1) X(pair_gap, npair, 1)                                                    \
  X(actuator_gear, nu, 1) X(actuator_gainprm, nu, 3) X(actuator_biasprm, nu, 3)                    \
  X(actuator_ctrlrange, nu, 2) X(actuator_forcerange, nu, 2)                                        \
  X(actuator_dynprm, nu, 3) X(actuator_actrange, nu, 2)                                             \
  X(eq_solref, neq, 2) X(eq_solimp, neq, 5) X(eq_data, neq, 11)                                     \
  X(wrap_prm, nwrap, 1) X(tendon_range, ntendon, 2) X(tendon_margin, ntendon, 1)                    \
  X(tendon_solref_lim, ntendon, 2) X(tendon_solimp_lim, ntendon, 5)                                 \
  X(tendon_stiffness, ntendon, 1) X(tendon_damping, ntendon, 1) X(tendon_lengthspring, ntendon, 2)  \
  X(tendon_length0, ntendon, 1) X(tendon_invweight0, ntendon, 1)

typedef struct ox_model_tables {
  /* sizes */
  int32_t nq, nv, nu, na, nbody, njnt, ngeom, nsite, nM, npair, nsensor, nsensordata;
  int32_t nvv;      /* nv*nv: size of dof_Mdense (index into qM of M(i,j), -1 where M is structurally zero) */
  int32_t nconmax;  /* sum of pair_maxcon: capacity of the per-env contact list         */
  int32_t nefcmax;  /* equality rows + 2*nlimited + sum of contact rows: capacity of the per-env efc list */
  int32_t nmocap;   /* mocap bodies (mocap_pos / mocap_quat, src/physics.rs:154-170) */
  int32_t neq;      /* equality constraints (eq_active, src/physics.rs:147-152) */
  int32_t ntendon, nwrap; /* fixed tendons (linear combinations of scalar joint coordinates) and their joint entries */
  /* mjOption subset */
  int32_t integrator, solver, cone, iterations, ls_iterations, disableflags;
  int32_t noslip_iterations;   /* noslip post-pass of the friction dimensions (0 = off, MuJoCo's default) */
  int32_t nfloss;              /* dofs with frictionloss > 0: one Huber-cost row each, after the equality rows */
  double timestep, gravity[3], tolerance, ls_tolerance, impratio, noslip_tolerance;
  /* medium (mjOption density / viscosity / wind): inertia-box fluid forces of mj_passive. nfluid = nbody when density or
   * viscosity is positive, else 0; body_fluid[11] per body = viscous torque and force coefficients (pi d^3 mu, 3 pi d mu),
   * quadratic drag coefficients of the three box faces (force, then torque), and the wind velocity */
  int32_t nfluid;
  int32_t ngravcomp;           /* nbody when any body has gravcomp != 0 (mj_passive adds -gravity * mass * gravcomp at its com), else 0 */
  double density, viscosity, wind[3];
  /* mjStatistic subset */
  double meaninertia;
#define OX_X(name, n, w) const int32_t* name;
  OX_MODEL_INT_TABLES(OX_X)
#undef OX_X
#define OX_X(name, n, w) const double* name;
  OX_MODEL_REAL_TABLES(OX_X)
#undef OX_X
} ox_model_tables;

typedef struct ox_model ox_model; /* immutable after construction; thread-safe to share */
typedef struct ox_batch ox_batch; /* nenv copies of mjData, SoA on one device, one stream */

/* ---- errors ---- */
OX_API const char* ox_last_error_message(void);
OX_API const char* ox_version(void);

/* ---- model (setup side of the boundary) ---- */
OX_API ox_status ox_model_from_xml_string(const char* xml, ox_model** out);
OX_API ox_status ox_model_from_xml_path(const char* path, ox_model** out);
OX_API void ox_model_free(ox_model* m);
/* Binary model format (SURVEY 8f N4; MuJoCo's counterpart is mj_saveModel / mj_loadModel on an .mjb file, which the reference
 * reaches through rusty_mujoco's mjModel but does not wrap): the compiled tables, options and names in one little-endian
 * blob, "OXB2MDL" magic + format version + table-layout fingerprint + FNV-1a checksum. A model loaded from it is
 * bit-identical to the one compiled from the XML (same model hash, so the same specialised kernel).
 * ox_model_serialize writes at most `capacity` bytes into `buf` and returns the size needed (call with NULL / 0 to size). */
OX_API int64_t ox_model_serialize(const ox_model* m, void* buf, int64_t capacity);
OX_API ox_status ox_model_deserialize(const void* buf, int64_t size, ox_model** out);
OX_API ox_status ox_model_save(const ox_model* m, const char* path);
OX_API ox_status ox_model_load(const char* path, ox_model** out);
OX_API const ox_model_tables* ox_model_get_tables(const ox_model* m);
/* name-addressed table access for bindings that cannot see the struct (ctypes, Rust sys crate) */
OX_API ox_status ox_model_int_table(const ox_model* m, const char* name, const int32_t** ptr, int32_t* count);
OX_API ox_status ox_model_real_table(const ox_model* m, const char* name, const double** ptr, int32_t* count);
OX_API int32_t ox_model_size(const ox_model* m, const char* name); /* "nq","nv",...; -1 if unknown */
OX_API int32_t ox_model_name2id(const ox_model* m, int32_t objtype, const char* name); /* -1 = None */
OX_API const char* ox_model_id2name(const ox_model* m, int32_t objtype, int32_t id);   /* "" if unnamed, NULL if bad id */

/* ---- batch ---- */
enum { OX_F32 = 0, OX_F64 = 1 };
enum { OX_MEM_HOST = 0, OX_MEM_DEVICE = 1 };
enum { OX_LAYOUT_ENV_MAJOR = 0 /* [env][elem] (AoS, what a Vec<mjData> would give) */,
       OX_LAYOUT_ELEM_MAJOR = 1 /* [elem][env] (native SoA) */ };
enum { OX_MODE_FUSED = 0 /* one launch per step, one thread per env */, OX_MODE_STAGED = 1 /* one launch per mj_step stage */,
       OX_MODE_COOP = 2 /* one launch per step, one lane group (16 / 32 lanes) per env, intermediates in shared memory:
                           any model with nv <= 32, Newton solver, Euler / implicitfast (csrc/ox_coop.cu) */ };

typedef struct ox_batch_config {
  int32_t nenv;
  int32_t device;        /* CUDA ordinal */
  int32_t precision;     /* OX_F32 throughput mode | OX_F64 validation mode */
  int32_t mode;          /* OX_MODE_FUSED | OX_MODE_STAGED | OX_MODE_COOP */
  int32_t iterations;    /* solver iteration cap; 0 = model's <option iterations> */
  int32_t ls_iterations; /* line-search iteration cap; 0 = model's */
  int32_t use_graph;     /* capture the per-step launch sequence in a CUDA graph */
  int32_t block_threads; /* 0 = default */
  int64_t env_id_offset; /* global env id of env 0 (multi-GPU sharding; keys the Philox control stream) */
  double tolerance;      /* <0 = model's, floored at 8*eps of `precision` (1e-6 in fp32; no effect in fp64) */
  int32_t specialize;    /* fused mode. 0: generic kernels (every mjData field stays current). 1 (default): the model-specialised
                            step kernel - compiled into the library for the spec_models, otherwise compiled at run time
                            (nvcc, cached on disk) when nenv >= 1024; generic kernel if neither is available.
                            2: always specialise at run time if needed; ox_batch_create fails if that is impossible. */
  int32_t lanes_per_warp; /* active envs per warp, 1..32; 0 = auto (thin warps while the batch cannot fill every SM scheduler) */
  int32_t coop_solver;   /* staged mode: warp-per-env Newton solver; -1 auto (on when eligible and nv > 12), 0 off, 1 on */
  int32_t reserved_;
} ox_batch_config;

OX_API void ox_batch_config_default(ox_batch_config* cfg);
OX_API ox_status ox_batch_create(const ox_model* m, const ox_batch_config* cfg, ox_batch** out);
OX_API void ox_batch_free(ox_batch* b);
OX_API int32_t ox_batch_nenv(const ox_batch* b);
OX_API void* ox_batch_stream(const ox_batch* b); /* cudaStream_t */

/* step family: asynchronous on the batch's stream */
OX_API ox_status ox_batch_step(ox_batch* b, int32_t nsteps);
OX_API ox_status ox_batch_forward(ox_batch* b);
/* Inverse dynamics (mj_inverse, continuous time) of every env, one launch on the batch's stream. From qpos, qvel, qacc,
 * ctrl, act, mocap, eq_active and the applied forces it writes
 *   qfrc_inverse = M(qpos) qacc + qfrc_bias - qfrc_passive - qfrc_constraint,   qfrc_constraint = J' efc_force,
 * where efc_force is the soft-constraint force at J qacc - aref (mj_invConstraint): the same function for PGS, CG and Newton
 * models, noslip not applied. It also writes every position- and velocity-dependent field ox_batch_forward writes (kinematics,
 * qM / qLD, bias, passive, tendons, contacts, constraint rows with the inverse efc_force and qfrc_constraint), the actuation
 * fields actuator_force / qfrc_actuator / act_dot, qfrc_smooth / qacc_smooth (which mj_inverse leaves stale), and sensordata
 * computed with the given qacc. Afterwards every derived field is readable. It never writes qpos, qvel, qacc,
 * qacc_warmstart, ctrl, act, time, the applied forces, mocap, eq_active, solver_niter, diverged, the statistics or the Philox
 * step counter; there is no divergence check and no auto-reset. */
OX_API ox_status ox_batch_inverse(ox_batch* b);
/* Action::apply + Physics::step + Observation::generate of Environment::step (reference src/lib.rs:63-66) in ONE call for the
 * whole batch: ctrl[nenv][nu] in (NULL = keep), one mj_step, qpos[nenv][nq] / qvel[nenv][nv] out (either may be NULL); env-major
 * `dtype` buffers in `mem`. With a model-specialised kernel and device memory or pinned host memory the step kernel reads and
 * writes the buffers itself (no extra launches, PCIe traffic overlaps the step); otherwise it is ox_batch_set + ox_batch_step +
 * ox_batch_get_many. Host outputs are complete on return. */
OX_API ox_status ox_batch_step_io(ox_batch* b, const void* ctrl, void* qpos, void* qvel, int32_t dtype, int32_t mem);
OX_API ox_status ox_batch_reset(ox_batch* b, const uint8_t* host_mask_or_null);
OX_API ox_status ox_batch_sync(ox_batch* b);

/* benchmark control source: fresh ctrl ~ U(-1,1) every step from Philox4x32-10 keyed on
 * (seed, global env id, step, actuator) generated on device. enable=0 returns to user ctrl. */
OX_API ox_status ox_batch_ctrl_philox(ox_batch* b, int32_t enable, uint64_t seed);
OX_API ox_status ox_batch_set_step_counter(ox_batch* b, int64_t step);
/* amplitude of the Philox control stream: ctrl = scale * U(-1,1) (default 1). Use a power of two to keep the CPU fp64 and
 * GPU fp32 control values bit-identical. 0.125 lets the humanoid settle into resting contact (ncon ~ 10) instead of thrashing. */
OX_API ox_status ox_batch_ctrl_philox_scale(ox_batch* b, double scale);

/* field ids for bulk / per-env access */
enum {
  OX_F_QPOS = 0, OX_F_QVEL, OX_F_CTRL, OX_F_QFRC_APPLIED, OX_F_XFRC_APPLIED, OX_F_QACC_WARMSTART,
  OX_F_TIME, OX_F_ACT,
  OX_F_QACC, OX_F_SENSORDATA, OX_F_XPOS, OX_F_XQUAT, OX_F_XMAT, OX_F_XIPOS, OX_F_XIMAT,
  OX_F_XANCHOR, OX_F_XAXIS, OX_F_GEOM_XPOS, OX_F_GEOM_XMAT, OX_F_SITE_XPOS, OX_F_SITE_XMAT,
  OX_F_SUBTREE_COM, OX_F_CINERT, OX_F_CDOF, OX_F_QM, OX_F_QLD, OX_F_QLDIAGINV, OX_F_CVEL,
  OX_F_CDOF_DOT, OX_F_QFRC_BIAS, OX_F_QFRC_PASSIVE, OX_F_ACTUATOR_FORCE, OX_F_QFRC_ACTUATOR,
  OX_F_QFRC_SMOOTH, OX_F_QACC_SMOOTH, OX_F_QFRC_CONSTRAINT,
  OX_F_CON_DIST, OX_F_CON_POS, OX_F_CON_FRAME,
  OX_F_EFC_J, OX_F_EFC_POS, OX_F_EFC_MARGIN, OX_F_EFC_D, OX_F_EFC_AREF, OX_F_EFC_FORCE,
  OX_F_ACT_DOT, OX_F_MOCAP_POS, OX_F_MOCAP_QUAT, OX_F_EQ_ACTIVE, OX_F_TEN_LENGTH, OX_F_TEN_J,
  OX_F_QFRC_INVERSE, /* written by ox_batch_inverse only; zeros until its first call */
  OX_F_COUNT_REAL,
  /* int32 fields */
  OX_F_NCON = 100, OX_F_NEFC, OX_F_SOLVER_NITER, OX_F_DIVERGED, OX_F_CON_PAIR
};
OX_API int32_t ox_batch_field_size(const ox_batch* b, int32_t field); /* elements per env; -1 bad field */

/* bulk I/O: `buf` holds nenv*field_size elements of `dtype` (OX_F32/OX_F64; int fields are int32)
 * in `layout`, living in `mem`. Stream-ordered; host copies complete before return. */
OX_API ox_status ox_batch_get(ox_batch* b, int32_t field, void* buf, int32_t dtype, int32_t mem, int32_t layout);
OX_API ox_status ox_batch_set(ox_batch* b, int32_t field, const void* buf, int32_t dtype, int32_t mem, int32_t layout);
/* several fields in one call: one stream synchronisation for all the device->host copies (the observation read of an
 * RL step: qpos + qvel [+ sensordata]). bufs[i] receives field fields[i]; same dtype / mem / layout for all. */
OX_API ox_status ox_batch_get_many(ox_batch* b, int32_t nfields, const int32_t* fields, void* const* bufs, int32_t dtype, int32_t mem, int32_t layout);
/* per-env slices, always fp64 at this boundary (reference types are f64 / [f64;N]) */
OX_API ox_status ox_batch_get1(ox_batch* b, int32_t field, int32_t env, int32_t offset, int32_t count, double* out);
OX_API ox_status ox_batch_set1(ox_batch* b, int32_t field, int32_t env, int32_t offset, int32_t count, const double* in);
OX_API ox_status ox_batch_get1_int(ox_batch* b, int32_t field, int32_t env, int32_t offset, int32_t count, int32_t* out);

/* Checkpoint / resume (SURVEY 5; the reference keeps no such API - its state is whatever the user copies out through the
 * getters of src/physics.rs:82-145, which is exactly this tuple): one record per env, env-major,
 *   [ time, qpos(nq), qvel(nv), act(na), ctrl(nu), qfrc_applied(nv), xfrc_applied(6 nbody), qacc_warmstart(nv),
 *     mocap_pos(3 nmocap), mocap_quat(4 nmocap), eq_active(neq) ]
 * = ox_batch_state_size() elements of `dtype`. Restoring a record and the Philox step counter reproduces the trajectory
 * bit for bit in the same precision (qacc_warmstart seeds the solver). */
OX_API int32_t ox_batch_state_size(const ox_batch* b);
OX_API ox_status ox_batch_get_state(ox_batch* b, void* buf, int32_t dtype, int32_t mem);
OX_API ox_status ox_batch_set_state(ox_batch* b, const void* buf, int32_t dtype, int32_t mem);
OX_API int64_t ox_batch_get_step_counter(const ox_batch* b);

/* run statistics accumulated on device since the last call (mean ncon, nefc, solver iterations,
 * number of divergence auto-resets); out[4]. */
OX_API ox_status ox_batch_stats(ox_batch* b, double* out4);
/* number of kernel launches issued by this batch so far (bench.py "gpu_launches") */
OX_API int64_t ox_batch_launch_count(const ox_batch* b);
/* which step kernel this batch launches: a spec name ("cheetah"), or the generic kernel */
OX_API const char* ox_batch_kernel_name(const ox_batch* b);
/* "" or the reason a batch that asked for a specialised kernel runs the generic one (no nvcc, compile error, ...) */
OX_API const char* ox_batch_jit_note(const ox_batch* b);
/* Run-time specialisation without a batch (and without a GPU): compile the model's step kernel with nvcc into the on-disk
 * cache ($OX_B200_CACHE_DIR, default ~/.cache/ox_b200) or find it there; the cubin path is copied into path_out. A later
 * ox_batch_create for the same model and precision then loads it from the cache. OX_B200_JIT=0 disables the mechanism. */
OX_API ox_status ox_jit_compile(const ox_model* m, int32_t precision, char* path_out, int32_t path_cap);
/* model-specialised kernels compiled into the library (every .xml under oxide_control_b200/spec_models at build time) */
OX_API int32_t ox_spec_count(void);
OX_API const char* ox_spec_name(int32_t i);
/* per-stage device time of one staged forward+integrate (ms), for profiles/: names via ox_stage_name */
OX_API ox_status ox_batch_stage_times(ox_batch* b, int32_t reps, double* out_ms, int32_t* nstage);
OX_API const char* ox_stage_name(int32_t i);

/* ---------------------------------------------------------------------------------------------
 * N1 (SURVEY 8f): batched Environment / Task — the direct caller of the step.
 * Mirrors reference src/lib.rs:8-26 (traits Task / Observation / Action) and :50-88 (Environment::reset / step,
 * enum TimeStep) for a whole batch, evaluated ON DEVICE so that an RL loop crosses PCIe once per step in each
 * direction (actions in; observation, reward, discount, finished out). The reference's user-written trait bodies
 * become a declarative task description, because user code cannot run inside the kernel:
 *   Observation::generate        -> concatenation of field slices                         (ox_obs_segment)
 *   Task::get_reward             -> bias + sum_k weight_k * f_k(field element)            (ox_reward_term)
 *   Task::should_finish_episode  -> any element outside [lo, hi], or time >= time_limit   (ox_finish_cond)
 *   Task::discount               -> constant
 *   Task::init_episode           -> mj_resetData, qpos0 + U(-a,a) on hinge/slide coordinates, qvel = U(-b,b);
 *                                   Philox4x32-10 keyed on (seed; global env id, episode index, word)
 *   Action::apply                -> ctrl[env][:] = action[env][:]  (Actuators::set for every actuator)
 * ------------------------------------------------------------------------------------------- */
typedef struct ox_env ox_env;
typedef struct ox_obs_segment { int32_t field, first, count; } ox_obs_segment;  /* real fields only */
enum { OX_REWARD_LINEAR = 0 /* w*x */, OX_REWARD_SQUARE = 1 /* w*x^2 */, OX_REWARD_ABS = 2 /* w*|x| */ };
typedef struct ox_reward_term { int32_t field, index, kind, reserved_; double weight; } ox_reward_term;
typedef struct ox_finish_cond { int32_t field, index; double lo, hi; } ox_finish_cond; /* finish if x < lo or x > hi */
typedef struct ox_task_spec {
  int32_t nobs;     const ox_obs_segment* obs;
  int32_t nreward;  const ox_reward_term* reward;
  int32_t nfinish;  const ox_finish_cond* finish;
  double reward_bias;
  double time_limit;       /* <= 0: none; otherwise finish once time >= time_limit - timestep/2 */
  double discount;         /* Task::discount, src/lib.rs:12 */
  double init_qpos_noise;  /* Task::init_episode, src/lib.rs:13 */
  double init_qvel_noise;
  uint64_t seed;
  int32_t frame_skip;      /* mj_steps per Environment::step (>= 1; the reference does exactly 1, src/lib.rs:65) */
  int32_t auto_reset;      /* 1: a finished env is re-initialised (init_episode) inside the same call, after its terminal
                              observation has been written, so the next step starts its next episode */
} ox_task_spec;

OX_API void ox_task_spec_default(ox_task_spec* spec);
/* Environment::new(physics, task), src/lib.rs:33-36. The env borrows the batch (which must outlive it). */
OX_API ox_status ox_env_create(ox_batch* b, const ox_task_spec* spec, ox_env** out);
OX_API void ox_env_free(ox_env* e);
OX_API int32_t ox_env_obs_dim(const ox_env* e);
/* Environment::reset, src/lib.rs:58-61: init_episode on every env, mj_forward (so derived fields / sensordata are
 * fresh for the first observation), then Observation::generate -> obs[nenv][obs_dim] (env-major, `dtype`, in `mem`). */
OX_API ox_status ox_env_reset(ox_env* e, void* obs, int32_t dtype, int32_t mem);
/* Environment::step, src/lib.rs:63-87: apply action[nenv][nu] (NULL = leave ctrl alone, e.g. the Philox stream),
 * frame_skip x mj_step, observation, reward, finish test. TimeStep::Step{observation,reward,discount} /
 * TimeStep::Finish{observation,reward} come back as arrays: obs[nenv][obs_dim], reward[nenv], discount[nenv]
 * (0 for a Finish), finished[nenv] (uint8). Any output pointer may be NULL. All buffers live in `mem`;
 * host buffers are complete on return. An env that MuJoCo's mj_check* auto-reset during the step also finishes. */
OX_API ox_status ox_env_step(ox_env* e, const void* action, void* obs, void* reward, void* discount, uint8_t* finished,
                             int32_t dtype, int32_t mem);
/* episode bookkeeping since creation: out[0] = finished episodes, out[1] = sum of their returns,
 * out[2] = sum of their lengths (env steps) */
OX_API ox_status ox_env_stats(ox_env* e, double* out3);

/* ---------------------------------------------------------------------------------------------
 * Multi-GPU (SURVEY 8e): one batch per device of the box driven from ONE host process - what a Rust host needs to use all
 * 8 GPUs without Python. Envs shard by global env id (rank r owns [env_id_offset + r*nenv, env_id_offset + (r+1)*nenv)),
 * one host thread per device issues its launches, no data-path collective exists. ox_group_stats is the only exchange:
 * 4 doubles per GPU summed by ncclAllReduce over NVLink (libnccl.so.2 via dlopen; host-side sum when NCCL is absent).
 * cfg->nenv = envs PER DEVICE; cfg->device is ignored; devices = NULL means ordinals 0..ndevices-1.
 * ------------------------------------------------------------------------------------------- */
typedef struct ox_group ox_group;
OX_API ox_status ox_group_create(const ox_model* m, const ox_batch_config* cfg, int32_t ndevices, const int32_t* devices_or_null, ox_group** out);
OX_API void ox_group_free(ox_group* g);
OX_API int32_t ox_group_size(const ox_group* g);
OX_API ox_batch* ox_group_batch(ox_group* g, int32_t rank);   /* borrowed: per-device I/O goes through the ox_batch_* calls */
OX_API ox_status ox_group_step(ox_group* g, int32_t nsteps);  /* asynchronous on every device's stream */
OX_API ox_status ox_group_sync(ox_group* g);
OX_API ox_status ox_group_reset(ox_group* g);
OX_API ox_status ox_group_ctrl_philox(ox_group* g, int32_t enable, uint64_t seed);
OX_API ox_status ox_group_stats(ox_group* g, double* out4);   /* totals over all devices, same layout as ox_batch_stats */
OX_API const char* ox_group_stats_backend(const ox_group* g); /* "nccl" or "host" */

/* Measurement aid (bench.py roofline): peak FMA throughput of the device's CUDA cores in TFLOP/s, measured with a
 * register-resident multiply-add kernel (8 independent chains per thread, every SM full), fp32 or fp64. */
OX_API ox_status ox_measure_fma_peak(int32_t device, int32_t precision, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* OX_B200_H */
