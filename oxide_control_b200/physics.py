"""Host-side mirror of oxide_control's `Physics` interface over the C ABI (include/ox_b200.h).

The reference's host language is Rust (absent in this image), so this module and the C++ header
include/ox_b200.hpp stand where `rust/ox_b200/src/lib.rs` would: same names, argument meaning and
error behaviour as /root/reference/src/physics.rs and src/error.rs, so that the tests read like
tests of the reference would. Nothing here computes physics: every method forwards to libox_b200.so.

  Physics           <- src/physics.rs:6-171   (one env; a BatchedPhysics of size 1, fp64)
  BatchedPhysics    <- new: nenv copies of mjData stepped together on one B200
  Actuators         <- src/physics.rs:65-79
  Error / *Error    <- src/error.rs:3-82
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _abi as A


# ---------------------------------------------------------------- errors (src/error.rs:3-15)
class Error(Exception):
    """Base of the reference's `enum Error` variants."""


class MujocoError(Error):
    """Error::Mujoco(MjError) - parse / load failures (src/error.rs:4, From<MjError> :17-21)."""


class MjsError(Error):
    """Error::Mjs(String) - model compile failures (src/error.rs:5, src/physics.rs:21)."""


class NameNotFound(Error):
    """Error::NameNotFound (src/error.rs:6)."""


class PhysicsDiverged(Error):
    """Error::PhysicsDiverged (src/error.rs:7). Raised only on request (check_diverged)."""


class JointTypeNotMatch(Error):
    """Error::JointTypeNotMatch{expected, found} (src/error.rs:8-11)."""


class CudaError(Error):
    """New variant: device / allocation / launch failure (no CPU fallback exists)."""


def _raise(status: int) -> None:
    msg = A.last_error()
    if status in (A.OX_ERR_PARSE, A.OX_ERR_IO):
        raise MujocoError(msg)
    if status == A.OX_ERR_COMPILE:
        raise MjsError(msg)
    if status == A.OX_ERR_CUDA:
        raise CudaError(msg)
    raise Error(f"ox_status {status}: {msg}")


def _check(status: int) -> None:
    if status != A.OX_OK:
        _raise(status)


# ---------------------------------------------------------------- typed ids (rusty_mujoco::ObjectId<O>, obj::*, joint::*)
@dataclass(frozen=True)
class ObjectId:
    objtype: int
    index: int


class obj:  # noqa: N801  (mirrors rusty_mujoco::obj)
    Body, Joint, Dof, Geom, Site = A.OBJ_BODY, A.OBJ_JOINT, A.OBJ_DOF, A.OBJ_GEOM, A.OBJ_SITE
    Actuator, Sensor, Equality, Plugin, Tendon = A.OBJ_ACTUATOR, A.OBJ_SENSOR, A.OBJ_EQUALITY, A.OBJ_PLUGIN, A.OBJ_TENDON


class joint:  # noqa: N801  (mirrors rusty_mujoco::joint: Qpos / Qvel widths per joint type)
    Free, Ball, Slide, Hinge = A.JNT_FREE, A.JNT_BALL, A.JNT_SLIDE, A.JNT_HINGE
    QPOS_WIDTH = {A.JNT_FREE: 7, A.JNT_BALL: 4, A.JNT_SLIDE: 1, A.JNT_HINGE: 1}
    QVEL_WIDTH = {A.JNT_FREE: 6, A.JNT_BALL: 3, A.JNT_SLIDE: 1, A.JNT_HINGE: 1}
    NAME = {A.JNT_FREE: "Free", A.JNT_BALL: "Ball", A.JNT_SLIDE: "Slide", A.JNT_HINGE: "Hinge"}


# ---------------------------------------------------------------- model
class Model:
    """Compiled model (the `mjModel` the reference owns at src/physics.rs:7). Immutable."""

    def __init__(self, handle: int):
        self._h = C.c_void_p(handle)
        self._cache = {}

    @staticmethod
    def from_xml_string(xml: str) -> "Model":
        h = C.c_void_p()
        _check(A.lib().ox_model_from_xml_string(xml.encode("utf-8"), C.byref(h)))
        return Model(h.value)

    @staticmethod
    def from_xml(path) -> "Model":
        h = C.c_void_p()
        _check(A.lib().ox_model_from_xml_path(str(path).encode("utf-8"), C.byref(h)))
        return Model(h.value)

    # binary model format (SURVEY 8f N4; MuJoCo: mj_saveModel / mj_loadModel)
    def save(self, path) -> None:
        _check(A.lib().ox_model_save(self._h, str(path).encode("utf-8")))

    @staticmethod
    def load(path) -> "Model":
        h = C.c_void_p()
        _check(A.lib().ox_model_load(str(path).encode("utf-8"), C.byref(h)))
        return Model(h.value)

    def to_bytes(self) -> bytes:
        n = A.lib().ox_model_serialize(self._h, None, 0)
        buf = C.create_string_buffer(n)
        assert A.lib().ox_model_serialize(self._h, buf, n) == n
        return buf.raw

    @staticmethod
    def from_bytes(data: bytes) -> "Model":
        h = C.c_void_p()
        _check(A.lib().ox_model_deserialize(data, len(data), C.byref(h)))
        return Model(h.value)

    def __del__(self):
        try:
            if self._h:
                A.lib().ox_model_free(self._h)
                self._h = None
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    @property
    def tables_ptr(self) -> int:
        """Address of the ox_model_tables struct (what the oracle in oracle/ consumes)."""
        return A.lib().ox_model_get_tables(self._h)

    def size(self, name: str) -> int:
        v = A.lib().ox_model_size(self._h, name.encode())
        if v < 0:
            raise Error(f"unknown model size '{name}'")
        return v

    def __getattr__(self, name: str):
        if name.startswith("_"):
            raise AttributeError(name)
        if name in self._cache:
            return self._cache[name]
        L = A.lib()
        v = L.ox_model_size(self._h, name.encode())
        if v >= 0:
            return v
        ip, cnt = C.POINTER(C.c_int32)(), C.c_int32()
        if L.ox_model_int_table(self._h, name.encode(), C.byref(ip), C.byref(cnt)) == A.OX_OK:
            arr = np.ctypeslib.as_array(ip, shape=(cnt.value,)).copy() if cnt.value else np.zeros(0, np.int32)
            self._cache[name] = arr
            return arr
        dp = C.POINTER(C.c_double)()
        if L.ox_model_real_table(self._h, name.encode(), C.byref(dp), C.byref(cnt)) == A.OX_OK:
            arr = np.ctypeslib.as_array(dp, shape=(cnt.value,)).copy() if cnt.value else np.zeros(0)
            if name in ("timestep", "tolerance", "ls_tolerance", "impratio", "meaninertia", "noslip_tolerance", "density", "viscosity"):
                arr = float(arr[0])
            self._cache[name] = arr
            return arr
        raise AttributeError(f"model has no table or size '{name}'")

    # src/physics.rs:56-62
    def jit_compile(self, precision: str = "f32") -> str:
        """Compile (or find cached) the run-time specialised step kernel of this model; needs nvcc, not a GPU. Returns the cubin path."""
        buf = C.create_string_buffer(4096)
        _check(A.lib().ox_jit_compile(self._h, A.F64 if precision == "f64" else A.F32, buf, 4096))
        return buf.value.decode()

    def object_id(self, objtype: int, name: str) -> Optional[ObjectId]:
        i = A.lib().ox_model_name2id(self._h, objtype, name.encode())
        return None if i < 0 else ObjectId(objtype, i)

    def object_name(self, oid: ObjectId) -> str:
        s = A.lib().ox_model_id2name(self._h, oid.objtype, oid.index)
        if s is None:
            raise Error(f"object id out of range: {oid}")
        return s.decode()


# ---------------------------------------------------------------- batched handle
class BatchedPhysics:
    """nenv independent copies of one model's mjData on one GPU (SURVEY.md 8b)."""

    def __init__(self, model: Model, nenv: int, *, precision: str = "f32", device: int = 0, mode: str = "fused",
                 iterations: int = 0, ls_iterations: int = 0, tolerance: float = -1.0, use_graph: bool = False,
                 block_threads: int = 0, env_id_offset: int = 0, specialize: bool = True, lanes_per_warp: int = 0, coop_solver: int = -1):
        self.model = model
        cfg = A.BatchConfig()
        A.lib().ox_batch_config_default(C.byref(cfg))
        cfg.nenv = nenv
        cfg.device = device
        cfg.precision = {"f32": A.F32, "f64": A.F64}[precision]
        cfg.mode = {"fused": A.MODE_FUSED, "staged": A.MODE_STAGED, "coop": A.MODE_COOP}[mode]
        cfg.iterations = iterations
        cfg.ls_iterations = ls_iterations
        cfg.tolerance = tolerance
        cfg.use_graph = int(use_graph)
        cfg.block_threads = block_threads
        cfg.env_id_offset = env_id_offset
        cfg.specialize = int(specialize)
        cfg.lanes_per_warp = lanes_per_warp
        cfg.coop_solver = coop_solver
        self.precision = precision
        self.nenv = nenv
        self._h = C.c_void_p()
        _check(A.lib().ox_batch_create(model.handle, C.byref(cfg), C.byref(self._h)))

    @staticmethod
    def from_xml_string(xml: str, nenv: int, **kw) -> "BatchedPhysics":
        return BatchedPhysics(Model.from_xml_string(xml), nenv, **kw)

    @classmethod
    def _borrowed(cls, handle, model: Model, nenv: int, precision: str) -> "BatchedPhysics":
        """View of a batch owned by someone else (a PhysicsGroup): never freed from here."""
        self = cls.__new__(cls)
        self.model, self.nenv, self.precision, self._h, self._owned = model, nenv, precision, C.c_void_p(handle), False
        return self

    def close(self):
        if getattr(self, "_h", None):
            if getattr(self, "_owned", True):
                A.lib().ox_batch_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    # ---- step family (src/physics.rs:44-54); asynchronous on the batch's stream
    def step(self, nsteps: int = 1) -> None:
        _check(A.lib().ox_batch_step(self._h, nsteps))

    def forward(self) -> None:
        _check(A.lib().ox_batch_forward(self._h))

    def inverse(self) -> None:
        """mj_inverse for every env (ox_batch_inverse): qfrc_inverse = M qacc + bias - passive - constraint at the current
        qpos / qvel / qacc, plus every derived field and sensordata. The state and qacc are left as they are."""
        _check(A.lib().ox_batch_inverse(self._h))

    def step_io(self, ctrl: Optional[np.ndarray] = None):
        """Action::apply + step + Observation::generate (src/lib.rs:63-66) for the whole batch in one call:
        ctrl[nenv, nu] in, one mj_step, (qpos[nenv, nq], qvel[nenv, nv]) out."""
        dt = np.float64 if self.precision == "f64" else np.float32
        code = A.F64 if self.precision == "f64" else A.F32
        q = np.empty((self.nenv, self.model.nq), dt)
        v = np.empty((self.nenv, self.model.nv), dt)
        c = None
        if ctrl is not None:
            c = np.ascontiguousarray(ctrl, dt)
            assert c.shape == (self.nenv, self.model.nu), c.shape
        _check(A.lib().ox_batch_step_io(self._h, c.ctypes.data_as(C.c_void_p) if c is not None else None, q.ctypes.data_as(C.c_void_p),
                                        v.ctypes.data_as(C.c_void_p), code, A.MEM_HOST))
        return q, v

    def step_io_ptr(self, ctrl_ptr: Optional[int], qpos_ptr: Optional[int], qvel_ptr: Optional[int], dtype_code: int, mem: int) -> None:
        """Raw-pointer form (pinned host or device buffers): the specialised step kernel does the I/O itself."""
        p = lambda x: C.c_void_p(x) if x else None
        _check(A.lib().ox_batch_step_io(self._h, p(ctrl_ptr), p(qpos_ptr), p(qvel_ptr), dtype_code, mem))

    def reset(self, mask: Optional[np.ndarray] = None) -> None:
        if mask is None:
            _check(A.lib().ox_batch_reset(self._h, None))
        else:
            m = np.ascontiguousarray(mask, dtype=np.uint8)
            assert m.shape == (self.nenv,)
            _check(A.lib().ox_batch_reset(self._h, m.ctypes.data_as(C.c_void_p)))
            self.sync()

    def sync(self) -> None:
        _check(A.lib().ox_batch_sync(self._h))

    def ctrl_philox(self, enable: bool, seed: int = 0x0B200) -> None:
        _check(A.lib().ox_batch_ctrl_philox(self._h, int(enable), seed))

    def ctrl_philox_scale(self, scale: float) -> None:
        _check(A.lib().ox_batch_ctrl_philox_scale(self._h, float(scale)))

    def set_step_counter(self, step: int) -> None:
        _check(A.lib().ox_batch_set_step_counter(self._h, step))

    # ---- bulk I/O
    # checkpoint / resume (ox_batch_get_state / ox_batch_set_state)
    def get_state(self, dtype=np.float64) -> np.ndarray:
        """[nenv, state_size] records: time, qpos, qvel, act, ctrl, qfrc_applied, xfrc_applied, qacc_warmstart."""
        n = A.lib().ox_batch_state_size(self._h)
        out = np.empty((self.nenv, n), dtype=dtype)
        _check(A.lib().ox_batch_get_state(self._h, out.ctypes.data_as(C.c_void_p), A.F64 if out.dtype == np.float64 else A.F32, A.MEM_HOST))
        return out

    def set_state(self, state: np.ndarray) -> None:
        state = np.ascontiguousarray(state, dtype=np.float64 if state.dtype != np.float32 else np.float32)
        assert state.shape == (self.nenv, A.lib().ox_batch_state_size(self._h)), state.shape
        _check(A.lib().ox_batch_set_state(self._h, state.ctypes.data_as(C.c_void_p), A.F64 if state.dtype == np.float64 else A.F32, A.MEM_HOST))

    def step_counter(self) -> int:
        return int(A.lib().ox_batch_get_step_counter(self._h))

    def field_size(self, field: str) -> int:
        n = A.lib().ox_batch_field_size(self._h, A.FIELD[field])
        if n < 0:
            raise Error(f"unknown field '{field}'")
        return n

    def get(self, field: str, dtype=np.float64, layout: str = "env_major") -> np.ndarray:
        """Download a field as [nenv, n] (env_major) or [n, nenv] (elem_major)."""
        n = self.field_size(field)
        is_int = field in A.INT_FIELDS
        dt = np.int32 if is_int else np.dtype(dtype)
        shape = (self.nenv, n) if layout == "env_major" else (n, self.nenv)
        out = np.empty(shape, dtype=dt)
        if n == 0:
            return out
        code = A.F64 if dt == np.float64 else A.F32
        lay = A.LAYOUT_ENV_MAJOR if layout == "env_major" else A.LAYOUT_ELEM_MAJOR
        _check(A.lib().ox_batch_get(self._h, A.FIELD[field], out.ctypes.data_as(C.c_void_p), code, A.MEM_HOST, lay))
        return out

    def set(self, field: str, values: np.ndarray, layout: str = "env_major") -> None:
        n = self.field_size(field)
        if n == 0:
            return
        v = np.asarray(values)
        dt = np.float32 if v.dtype == np.float32 else np.float64
        v = np.ascontiguousarray(v, dtype=dt)
        shape = (self.nenv, n) if layout == "env_major" else (n, self.nenv)
        if v.shape != shape:
            raise Error(f"set('{field}'): expected shape {shape}, got {v.shape}")
        code = A.F64 if dt == np.float64 else A.F32
        lay = A.LAYOUT_ENV_MAJOR if layout == "env_major" else A.LAYOUT_ELEM_MAJOR
        _check(A.lib().ox_batch_set(self._h, A.FIELD[field], v.ctypes.data_as(C.c_void_p), code, A.MEM_HOST, lay))
        self.sync()  # the numpy temporary may die right after this call

    def get_ptr(self, field: str, ptr: int, dtype_code: int, mem: int, layout: int) -> None:
        _check(A.lib().ox_batch_get(self._h, A.FIELD[field], C.c_void_p(ptr), dtype_code, mem, layout))

    def get_many_ptr(self, fields: Sequence[str], ptrs: Sequence[int], dtype_code: int, mem: int, layout: int) -> None:
        """Several fields, one stream synchronisation (the observation read of an RL step)."""
        n = len(fields)
        ids = (C.c_int32 * n)(*[A.FIELD[f] for f in fields])
        bufs = (C.c_void_p * n)(*ptrs)
        _check(A.lib().ox_batch_get_many(self._h, n, ids, bufs, dtype_code, mem, layout))

    def set_ptr(self, field: str, ptr: int, dtype_code: int, mem: int, layout: int) -> None:
        _check(A.lib().ox_batch_set(self._h, A.FIELD[field], C.c_void_p(ptr), dtype_code, mem, layout))

    # ---- per-env slices (fp64 at the boundary)
    def get1(self, field: str, env: int, offset: int = 0, count: Optional[int] = None) -> np.ndarray:
        if count is None:
            count = self.field_size(field) - offset
        if field in A.INT_FIELDS:
            out = np.zeros(count, np.int32)
            st = A.lib().ox_batch_get1_int(self._h, A.FIELD[field], env, offset, count, out.ctypes.data_as(C.POINTER(C.c_int32)))
        else:
            out = np.zeros(count, np.float64)
            st = A.lib().ox_batch_get1(self._h, A.FIELD[field], env, offset, count, out.ctypes.data_as(C.POINTER(C.c_double)))
        if st == A.OX_ABSENT:
            return None
        _check(st)
        return out

    def set1(self, field: str, env: int, values: Sequence[float], offset: int = 0):
        v = np.ascontiguousarray(np.atleast_1d(values), dtype=np.float64)
        st = A.lib().ox_batch_set1(self._h, A.FIELD[field], env, offset, v.size, v.ctypes.data_as(C.POINTER(C.c_double)))
        if st == A.OX_ABSENT:
            return None
        _check(st)
        return ()

    # ---- diagnostics
    def diverged(self) -> np.ndarray:
        """Per-env count of mj_checkPos/Vel/Acc auto-resets (home of Error::PhysicsDiverged)."""
        return self.get("diverged")[:, 0]

    def check_diverged(self) -> None:
        if int(self.diverged().sum()) > 0:
            raise PhysicsDiverged("one or more environments diverged and were auto-reset")

    def stats(self) -> dict:
        out = (C.c_double * 4)()
        _check(A.lib().ox_batch_stats(self._h, out))
        return {"sum_ncon": out[0], "sum_nefc": out[1], "sum_niter": out[2], "diverged": out[3]}

    def kernel_name(self) -> str:
        return A.lib().ox_batch_kernel_name(self._h).decode()

    def jit_note(self) -> str:
        return (A.lib().ox_batch_jit_note(self._h) or b"").decode()

    def launch_count(self) -> int:
        return int(A.lib().ox_batch_launch_count(self._h))

    def stage_times(self, reps: int = 10) -> dict:
        ms = (C.c_double * 32)()
        n = C.c_int32()
        _check(A.lib().ox_batch_stage_times(self._h, reps, ms, C.byref(n)))
        return {A.lib().ox_stage_name(i).decode(): ms[i] for i in range(n.value)}


# ---------------------------------------------------------------- single-env handle (src/physics.rs)
class PhysicsGroup:
    """One batch per GPU of the box, driven from this one process (ox_group_* in include/ox_b200.h): envs shard by global
    env id, one host thread per device issues its launches, the only exchange is the NCCL all-reduce of 4 statistics."""

    def __init__(self, model: Model, nenv_per_device: int, ndevices: int, *, precision: str = "f32", devices: Optional[Sequence[int]] = None,
                 env_id_offset: int = 0, specialize: int = 1, mode: str = "fused"):
        cfg = A.BatchConfig()
        A.lib().ox_batch_config_default(C.byref(cfg))
        cfg.nenv, cfg.precision, cfg.env_id_offset = nenv_per_device, {"f32": A.F32, "f64": A.F64}[precision], env_id_offset
        cfg.specialize, cfg.mode = int(specialize), {"fused": A.MODE_FUSED, "staged": A.MODE_STAGED, "coop": A.MODE_COOP}[mode]
        devs = (C.c_int32 * ndevices)(*devices) if devices is not None else None
        self.model, self._h = model, C.c_void_p()
        _check(A.lib().ox_group_create(model.handle, C.byref(cfg), ndevices, devs, C.byref(self._h)))
        self.size = A.lib().ox_group_size(self._h)
        self.batches = [BatchedPhysics._borrowed(A.lib().ox_group_batch(self._h, r), model, nenv_per_device, precision) for r in range(self.size)]

    def close(self):
        if getattr(self, "_h", None):
            for b in self.batches:
                b._h = None
            A.lib().ox_group_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def step(self, nsteps: int = 1) -> None:
        _check(A.lib().ox_group_step(self._h, nsteps))

    def sync(self) -> None:
        _check(A.lib().ox_group_sync(self._h))

    def reset(self) -> None:
        _check(A.lib().ox_group_reset(self._h))

    def ctrl_philox(self, enable: bool, seed: int = 0x0B200) -> None:
        _check(A.lib().ox_group_ctrl_philox(self._h, int(enable), seed))

    def stats(self) -> dict:
        out = (C.c_double * 4)()
        _check(A.lib().ox_group_stats(self._h, out))
        return {"sum_ncon": out[0], "sum_nefc": out[1], "sum_niter": out[2], "diverged": out[3]}

    def stats_backend(self) -> str:
        return A.lib().ox_group_stats_backend(self._h).decode()


def measure_fma_peak(device: int = 0, precision: str = "f32") -> float:
    """Measured FMA peak of the device's CUDA cores, TFLOP/s (ox_measure_fma_peak)."""
    out = C.c_double()
    _check(A.lib().ox_measure_fma_peak(device, A.F64 if precision == "f64" else A.F32, C.byref(out)))
    return out.value


class Actuators:
    """src/physics.rs:65-79: the only thing an Action may touch."""

    def __init__(self, physics: "Physics"):
        self._p = physics

    def set(self, id: ObjectId, control: float) -> None:
        self._p.set_ctrl(id, control)


class _Data:
    """Read-only view standing where `Physics::data() -> &mjData` (src/physics.rs:30-32) gives access
    to fields Physics does not wrap (qacc, sensordata, xpos, ncon, ...)."""

    def __init__(self, b: BatchedPhysics):
        self._b = b

    def __getattr__(self, name: str):
        if name.startswith("_"):
            raise AttributeError(name)
        if name not in A.FIELD:
            raise AttributeError(f"mjData field '{name}' is not exposed")
        v = self._b.get1(name, 0)
        if name in ("ncon", "nefc", "solver_niter", "time"):
            return v[0].item()
        return v


class Physics:
    """One environment. Method-for-method mirror of /root/reference/src/physics.rs."""

    def __init__(self, model: Model, **kw):
        kw.setdefault("precision", "f64")
        # data() stands for &mjData: every derived field must be current after step(), which only the generic kernels
        # guarantee (the model-specialised kernel writes back state, qacc, sensordata and counters only - see
        # field_live() in csrc/ox_batch_internal.cuh; reading anything else after such a step is an error)
        kw.setdefault("specialize", False)
        self._model = model
        self._b = BatchedPhysics(model, 1, **kw)

    # constructors, src/physics.rs:12-24
    @staticmethod
    def from_xml(xml_path, **kw) -> "Physics":
        return Physics(Model.from_xml(xml_path), **kw)

    @staticmethod
    def from_xml_string(xml_string: str, **kw) -> "Physics":
        return Physics(Model.from_xml_string(xml_string), **kw)

    # src/physics.rs:26-42
    def model(self) -> Model:
        return self._model

    def data(self) -> _Data:
        return _Data(self._b)

    def data_mut(self) -> BatchedPhysics:
        return self._b

    def model_data(self):
        return self._model, self.data()

    def model_datamut(self):
        return self._model, self._b

    # src/physics.rs:44-54 (infallible, like the reference)
    def step(self) -> None:
        self._b.step(1)
        self._b.sync()

    def forward(self) -> None:
        self._b.forward()
        self._b.sync()

    # extension: mj_inverse; the result is data().qfrc_inverse
    def inverse(self) -> None:
        self._b.inverse()
        self._b.sync()

    def reset(self) -> None:
        self._b.reset()
        self._b.sync()

    # src/physics.rs:56-62
    def object_id(self, objtype: int, name: str) -> Optional[ObjectId]:
        return self._model.object_id(objtype, name)

    def object_name(self, oid: ObjectId) -> str:
        return self._model.object_name(oid)

    # src/physics.rs:73-79
    def actuators(self) -> Actuators:
        return Actuators(self)

    # src/physics.rs:82-87
    def time(self) -> float:
        return float(self._b.get1("time", 0)[0])

    def set_time(self, time: float) -> None:
        self._b.set1("time", 0, [time])

    # src/physics.rs:89-94
    def ctrl(self, id: ObjectId) -> float:
        return float(self._b.get1("ctrl", 0, id.index, 1)[0])

    def set_ctrl(self, id: ObjectId, value: float) -> None:
        self._b.set1("ctrl", 0, [value], id.index)

    # src/physics.rs:96-102: Some(activation) for a stateful actuator (dyntype integrator / filter / filterexact), None otherwise
    def _actadr(self, id: ObjectId) -> int:
        return int(self._model.actuator_actadr[id.index]) if self._model.na else -1

    def act(self, id: ObjectId) -> Optional[float]:
        adr = self._actadr(id)
        return None if adr < 0 else float(self._b.get1("act", 0, adr, 1)[0])

    def set_act(self, id: ObjectId, value: float) -> Optional[tuple]:
        adr = self._actadr(id)
        if adr < 0:
            return None
        self._b.set1("act", 0, [value], adr)
        return ()

    # src/physics.rs:104-116
    def _jnt(self, id: ObjectId, expected: Optional[int]):
        jt = int(self._model.jnt_type[id.index])
        if expected is not None and jt != expected:
            raise JointTypeNotMatch(f"expected {joint.NAME[expected]}, found {joint.NAME[jt]}")
        return jt

    def qpos(self, id: ObjectId, jtype: Optional[int] = None):
        jt = self._jnt(id, jtype)
        v = self._b.get1("qpos", 0, int(self._model.jnt_qposadr[id.index]), joint.QPOS_WIDTH[jt])
        return float(v[0]) if v.size == 1 else v

    def set_qpos(self, id: ObjectId, qpos, jtype: Optional[int] = None) -> None:
        jt = self._jnt(id, jtype)
        v = np.atleast_1d(np.asarray(qpos, dtype=np.float64))
        assert v.size == joint.QPOS_WIDTH[jt]
        self._b.set1("qpos", 0, v, int(self._model.jnt_qposadr[id.index]))

    def qvel(self, id: ObjectId, jtype: Optional[int] = None):
        jt = self._jnt(id, jtype)
        v = self._b.get1("qvel", 0, int(self._model.jnt_dofadr[id.index]), joint.QVEL_WIDTH[jt])
        return float(v[0]) if v.size == 1 else v

    def set_qvel(self, id: ObjectId, qvel, jtype: Optional[int] = None) -> None:
        jt = self._jnt(id, jtype)
        v = np.atleast_1d(np.asarray(qvel, dtype=np.float64))
        assert v.size == joint.QVEL_WIDTH[jt]
        self._b.set1("qvel", 0, v, int(self._model.jnt_dofadr[id.index]))

    # src/physics.rs:118-123
    def qacc_warmstart(self, id: ObjectId) -> float:
        return float(self._b.get1("qacc_warmstart", 0, id.index, 1)[0])

    def set_qacc_warmstart(self, id: ObjectId, value: float) -> None:
        self._b.set1("qacc_warmstart", 0, [value], id.index)

    # src/physics.rs:125-131: no plugins in the supported subset
    def plugin_state(self, id: ObjectId) -> Optional[float]:
        return None

    def set_plugin_state(self, id: ObjectId, value: float) -> Optional[tuple]:
        return None

    # src/physics.rs:133-145
    def qfrc_applied(self, id: ObjectId) -> float:
        return float(self._b.get1("qfrc_applied", 0, id.index, 1)[0])

    def set_qfrc_applied(self, id: ObjectId, value: float) -> None:
        self._b.set1("qfrc_applied", 0, [value], id.index)

    def xfrc_applied(self, id: ObjectId) -> np.ndarray:
        return self._b.get1("xfrc_applied", 0, 6 * id.index, 6)

    def set_xfrc_applied(self, id: ObjectId, value) -> None:
        v = np.asarray(value, dtype=np.float64)
        assert v.shape == (6,)
        self._b.set1("xfrc_applied", 0, v, 6 * id.index)

    # src/physics.rs:147-152: equality constraints (connect, joint) can be switched on and off at run time
    def eq_active(self, id: ObjectId) -> bool:
        if not self._model.neq:
            raise Error("model has no equality constraints (neq = 0)")
        return bool(self._b.get1("eq_active", 0, id.index, 1)[0] != 0)

    def set_eq_active(self, id: ObjectId, value: bool) -> None:
        if not self._model.neq:
            raise Error("model has no equality constraints (neq = 0)")
        self._b.set1("eq_active", 0, [1.0 if value else 0.0], id.index)

    # src/physics.rs:154-170: None when the body is not a mocap body
    def _mocapid(self, id: ObjectId) -> int:
        return int(self._model.body_mocapid[id.index]) if self._model.nmocap else -1

    def mocap_pos(self, id: ObjectId):
        mid = self._mocapid(id)
        return None if mid < 0 else self._b.get1("mocap_pos", 0, 3 * mid, 3)

    def set_mocap_pos(self, id: ObjectId, pos):
        mid = self._mocapid(id)
        if mid < 0:
            return None
        v = np.asarray(pos, dtype=np.float64)
        assert v.shape == (3,)
        self._b.set1("mocap_pos", 0, v, 3 * mid)
        return ()

    def mocap_quat(self, id: ObjectId):
        mid = self._mocapid(id)
        return None if mid < 0 else self._b.get1("mocap_quat", 0, 4 * mid, 4)

    def set_mocap_quat(self, id: ObjectId, quat):
        mid = self._mocapid(id)
        if mid < 0:
            return None
        v = np.asarray(quat, dtype=np.float64)
        assert v.shape == (4,)
        self._b.set1("mocap_quat", 0, v, 4 * mid)
        return ()
