"""Inverse dynamics (ox_batch_inverse, MuJoCo's mj_inverse): qfrc_inverse = M qacc + qfrc_bias - qfrc_passive - qfrc_constraint
with the soft-constraint force at the given qacc. Three restatements must agree: the product's stage code (on the host through
tests/native and on the B200 through k_inverse, both M qacc + bias), the oracle (RNE with the acceleration term) and the dense
checker (dense M, Kane bias, autograd constraint forces). The inverse entry points of the checkers live in
tests/inverse_support.py and tests/dense_inverse.py. CPU tests first, then the gpu-marked ones."""
import os
import re
import subprocess

import numpy as np
import pytest

import oxide_control_b200 as ox
from oxide_control_b200 import _abi as A
from inverse_support import InverseHostBatch, InverseOracle
from support import SEED, random_state, rel_err
from tests_util import quat2mat
from zoo_models import HOPPER, NOCONTACT, ZOO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODELS = {**{k: v["xml"] for k, v in ox.models.CONFIGS.items()}, **ZOO}
DERIVED = ["xpos", "xquat", "xmat", "xipos", "ximat", "xanchor", "xaxis", "geom_xpos", "geom_xmat", "site_xpos", "site_xmat",
           "subtree_com", "cinert", "cdof", "qM", "qLD", "cvel", "cdof_dot", "qfrc_bias", "qfrc_passive", "actuator_force",
           "qfrc_actuator", "qfrc_smooth", "qacc_smooth", "qacc", "qacc_warmstart", "qfrc_constraint", "sensordata",
           "efc_D", "efc_aref", "efc_pos", "efc_force", "con_dist", "con_pos", "con_frame"]
UNTOUCHED = ["qpos", "qvel", "qacc", "qacc_warmstart", "time", "ctrl", "act"]
# fields that depend on qpos / qvel (and ctrl) only: after an inverse they equal what ox_batch_forward computes
QACC_FREE = ["xpos", "xquat", "xmat", "xipos", "subtree_com", "cinert", "cdof", "qM", "qLD", "cvel", "cdof_dot", "qfrc_bias",
             "qfrc_passive", "actuator_force", "qfrc_actuator", "qfrc_smooth", "qacc_smooth"]


def inputs(m, nenv, seed):
    """random state with free bodies 5 cm lower (contacts right away), controls, applied forces and a random qacc"""
    rng = np.random.default_rng(seed)
    qpos, qvel = random_state(m, nenv, seed=seed)
    for j in range(m.njnt):
        if int(m.jnt_type[j]) == 0:
            qpos[:, int(m.jnt_qposadr[j]) + 2] -= 0.05
    xfrc = rng.normal(0, 1.0, (nenv, 6 * m.nbody))
    xfrc[:, :6] = 0
    return dict(qpos=qpos, qvel=qvel, ctrl=rng.uniform(-1, 1, (nenv, m.nu)), qfrc_applied=rng.normal(0, 0.5, (nenv, m.nv)),
                xfrc_applied=xfrc, qacc=rng.normal(0, 2.0, (nenv, m.nv)))


def oracle_inverse(m, inp, e):
    od = InverseOracle(m)
    for f, v in inp.items():
        if v.shape[1]:
            od.field(f)[:] = v[e]
    od.inverse()
    return od


def check_against_oracle(m, get, nenv, ods, tol):
    assert np.array_equal(get("ncon")[:, 0], [od.int("ncon") for od in ods])
    assert np.array_equal(get("nefc")[:, 0], [od.int("nefc") for od in ods])
    for f in ["qfrc_inverse"] + DERIVED:
        got = get(f)
        if not got.shape[1]:
            continue
        ref = np.stack([od.field(f) for od in ods])
        if f.startswith("efc_") or f.startswith("con_"):   # only the first nefc / ncon entries are defined
            per = got.shape[1] // max(1, (m.nefcmax if f.startswith("efc_") else m.nconmax))
            for e, od in enumerate(ods):
                n = (od.int("nefc") if f.startswith("efc_") else od.int("ncon")) * per
                assert rel_err(got[e, :n], ref[e, :n]) <= tol, (f, e, rel_err(got[e, :n], ref[e, :n]))
        else:
            assert rel_err(got, ref) <= tol, (f, rel_err(got, ref))


def mul_m(m, qM, v):
    """M v from the sparse qM of one env (MuJoCo's layout: dof_Madr, the chain of dof_parentid)"""
    res = np.zeros(m.nv)
    for i in range(m.nv):
        adr = int(m.dof_Madr[i])
        res[i] += qM[adr] * v[i]
        j, adr = int(m.dof_parentid[i]), adr + 1
        while j >= 0:
            res[i] += qM[adr] * v[j]
            res[j] += qM[adr] * v[i]
            j, adr = int(m.dof_parentid[j]), adr + 1
    return res


# ------------------------------------------------------------------------------------------------ closed forms
def _hinge_inertia(m, body, axis):
    R = quat2mat(np.asarray(m.body_iquat[4 * body:4 * body + 4]))
    I = R @ np.diag(np.asarray(m.body_inertia[3 * body:3 * body + 3])) @ R.T
    return float(axis @ I @ axis)


def _closed_form_cases(name, qpos, qvel, qacc):
    m = ox.Model.from_xml_string(ox.models.CONFIGS[name]["xml"])
    g = -float(np.asarray(m.gravity)[2])
    ay = np.array([0.0, 1.0, 0.0])
    out = np.zeros_like(qacc)
    if name == "pendulum":
        mass, ipos = float(m.body_mass[1]), np.asarray(m.body_ipos[3:6])
        assert abs(ipos[0]) < 1e-12 and abs(ipos[1]) < 1e-12
        d = -ipos[2]                                     # com on the pole's axis, below the hinge
        I = _hinge_inertia(m, 1, ay) + mass * d * d + float(m.dof_armature[0])
        th, w, a = qpos[:, 0], qvel[:, 0], qacc[:, 0]
        # rotation about +y moves the com to (-d sin th, 0, -d cos th): gravity's torque about +y is -m g d sin th
        out[:, 0] = I * a + mass * g * d * np.sin(th) + float(m.dof_damping[0]) * w
    else:   # cartpole: slider x, hinge th about +y, pole com at height l above the hinge
        mc, mp, ipos = float(m.body_mass[1]), float(m.body_mass[2]), np.asarray(m.body_ipos[6:9])
        assert abs(ipos[0]) < 1e-12 and abs(ipos[1]) < 1e-12 and np.allclose(m.body_ipos[3:6], 0)
        l, Ip = ipos[2], _hinge_inertia(m, 2, ay)
        th, w = qpos[:, 1], qvel[:, 1]
        M11, M12, M22 = mc + mp + float(m.dof_armature[0]), mp * l * np.cos(th), Ip + mp * l * l + float(m.dof_armature[1])
        out[:, 0] = M11 * qacc[:, 0] + M12 * qacc[:, 1] - mp * l * np.sin(th) * w * w + float(m.dof_damping[0]) * qvel[:, 0]
        out[:, 1] = M12 * qacc[:, 0] + M22 * qacc[:, 1] - mp * g * l * np.sin(th) + float(m.dof_damping[1]) * w
    return m, out


@pytest.mark.parametrize("name", ["pendulum", "cartpole"])
def test_closed_form_on_oracle_and_host_instantiation(name):
    m0 = ox.Model.from_xml_string(ox.models.CONFIGS[name]["xml"])
    nenv = 8
    rng = np.random.default_rng(5)
    qpos, qvel = random_state(m0, nenv, seed=5)
    qpos[:, -1] += rng.uniform(-2.5, 2.5, nenv)        # large angles: sin th far from th
    qacc = rng.normal(0, 3.0, (nenv, m0.nv))
    m, ref = _closed_form_cases(name, qpos, qvel, qacc)
    hb = InverseHostBatch(m, nenv, "f64")
    hb.set("qpos", qpos); hb.set("qvel", qvel); hb.set("qacc", qacc)
    hb.inverse()
    assert hb.get("nefc").sum() == 0
    assert rel_err(hb.get("qfrc_inverse"), ref) <= 1e-12, rel_err(hb.get("qfrc_inverse"), ref)
    inp = dict(qpos=qpos, qvel=qvel, qacc=qacc)
    ods = [oracle_inverse(m, inp, e) for e in range(nenv)]
    got = np.stack([od.field("qfrc_inverse") for od in ods])
    assert rel_err(got, ref) <= 1e-12, rel_err(got, ref)


# ------------------------------------------------------------------------------------------------ host instantiation vs oracle
@pytest.mark.parametrize("name", list(MODELS))
def test_host_instantiation_matches_oracle_fp64(name):
    m = ox.Model.from_xml_string(MODELS[name])
    nenv = 6
    inp = inputs(m, nenv, seed=41)
    hb = InverseHostBatch(m, nenv, "f64")
    for f, v in inp.items():
        if v.shape[1]:
            hb.set(f, v)
    if m.na:
        hb.set("act", np.random.default_rng(42).uniform(-0.5, 0.5, (nenv, m.na)))
    before = {f: hb.get(f) for f in UNTOUCHED}
    hb.inverse()
    inp_o = dict(inp, **({"act": hb.get("act")} if m.na else {}))
    ods = [oracle_inverse(m, inp_o, e) for e in range(nenv)]
    check_against_oracle(m, hb.get, nenv, ods, 1e-9)
    for f, v in before.items():    # mj_inverse does not touch the state, qacc or the warm start
        assert np.array_equal(hb.get(f), v), f


# ------------------------------------------------------------------------------------------------ oracle vs dense checker
GOLDEN_MODELS = {**{k: v["xml"] for k, v in ox.models.CONFIGS.items()}, **ZOO, **NOCONTACT, "hopper": HOPPER}
GOLDEN_INPUTS = ("qpos", "qvel", "ctrl", "act", "mocap_pos", "mocap_quat", "eq_active")


@pytest.mark.parametrize("name", list(GOLDEN_MODELS))
def test_oracle_matches_dense_checker(name):
    """At the golden fixtures' states (most in contact), the oracle's RNE route and the dense checker's M qacc + Kane bias with
    autograd constraint forces give the same qfrc_inverse: both cones, frictionloss, equalities, tendons, fluid, gravcomp."""
    import json
    import dense_checker as dc
    import dense_inverse
    with open(os.path.join(ROOT, "tests", "golden", f"dense_{name}.json")) as f:
        cases = json.load(f)["cases"]
    m = ox.Model.from_xml_string(GOLDEN_MODELS[name])
    dm = dc.DenseModel(m)
    rng = np.random.default_rng(43)
    contact = [c for c in cases if c["output"]["ncon"] > 0]
    picked = (contact[:3] + [c for c in cases if c["output"]["ncon"] == 0][:1]) if m.npair else cases[:4]
    for case in picked:
        i = case["input"]
        qacc = rng.normal(0, 2.0, m.nv)
        od = InverseOracle(m)
        for f in GOLDEN_INPUTS:
            if len(i.get(f, ())):
                od.field(f)[:] = i[f]
        od.field("qacc")[:] = qacc
        od.inverse()
        r = dense_inverse.inverse(dm, np.array(i["qpos"]), np.array(i["qvel"]), qacc,
                                  mocap=(np.array(i.get("mocap_pos", [])), np.array(i.get("mocap_quat", []))),
                                  eq_active=np.array(i["eq_active"]) if "eq_active" in i else None)
        assert r["ncon"] == od.int("ncon") and r["nefc"] == od.int("nefc")
        assert rel_err(od.field("qfrc_inverse"), r["qfrc_inverse"]) <= 1e-9, rel_err(od.field("qfrc_inverse"), r["qfrc_inverse"])
        assert rel_err(od.field("qfrc_constraint"), r["qfrc_constraint"]) <= 1e-9


# ------------------------------------------------------------------------------------------------ inverse <-> forward
def _tight(xml, tol):
    return re.sub(r"<option([^>]*?)(/?)>", lambda mo: "<option" + re.sub(r'\s(tolerance|iterations)="[^"]*"', "", mo.group(1))
                  + f' tolerance="{tol}" iterations="500"' + mo.group(2) + ">", xml, count=1)


# Newton (pyramidal: cheetah, humanoid, zoo_a; elliptic: zoo_j) and CG (elliptic: zoo_n)
ROUNDTRIP = {"cheetah": ox.models.CHEETAH, "humanoid": ox.models.HUMANOID, "zoo_a": ZOO["zoo_a"], "zoo_j": ZOO["zoo_j"], "zoo_n": ZOO["zoo_n"]}


@pytest.mark.parametrize("name", list(ROUNDTRIP))
def test_round_trip_inverse_then_forward(name):
    """qacc -> inverse -> qfrc_applied := qfrc_inverse - qfrc_actuator -> forward recovers qacc. The forward solve stops at its
    tolerance (1e-14 here, on the gradient scaled by 1 / (meaninertia nv)); with the condition of these models that bounds the
    recovered qacc to 1e-7 relative (max |a - b| / max(1, |b|)). Newton on a pyramidal model lands on the exact minimiser."""
    m = ox.Model.from_xml_string(_tight(ROUNDTRIP[name], 1e-14))
    assert int(m.solver) in (1, 2)
    inp = inputs(m, 4, seed=44)
    for e in range(4):
        od = oracle_inverse(m, dict(inp, xfrc_applied=np.zeros_like(inp["xfrc_applied"])), e)
        qacc = od.field("qacc").copy()
        od.field("qfrc_applied")[:] = od.field("qfrc_inverse") - od.field("qfrc_actuator")
        od.field("xfrc_applied")[:] = 0
        od.forward()
        assert rel_err(od.field("qacc"), qacc) <= 1e-7, (e, rel_err(od.field("qacc"), qacc))


@pytest.mark.parametrize("name", ["pendulum", "cartpole", "acrobot", "cheetah", "humanoid", "zoo_a", "zoo_b", "zoo_j", "zoo_n"])
def test_forward_then_inverse_gives_the_solver_gradient(name):
    """After a forward solve, qfrc_inverse - (qfrc_applied + qfrc_actuator + J'xfrc) is the solver's final gradient
    M qacc - qfrc_smooth - qfrc_constraint: zero to round-off without contacts, the solver's residual with them."""
    m = ox.Model.from_xml_string(MODELS[name])
    inp = inputs(m, 4, seed=45)
    for e in range(4):
        od = InverseOracle(m)
        for f in ("qpos", "qvel", "ctrl", "qfrc_applied", "xfrc_applied"):
            if inp[f].shape[1]:
                od.field(f)[:] = inp[f][e]
        od.forward()
        qacc, smooth, cons = od.field("qacc").copy(), od.field("qfrc_smooth").copy(), od.field("qfrc_constraint").copy()
        xfrc_gen = smooth - (od.field("qfrc_passive") - od.field("qfrc_bias") + od.field("qfrc_applied") + od.field("qfrc_actuator"))
        grad = mul_m(m, od.field("qM"), qacc) - smooth - cons
        od.inverse()
        lhs = od.field("qfrc_inverse") - (od.field("qfrc_applied") + od.field("qfrc_actuator") + xfrc_gen)
        tol = 1e-11 if od.int("nefc") == 0 else 1e-6
        assert np.max(np.abs(lhs - grad)) <= tol * max(1.0, np.max(np.abs(smooth))), (e, np.max(np.abs(lhs - grad)))


# ------------------------------------------------------------------------------------------------ surface
def test_null_batch_is_refused():
    assert A.lib().ox_batch_inverse(None) == A.OX_ERR_INVALID
    assert "null batch" in A.last_error()
    assert A.FIELD["qfrc_inverse"] == 51 and A.FIELD["ten_J"] == 50


def test_rust_wrapper_declares_inverse():
    src = open(os.path.join(ROOT, "rust", "ox_b200", "src", "lib.rs")).read()
    impls = re.split(r"\nimpl ", src)
    for ty in ("BatchedPhysics {", "Physics {"):
        body = next(b for b in impls if b.startswith(ty))
        assert re.search(r"pub fn inverse\(&mut self\)", body), ty
    sys_src = open(os.path.join(ROOT, "rust", "ox_b200-sys", "src", "lib.rs")).read()
    assert "pub fn ox_batch_inverse(b: *mut ox_batch) -> ox_status;" in sys_src
    assert "pub const OX_F_QFRC_INVERSE: i32 = 51;" in sys_src


def test_cpp_snippet_calling_inverse_compiles(tmp_path):
    src = tmp_path / "inv.cpp"
    src.write_text('#include <variant>\n#include "ox_b200.hpp"\n'
                   "void f(ox_b200::BatchedPhysics& b, ox_b200::Physics& p) { b.inverse(); p.inverse(); }\n"
                   "int field() { return OX_F_QFRC_INVERSE; }\n")
    subprocess.check_call(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-I" + os.path.join(ROOT, "include"), str(src)])


# ================================================================================================ GPU
def _load(b, m, inp, act=None):
    for f, v in inp.items():
        if v.shape[1]:
            b.set(f, v)
    if act is not None:
        b.set("act", act)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODELS))
def test_gpu_inverse_matches_oracle_fp64(name):
    m = ox.Model.from_xml_string(MODELS[name])
    nenv = 64
    inp = inputs(m, nenv, seed=51)
    act = np.random.default_rng(52).uniform(-0.5, 0.5, (nenv, m.na)) if m.na else None
    b = ox.BatchedPhysics(m, nenv, precision="f64")
    _load(b, m, inp, act)
    before = {f: b.get(f) for f in UNTOUCHED if b.field_size(f)}
    n0 = b.launch_count()
    b.inverse(); b.sync()
    assert b.launch_count() - n0 == 1
    ods = [oracle_inverse(m, dict(inp, **({"act": act} if m.na else {})), e) for e in range(nenv)]
    check_against_oracle(m, b.get, nenv, ods, 1e-9)   # no solve: the elliptic models need no looser gate
    for f, v in before.items():
        assert np.array_equal(b.get(f), v), f


BATCH_KINDS = {"fused": dict(), "generic": dict(specialize=False), "staged_coop": dict(mode="staged", coop_solver=1),
               "staged_graph": dict(mode="staged", use_graph=True), "coop": dict(mode="coop")}


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cheetah", "humanoid"])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_gpu_inverse_identical_on_every_batch_kind(name, precision):
    """The same inputs give bit-identical qfrc_inverse whatever the batch runs its steps with, also after steps of that kind
    (the coop step stores rows env-contiguously, the specialised step keeps intermediates on chip)."""
    m = ox.Model.from_xml_string(ox.models.CONFIGS[name]["xml"])
    nenv = 96
    inp = inputs(m, nenv, seed=53)
    outs = {}
    for kind, kw in BATCH_KINDS.items():
        b = ox.BatchedPhysics(m, nenv, precision=precision, **kw)
        b.ctrl_philox(True, SEED); b.step(3)
        b.ctrl_philox(False)
        _load(b, m, inp)
        b.inverse(); b.sync()
        nefc = b.get("nefc")[:, 0]
        efc = b.get("efc_force", dtype=np.float64)
        outs[kind] = (b.get("qfrc_inverse", dtype=np.float64), b.get("sensordata", dtype=np.float64), nefc,
                      np.concatenate([efc[e, :n] for e, n in enumerate(nefc)]))   # rows past nefc hold whatever earlier steps left
    for kind, o in outs.items():
        for a, r in zip(o, outs["fused"]):
            assert np.array_equal(a, r), kind


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODELS))
def test_gpu_fp32_inverse_normwise(name):
    """fp32 against the fp64 oracle, per env: |qfrc_inverse - ref| <= c eps32 (|M| |qacc| + |bias| + |passive| + |J'| |f|)
    (2-norms, |M| and |J'| Frobenius). Measured worst ratio on a B200: see C_FP32."""
    m = ox.Model.from_xml_string(MODELS[name])
    nenv = 64
    inp = inputs(m, nenv, seed=54)
    b = ox.BatchedPhysics(m, nenv, precision="f32")
    _load(b, m, inp)
    b.inverse(); b.sync()
    got = b.get("qfrc_inverse")
    worst = 0.0
    for e in range(nenv):
        od = oracle_inverse(m, inp, e)
        nefc = od.int("nefc")
        J = od.field("efc_J")[:nefc * m.nv].reshape(nefc, m.nv)
        M = np.zeros((m.nv, m.nv))
        for i in range(m.nv):
            M[:, i] = mul_m(m, od.field("qM"), np.eye(m.nv)[i])
        scale = (np.linalg.norm(M) * np.linalg.norm(inp["qacc"][e]) + np.linalg.norm(od.field("qfrc_bias")) + np.linalg.norm(od.field("qfrc_passive"))
                 + np.linalg.norm(J) * np.linalg.norm(od.field("efc_force")[:nefc]))
        worst = max(worst, np.linalg.norm(got[e] - od.field("qfrc_inverse")) / (np.finfo(np.float32).eps * max(scale, 1e-30)))
    print(f"{name}: worst normwise fp32 error {worst:.3g} eps32")
    assert worst <= C_FP32, worst


# measured on one NVIDIA B200 (1000 W, 1965 MHz): worst ratio 1.57e3 (zoo_q), 650 (zoo_n), 404 (zoo_g), 358 (cheetah),
# 67 (humanoid), <= 5 on the contact-free models; the bound is 2.5 x the worst
C_FP32 = 4000.0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cheetah", "humanoid"])
def test_gpu_inverse_does_not_perturb_the_simulation(name):
    m = ox.Model.from_xml_string(ox.models.CONFIGS[name]["xml"])
    nenv = 128
    qpos, qvel = random_state(m, nenv, seed=55)
    a, t = ox.BatchedPhysics(m, nenv, precision="f32"), ox.BatchedPhysics(m, nenv, precision="f32")
    assert "generic" not in a.kernel_name()
    for b in (a, t):
        b.set("qpos", qpos); b.set("qvel", qvel); b.ctrl_philox(True, SEED); b.step(5)
    n0 = a.launch_count()
    a.inverse()
    assert a.launch_count() - n0 == 1
    a.sync()
    for f in ("xpos", "qM", "efc_force", "qfrc_constraint", "qfrc_inverse"):   # readable after the inverse, no stale refusal
        a.get(f)
    for b in (a, t):
        b.step(5); b.sync()
    for f in ("qpos", "qvel", "qacc", "sensordata", "ctrl"):
        assert np.array_equal(a.get(f), t.get(f)), f


@pytest.mark.gpu
@pytest.mark.parametrize("nenv", [1, 33, 1000])
def test_gpu_inverse_ragged_sizes_and_forward_fields(nenv):
    m = ox.Model.from_xml_string(ox.models.CHEETAH)
    inp = inputs(m, nenv, seed=56)
    b = ox.BatchedPhysics(m, nenv, precision="f64")
    _load(b, m, inp)
    b.inverse(); b.sync()
    inv = {f: b.get(f) for f in QACC_FREE + ["qfrc_inverse"]}
    for e in sorted({0, nenv // 2, nenv - 1}):
        od = oracle_inverse(m, inp, e)
        assert rel_err(inv["qfrc_inverse"][e], od.field("qfrc_inverse")) <= 1e-9
    b.forward(); b.sync()
    for f in QACC_FREE:    # what does not depend on qacc equals ox_batch_forward's values
        assert rel_err(inv[f], b.get(f)) <= 1e-12, f
