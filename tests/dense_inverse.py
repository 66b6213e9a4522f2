"""Inverse dynamics (mj_inverse, continuous time) restated with the dense whole-step checker's machinery (tests/dense_checker.py,
which stays as it is): dense M, Kane bias, the passive force, and constraint forces by autograd from the same row penalties and
cone cost its solver minimises. Test infrastructure only."""
from __future__ import annotations

import numpy as np
import torch

from dense_checker import DenseModel, Kin, _T, collide, constraints, fluid_force, mass_matrix_and_bias, passive_force, tendons


def _row_penalty(xt, D, ne, floss, ell):
    """The constraint part of the objective solve_qacc_autodiff minimises, as a function of x = J qacc - aref (torch)."""
    n, nf = len(D), len(floss)
    Dt = _T(D)
    inell = np.zeros(n, bool)
    for r0, dim, _, _ in ell:
        inell[r0:r0 + dim] = True
    two_sided = _T((np.arange(n) < ne + nf).astype(float))
    quad = torch.where(two_sided > 0, xt, torch.clamp(xt, max=0.0))
    rowc = 0.5 * Dt * quad ** 2
    if nf:
        fl = np.zeros(n)
        fl[ne:ne + nf] = floss
        flt, band = _T(fl), _T(np.where(fl > 0, fl / np.asarray(D), np.inf))
        rowc = torch.where(torch.abs(xt) >= band, flt * (torch.abs(xt) - 0.5 * flt / Dt), rowc)
    pc = torch.sum(rowc * _T((~inell).astype(float)))
    for r0, dim, mu, fri in ell:
        xc = xt[r0:r0 + dim]
        N = xc[0] * mu
        U = xc[1:] * _T(fri)
        Tn = torch.sqrt(torch.sum(U * U))
        if N >= mu * Tn:
            continue
        if mu * N + Tn <= 0:
            pc = pc + 0.5 * torch.sum(Dt[r0:r0 + dim] * xc ** 2)
        else:
            pc = pc + 0.5 * Dt[r0] / (mu * mu * (1 + mu * mu)) * (N - mu * Tn) ** 2
    return pc


def inverse(dm: DenseModel, qpos, qvel, qacc, mocap=None, eq_active=None):
    """mj_inverse (continuous time): qfrc_inverse = M qacc + c - passive - J' f with the dense M, the Kane bias c, the passive
    force (springs, dampers, fluid, gravity compensation) and f = -d(penalty)/dx at x = J qacc - aref, by autograd. Applied and
    actuator forces do not enter. Returns qfrc_inverse, the row forces and the pieces."""
    qpos, qvel, qacc = np.asarray(qpos, float), np.asarray(qvel, float), np.asarray(qacc, float)
    kin = Kin(dm, qpos, qvel, mocap)
    tendons(dm, kin, qpos)
    M, c = mass_matrix_and_bias(dm, kin)
    passive = passive_force(dm, qpos, qvel)
    if not dm.dis("passive"):
        passive = passive + fluid_force(dm, kin)
        if dm.m.ngravcomp and not dm.dis("gravity"):
            gc = np.asarray(dm.m.body_gravcomp, float)
            for b in range(1, dm.nbody):
                if gc[b]:
                    com = kin.P[b] + kin.R[b] @ dm.body_ipos[3 * b:3 * b + 3]
                    passive = passive + kin.point_jac(b, com).T @ (-dm.gravity * dm.body_mass[b] * gc[b])
    cons = collide(dm, kin)
    J, D, aref, ne = constraints(dm, kin, qpos, qvel, cons, eq_active)
    force = np.zeros(J.shape[0])
    if J.shape[0]:
        xt = _T(J @ qacc - aref).requires_grad_(True)
        pc = _row_penalty(xt, D, ne, dm._floss, dm._ell)
        if pc.requires_grad:
            gx, = torch.autograd.grad(pc, xt, allow_unused=True)
            if gx is not None:
                force = -gx.numpy()
    qfrc_constraint = J.T @ force if len(force) else np.zeros(dm.nv)
    return dict(qfrc_inverse=M @ qacc + c - passive - qfrc_constraint, efc_force=force, qfrc_constraint=qfrc_constraint, M=M,
                qfrc_bias=c, qfrc_passive=passive, ncon=len(cons), nefc=J.shape[0])
