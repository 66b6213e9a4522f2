// Lane-group dense solves shared by the warp-per-env Newton solve (k_solve_coop, ox_solve_coop.cu) and the group-per-env
// step kernel (k_step_coop, ox_coop.cu). One group of G lanes (16 or 32, within one warp) owns one environment, lane = dof:
//   * every dof-vector (qacc, M*qacc, grad, search, ...) is one register per lane,
//   * lane i owns row i of the dense Hessian H = M + J' D J in G registers: the rank-1 row updates read the staged J row
//     with broadcast shared-memory loads, the right-looking Cholesky exchanges one shuffle per (column, row) pair, the
//     triangular solves one shuffle per column. Only this block is unrolled (about 3 k instructions, one call site); v1
//     unrolled everything at three call sites (34 k instructions, `no_instruction` 10.7 cycles per issue -
//     profiles/r1_ncu_coop_v1_humanoid_f32_4096.txt), v2/v3 kept H in shared memory (4 instructions and a shared-memory
//     round trip per multiply-add); M's row also stays in registers,
//   * constraint rows are dealt round-robin over lanes (row r -> lane r % G) for jar / Jv / line search,
//   * the first COOP_SROWS rows of J are staged once per solve into shared memory ([row][dof], padded): the batch stores J
//     [element][env] (lane = env layout), which a lane = dof group can only gather from.
// Same algorithm, stopping rules and warm start as Env::fwd_constraint (ox_stages.cuh); only the summation order differs.
#pragma once

#include "ox_stages.cuh"

namespace ox {

constexpr int COOP_SROWS = 32;  // rows of J staged in shared memory per group; the rest is read from the batch

template <int G>
struct LaneGroup {
  int lane;        // lane in group
  unsigned mask;   // lanes of this group within the warp
  __device__ __forceinline__ void sync() const { __syncwarp(mask); }
  template <typename V> __device__ __forceinline__ V shfl(V v, int src) const { return __shfl_sync(mask, v, src, G); }
  template <typename V> __device__ __forceinline__ V sum(V v) const {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o, G);
    return v;
  }
};

// index of element i of one environment's batch field: the arena keeps it at i * stride + env; a per-group view of one
// environment (k_step_coop) is {1, 0}
struct ElemAt {
  uint32_t stride, env;
  __device__ __forceinline__ uint32_t operator()(int i) const { return (uint32_t)i * stride + env; }
};

// row `lane` of the dense mass matrix from the sparse qM (0 beyond nv / for idle lanes)
template <typename T, int G>
__device__ __forceinline__ void group_load_mrow(const LaneGroup<G>& g, const DevModel<T>& m, const T* qM, ElemAt at, T (&Mr)[G]) {
  const int nv = m.h().nv;
#pragma unroll
  for (int j = 0; j < G; j++) {
    Mr[j] = 0;
    if (j < nv && g.lane < nv) {
      const int idx = m.dof_Mdense(g.lane * nv + j);
      if (idx >= 0) Mr[j] = qM[at(idx)];
    }
  }
}

// H (symmetric positive definite, nv x nv): lane i passes row i in Hr[0..nv); returns x_i of H x = rhs. Destroys Hr.
// sL: [G][G + 1] shared scratch for the back substitution.
template <typename T, int G>
__device__ __forceinline__ T group_chol_solve(const LaneGroup<G>& g, T (&Hr)[G], T rhs, int nv, T* sL) {
  // right-looking Cholesky on the register rows: at step kk lane i >= kk turns H[i][kk] into L[i][kk] and every lane
  // subtracts L[i][kk] * L[j][kk] (lane j's value, one shuffle) from H[i][j]. Entries above the diagonal and the rows
  // of idle lanes hold finite garbage that is never read.
  T dinv = 1;
#pragma unroll
  for (int kk = 0; kk < G; kk++) {
    if (kk < nv) {  // group-uniform
      const T piv = g.shfl(Hr[kk], kk);
      const T inv = ox_rsqrt(ox_max(piv, (T)OX_MINVAL));  // 1 / L[kk][kk]; the diagonal itself is never needed
      const T lik = Hr[kk] * inv;
      Hr[kk] = lik;
      if (g.lane == kk) dinv = inv;
#pragma unroll
      for (int j = kk + 1; j < G; j++) Hr[j] -= lik * g.shfl(lik, j);
    }
  }
  T acc = rhs, y = 0;
#pragma unroll
  for (int kk = 0; kk < G; kk++) {  // L y = rhs, column-oriented
    if (kk < nv) {
      const T yk = g.shfl(acc * dinv, kk);
      if (g.lane == kk) y = yk;
      if (g.lane > kk) acc -= Hr[kk] * yk;
    }
  }
  // L' x = y, column-oriented: lane j needs L[kk][j], which sits in lane kk's register j - so the factor goes through
  // shared memory once (row kk contiguous: conflict-free reads) instead of one butterfly reduction per column
#pragma unroll
  for (int j = 0; j < G; j++) sL[g.lane * (G + 1) + j] = Hr[j];
  g.sync();
  T x = 0;
  acc = y;
  for (int kk = nv - 1; kk >= 0; kk--) {
    const T xk = g.shfl(acc * dinv, kk);
    if (g.lane == kk) x = xk;
    if (g.lane < kk) acc -= sL[kk * (G + 1) + g.lane] * xk;
  }
  g.sync();
  return x;
}

// The Newton solve of one environment (Env::fwd_constraint, rows over lanes): qacc, qacc_warmstart, qfrc_constraint,
// efc_force and solver_niter from qM, qfrc_smooth, qacc_smooth, qacc_warmstart and the constraint rows (efc_J, efc_D,
// efc_aref, nefc, ne). Batch element i is b.field[at(i)]. Scratch: sJ [COOP_SROWS][G + 1], sL [G][G + 1], srow 5 x RCAP.
// An environment with at most RCAP rows keeps its per-row scalars in srow (stride 1); otherwise they live in the batch's
// own row arrays (efc_D and efc_aref read in place; jar, Jv and force in s_Jaref, s_Jv, efc_force). Ends with a group sync.
template <typename T, int G, int RCAP>
__device__ __forceinline__ void group_newton(const LaneGroup<G>& g, const DevModel<T>& m, const DevBatch<T>& b, ElemAt at, T* sJ, T* sL, T* srow) {
  const BlobHeader& h = m.h();
  const int nv = h.nv, lane = g.lane;
  const bool me = lane < nv;
  const int nefc = b.nefc[at.env], ne = b.ne[at.env];   // rows below ne are equality rows: active on both sides
  if (nefc == 0) {
    if (me) {
      const T a = b.qacc_smooth[at(lane)];
      b.qacc[at(lane)] = a; b.qacc_warmstart[at(lane)] = a; b.qfrc_constraint[at(lane)] = 0;
    }
    if (lane == 0) b.solver_niter[at.env] = 0;
    g.sync();
    return;
  }
  const bool small = RCAP > 0 && nefc <= RCAP;
  const uint32_t rs = small ? 1u : at.stride;
  T* rowD = small ? srow : b.efc_D + at.env;
  T* rowA = small ? rowD + RCAP : b.efc_aref + at.env;
  T* rowJar = small ? rowA + RCAP : b.s_Jaref + at.env;
  T* rowJv = small ? rowJar + RCAP : b.s_Jv + at.env;
  T* rowF = small ? rowJv + RCAP : b.efc_force + at.env;
#define ROW(arr, r) arr[(uint32_t)(r) * rs]
  const int nsm = nefc < COOP_SROWS ? nefc : COOP_SROWS;
  for (int r = 0; r < nsm; r++)
    sJ[r * (G + 1) + lane] = me ? b.efc_J[at(r * nv + lane)] : (T)0;
  if (small)
    for (int r = lane; r < nefc; r += G) { rowD[r] = b.efc_D[at(r)]; rowA[r] = b.efc_aref[at(r)]; }
  g.sync();
  auto Jat = [&](int r, int i) -> T { return r < COOP_SROWS ? sJ[r * (G + 1) + i] : b.efc_J[at(r * nv + i)]; };

  const T fs = me ? b.qfrc_smooth[at(lane)] : (T)0, as = me ? b.qacc_smooth[at(lane)] : (T)0, aw = me ? b.qacc_warmstart[at(lane)] : (T)0;
  T Mrow[G];
  group_load_mrow(g, m, b.qM, at, Mrow);
  auto Mdot = [&](T x) -> T {  // (M x)_lane, x distributed one element per lane
    T acc = 0;
#pragma unroll
    for (int j = 0; j < G; j++)
      if (j < nv) acc += Mrow[j] * g.shfl(x, j);
    return acc;
  };
  auto Jdot = [&](T x, T* out, bool minus_aref) {  // out[r] = J_r . x (- aref_r), rows round-robin over lanes
    for (int r0 = 0; r0 < nefc; r0 += G) {
      const int r = r0 + lane;
      T acc = 0;
#pragma unroll 4
      for (int i = 0; i < nv; i++) {
        const T xi = g.shfl(x, i);
        if (r < nefc) acc += Jat(r, i) * xi;
      }
      if (r < nefc) ROW(out, r) = minus_aref ? acc - ROW(rowA, r) : acc;
    }
    g.sync();
  };

  // warm start: cheaper of cost(qacc_warmstart), cost(qacc_smooth), through one evaluation site
  bool use_smooth = true;
  if (!(h.disableflags & OX_DSBL_WARMSTART)) {
    T cand[2];
#pragma unroll 1
    for (int c = 0; c < 2; c++) {
      const T x = c ? as : aw;
      const T Mx = Mdot(x);
      T cc = me ? (T)0.5 * (Mx - fs) * (x - as) : (T)0;
      Jdot(x, rowJv, true);
      for (int r = lane; r < nefc; r += G) {
        const T v = ROW(rowJv, r);
        if (v < 0 || r < ne) cc += (T)0.5 * ROW(rowD, r) * v * v;
      }
      cand[c] = g.sum(cc);
      g.sync();
    }
    use_smooth = cand[0] > cand[1];
  }
  T a = use_smooth ? as : aw;
  T Ma = Mdot(a);
  Jdot(a, rowJar, true);

  T fc = 0, gauss = 0, cost = 0, grad = 0, Mgrad = 0, gnorm = 0, search = 0;
  const T tol = (T)h.tolerance;
  const T mscale = (T)h.meaninertia * (T)(nv > 1 ? nv : 1);
  const T scale = (T)1 / mscale;
  const int maxiter = h.iterations;
  int iter = 0;
  bool init = true;
#pragma unroll 1
  for (;;) {
    if (!init) {
      if (iter >= maxiter) break;
      // ---- exact line search on the convex piecewise-quadratic phi(alpha)
      const T snorm = ox_sqrt(g.sum(search * search));
      if (snorm < (T)OX_MINVAL) break;
      const T gtol = tol * (T)h.ls_tolerance * snorm * mscale;
      const T Mv = Mdot(search);
      Jdot(search, rowJv, false);
      const T qg1 = g.sum(me ? search * (Ma - fs) : (T)0), qg2 = g.sum(me ? (T)0.5 * search * Mv : (T)0);
      T p0c = 0, p0d0 = 0, cur_a = 0, cur_c = 0, cur_d0 = 0, cur_d1 = 1, lo_a = 0, hi_a = 0;
      bool have_hi = false, stop = false;
#pragma unroll 1
      for (int it = -1; it < h.ls_iterations && !stop; it++) {  // it = -1 evaluates alpha = 0
        T an = 0;
        if (it >= 0) {
          an = cur_a - cur_d0 / cur_d1;
          if (have_hi && !(an > lo_a && an < hi_a)) an = (T)0.5 * (lo_a + hi_a);
          if (ox_abs(an - cur_a) <= Eps<T>::v() * ox_abs(an)) break;
        }
        T c = 0, d0 = 0, d1 = 0, s0 = 0;
        for (int r = lane; r < nefc; r += G) {
          const T ja = ROW(rowJar, r), jvr = ROW(rowJv, r);
          const T x = ja + an * jvr;
          if (x < 0 || r < ne) {
            const T Dx = ROW(rowD, r) * x, Dj = ROW(rowD, r) * jvr;
            c += (T)0.5 * Dx * x;
            d0 += Dx * jvr;
            d1 += Dj * jvr;
            s0 += ox_abs(Dx * jvr);
          }
        }
        cur_a = an;
        cur_c = an * an * qg2 + an * qg1 + gauss + g.sum(c);
        cur_d0 = 2 * an * qg2 + qg1 + g.sum(d0);
        cur_d1 = 2 * qg2 + g.sum(d1);
        const T cur_s0 = ox_abs(2 * an * qg2) + ox_abs(qg1) + g.sum(s0);
        if (cur_d1 < (T)OX_MINVAL) cur_d1 = (T)OX_MINVAL;
        if (it < 0) {
          p0c = cur_c; p0d0 = cur_d0;
          if (!(p0d0 < 0)) stop = true;
        } else {
          if (ox_abs(cur_d0) < gtol || ox_abs(cur_d0) <= 8 * Eps<T>::v() * cur_s0) break;
          if (cur_d0 < 0) lo_a = cur_a; else { hi_a = cur_a; have_hi = true; }
        }
      }
      if (stop) break;
      const T alpha = cur_c <= p0c ? cur_a : (T)0;
      if (alpha == 0) break;
      a += alpha * search;
      Ma += alpha * Mv;
      for (int r = lane; r < nefc; r += G) ROW(rowJar, r) += alpha * ROW(rowJv, r);
      g.sync();
    }
    const T oldcost = cost;
    // ---- efc_force, qfrc_constraint, cost at (a, Ma, jar)
    {
      T crow = 0;
      for (int r = lane; r < nefc; r += G) {
        const T ja = ROW(rowJar, r);
        T f = 0;
        if (ja < 0 || r < ne) { f = -ROW(rowD, r) * ja; crow += (T)0.5 * ROW(rowD, r) * ja * ja; }
        ROW(rowF, r) = f;
      }
      g.sync();
      fc = 0;
      for (int r = 0; r < nefc; r++) {
        const T f = ROW(rowF, r);
        if (f != 0 && me) fc += Jat(r, lane) * f;
      }
      gauss = g.sum(me ? (T)0.5 * (Ma - fs) * (a - as) : (T)0);
      cost = g.sum(crow) + gauss;
    }
    // ---- gradient, H = M + J' D_active J (row `lane` in registers), Cholesky, Mgrad = H^-1 grad
    {
      grad = me ? Ma - fs - fc : (T)0;
      gnorm = ox_sqrt(g.sum(grad * grad));
      // static indices only: the j loops are fully unrolled, the row loop is not
      T Hreg[G];
#pragma unroll
      for (int j = 0; j < G; j++) Hreg[j] = Mrow[j];
      for (int r = 0; r < nefc; r++) {
        if (!(ROW(rowJar, r) < 0 || r < ne)) continue;  // group-uniform
        if (r < COOP_SROWS) {
          const T* jr = sJ + r * (G + 1);  // padding columns nv..G-1 are zero
          const T s = ROW(rowD, r) * jr[lane];
#pragma unroll
          for (int j = 0; j < G; j++) Hreg[j] += s * jr[j];  // broadcast reads
        } else {
          const T Jri = me ? b.efc_J[at(r * nv + lane)] : (T)0;
          const T s = ROW(rowD, r) * Jri;
#pragma unroll
          for (int j = 0; j < G; j++) Hreg[j] += s * g.shfl(Jri, j);
        }
      }
      Mgrad = group_chol_solve(g, Hreg, grad, nv, sL);
    }
    if (init) {
      init = false;
      if (scale * gnorm < tol) break;
    } else {
      iter++;
      const T improvement = scale * (oldcost - cost), gradient = scale * gnorm;
      if (improvement < tol || gradient < tol) break;
      if (oldcost - cost <= OX_FLOOR_MULT * Eps<T>::v() * (ox_abs(oldcost) + ox_abs(cost))) break;
    }
    search = -Mgrad;
  }
  if (me) { b.qacc[at(lane)] = a; b.qacc_warmstart[at(lane)] = a; b.qfrc_constraint[at(lane)] = fc; }
  if (small)
    for (int r = lane; r < nefc; r += G) b.efc_force[at(r)] = ROW(rowF, r);
  if (lane == 0) b.solver_niter[at.env] = iter;
  g.sync();
#undef ROW
}

}  // namespace ox
