// Cooperative step kernel: ONE LANE GROUP (G = 16 or 32 lanes) PER ENVIRONMENT for the whole of mj_step, the mapping north_star
// asks for ("one environment per warp or per thread group, shuffle reductions for the small dense solves").
//
// Why: thread-per-env gives a humanoid-class batch (4096 envs, nv = 27) only 128 warps for 592 schedulers, each streaming a
// 50 k-instruction straight-line body at ~12 cycles per instruction (profiles/r2_notes.md); only the Newton solve ran one
// warp per env (ox_solve_coop.cu). Here every stage does:
//   * per-env mjData intermediates live in SHARED MEMORY (a per-group DevBatch view, stride 1), the model tables next to them
//     (one TMA bulk copy per CTA); only the state crosses HBM - plus the constraint rows and the contact list, which are
//     too large for shared memory (humanoid: 342 x 27 words of J) and live env-contiguous in the batch's own arena regions;
//   * the arithmetic is the SAME per-item code as the thread-per-env kernels (Env::kin_body, cinert_body, mass_row, vel_body,
//     rne_fwd_body, collide_pair, contact_rows, ... in ox_stages.cuh): a loop over bodies / joints / dofs / geoms / pairs /
//     contacts hands item i to lane i % G; tree passes run level by level (parents before children, or children gathered
//     by their parent - no atomics, deterministic summation order) with a group barrier between levels;
//   * the dense solves (qacc_smooth = M^-1 f, the Newton step, Euler's implicit damping) are the register-row Cholesky of
//     ox_group_solve.cuh: lane i owns row i, one shuffle per (column, row) pair;
//   * the Newton solver is group_newton (ox_group_solve.cuh), the one k_solve_coop runs, with rows dealt round-robin to lanes.
// Generic: any model the compiler accepts with nv <= G, the Newton solver and Euler / implicitfast integration (others keep
// the thread-per-env kernels). No model-specific code is generated.
#include "ox_kernels.cuh"
#include "ox_group_solve.cuh"
#include "ox_spec.cuh"   // StepArgs

#ifndef OX_COOP_THREADS
#define OX_COOP_THREADS 128
#endif

namespace ox {

constexpr int COOP_THREADS = OX_COOP_THREADS;  // 128: 4 (G = 32) or 8 (G = 16) envs per CTA; the register rows of the dense solves want > 128 registers per thread

// ---- per-group shared-memory layout: [DevBatch<T> view][int scalars + body levels][real fields][solver scratch]
template <typename T>
struct CoopSizes {
  int nq, nv, nu, na, nb, nj, ng, ns, nM, ncm, nem, nsd, nmc, neq, nten;
  OX_HD static CoopSizes from(const BlobHeader& h) {
    CoopSizes s;
    s.nq = h.nq; s.nv = h.nv; s.nu = h.nu; s.na = h.na; s.nb = h.nbody; s.nj = h.njnt; s.ng = h.ngeom; s.ns = h.nsite; s.nM = h.nM;
    s.ncm = h.nconmax > 1 ? h.nconmax : 1; s.nem = h.nefcmax > 1 ? h.nefcmax : 1; s.nsd = h.nsensordata; s.nmc = h.nmocap; s.neq = h.neq; s.nten = h.ntendon;
    return s;
  }
};
constexpr int COOP_NINT = 16;  // int scalars (ncon, nefc, ...) rounded up

// words of T of shared memory one group needs (G enters through the solver scratch)
template <typename T>
OX_HD size_t coop_group_bytes(const CoopSizes<T>& z, int G) {
  const long nq = z.nq, nv = z.nv, nu = z.nu, na = z.na, nb = z.nb, nj = z.nj, ng = z.ng, ns = z.ns, nM = z.nM, nsd = z.nsd, nmc = z.nmc, neq = z.neq, nten = z.nten;
  (void)nq; (void)nv; (void)nu; (void)na; (void)nb; (void)nj; (void)ng; (void)ns; (void)nM; (void)nsd; (void)nmc; (void)neq; (void)nten;
  size_t words = 0;
#define OX_X(name, cnt) words += (size_t)((cnt) > 0 ? (cnt) : 1);
  OX_BATCH_REAL_FIELDS_SMALL(OX_X)
#undef OX_X
  words += (size_t)COOP_SROWS * (G + 1) + (size_t)G * (G + 1);
  size_t bytes = sizeof(DevBatch<T>) + (COOP_NINT + (size_t)z.nb) * sizeof(int32_t);
  bytes = (bytes + 15) / 16 * 16 + words * sizeof(T);
  return (bytes + 15) / 16 * 16;
}

#if defined(__CUDACC__)

template <typename T, int G>
struct Coop : LaneGroup<G> {
  using LaneGroup<G>::lane;
  using LaneGroup<G>::mask;
  using LaneGroup<G>::sync;
  using LaneGroup<G>::sum;
  using E = Env<T, DevModel<T>, true>;
  E& env;
  int32_t* level;          // [nbody] depth of each body in the tree (world = 0)
  int maxlevel;
  T* sJ;                   // [COOP_SROWS][G + 1]
  T* sL;                   // [G][G + 1]

  __device__ __forceinline__ bool gany(bool p) const { return __ballot_sync(mask, p) != 0u; }
  // exclusive prefix sum over the lanes of the group
  __device__ __forceinline__ int gscan_excl(int v) const {
    int x = v;
#pragma unroll
    for (int o = 1; o < G; o <<= 1) {
      const int y = __shfl_up_sync(mask, x, o, G);
      if (lane >= o) x += y;
    }
    return x - v;
  }

  // ------------------------------------------------------------------ tree helpers
  __device__ void compute_levels() {
    const auto& m = env.m;
    const int nb = m.h().nbody;
    int mx = 0;
    for (int i = lane; i < nb; i += G) {
      int d = 0;
      for (int p = i; p > 0; p = m.body_parentid(p)) d++;
      level[i] = d;
      mx = d > mx ? d : mx;
    }
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) { const int y = __shfl_xor_sync(mask, mx, o, G); mx = y > mx ? y : mx; }
    maxlevel = mx;
    sync();
  }
  // f(i) for every body of each level in turn, parents first
  template <class F> __device__ __forceinline__ void down(int first_level, F f) const {
    const int nb = env.m.h().nbody;
    for (int lv = first_level; lv <= maxlevel; lv++) {
      for (int i = lane; i < nb; i += G)
        if (level[i] == lv) f(i);
      sync();
    }
  }
  // field[w*p .. w*p+w) += sum over children c of p (ascending c) of field[w*c ..), deepest parents first; bodies above
  // `top_level` (0 = include the world) are left alone
  template <int W> __device__ __forceinline__ void gather_up(T* field, int top_level) const {
    const auto& m = env.m;
    const int nb = m.h().nbody;
    for (int lv = maxlevel - 1; lv >= top_level; lv--) {
      for (int p = lane; p < nb; p += G) {
        if (level[p] != lv) continue;
        T acc[W];
#pragma unroll
        for (int k = 0; k < W; k++) acc[k] = field[W * p + k];
        for (int c = p + 1; c < nb; c++) {
          if (m.body_parentid(c) != p) continue;
#pragma unroll
          for (int k = 0; k < W; k++) acc[k] += field[W * c + k];
        }
#pragma unroll
        for (int k = 0; k < W; k++) field[W * p + k] = acc[k];
      }
      sync();
    }
  }
  template <class F> __device__ __forceinline__ void each(int n, F f) const {
    for (int i = lane; i < n; i += G) f(i);
  }

  // ------------------------------------------------------------------ forward dynamics up to the constraint rows
  __device__ void fwd_position() const {
    const auto& m = env.m;
    const auto& h = m.h();
    const DevBatch<T>& b = env.b;
    const int nb = h.nbody;
    down(0, [&](int i) { env.kin_body(i); });
    each(h.ngeom, [&](int g) { env.kin_geom(g); });
    each(h.nsite, [&](int s) { env.kin_site(s); });
    // subtree com: mass-weighted sums gathered up the tree, then normalised
    each(nb, [&](int i) {
      const T mi = m.body_mass(i);
      for (int k = 0; k < 3; k++) b.subtree_com[3 * i + k] = b.xipos[3 * i + k] * mi;
    });
    sync();
    gather_up<3>(b.subtree_com, 0);
    each(nb, [&](int i) {
      const T sm = m.body_subtreemass(i);
      for (int k = 0; k < 3; k++) b.subtree_com[3 * i + k] = sm < (T)OX_MINVAL ? b.xipos[3 * i + k] : b.subtree_com[3 * i + k] / sm;
    });
    sync();
    each(nb, [&](int i) {
      if (i == 0) { for (int k = 0; k < 10; k++) b.cinert[k] = 0; } else env.cinert_body(i);
    });
    each(h.njnt, [&](int j) { env.cdof_joint(j); });
    sync();
    // composite inertias: own + children, gathered up to the bodies below the world; then one row of M per dof
    each(10 * nb, [&](int k) { b.crb[k] = b.cinert[k]; });
    sync();
    gather_up<10>(b.crb, 1);
    each(h.nv, [&](int i) { env.mass_row(i); });
    // narrowphase: one candidate pair per lane, contacts into the static slots of the pair
    each(h.nconmax > 0 ? h.nconmax : 1, [&](int c) { b.con_active[c] = 0; });
    sync();
    int mine = 0;
    if (!(env.dis(OX_DSBL_CONTACT) || env.dis(OX_DSBL_CONSTRAINT))) each(h.npair, [&](int p) { env.collide_pair(p, mine); });
    const int ncon = sum(mine);
    if (lane == 0) b.ncon[0] = ncon;
    sync();
  }
  __device__ void fwd_velocity() const {
    const auto& m = env.m;
    const auto& h = m.h();
    const DevBatch<T>& b = env.b;
    if (lane < 6) b.cvel[lane] = 0;
    if (lane == 0) {
      T a0[6] = {0, 0, 0, 0, 0, 0};
      if (!env.dis(OX_DSBL_GRAVITY)) { a0[3] = -(T)h.grav(0); a0[4] = -(T)h.grav(1); a0[5] = -(T)h.grav(2); }
      for (int k = 0; k < 6; k++) { b.cacc[k] = a0[k]; b.cfrc[k] = 0; }
    }
    each(h.nv, [&](int i) { b.qfrc_passive[i] = 0; });
    each(h.ntendon, [&](int i) { env.tendon_length(i); });
    sync();
    down(1, [&](int i) { env.vel_body(i); });
    if (!env.dis(OX_DSBL_PASSIVE)) {
      each(h.njnt, [&](int j) { env.passive_joint(j); });
      sync();
      each(h.nv, [&](int i) { b.qfrc_passive[i] -= m.dof_damping(i) * b.qvel[i]; });
      if (h.ntendon > 0) {   // a tendon touches several dofs: one lane applies them in order
        sync();
        if (lane == 0) for (int i = 0; i < h.ntendon; i++) env.passive_tendon(i);
      }
      if (h.nfluid > 0) {    // fluid drag: a body's wrench touches its whole dof chain, same rule
        sync();
        if (lane == 0) for (int bd = 1; bd < h.nfluid; bd++) env.passive_fluid(bd);
      }
      if (h.ngravcomp > 0 && !env.dis(OX_DSBL_GRAVITY)) {
        sync();
        if (lane == 0) for (int bd = 1; bd < h.ngravcomp; bd++) env.passive_gravcomp(bd);
      }
    }
    down(1, [&](int i) { env.rne_fwd_body(i); });
    gather_up<6>(b.cfrc, 1);
    each(h.nv, [&](int i) { env.rne_bias_dof(i); });
    sync();
  }
  // constraint rows: counts per item, exclusive scan across the group, rows written in place - same row order as the serial code
  __device__ void make_constraint() const {
    const auto& m = env.m;
    const auto& h = m.h();
    const DevBatch<T>& b = env.b;
    int base = 0;
    if (!env.dis(OX_DSBL_CONSTRAINT)) {
      if (!env.dis(OX_DSBL_EQUALITY)) {
        for (int i0 = 0; i0 < h.neq; i0 += G) {
          const int i = i0 + lane;
          const int cnt = i < h.neq ? env.equality_count(i) : 0;
          int r = base + gscan_excl(cnt);
          if (cnt) env.equality_rows(i, r);
          base += sum(cnt);
        }
      }
      if (lane == 0) b.ne[0] = base;
      if (!env.dis(OX_DSBL_LIMIT)) {
        for (int j0 = 0; j0 < h.njnt; j0 += G) {
          const int j = j0 + lane;
          const int cnt = j < h.njnt ? env.limit_count(j) : 0;
          int r = base + gscan_excl(cnt);
          if (cnt) env.limit_rows(j, r);
          base += sum(cnt);
        }
        for (int i0 = 0; i0 < h.ntendon; i0 += G) {
          const int i = i0 + lane;
          const int cnt = i < h.ntendon ? env.tendon_limit_count(i) : 0;
          int r = base + gscan_excl(cnt);
          if (cnt) env.tendon_limit_rows(i, r);
          base += sum(cnt);
        }
      }
      for (int c0 = 0; c0 < h.nconmax; c0 += G) {
        const int c = c0 + lane;
        int cnt = 0, p = 0;
        if (c < h.nconmax && b.con_active[c]) {
          p = b.con_pair[c];
          if (b.con_dist[c] < m.pair_margin(p) - m.pair_gap(p)) cnt = m.pair_dim(p) == 1 ? 1 : 2 * (m.pair_dim(p) - 1);
          else b.con_efcadr[c] = -1;
        }
        int r = base + gscan_excl(cnt);
        if (cnt) env.contact_rows(c, p, r);
        base += sum(cnt);
      }
    }
    if (lane == 0) { b.nefc[0] = base; if (env.dis(OX_DSBL_CONSTRAINT)) b.ne[0] = 0; }
    sync();
  }
  __device__ void actuation_and_smooth() const {
    const auto& m = env.m;
    const auto& h = m.h();
    const DevBatch<T>& b = env.b;
    each(h.nu, [&](int i) { (void)env.actuator_one(i); });
    sync();
    each(h.nv, [&](int d) {   // gather the actuators of this dof in index order (several may drive one joint)
      T f = 0;
      if (!env.dis(OX_DSBL_ACTUATION))
        for (int i = 0; i < h.nu; i++)
          if (m.jnt_dofadr(m.actuator_trnid(i)) == d) f += m.actuator_gear(i) * b.actuator_force[i];
      b.qfrc_actuator[d] = f;
      b.qfrc_smooth[d] = b.qfrc_passive[d] - b.qfrc_bias[d] + b.qfrc_applied[d] + f;
    });
    sync();
    if (applied) {
      if (lane == 0) env.apply_xfrc();
      sync();
    }
    T Mr[G];
    group_load_mrow(*this, m, b.qM, ElemAt{1, 0}, Mr);
    const T as = group_chol_solve(*this, Mr, lane < h.nv ? b.qfrc_smooth[lane] : (T)0, h.nv, sL);
    if (lane < h.nv) b.qacc_smooth[lane] = as;
    sync();
  }
  int applied = 1;

  bool live = true;   // false: a group of the tail CTA beyond nenv - it only keeps the CTA barriers company
  // CTA-wide barrier between stages: the warps of a CTA then stream the same part of the ~700 KB body at the same time and
  // share its instruction-cache fills, at the price of waiting for the slowest env of the CTA in the solver (humanoid 4096
  // envs: 1.19 -> 0.90 ms per step, 300 steps in one launch 2.5 x faster than without)
  __device__ __forceinline__ void stage_barrier() const { __syncthreads(); }
  __device__ void forward(bool skipsensor) const {
    if (live) fwd_position();
    stage_barrier();
    if (live) fwd_velocity();
    stage_barrier();
    if (live) make_constraint();
    stage_barrier();
    if (live) actuation_and_smooth();
    stage_barrier();
    if (live) group_newton<T, G, 0>(*this, env.m, env.b, ElemAt{1, 0}, sJ, sL, nullptr);   // per-row scalars stay in the arena
    stage_barrier();
    if (live && !skipsensor && env.m.h().nsensor > 0) {
      if (lane == 0) env.sensors();
      sync();
    }
  }

  // ------------------------------------------------------------------ checks, reset, integration
  __device__ bool bad_state() const {
    const auto& h = env.m.h();
    const DevBatch<T>& b = env.b;
    bool bad = false;
    each(h.nq, [&](int i) { bad |= ox_bad(b.qpos[i]); });
    each(h.nv, [&](int i) { bad |= ox_bad(b.qvel[i]); });
    each(h.na, [&](int i) { bad |= ox_bad(b.act[i]); });
    return gany(bad);
  }
  __device__ bool bad_acc() const {
    bool bad = false;
    each(env.m.h().nv, [&](int i) { bad |= ox_bad(env.b.qacc[i]); });
    return gany(bad);
  }
  __device__ void reset() const {
    if (lane == 0) { env.reset_data(); env.b.diverged[0] += 1; }
    sync();
  }
  __device__ void euler() const {
    const auto& m = env.m;
    const auto& h = m.h();
    const DevBatch<T>& b = env.b;
    const int nv = h.nv;
    const bool fast = h.integrator == OX_INT_IMPLICITFAST;
    const T dt = (T)h.timestep;
    T qa = lane < nv ? b.qacc[lane] : (T)0;
    if (fast || (h.any_damping && !env.dis(OX_DSBL_EULERDAMP))) {
      // (M + h B) qacc' = qfrc_smooth + qfrc_constraint, B as in Env::euler (joint damping; implicitfast: - actuator velocity derivative)
      T d = lane < nv ? dt * m.dof_damping(lane) : (T)0;
      if (fast && !env.dis(OX_DSBL_ACTUATION) && lane < nv) {
        const bool clamp = !env.dis(OX_DSBL_CLAMPCTRL);
        for (int i = 0; i < h.nu; i++) {
          if (m.jnt_dofadr(m.actuator_trnid(i)) != lane) continue;
          const bool gaff = m.actuator_gaintype(i) == OX_GAIN_AFFINE, baff = m.actuator_biastype(i) == OX_BIAS_AFFINE;
          if (!gaff && !baff) continue;
          if (m.actuator_forcelimited(i)) {
            const T f = b.actuator_force[i];
            if (f <= m.actuator_forcerange(2 * i) || f >= m.actuator_forcerange(2 * i + 1)) continue;
          }
          T input = b.ctrl[i];
          if (m.actuator_ctrllimited(i) && clamp) input = ox_clip(input, m.actuator_ctrlrange(2 * i), m.actuator_ctrlrange(2 * i + 1));
          if (m.actuator_dyntype(i) != OX_DYN_NONE) input = b.act[m.actuator_actadr(i)];
          const T gear = m.actuator_gear(i);
          d -= dt * gear * gear * ((gaff ? m.actuator_gainprm(3 * i + 2) * input : (T)0) + (baff ? m.actuator_biasprm(3 * i + 2) : (T)0));
        }
      }
      T Hr[G];
      group_load_mrow(*this, m, b.qM, ElemAt{1, 0}, Hr);
#pragma unroll
      for (int j = 0; j < G; j++)
        if (j == lane) Hr[j] += d;   // static register indices only (a runtime index would push the row into local memory)
      qa = group_chol_solve(*this, Hr, lane < nv ? b.qfrc_smooth[lane] + b.qfrc_constraint[lane] : (T)0, nv, sL);
    }
    // mj_advance: activations, velocities, then positions with the new velocities, time
    each(h.nu, [&](int i) {
      if (m.actuator_dyntype(i) == OX_DYN_NONE) return;
      const int aa = m.actuator_actadr(i);
      b.act[aa] = env.next_activation(i, b.act[aa], b.act_dot[aa]);
    });
    if (lane < nv) b.qvel[lane] += dt * qa;
    sync();
    each(h.njnt, [&](int j) { env.integrate_pos_joint(b.qpos, b.qvel, dt, j); });
    if (lane == 0) b.time[0] += dt;
    sync();
  }
  __device__ void step() const {
    if (live && bad_state()) reset();
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) {   // ONE call site of forward(): the second pass is mj_checkAcc's reset-and-redo
      forward(false);
      // (with CTA barriers inside forward() every group of the CTA must take the same number of passes)
      const bool mine = live && bad_acc();
      const bool redo = !pass && __syncthreads_or(mine) != 0;
      if (!redo) break;
      if (mine) reset();
    }
    if (!live) return;
    if (lane == 0) env.accumulate_stats();
    euler();
  }
};

template <typename T, int G>
__global__ void __launch_bounds__(COOP_THREADS, COOP_THREADS >= 256 ? 1 : 2) k_step_coop(const unsigned char* __restrict__ gblob, int bytes, DevBatch<T> g, StepArgs a, int group_bytes) {
  DevModel<T> m{stage_model(gblob, bytes)};
  extern __shared__ __align__(128) unsigned char ox_smem[];
  constexpr int GPC = COOP_THREADS / G;
  const int gic = threadIdx.x / G, gl = threadIdx.x % G;
  const int e_raw = blockIdx.x * GPC + gic;
  const bool live = e_raw < g.nenv;            // the spare groups of a tail CTA do no work but join the CTA barriers
  const int e = live ? e_raw : g.nenv - 1;
  const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (((threadIdx.x & 31) / G) * G));
  const BlobHeader& h = m.h();
  unsigned char* base = ox_smem + ((bytes + 127) / 128) * 128 + (size_t)gic * group_bytes;
  DevBatch<T>* lb = reinterpret_cast<DevBatch<T>*>(base);
  int32_t* ib = reinterpret_cast<int32_t*>(base + sizeof(DevBatch<T>));
  T* rb = reinterpret_cast<T*>(base + (sizeof(DevBatch<T>) + (COOP_NINT + (size_t)h.nbody) * sizeof(int32_t) + 15) / 16 * 16);
  const CoopSizes<T> z = CoopSizes<T>::from(h);
  if (gl == 0) {
    const long nq = z.nq, nv = z.nv, nu = z.nu, na = z.na, nb = z.nb, nj = z.nj, ng = z.ng, ns = z.ns, nM = z.nM, ncm = z.ncm, nem = z.nem, nsd = z.nsd, nmc = z.nmc, neq = z.neq, nten = z.nten;
    (void)nq; (void)nv; (void)nu; (void)na; (void)nb; (void)nj; (void)ng; (void)ns; (void)nM; (void)ncm; (void)nem; (void)nsd; (void)nmc; (void)neq; (void)nten;
    lb->nenv = 1; lb->stride = 1; lb->lanes = 32;
    T* p = rb;
#define OX_X(name, cnt) lb->name = p; p += ((cnt) > 0 ? (cnt) : 1);
    OX_BATCH_REAL_FIELDS_SMALL(OX_X)
#undef OX_X
    // rows and contacts: the batch's own arena regions, addressed env-contiguously ([env][element]) in this mode
#define OX_X(name, cnt) lb->name = g.name + (size_t)e * (size_t)((cnt) > 0 ? (cnt) : 1);
    OX_BATCH_REAL_FIELDS_ROWS(OX_X)
    OX_BATCH_INT_FIELDS_ROWS(OX_X)
#undef OX_X
    int32_t* q = ib;
#define OX_X(name, cnt) lb->name = q; q += 1;
    OX_BATCH_INT_FIELDS_SCALAR(OX_X)
#undef OX_X
  }
  __syncwarp(gmask);
  T* scratch = rb;
  {
    const long nq = z.nq, nv = z.nv, nu = z.nu, na = z.na, nb = z.nb, nj = z.nj, ng = z.ng, ns = z.ns, nM = z.nM, nsd = z.nsd, nmc = z.nmc, neq = z.neq, nten = z.nten;
    (void)nq; (void)nv; (void)nu; (void)na; (void)nb; (void)nj; (void)ng; (void)ns; (void)nM; (void)nsd; (void)nmc; (void)neq; (void)nten;
#define OX_X(name, cnt) scratch += ((cnt) > 0 ? (cnt) : 1);
    OX_BATCH_REAL_FIELDS_SMALL(OX_X)
#undef OX_X
  }
  Env<T, DevModel<T>, true> env(m, *lb, 0);
  env.slots = true;
  Coop<T, G> c{{gl, gmask}, env, ib + COOP_NINT, 0, scratch, scratch + COOP_SROWS * (G + 1)};
  c.applied = a.applied;
  c.live = live;
  c.compute_levels();
  const DevBatch<T>& b = *lb;
  const uint32_t S = (uint32_t)g.stride, ue = (uint32_t)e;
#define GA(field, i) g.field[(uint32_t)(i) * S + ue]
  // ---- state in (SURVEY 8d): qpos, qvel, act, ctrl, qacc_warmstart, time (+ applied forces when a user has written them)
  if (live) {
  c.each(h.nq, [&](int i) { b.qpos[i] = GA(qpos, i); });
  c.each(h.nv, [&](int i) { b.qvel[i] = GA(qvel, i); b.qacc_warmstart[i] = GA(qacc_warmstart, i); b.qfrc_applied[i] = a.applied ? GA(qfrc_applied, i) : (T)0; b.qacc[i] = 0; });
  c.each(h.nu, [&](int i) { b.ctrl[i] = GA(ctrl, i); });
  c.each(h.na, [&](int i) { b.act[i] = GA(act, i); b.act_dot[i] = 0; });
  c.each(3 * h.nmocap, [&](int i) { b.mocap_pos[i] = GA(mocap_pos, i); });
  c.each(4 * h.nmocap, [&](int i) { b.mocap_quat[i] = GA(mocap_quat, i); });
  c.each(h.neq, [&](int i) { b.eq_active[i] = GA(eq_active, i); });
  c.each(6 * h.nbody, [&](int i) { b.xfrc_applied[i] = a.applied ? GA(xfrc_applied, i) : (T)0; });
  if (gl == 0) {
    b.time[0] = GA(time, 0);
    b.diverged[0] = g.diverged[ue]; b.acc_ncon[0] = g.acc_ncon[ue]; b.acc_nefc[0] = g.acc_nefc[ue]; b.acc_niter[0] = g.acc_niter[ue];
    b.ncon[0] = 0; b.nefc[0] = 0; b.solver_niter[0] = 0; b.ne[0] = 0;
  }
  }
  __syncwarp(gmask);
  const int32_t div0 = b.diverged[0];
  const long long step0 = a.d_step ? *a.d_step : a.step0;
  for (int s = 0; s < a.nsteps; s++) {
    // a spare group fills its own view too (never written back): a `live` test here costs k_step_coop<double, 32> a spill
    if (a.philox) {
      if (gl == 0) env.fill_ctrl_philox(a.seed, a.env_id_offset + e, step0 + s, (T)a.ctrl_scale);
      __syncwarp(gmask);
    }
    c.step();
  }
  if (!live) return;
  // ---- state out: qpos, qvel, act, time, qacc, qacc_warmstart, sensordata, counters (+ what an auto-reset cleared)
  const bool did_reset = b.diverged[0] != div0;
  c.each(h.nq, [&](int i) { GA(qpos, i) = b.qpos[i]; });
  c.each(h.nv, [&](int i) { GA(qvel, i) = b.qvel[i]; GA(qacc, i) = b.qacc[i]; GA(qacc_warmstart, i) = b.qacc_warmstart[i]; });
  c.each(h.na, [&](int i) { GA(act, i) = b.act[i]; GA(act_dot, i) = b.act_dot[i]; });
  c.each(h.nsensordata, [&](int i) { GA(sensordata, i) = b.sensordata[i]; });
  if (a.philox || did_reset) c.each(h.nu, [&](int i) { GA(ctrl, i) = b.ctrl[i]; });
  if (did_reset) {
    c.each(3 * h.nmocap, [&](int i) { GA(mocap_pos, i) = b.mocap_pos[i]; });
    c.each(4 * h.nmocap, [&](int i) { GA(mocap_quat, i) = b.mocap_quat[i]; });
    c.each(h.neq, [&](int i) { GA(eq_active, i) = b.eq_active[i]; });
    c.each(h.nv, [&](int i) { GA(qfrc_applied, i) = b.qfrc_applied[i]; });
    c.each(6 * h.nbody, [&](int i) { GA(xfrc_applied, i) = b.xfrc_applied[i]; });
  }
  if (gl == 0) {
    GA(time, 0) = b.time[0];
    g.diverged[ue] = b.diverged[0]; g.acc_ncon[ue] = b.acc_ncon[0]; g.acc_nefc[ue] = b.acc_nefc[0]; g.acc_niter[ue] = b.acc_niter[0];
    g.ncon[ue] = b.ncon[0]; g.nefc[ue] = b.nefc[0]; g.solver_niter[ue] = b.solver_niter[0];
  }
#undef GA
}

#endif  // __CUDACC__

// ---- host side
template <typename T> static int coop_group_size(const ox_model_tables& t) { return t.nv <= 16 ? 16 : 32; }

bool step_coop_eligible(const ox_model_tables& t) {
  for (int i = 0; i < t.nu; i++)
    if (t.actuator_trntype[i] != OX_TRN_JOINT) return false;   // the lane = dof gather of the actuator forces knows joint transmissions only
  return t.nv >= 1 && t.nv <= 32 && t.solver == OX_SOL_NEWTON && t.noslip_iterations == 0 && t.nfloss == 0 && t.cone == OX_CONE_PYRAMIDAL && (t.integrator == OX_INT_EULER || t.integrator == OX_INT_IMPLICITFAST);
}
template <typename T>
static size_t coop_group_bytes_host(const ox_model_tables& t, int G) {
  CoopSizes<T> z;
  z.nq = t.nq; z.nv = t.nv; z.nu = t.nu; z.na = t.na; z.nb = t.nbody; z.nj = t.njnt; z.ng = t.ngeom; z.ns = t.nsite; z.nM = t.nM;
  z.ncm = t.nconmax > 1 ? t.nconmax : 1; z.nem = t.nefcmax > 1 ? t.nefcmax : 1; z.nsd = t.nsensordata; z.nmc = t.nmocap; z.neq = t.neq; z.nten = t.ntendon;
  return coop_group_bytes<T>(z, G);
}
size_t step_coop_smem(const ox_model_tables& t, int blob_bytes, bool f64) {
  const int G = t.nv <= 16 ? 16 : 32;
  const size_t gb = f64 ? coop_group_bytes_host<double>(t, G) : coop_group_bytes_host<float>(t, G);
  return (size_t)((blob_bytes + 127) / 128) * 128 + (size_t)(COOP_THREADS / G) * gb;
}
cudaError_t step_coop_prepare(const ox_model_tables& t, int blob_bytes, bool f64) {
  const size_t smem = step_coop_smem(t, blob_bytes, f64);
  if (smem > 227 * 1024) return cudaErrorInvalidValue;
  const int G = t.nv <= 16 ? 16 : 32;
  if (f64) return G == 16 ? cudaFuncSetAttribute(k_step_coop<double, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                          : cudaFuncSetAttribute(k_step_coop<double, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  return G == 16 ? cudaFuncSetAttribute(k_step_coop<float, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                 : cudaFuncSetAttribute(k_step_coop<float, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}
template <typename T>
static cudaError_t launch_coop_step(cudaStream_t stream, const ox_model_tables& t, const unsigned char* blob, int bytes, const DevBatch<T>& g, const StepArgs& a) {
  const int G = t.nv <= 16 ? 16 : 32;
  const int gpc = COOP_THREADS / G, grid = (g.nenv + gpc - 1) / gpc;
  const size_t gb = coop_group_bytes_host<T>(t, G);
  const size_t smem = (size_t)((bytes + 127) / 128) * 128 + (size_t)gpc * gb;
  if (G == 16) k_step_coop<T, 16><<<grid, COOP_THREADS, smem, stream>>>(blob, bytes, g, a, (int)gb);
  else k_step_coop<T, 32><<<grid, COOP_THREADS, smem, stream>>>(blob, bytes, g, a, (int)gb);
  return cudaPeekAtLastError();
}
cudaError_t launch_step_coop_f32(cudaStream_t s, const ox_model_tables& t, const unsigned char* blob, int bytes, const DevBatch<float>& g, const StepArgs& a) { return launch_coop_step<float>(s, t, blob, bytes, g, a); }
cudaError_t launch_step_coop_f64(cudaStream_t s, const ox_model_tables& t, const unsigned char* blob, int bytes, const DevBatch<double>& g, const StepArgs& a) { return launch_coop_step<double>(s, t, blob, bytes, g, a); }

}  // namespace ox
