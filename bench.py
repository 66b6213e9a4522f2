#!/usr/bin/env python
"""bench.py - env-steps/s of the batched mj_step hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  # the CPU path (restated oracle) on the host cores
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # also write the state after the last timed step as DIR/<field>.npy

A "step" is one mj_step of every environment of the batch (cheetah, 8192 envs per GPU, fresh Philox
controls every step). `value` is whole-job env-steps/s with inputs resident in HBM; `e2e` is the same
metric through the C ABI with HOST buffers (controls H2D and observations D2H every step, inside the
timed region). PyTorch is plumbing only here: NCCL barrier / max-reduction and CUDA events on the
library's stream; all physics runs in libox_b200.so.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (it may be read-only)

SEED = 0x0B200
METRIC = "env-steps/sec"
UNIT = "env-steps/s"
# --dump-outputs: what a caller reads back after BatchedPhysics.step (fields of size 0 in a model are skipped), at most
# DUMP_BYTES of array data in all (with the .npy headers, under 64 MB); above that a fixed, seeded sample of environments
# (the same rows on every run) is written
DUMP_FIELDS = ("qpos", "qvel", "qacc", "act", "sensordata")
DUMP_BYTES = 60 << 20


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cheetah", choices=["pendulum", "cartpole", "acrobot", "cheetah", "humanoid"])
    ap.add_argument("--nenv", type=int, default=0, help="envs per GPU (0 = the BASELINE config's)")
    ap.add_argument("--precision", default="", choices=["", "f32", "f64"])
    ap.add_argument("--mode", default="fused", choices=["fused", "staged", "coop"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--block", type=int, default=0)
    ap.add_argument("--lanes", type=int, default=0, help="active envs per warp (0 = library default)")
    ap.add_argument("--iterations", type=int, default=0)
    ap.add_argument("--ls-iterations", type=int, default=0)
    ap.add_argument("--stage-times", action="store_true", help="also print per-stage device times (staged kernels)")
    ap.add_argument("--no-spec", action="store_true", help="use the generic fused kernel instead of the model-specialised one")
    ap.add_argument("--ctrl-scale", type=float, default=1.0, help="amplitude of the Philox control stream (power of two; 0.125 = the "
                    "resting-contact regime of the humanoid)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the state after the last timed step as DIR/<field>.npy (batch precision; single rank only)")
    return ap.parse_args()


def initial_state(model, nenv_total, lo, hi, seed=20261018):
    """Seeded initial states (SURVEY 8d), drawn row by row so env g gets the same state for any GPU count."""
    rng = np.random.default_rng(seed)
    nq, nv = model.nq, model.nv
    u = rng.uniform(-0.1, 0.1, (nenv_total, nq))[lo:hi]
    g = rng.normal(0.0, 1.0, (nenv_total, nq + nv))[lo:hi]
    qpos = np.tile(np.asarray(model.qpos0, dtype=np.float64), (hi - lo, 1))
    for j in range(model.njnt):
        jt, a = int(model.jnt_type[j]), int(model.jnt_qposadr[j])
        if jt in (2, 3):
            qpos[:, a] += u[:, a]
        else:
            if jt == 0:
                qpos[:, a + 2] += u[:, a + 2] + 0.1
                a += 3
            q = qpos[:, a:a + 4] + 0.05 * g[:, a:a + 4]
            qpos[:, a:a + 4] = q / np.linalg.norm(q, axis=1, keepdims=True)
    qvel = 0.1 * g[:, nq:]
    return qpos, qvel


def algorithmic_bytes_per_env_step(model, real_bytes):
    """SURVEY 8d: reads (nq + 2nv + nu + na + 1) + writes (nq + 3nv + na + 1) words."""
    return (2 * model.nq + 5 * model.nv + model.nu + 2 * model.na + 2) * real_bytes


def algorithmic_flops_per_env_step(model, ncon, nefc, niter, n_ls=5.0):
    """SURVEY Appendix C.3 flop model evaluated with measured mean ncon / nefc / solver iterations."""
    nb, nv, nM, ng, nu = model.nbody - 1, model.nv, model.nM, model.ngeom, model.nu
    depth = []
    for i in range(nv):
        d, a = 1, int(model.dof_parentid[i])
        while a >= 0:
            d, a = d + 1, int(model.dof_parentid[a])
        depth.append(d)
    sd2 = float(sum(d * d for d in depth))
    dbar = float(np.mean(depth)) if depth else 0.0
    fwd = (200 * nb + 76 * ng) + (104 * nb + 12 * nv) + (10 * nb + 40 * nv + 11 * nM) + 2 * sd2 + 32 * nv + (110 * nb + 23 * nv) \
        + (4 * nv + 6 * nu) + (50 * model.npair + 30 * ncon) + (35 * dbar * ncon + 30 * nefc + 2 * nefc * nv) + (4 * nM + nv)
    newton = nefc * nv * (nv + 1) + nv ** 3 / 3 + 2 * nv * nv + 6 * nefc * nv + 4 * nM + n_ls * 8 * nefc
    integ = 2 * sd2 + 8 * nM
    nfwd = 4 if model.integrator == 1 else 1
    return nfwd * (fwd + niter * newton) + integ


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML; nvidia-smi fallback)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if mask & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop_evt.wait(0.02)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def dump_outputs(b, out_dir, dtype):
    """Writes DUMP_FIELDS of the batch as out_dir/<field>.npy ([nenv, n] in dtype; [sampled envs, n] above DUMP_BYTES)."""
    fields = [f for f in DUMP_FIELDS if b.field_size(f) > 0]
    row_bytes = sum(b.field_size(f) for f in fields) * np.dtype(dtype).itemsize
    rows = None
    if row_bytes * b.nenv > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(SEED).choice(b.nenv, DUMP_BYTES // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for f in fields:
        a = b.get(f, dtype=dtype)
        np.save(os.path.join(out_dir, f"{f}.npy"), a if rows is None else a[rows])


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


def cpu_oracle_rate(model, cfgname, steps, warmup, budget_s=20.0, ctrl_scale=1.0):
    """Times the restated CPU oracle on all host cores on a bounded sample of the workload."""
    from support import oracle_bench, oracle_lib
    oracle_lib().oxo_set_ctrl_scale(C.c_double(ctrl_scale))
    threads = max(1, oracle_lib().oxo_hardware_threads())
    q, v = initial_state(model, 2 * threads, 0, 2 * threads)
    sec, _ = oracle_bench(model, q, v, 20, threads)  # calibration (also warms the threads)
    rate = max(1.0, 2 * threads * 20 / max(sec, 1e-6))
    total_steps = steps + warmup
    nenv_s = int(min(8192, max(threads, rate * budget_s / max(1, total_steps))))
    nenv_s = max(threads, nenv_s // threads * threads)
    q, v = initial_state(model, nenv_s, 0, nenv_s)
    if warmup > 0:
        oracle_bench(model, q, v, warmup, threads, SEED, 0, 0)
    sec, stats = oracle_bench(model, q, v, steps, threads, SEED, 0, warmup)
    value = nenv_s * steps / sec
    return {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{nenv_s} {cfgname} envs x {steps} steps (after {warmup} warm-up steps), restated CPU oracle "
                      f"(not libmujoco), fp64, {threads} threads, same Philox controls",
            "seconds": sec, "mean_ncon": stats[0], "mean_nefc": stats[1], "mean_solver_iters": stats[2]}, nenv_s


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path on the host cores. The real path (oxide_control -> rusty_mujoco ->
    libmujoco 3.3.2) cannot be built here (SURVEY F3/F6), so this is the restated oracle port, labelled as such."""
    if rank != 0:
        return
    import oxide_control_b200 as ox
    cfg = ox.models.CONFIGS[args.config]
    model = ox.Model.from_xml_string(cfg["xml"])
    t0 = time.time()
    base, nenv_s = cpu_oracle_rate(model, args.config, args.steps, args.warmup, budget_s=60.0, ctrl_scale=args.ctrl_scale)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * base["seconds"] / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{cfg['label']}: bounded sample of {nenv_s} envs per step on the host CPU"},
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.time() - t0,
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs applies to the CUDA path only")
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import oxide_control_b200 as ox
    from oxide_control_b200 import _abi as A
    from oxide_control_b200 import sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    if args.dump_outputs and world > 1:
        raise SystemExit("bench.py: --dump-outputs writes one batch; run it with a single rank")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cfg = ox.models.CONFIGS[args.config]
    model = ox.Model.from_xml_string(cfg["xml"])
    nenv = args.nenv or cfg["nenv"]
    precision = args.precision or cfg["precision"]
    real_bytes = 8 if precision == "f64" else 4
    K, W = args.steps, max(args.warmup, 3)

    b = ox.BatchedPhysics(model, nenv, precision=precision, device=local_rank, mode=args.mode, env_id_offset=rank * nenv,
                          block_threads=args.block, lanes_per_warp=args.lanes, iterations=args.iterations, ls_iterations=args.ls_iterations, specialize=not args.no_spec)
    lo, hi = sharding.shard_range(rank, world, nenv)   # global env ids of this rank: they key the Philox control stream
    qpos, qvel = initial_state(model, world * nenv, lo, hi)
    b.set("qpos", qpos)
    b.set("qvel", qvel)
    b.ctrl_philox(True, SEED)
    if args.ctrl_scale != 1.0:
        b.ctrl_philox_scale(args.ctrl_scale)
    stream = torch.cuda.ExternalStream(A.lib().ox_batch_stream(b.handle), device=local_rank)
    flush_buf = None if args.no_flush else torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        return sharding.max_over_ranks(x, device="cuda")   # NCCL all-reduce(MAX) of one double; the only collectives of the job are
                                                           # these report-boundary reductions (none touches the step)
    def sum_over_ranks(vec):
        tot = sharding.gather_stats(dict(zip(("sum_ncon", "sum_nefc", "sum_niter", "diverged"), vec)), device="cuda")
        return [tot[k] for k in ("sum_ncon", "sum_nefc", "sum_niter", "diverged")]

    # ---------------- device-resident throughput: W warm-up steps, then exactly K timed steps
    b.step(W)
    b.sync()
    b.stats()  # clear accumulators
    launches0 = b.launch_count()
    sampler = ClockSampler(local_rank)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    barrier()
    sampler.start()
    with torch.cuda.stream(stream):
        for i in range(K):
            if flush_buf is not None:
                flush_buf.zero_()  # evict L2 between timed steps (outside the event pair)
            evs[i][0].record(stream)
            b.step(1)
            evs[i][1].record(stream)
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs:   # before the runs below step the batch further
        dump_outputs(b, args.dump_outputs, np.float64 if precision == "f64" else np.float32)
    dev_ms = float(sum(s.elapsed_time(e) for s, e in evs))
    launches = b.launch_count() - launches0
    stats = b.stats()
    total_ms = max_over_ranks(dev_ms)
    value = world * nenv * K / (total_ms * 1e-3)
    st = sum_over_ranks([stats["sum_ncon"], stats["sum_nefc"], stats["sum_niter"], stats["diverged"]])
    denom = float(world * nenv * K)
    mean_ncon, mean_nefc, mean_iter = st[0] / denom, st[1] / denom, st[2] / denom

    # ---------------- resident, no flush, K steps in ONE launch (what an on-device RL loop sees)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with torch.cuda.stream(stream):
        e0.record(stream)
        b.step(K)
        e1.record(stream)
    barrier()
    resident_ms = max_over_ranks(float(e0.elapsed_time(e1)))
    value_resident = world * nenv * K / (resident_ms * 1e-3)

    # ---------------- end to end through the C ABI with host buffers
    e2e = None
    if not args.no_e2e:
        nu, nq, nv = model.nu, model.nq, model.nv
        npool = 8
        rng = np.random.default_rng(7 + rank)
        ctrl_pool = [torch.from_numpy((args.ctrl_scale * rng.uniform(-1, 1, (nenv, nu))).astype(np.float32)).pin_memory() for _ in range(npool)]
        obs_q = torch.empty((nenv, nq), dtype=torch.float32).pin_memory()
        obs_v = torch.empty((nenv, nv), dtype=torch.float32).pin_memory()
        b.ctrl_philox(False, SEED)
        Ke = K
        def e2e_step(i):
            b.set_ptr("ctrl", ctrl_pool[i % npool].data_ptr(), A.F32, A.MEM_HOST, A.LAYOUT_ENV_MAJOR)
            b.step(1)
            b.get_many_ptr(("qpos", "qvel"), (obs_q.data_ptr(), obs_v.data_ptr()), A.F32, A.MEM_HOST, A.LAYOUT_ENV_MAJOR)
        for i in range(3):
            e2e_step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(Ke):
            e2e_step(i)
        b.sync()
        t1 = time.perf_counter()
        barrier()
        e2e3_s = max_over_ranks(t1 - t0)
        # the same crossing through the single-call form (ox_batch_step_io): the specialised step kernel reads the pinned
        # controls and writes the pinned qpos / qvel itself, so the PCIe traffic overlaps the step and no pack kernels launch
        def e2e_step_io(i):
            b.step_io_ptr(ctrl_pool[i % npool].data_ptr(), obs_q.data_ptr(), obs_v.data_ptr(), A.F32, A.MEM_HOST)
        for i in range(3):
            e2e_step_io(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(Ke):
            e2e_step_io(i)
        b.sync()
        t1 = time.perf_counter()
        barrier()
        e2e_s = max_over_ranks(t1 - t0)
        e2e = {"value": world * nenv * Ke / e2e_s, "unit": UNIT, "h2d_bytes_per_step": nenv * nu * 4,
               "d2h_bytes_per_step": nenv * (nq + nv) * 4, "ms_per_step": 1e3 * e2e_s / Ke,
               "three_call_value": world * nenv * Ke / e2e3_s, "three_call_ms_per_step": 1e3 * e2e3_s / Ke,
               "timing": "host wall clock around K x ox_batch_step_io(ctrl pinned host -> qpos, qvel pinned host), which returns "
                         "after the outputs are complete; the step kernel reads / writes the pinned buffers over PCIe itself. "
                         "three_call_* = the same loop as ox_batch_set(ctrl) + ox_batch_step(1) + ox_batch_get_many(qpos, qvel). "
                         "No L2 flush inside this loop (value is measured with one), so e2e can exceed value; max over ranks"}
        finite = bool(np.isfinite(obs_q.numpy()).all())
        # ---------------- N1: the same loop through the on-device Environment / Task layer (ox_env_step): actions in,
        # observation + reward + discount + finished out, reward / finish / auto-reset evaluated on the GPU
        import oxide_control_b200 as ox
        task = ox.TaskSpec(obs=[("qpos", 0, nq), ("qvel", 0, nv)], reward=[("qvel", 0, "linear", 1.0)] + [("ctrl", i, "square", -0.1) for i in range(nu)],
                           time_limit=1000 * model.timestep, discount=0.99, init_qpos_noise=0.1, init_qvel_noise=0.1, seed=SEED)
        env = ox.BatchedEnvironment(b, task)
        obs = torch.empty((nenv, env.obs_dim), dtype=torch.float32).pin_memory()
        rew = torch.empty(nenv, dtype=torch.float32).pin_memory()
        dis = torch.empty(nenv, dtype=torch.float32).pin_memory()
        fin = torch.empty(nenv, dtype=torch.uint8).pin_memory()
        def env_step(i):
            env.step_ptr(ctrl_pool[i % npool].data_ptr(), obs.data_ptr(), rew.data_ptr(), dis.data_ptr(), fin.data_ptr(), A.F32, A.MEM_HOST)
        for i in range(3):
            env_step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(Ke):
            env_step(i)
        b.sync()
        t1 = time.perf_counter()
        barrier()
        env_s = max_over_ranks(t1 - t0)
        env_line = {"value": world * nenv * Ke / env_s, "unit": UNIT, "h2d_bytes_per_step": nenv * nu * 4,
                    "d2h_bytes_per_step": nenv * (env.obs_dim * 4 + 4 + 4 + 1), "ms_per_step": 1e3 * env_s / Ke,
                    "timing": "host wall clock around K x ox_env_step(action pinned host -> obs, reward, discount, finished pinned host); "
                              "reward, finish test and auto-reset on device; max over ranks"}
        finite = finite and bool(np.isfinite(obs.numpy()).all())
        env.close()
        b.ctrl_philox(True, SEED)
    else:
        finite = True
        env_line = None

    # ---------------- roofline of the dominant kernel (the step kernel: the only kernel of a step)
    peaks, peak_src = load_peaks()
    step_ms = dev_ms / K  # this rank's average launch duration
    alg_bytes = algorithmic_bytes_per_env_step(model, real_bytes) * nenv
    achieved = alg_bytes / (step_ms * 1e-3) / 1e9
    flops = algorithmic_flops_per_env_step(model, mean_ncon, mean_nefc, mean_iter)
    fp_nominal = 148 * 128 * 2 * peaks.get("sm_max_mhz", 1965.0) * 1e6 / 1e12 * (0.5 if precision == "f64" else 1.0)
    fp_peak = ox.measure_fma_peak(local_rank, precision)   # measured on this GPU, now: register-resident FMA chains on every SM
    fp_achieved = flops * nenv / (step_ms * 1e-3) / 1e12
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                "peak_source": f"{peak_src} copy bandwidth (burst)", "kernel": (f"k_step_spec<Spec_{args.config},{precision}>" if b.kernel_name() == args.config else f"{b.kernel_name()} <{precision}>"),
                "algorithmic_bytes_per_env_step": algorithmic_bytes_per_env_step(model, real_bytes),
                "fp_model_flops_per_env_step": flops, "fp_achieved_tflops": fp_achieved, "fp_peak_tflops_measured": fp_peak,
                "fp_peak_tflops_nominal": fp_nominal, "fp_frac": fp_achieved / fp_peak,
                "note": "latency/issue-bound physics: both fractions are small by construction (SURVEY 8d)"}
    # per-launch DRAM traffic and issue-slot utilisation of the same kernel from the committed ncu capture (profiles/ncu_summary.json,
    # written by tools/ncu_summary.py from an `ncu --set full` report); the keys are present only for configurations that were captured
    spath = os.path.join(ROOT, "profiles", "ncu_summary.json")
    roofline["traffic"] = None
    if os.path.exists(spath):
        try:
            with open(spath) as f:
                cap = json.load(f).get(f"{args.config}_{precision}_{nenv}")
            if cap:
                roofline["traffic"] = cap.get("dram_bytes_per_launch")
                roofline["issue_slot_util_pct_ncu"] = cap.get("issue_active_pct")
                roofline["ncu_source"] = cap.get("source")
        except Exception:
            pass

    # ---------------- CPU baseline beside it (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu, _ = cpu_oracle_rate(model, args.config, min(K, 200), min(W, 100), budget_s=15.0, ctrl_scale=args.ctrl_scale)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "mean_ncon", "mean_nefc", "mean_solver_iters")}

    stage_times = b.stage_times(5) if args.stage_times else None

    if rank == 0:
        arena_mb = None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": precision, "data": "synthetic",
            "config": {"workload": f"{cfg['label']}: {nenv} envs per GPU, fresh Philox {args.ctrl_scale:g}*U(-1,1) controls every step, "
                                   f"{'RK4' if model.integrator == 1 else 'Euler'}, Newton solver, mode={args.mode}, kernel={b.kernel_name()}",
                       "envs_per_gpu": nenv, "parallelism": f"env-sharded x{world}, no data-path collective",
                       "l2": "none (state resident by design)" if args.no_flush else
                             "L2 flushed (256 MiB memset) between timed steps, outside the per-step event pairs"},
            "e2e": e2e, "env_step": env_line, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "value_resident_one_launch": value_resident, "ms_per_step_resident": resident_ms / K,
            "mean_ncon": mean_ncon, "mean_nefc": mean_nefc, "mean_solver_iters": mean_iter, "diverged_resets": st[3],
            "finite": finite, "timing": "CUDA events on the library's stream around every step, summed; max over ranks",
        }
        if stage_times:
            line["stage_times_ms"] = stage_times
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
