"""Device time of ox_batch_inverse next to ox_batch_forward on the same batch (DESIGN 3.6).

Workloads: cheetah with 8192 envs and humanoid with 4096 envs (the two flagship sizes of bench.py), fp32 and fp64, default
batch configuration. The state is seeded: hinge and slide joints perturbed, free roots lowered by up to 5 cm (few envs end
up in contact); qacc is the forward solution perturbed by noise. Protocol: CUDA events on the library's stream around each call, L2 flushed (256 MiB
memset) between calls outside the event pairs, warm-up calls first, then --calls timed calls of each, alternating
inverse / forward so that both see the same clocks. One JSON line per workload plus a header line with the device name, power
limit and maximum SM clock read in the same run; --out also writes them to a file.

    python tools/inverse_bench.py --calls 300 --out profiles/inverse_b200.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

WORKLOADS = [("cheetah", 8192), ("humanoid", 4096)]


def device_info() -> dict:
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                                      text=True, timeout=30).strip()
        pl, clk = [s.strip() for s in out.split(",")]
        info.update(power_limit=pl, max_sm_clock=clk)
    except Exception as e:   # noqa: BLE001  (reported, not hidden)
        info.update(power_limit=f"unavailable ({e})", max_sm_clock="unavailable")
    return info


def run(name: str, nenv: int, precision: str, calls: int, warmup: int) -> dict:
    import torch
    import oxide_control_b200 as ox
    from oxide_control_b200 import _abi as A
    m = ox.Model.from_xml_string(ox.models.CONFIGS[name]["xml"])
    rng = np.random.default_rng(7)
    b = ox.BatchedPhysics(m, nenv, precision=precision)
    qpos = np.tile(np.asarray(m.qpos0, float), (nenv, 1))
    for j in range(m.njnt):
        a = int(m.jnt_qposadr[j])
        if int(m.jnt_type[j]) == 0:
            qpos[:, a + 2] -= 0.05 * rng.uniform(0, 1, nenv)       # free root lowered: contacts
        elif int(m.jnt_type[j]) in (2, 3):
            qpos[:, a] += rng.uniform(-0.1, 0.1, nenv)
    b.set("qpos", qpos)
    b.set("qvel", rng.normal(0, 0.1, (nenv, m.nv)))
    b.set("ctrl", rng.uniform(-1, 1, (nenv, m.nu)))
    b.forward()
    b.sync()
    b.set("qacc", b.get("qacc") + rng.normal(0, 1.0, (nenv, m.nv)))
    stream = torch.cuda.ExternalStream(A.lib().ox_batch_stream(b.handle))
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    for _ in range(warmup):
        b.inverse()
        b.forward()
    b.sync()
    torch.cuda.synchronize()
    ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(calls)] for k in ("inverse", "forward")}
    n0 = b.launch_count()
    with torch.cuda.stream(stream):
        for i in range(calls):
            for k, fn in (("inverse", b.inverse), ("forward", b.forward)):
                flush.zero_()                      # evict L2 between calls, outside the event pair
                ev[k][i][0].record(stream)
                fn()
                ev[k][i][1].record(stream)
    torch.cuda.synchronize()
    launches = b.launch_count() - n0
    res = {"model": name, "nenv": nenv, "precision": precision, "calls": calls, "warmup": warmup, "kernel": b.kernel_name(),
           "launches_per_call": launches / (2 * calls), "mean_ncon": float(b.get("ncon").mean()), "mean_nefc": float(b.get("nefc").mean())}
    for k in ev:
        ms = np.array([s.elapsed_time(e) for s, e in ev[k]])
        res[k] = {"mean_ms": float(ms.mean()), "median_ms": float(np.median(ms)), "p10_ms": float(np.percentile(ms, 10)),
                  "p90_ms": float(np.percentile(ms, 90)), "env_calls_per_s": float(nenv / (ms.mean() * 1e-3))}
    res["inverse_over_forward_time"] = res["inverse"]["mean_ms"] / res["forward"]["mean_ms"]
    return res


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--calls", type=int, default=300, help="timed calls of each entry point (>= 200)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    args = ap.parse_args()
    if args.calls < 200:
        ap.error("--calls must be >= 200")
    import torch
    if not torch.cuda.is_available():
        sys.exit("inverse_bench: no CUDA device (this measurement needs the B200)")
    lines = [{"header": device_info(), "l2": "flushed (256 MiB memset) between calls, outside the event pairs",
              "timing": "CUDA events on the batch's stream around each call; inverse and forward alternate"}]
    print(json.dumps(lines[0]), flush=True)
    for name, nenv in WORKLOADS:
        for precision in ("f32", "f64"):
            r = run(name, nenv, precision, args.calls, args.warmup)
            print(json.dumps(r), flush=True)
            lines.append(r)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
