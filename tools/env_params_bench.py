"""Throughput cost of per-env tendon and actuator parameters: one JSON line comparing, in the same process and
alternated window by window, three configurations of the flagship env (tr_env straight, reset_pool="auto"):

  off      -- no per-env parameters (the default kernels)
  nominal  -- per-env kernels, every row the nominal row (param ranges of scale 1)
  ranges   -- per-env kernels, every field redrawn in nominal x [0.8, 1.2] at each reset

bench.py's protocol: a reset, 200 untimed settle steps, then timed single steps between CUDA events, with the L2 flushed
between timed steps when the state working set would fit it.  Usage:

    python tools/env_params_bench.py --xml flat --envs 131072 [--steps 30 --reps 5]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

CTRL_LO, CTRL_HI = -0.45, -0.15   # bench.py's control range
L2_BYTES = 126 * 2 ** 20


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "power_limit": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--xml", default="flat")
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--steps", type=int, default=30, help="timed steps per window")
    ap.add_argument("--reps", type=int, default=5, help="windows per configuration (alternated)")
    ap.add_argument("--settle", type=int, default=200)
    args = ap.parse_args()

    import torch
    from tensegrity_rl_b200 import TensegrityVecEnv, lib

    dev = torch.device("cuda", 0)
    n = args.envs
    configs = {"off": None, "nominal": {f: (1.0, 1.0) for f in lib.PARAM}, "ranges": {f: (0.8, 1.2) for f in lib.PARAM}}
    envs = {}
    for k, pr in configs.items():
        envs[k] = TensegrityVecEnv(n, xml_file=args.xml, env="tr_env", seed=0, auto_reset=True,
                                   desired_action="straight", reset_pool="auto", param_ranges=pr)
        envs[k].reset_tensor()
        g = torch.Generator(device=dev); g.manual_seed(777)
        for _ in range(args.settle):
            envs[k].step_tensor(CTRL_LO + (CTRL_HI - CTRL_LO) * torch.rand(n, 6, generator=g, device=dev, dtype=torch.float64),
                                want_info=False)
    torch.cuda.synchronize()
    obs_dim = envs["off"].obs_dim
    flush = n * (96 * 8 + obs_dim * 8 + 6 * 8) < 2 * L2_BYTES
    scratch = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=dev) if flush else None
    g = torch.Generator(device=dev); g.manual_seed(1234)
    ms = {k: [] for k in configs}
    for rep in range(args.reps):
        for k, env in envs.items():
            ctrl = CTRL_LO + (CTRL_HI - CTRL_LO) * torch.rand(args.steps, n, 6, generator=g, device=dev, dtype=torch.float64)
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
            torch.cuda.synchronize()
            for s in range(args.steps):
                if flush:
                    scratch.fill_(s & 255)
                ev[s][0].record()
                env.step_tensor(ctrl[s], want_info=True)
                ev[s][1].record()
            torch.cuda.synchronize()
            ms[k].append(sum(a.elapsed_time(b) for a, b in ev))
    rate = {k: [n * args.steps / (t * 1e-3) for t in v] for k, v in ms.items()}
    med = {k: sorted(v)[len(v) // 2] for k, v in rate.items()}
    out = {"metric": "env_steps_per_s", "xml": args.xml, "envs": n, "reset_pool": envs["off"].reset_pool,
           "steps_per_window": args.steps, "windows": args.reps, "settle": args.settle,
           "l2": "flush between timed steps" if flush else "working set > 126 MB L2",
           "median": med, "windows_env_steps_per_s": rate,
           "ratio_nominal_vs_off": med["nominal"] / med["off"], "ratio_ranges_vs_off": med["ranges"] / med["off"],
           "spread_off": (max(rate["off"]) - min(rate["off"])) / med["off"]}
    out.update(gpu_info())
    print(json.dumps(out), flush=True)
    for env in envs.values():
        env.close()


if __name__ == "__main__":
    main()
