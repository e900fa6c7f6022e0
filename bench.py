#!/usr/bin/env python
"""bench.py -- env-steps/s of the tensegrity hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--envs E] [--impl reference] [--dump-outputs bench_outputs]

A "step" is one env step (frame_skip = 20 substeps + obs/reward/done, in-kernel auto reset) of ALL envs of a
rank: flat-ground XML, tr_env `straight`, fp64, uniform random ctrl in [-0.45, -0.15] drawn on the device
before the timed region (BASELINE configs[1] inputs at the per-GPU env count of configs[4]).  The timed window is
STEADY STATE: `--settle` untimed steps after the reset (contacts and Newton iterations per step grow for the first
~100 steps while the tendons contract); the post-reset transient is reported beside it.  Prints ONE JSON
line (rank 0).  `value` = whole-job env-steps/s with inputs resident in HBM, device-timed (CUDA events on the
launching stream), max over ranks; `e2e` = the same through the public host API (pinned host ctrl in, host
obs/reward/done out, copies inside the timed region); `roofline` / `cpu_baseline` per the round contract.
`--impl reference` times the CPU restatement of the reference path (the oracle; MuJoCo itself is not
installable here) on all host threads -- rank 0 only.
`--dump-outputs DIR` writes what the last timed step returned on rank 0 (obs, reward, done) as .npy files, so that
two builds run with the same arguments (identical seeded inputs) can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env-steps/sec (whole box, device-timed)"
UNIT = "env-steps/s"
CTRL_LO, CTRL_HI = -0.45, -0.15
L2_BYTES = 126 * 2 ** 20
DUMP_BYTES = 64 * 2 ** 20


def algorithmic_bytes(obs_dim):
    """SURVEY 8(d): state read + written once (71 doubles each way), ctrl in, obs / reward / done out."""
    return 2 * 71 * 8 + 6 * 8 + obs_dim * 8 + 8 + 1


def flops_per_env_step(ncon, niter_per_sub, frame_skip=20):
    """SURVEY 8(d) FLOP model (FMA = 2): per substep 3.0k + 0.45k*ncon + n_iter*(1.5k + 0.9k*ncon)."""
    return frame_skip * (3.0e3 + 0.45e3 * ncon + niter_per_sub * (1.5e3 + 0.9e3 * ncon))


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons while the timed region runs (recipe in B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); smax = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def run_reference(args, rank):
    """CPU arm: the oracle port of the reference path on all host threads (rank 0 only)."""
    if rank != 0:
        return
    from oracle import oracle as O
    threads = O.lib().tsgo_max_threads()
    n_envs = args.ref_envs or 128 * threads          # ~5-10 s of host work at the default --steps / --warmup
    b = O.Batch("flat", n_envs, seed=0)
    b.step(50, lo=0.15, hi=0.15)           # the reset warm-up (50 env steps), untimed, like the GPU arm's reset
    for _ in range(args.warmup):
        b.step(1, lo=CTRL_LO, hi=CTRL_HI)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        b.step(1, lo=CTRL_LO, hi=CTRL_HI)
    dt = time.perf_counter() - t0
    b.close()
    value = n_envs * args.steps / dt
    sample = "%d envs x %d env-steps (each 20 substeps), flat XML, random ctrl, %d host threads" % (n_envs, args.steps, threads)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "flat_random_ctrl_fp64 (CPU restatement of the reference path; MuJoCo 2.3.7 is not installable here)",
                   "envs": n_envs, "frame_skip": 20},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def dump_outputs(out_dir, obs, rew, done):
    """obs / reward (float64) and done (float32) of one step as DIR/<name>.npy, with env_index.npy naming the env of
    each row: every env when that fits in DUMP_BYTES, else a fixed seeded sample of envs in ascending order."""
    import numpy as np
    import torch
    n = obs.shape[0]
    row_bytes = (obs.shape[1] + 2) * 8 + 4           # obs, reward, env_index in float64; done in float32
    rows = np.arange(n)
    if n * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // row_bytes, replace=False))
    idx = torch.as_tensor(rows, device=obs.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("obs", obs), ("reward", rew), ("done", done.float())):
        np.save(os.path.join(out_dir, name + ".npy"), t[idx].cpu().numpy())
    np.save(os.path.join(out_dir, "env_index.npy"), rows.astype(np.float64))


def cpu_baseline_sample(seconds=12.0):
    from oracle import oracle as O
    threads = O.lib().tsgo_max_threads()
    n_envs = 32 * threads
    b = O.Batch("flat", n_envs, seed=0)
    b.step(50, lo=0.15, hi=0.15)
    b.step(2, lo=CTRL_LO, hi=CTRL_HI)
    t0 = time.perf_counter(); n = 0
    while time.perf_counter() - t0 < seconds:
        n += b.step(5, lo=CTRL_LO, hi=CTRL_HI)
    dt = time.perf_counter() - t0
    b.close()
    return {"value": n / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d envs, %d env-steps in %.1f s, flat XML random ctrl, oracle (our CPU restatement, not MuJoCo), "
                      "%d threads" % (n_envs, n, dt, threads)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--envs", type=int, default=131072, help="envs per GPU (weak scaling)")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--ref-envs", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--sweep", default="4096,65536", help="extra env counts timed briefly at N=1 (reported in config)")
    ap.add_argument("--settle", type=int, default=200, help="untimed env steps between the reset and the timed window")
    ap.add_argument("--no-workloads", action="store_true", help="skip the policy-rollout sub-results (BASELINE configs[2], [3])")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write obs / reward / done of the last timed step (rank 0's envs) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs needs --impl native")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from tensegrity_rl_b200 import TensegrityVecEnv

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # the JSON line must be the only thing on stdout: NCCL prints its version banner there when NCCL_DEBUG is set
        # (at communicator creation), so stdout points at stderr until the first collective has run
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier(device_ids=[local_rank])
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    n = args.envs

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def settle(env, n_envs, steps, seed):
        """untimed random-ctrl steps (same distribution as the timed ones)"""
        g = torch.Generator(device=dev); g.manual_seed(seed)
        for k in range(steps):
            c = CTRL_LO + (CTRL_HI - CTRL_LO) * torch.rand(n_envs, 6, generator=g, device=dev, dtype=torch.float64)
            env.step_tensor(c, want_info=False)

    def timed_run(env, n_envs, steps, warmup, flush):
        g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
        ctrl = CTRL_LO + (CTRL_HI - CTRL_LO) * torch.rand(steps + warmup, n_envs, 6, generator=g, device=dev, dtype=torch.float64)
        scratch = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=dev) if flush else None
        for k in range(warmup):
            env.step_tensor(ctrl[k], want_info=False)
        stats = torch.zeros(8, dtype=torch.float64, device=dev)   # reward sum, dones, then per-step means of ncon / niter / nls / overflow / bad
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        l0 = env.launches
        barrier()
        for k in range(steps):
            if flush:
                scratch.fill_(k & 255)       # evict L2 between timed iterations (outside the event pair)
            ev[k][0].record()
            obs, rew, done = env.step_tensor(ctrl[warmup + k], want_info=True)
            ev[k][1].record()
            stats[0] += rew.sum(); stats[1] += done.sum()
            stats[2:5] += env.info[:, 19:22].sum(0); stats[5:7] += env.info[:, 28:30].sum(0)
        if world > 1:                        # the only collective of the path: episode statistics
            dist.all_reduce(stats)
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in ev)
        return ms, env.launches - l0, stats

    env = TensegrityVecEnv(n, xml_file="flat", env="tr_env", device=local_rank, seed=0, env_id_base=rank * n,
                           auto_reset=True, desired_action="straight", reset_pool="auto")
    env.reset_tensor()
    torch.cuda.synchronize()
    state_bytes = n * (96 * 8 + env.obs_dim * 8 + 6 * 8)
    flush = state_bytes < 2 * L2_BYTES
    # the post-reset transient (steps W .. W+10 after the reset), for comparison with round 1's window
    ms_tr, _, st_tr = timed_run(env, n, 10, args.warmup, flush)
    transient = {"value": world * n * 10 / (ms_tr * 1e-3), "window": "env steps %d..%d after the reset" % (args.warmup, args.warmup + 10),
                 "mean_contacts": float(st_tr[2].item()) / (world * n * 10), "newton_iters_per_substep": float(st_tr[3].item()) / (world * n * 10 * 20)}
    settle(env, n, max(0, args.settle - args.warmup - 10), 777 + rank)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms, launches, stats = timed_run(env, n, args.steps, args.warmup, flush)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:   # env.obs / reward / done still hold the last timed step's results
        dump_outputs(args.dump_outputs, env.obs, env.reward, env.done)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * n * args.steps / (ms_max * 1e-3)

    # solver statistics averaged over ALL timed steps (for the FLOP model) and contact overflow / bad-state counters
    tot = world * n * args.steps
    ncon, niter, nls = float(stats[2].item()) / tot, float(stats[3].item()) / tot / 20, float(stats[4].item()) / tot / 20
    overflow, bad = float(stats[5].item()), float(stats[6].item())
    done_frac = float(stats[1].item()) / tot

    # ---- e2e: public host API, pinned host buffers, H2D + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        hc = torch.empty(n, 6, dtype=torch.float64).pin_memory()
        ho = torch.empty(n, env.obs_dim, dtype=torch.float64).pin_memory()
        hr = torch.empty(n, dtype=torch.float64).pin_memory()
        hd = torch.empty(n, dtype=torch.uint8).pin_memory()
        dc = torch.empty(n, 6, dtype=torch.float64, device=dev)
        gen = torch.Generator(); gen.manual_seed(99 + rank)
        ksteps, kwarm = args.steps, args.warmup
        hsrc = CTRL_LO + (CTRL_HI - CTRL_LO) * torch.rand(ksteps + kwarm, n, 6, generator=gen, dtype=torch.float64)
        # same steady-state workload as the device-timed loop: the envs simply keep stepping

        def host_step(k):
            hc.copy_(hsrc[k])                            # the caller's actions land in pinned memory
            dc.copy_(hc, non_blocking=True)              # H2D
            obs, rew, done = env.step_tensor(dc, want_info=False)
            ho.copy_(obs, non_blocking=True); hr.copy_(rew, non_blocking=True); hd.copy_(done, non_blocking=True)  # D2H
            torch.cuda.synchronize()
        for k in range(kwarm):
            host_step(k)
        barrier()
        t0 = time.perf_counter()
        for k in range(ksteps):
            host_step(kwarm + k)
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": world * n * ksteps / float(dt.item()), "unit": UNIT, "h2d_bytes_per_step": world * n * 6 * 8,
               "d2h_bytes_per_step": world * n * (env.obs_dim * 8 + 8 + 1), "steps": ksteps,
               "warmup": kwarm,
               "api": "TensegrityVecEnv.step_tensor with pinned host ctrl/obs/reward/done copies, wall clock, no L2 flush"}

    sweep = {}
    if rank == 0 and world == 1 and args.sweep:
        for s in [int(x) for x in args.sweep.split(",") if x]:
            if s == n:
                continue
            e2 = TensegrityVecEnv(s, xml_file="flat", env="tr_env", device=local_rank, seed=0, auto_reset=True, reset_pool="auto")
            e2.reset_tensor()
            settle(e2, s, 100, 555)
            m2, _, _ = timed_run(e2, s, 10, 3, True)
            sweep[str(s)] = s * 10 / (m2 * 1e-3)
            e2.close()
            if s <= 8192:   # BASELINE configs[1] proper: random ctrl, no resets inside the run (no pool slots to warm up)
                e2 = TensegrityVecEnv(s, xml_file="flat", env="tr_env", device=local_rank, seed=0, auto_reset=False, reset_pool=0)
                e2.reset_tensor()
                settle(e2, s, 100, 555)
                m2, _, _ = timed_run(e2, s, 10, 3, True)
                sweep["%d_no_auto_reset" % s] = s * 10 / (m2 * 1e-3)
                e2.close()
        # optional fp32 mode (north_star: 1e-4 tolerance class; the headline stays f64)
        try:
            e2 = TensegrityVecEnv(n, xml_file="flat", env="tr_env", device=local_rank, seed=0, auto_reset=True, reset_pool="auto", precision="f32")
            e2.reset_tensor()
            settle(e2, n, 100, 555)
            m2, _, _ = timed_run(e2, n, 10, 3, flush)
            sweep["fp32_%d" % n] = n * 10 / (m2 * 1e-3)
            e2.close()
        except Exception as ex:  # noqa: BLE001
            sweep["fp32_%d" % n] = "failed: %s" % ex

    # ---- sub-results for the other BASELINE configs (pretrained SAC actor in the loop, device resident), and the
    # same-total-N strong-scaling line of SURVEY 8(d) C5 at N > 1
    workloads = {}
    if not args.no_workloads:
        from tensegrity_rl_b200 import SacActor
        from tensegrity_rl_b200.rollout import rollout
        specs = [("configs[2] forward_uneven", "uneven", "tensegrity_env", dict(desired_action="straight", desired_direction=1), "forward", 65536),
                 ("configs[3] track_flat", "flat", "tr_env", dict(desired_action="tracking"), "traj_track", 262144)]
        for name, xml, ek, kw, pol, ne in specs:
            try:
                v = TensegrityVecEnv(ne, xml_file=xml, env=ek, device=local_rank, seed=3, env_id_base=rank * ne, auto_reset=True,
                                     reset_pool="auto", **kw)
                actor = SacActor(pol, device=dev, seed=3 + rank)
                v.reset_tensor()
                rollout(v, actor, 25, False)            # untimed: policy-driven steps after the reset
                barrier()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                st = rollout(v, actor, 15, False)
                b.record()
                barrier()
                tms = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
                if world > 1:
                    dist.all_reduce(tms, op=dist.ReduceOp.MAX)
                workloads[name] = {"env_steps_per_s": world * ne * 15 / (float(tms.item()) * 1e-3), "envs_per_gpu": ne, "xml": xml,
                                   "env": ek, "policy": pol, "stochastic": True, "timed_steps": 15, "untimed_steps_after_reset": 25,
                                   "mean_contacts": float(v.info[:, 19].mean()), "newton_iters_per_substep": float(v.info[:, 20].mean()) / 20}
                v.close()
            except Exception as ex:  # noqa: BLE001
                workloads[name] = {"failed": str(ex)}
    strong = None
    if world > 1:
        ns = max(1, n // world)
        v = TensegrityVecEnv(ns, xml_file="flat", env="tr_env", device=local_rank, seed=0, env_id_base=rank * ns, auto_reset=True,
                             desired_action="straight", reset_pool="auto")
        v.reset_tensor()
        settle(v, ns, 100, 555 + rank)
        m3, _, _ = timed_run(v, ns, 10, 3, True)
        t3 = torch.tensor([m3], dtype=torch.float64, device=dev)
        dist.all_reduce(t3, op=dist.ReduceOp.MAX)
        strong = {"total_envs": ns * world, "envs_per_gpu": ns, "value": world * ns * 10 / (float(t3.item()) * 1e-3), "unit": UNIT,
                  "note": "same total env count as the 1-GPU line, split over the ranks (strong scaling)"}
        v.close()

    if rank == 0:
        obs_dim = env.obs_dim
        balg = algorithmic_bytes(obs_dim)
        kernel_ms = ms_max / args.steps          # one step kernel launch per step (+ a masked reset launch)
        achieved = balg * n / (kernel_ms * 1e-3) / 1e9
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:  # noqa: BLE001
            pass
        peak = peaks.get("hbm_gbs", 6650.0)
        traffic, traffic_note = None, "no ncu capture committed"
        try:   # dram__bytes_read + dram__bytes_write of ONE step-kernel launch from the committed ncu --set full capture
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            traffic = tj["bytes_per_env_step"] * n
            traffic_note = "ncu --set full at %d envs (profiles/r2_traffic.json)%s" % (
                tj["envs"], "" if tj["envs"] == n else ", scaled per env to %d" % n)
        except Exception:  # noqa: BLE001
            pass
        fl = flops_per_env_step(ncon, niter)
        tflops = fl * n / (kernel_ms * 1e-3) / 1e12
        fp64_peak, fp64_src = 37.0, "nominal 148 SM x 64 DFMA/clk x 2 x 1.965 GHz"
        try:   # DFMA peak measured on this pool's B200s with tools/proto/peak_fma.cu
            fp64_peak = json.load(open(os.path.join(ROOT, "profiles", "r1c_vector_peaks.json")))["fp64_dfma_tflops"]
            fp64_src = "measured DFMA peak on this pool's B200s (profiles/r1c_vector_peaks.json; MEASURED_PEAKS.json holds no fp64 figure)"
        except Exception:  # noqa: BLE001
            pass
        cfgk = env.kernel_config()
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "flat_random_ctrl_fp64: 3prism_jonathan_steady_side.xml, tr_env straight, ctrl~U[-0.45,-0.15], "
                                   "%d envs/GPU (BASELINE configs[1] inputs at the configs[4] per-GPU env count)" % n,
                       "envs_per_gpu": n, "frame_skip": 20, "obs_dim": obs_dim, "auto_reset": True, "reset_pool_slots": env.reset_pool,
                       "l2": "flush between timed steps" if flush else "state+obs working set %.0f MB > 126 MB L2" % (state_bytes / 2 ** 20),
                       "window": "steady state: %d untimed env steps after the reset, then %d warm-up + %d timed" % (args.settle, args.warmup, args.steps),
                       "transient": transient,
                       "done_fraction_per_step": done_frac, "mean_contacts": ncon, "newton_iters_per_substep": niter,
                       "linesearch_evals_per_substep": nls, "contact_overflow": overflow, "bad_state": bad,
                       "stats": "averaged over all timed steps",
                       "kernel": cfgk, "sweep_env_steps_per_s": sweep, "workloads": workloads, "strong_scaling": strong},
            "clocks": clocks, "gpu_launches": launches,
            # SURVEY 8(d): neither HBM nor tensor cores bind this path; the nominal bound is the FP64 (DFMA) pipe, so the
            # roofline is reported on that axis (algorithmic flops of the measured contact / iteration counts), HBM beside it
            "roofline": {"bound": "fp64", "achieved": tflops, "peak": fp64_peak, "unit": "TFLOP/s", "frac": tflops / fp64_peak,
                         "traffic": traffic, "traffic_note": traffic_note, "peak_source": fp64_src,
                         "algorithmic_flops_per_env_step": fl,
                         "flop_model": "SURVEY 8(d): 20 x [3.0k + 0.45k ncon + n_iter (1.5k + 0.9k ncon)], FMA = 2, with the measured means",
                         "hbm": {"achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                                 "algorithmic_bytes_per_env_step": balg, "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"},
                         "note": "latency bound: 6 resident warps per SM (shared memory: 3.6 KB per env, ten envs per warp) walking "
                                 "dependent fp64 chains in lock step; no pipe is above 15 % busy (profiles/r2_*)"},
        }
        if e2e:
            out["e2e"] = e2e
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline_sample()
        print(json.dumps(out), flush=True)
    env.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
