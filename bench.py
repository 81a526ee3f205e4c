#!/usr/bin/env python3
"""bench.py — env-steps/sec of jvrc_walk (BASELINE.json metric) on N x B200, one JSON line on rank 0.

A "step" is one pass of the rollout hot path over one batch: one control step (25 physics substeps + reward +
observation + termination + auto-reset) for every environment of the batch — the work of
BaseHumanoidEnv.step x num_envs in the reference.  Workload: BASELINE.json configs[1], jvrc_walk, 4096
environments per GPU (weak scaling: envs shard by index, no data-path collective), actions ~ N(0, 0.223^2)
(the action distribution of the reference's freshly initialised Gaussian_FF_Actor: output layer x0.01,
std_dev 0.223), synthetic, generated up front.

  value   device-resident: actions already in HBM, one lhw_sim_step launch per step.
  e2e     the same steps through the host-facing API: actions from pinned host memory (H2D every step),
          observation / reward / done read back to pinned host memory (D2H every step).
  roofline  the step kernel: algorithmic HBM bytes per env-step (SURVEY.md §8d) x envs / CUDA-event time of
          the launches, against the measured HBM peak (MEASURED_PEAKS.json).  The kernel is ALU/latency bound;
          the honest secondary bound is reported beside it as roofline.issue (warp-instruction issue rate, instruction
          count per env-step from the committed ncu capture); roofline.traffic = DRAM bytes of that capture.  Both come
          from profiles/ncu_counters.json and are only used when that capture was taken on the step kernels of THIS
          build (md5 of their SASS, learninghumanoidwalking_b200/build.py); otherwise they are null and say why.
  train_iter  (every N) whole PPO iterations the way the reference defines fps (rl/algos/ppo.py:468-595: sampling +
          optimisation): 4096 envs/GPU x 400 steps, GAE, advantage normalisation, 3 epochs of minibatch updates with
          run_experiment.py's default flags, every optimiser step containing the gradient exchange across the N GPUs;
          `exchange_us` = that exchange step alone (all-reduce + 2 x clip + 2 x Adam), fused peer-memory kernels vs NCCL.
  cpu_baseline / --impl reference   the CPU restatement (oracle/, "port": the reference's own MuJoCo path is
          not installable here) on the box's host cores, same workload, bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env-steps/sec jvrc_walk"
UNIT = "env-steps/s"
SIGMA = 0.223
ALG_BYTES = {32: 1220, 64: 2288}   # SURVEY.md §8d: state read+write, action read, obs/reward/done write


TRAINED_ACTOR = os.path.join(ROOT, "tests", "golden", "trained_actor_jvrc_walk.pt")


def ncu_counters(workload: str, precision: int):
    """(dram bytes, warp instructions) per 4096-env launch from the committed ncu capture, or (None, reason).  The capture is
    only valid for the kernels it was taken on: profiles/ncu_counters.json records the md5 of their SASS (build_record.json).  Under ncu the
    state record is L2 resident when the launch starts (no flush between replays), so the DRAM traffic is BELOW the
    algorithmic bytes; nothing is re-read."""
    try:
        from learninghumanoidwalking_b200.build import step_kernel_sass_md5
        c = json.load(open(os.path.join(ROOT, "profiles", "ncu_counters.json")))
        if c.get("step_kernel_sass_md5") != step_kernel_sass_md5():
            return None, (f"profiles/ncu_counters.json was captured on step-kernel SASS {c.get('step_kernel_sass_md5')}, "
                          f"this build is {step_kernel_sass_md5()}")
        w = c["launch_4096_envs"].get(f"{workload}/fp{precision}")
        if w is None:
            return None, "no capture of this workload / precision"
        return (float(w["dram_bytes"]), float(w["warp_instructions"])), c.get("source")
    except Exception as e:
        return None, f"no usable profiles/ncu_counters.json ({type(e).__name__})"


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 8 and r[4 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def effective_cpus() -> int:
    """Host cores this process may really use: affinity mask capped by the cgroup CPU quota (the GPU boxes expose 128
    logical CPUs but a container quota of 16)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(round(int(q) / int(per)))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, int(round(q / per))))
        except Exception:
            pass
    return n


WORKLOADS = {
    "jvrc_walk": dict(model="jvrc_walk", metric="env-steps/sec jvrc_walk",
                      desc="jvrc_walk {n} envs/GPU (BASELINE configs[1]), JVRC-1 sim_dt=0.001 control_dt=0.025 flat terrain"),
    "jvrc_step": dict(model="jvrc_step", metric="env-steps/sec jvrc_step",
                      desc="jvrc_step footstep-plan task {n} envs/GPU (BASELINE configs[2]), JVRC-1 sim_dt=0.001 control_dt=0.025, "
                           "20 stepping-stone slabs per env (footstep sequences, floor dropped in FORWARD mode, 0.1 m stairs: "
                           "iteration_count = inf) in the kernel"),
    "jvrc_walk_terrain": dict(model="jvrc_walk_terrain", metric="env-steps/sec jvrc_walk uneven/compliant terrain",
                              desc="jvrc_walk on uneven / compliant terrain {n} envs/GPU (BASELINE configs[4]; an EXTENSION — the reference "
                                   "has only the unused manip_hfield hook): 20 terraces re-posed with the hook's ranges, contact solref 0.04 s"),
    "h1": dict(model="h1", metric="env-steps/sec h1 standing",
               desc="h1 standing task {n} envs/GPU (BASELINE configs[3]), Unitree H1 sim_dt=0.001 control_dt=0.025, observation "
                    "noise + dynamics randomisation (damping, frictionloss, mass, CoM) + random pushes in the kernel"),
}


def cpu_reference(n_envs: int, seconds: float, warmup: int, seed: int, nthreads: int = 0, model: str = "jvrc_walk"):
    """The oracle (CPU port of the reference path) on the host cores, run for about `seconds` of wall time
    (a bounded sample of the same workload): env-steps/s, threads used, elapsed, control steps done."""
    import numpy as np
    from oracle.oracle import Oracle
    o = Oracle(model)
    nthreads = nthreads or effective_cpus()
    envs = o.make_envs(n_envs, seed=seed)
    o.batch_reset(envs, n_envs, nthreads)
    rng = np.random.RandomState(seed)
    for _ in range(warmup):
        o.batch_step(envs, n_envs, rng.normal(size=(n_envs, o.nu)) * SIGMA, 400, nthreads)
    steps, t0 = 0, time.perf_counter()
    while True:
        a = rng.normal(size=(n_envs, o.nu)) * SIGMA
        o.batch_step(envs, n_envs, a, 400, nthreads)
        steps += 1
        dt = time.perf_counter() - t0
        if dt >= seconds or steps >= 400:
            break
    return n_envs * steps / dt, nthreads, dt, steps


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """arrays: name -> [num_envs, ...] numpy array.  Float arrays keep their width, integer flags become float32.  Above
    DUMP_LIMIT_BYTES the same fixed, seeded sample of environment rows is taken from every array."""
    import numpy as np
    arrays = {k: v.astype(v.dtype if v.dtype in (np.float32, np.float64) else np.float32) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(v.nbytes // n for v in arrays.values())
    if n * row_bytes > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // row_bytes, replace=False))
        arrays = {k: v[rows] for k, v in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20, help="untimed control steps before the timed region (after the fixed "
                    "150-step pre-roll that brings the batch to its steady-state mix of episode ages)")
    ap.add_argument("--actions", default="noise", choices=["noise", "zero", "policy"],
                    help="noise: open loop N(0, 0.223^2) (headline); zero: a = 0, standing, 8 contacts (SURVEY 8d regime ii); "
                         "policy: closed loop, freshly initialised Gaussian_FF_Actor + exploration noise (regime i)")
    ap.add_argument("--no-train-iter", action="store_true")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=4096, help="environments per GPU")
    ap.add_argument("--precision", type=int, default=int(os.environ.get("LHW_BENCH_PRECISION", "64")), choices=[32, 64])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--workload", default="jvrc_walk", choices=sorted(WORKLOADS),
                    help="jvrc_walk: the configuration BASELINE.json's metric is quoted on (default); jvrc_step: configs[2]; h1: configs[3]; jvrc_walk_terrain: configs[4] (extension)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (obs, reward, done, ended of rank 0's "
                         "environments) to DIR/<name>.npy as float32 / float64, at most 64 MB in all (a fixed, seeded sample of "
                         "environments beyond that), so that two builds can be compared output for output on the same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the reference arm runs for a wall-time budget, not a fixed number of steps)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K, W = args.steps, max(3, args.warmup)
    PREROLL = 150    # untimed control steps BEFORE the W warm-up steps, whatever W the caller passes: >= 3 x the mean episode
    #                  length under the noisy actions, so that the timed steps see the steady-state mix of episode ages
    wl = WORKLOADS[args.workload]
    metric = wl["metric"]
    config = {"workload": wl["desc"].format(n=args.envs),
              "envs_per_gpu": args.envs, "global_envs": args.envs * world, "actions": f"N(0,{SIGMA}^2) synthetic, pre-generated",
              "parallelism": f"env-sharded x{world}; step kernel: no data-path collective; train_iter: one gradient exchange per optimiser step",
              "actions_regime": args.actions, "preroll_steps": PREROLL}

    if args.impl == "reference":
        # the reference's own Ray+MuJoCo path cannot be installed here (mujoco/ray absent, no network):
        # this arm times the CPU port (oracle/) on all host cores, rank 0 only, on the SAME number of environments.
        if rank != 0:
            return
        n_sample = args.envs * world
        sps, threads, dt, steps_ref = cpu_reference(n_sample, 15.0, 2, args.seed, model=wl["model"])
        print(json.dumps({"metric": metric, "value": sps, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
                          "ms_per_step": 1e3 * dt / steps_ref, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "f64", "data": "synthetic", "impl": "reference", "config": config,
                          "cpu_baseline": {"value": sps, "unit": UNIT, "cores": threads, "kind": "port",
                                           "sample": f"{n_sample} envs (= the GPU arm's global batch) x {steps_ref} control steps ({dt:.1f} s) "
                                                     f"after 2 warm-up steps, OpenMP over envs; threads = cgroup CPU quota ({threads} of "
                                                     f"{os.cpu_count()} logical CPUs); reference Ray+MuJoCo path not runnable on this box "
                                                     "(mujoco/ray not installable)"},
                          "e2e": {"value": sps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    import torch.distributed as dist
    from learninghumanoidwalking_b200 import _lib
    from learninghumanoidwalking_b200.envs import BatchedHumanoidEnv
    from learninghumanoidwalking_b200.rl import FF_V, DeviceRolloutWorker, Gaussian_FF_Actor

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints its version banner on the process's stdout (fd 1) when NCCL_DEBUG=VERSION is set in the environment;
        # stdout carries exactly ONE JSON line, so fd 1 points at stderr while the communicator comes up
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()     # before the warm-up: nvidia-smi needs a few hundred ms before its first sample
    n = args.envs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def make_policy(env):
        torch.manual_seed(args.seed)
        pol = Gaussian_FF_Actor(env.obs_dim, env.act_dim, init_std=SIGMA).to(dev)
        cri = FF_V(env.obs_dim).to(dev)
        pol.obs_mean = cri.obs_mean = torch.tensor(env.obs_mean, dtype=torch.float32, device=dev)
        pol.obs_std = cri.obs_std = torch.tensor(env.obs_std, dtype=torch.float32, device=dev)
        return pol, cri

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def timed_steps(env, regime, warm, steps, seed_off=0, do_flush=True):
        """`steps` control steps of `env` after `warm` untimed ones; returns the per-step CUDA-event times (the event pair
        brackets the step launch only; action generation and the L2 flush sit outside it)."""
        A, nn = env.act_dim, env.num_envs
        g = torch.Generator(device=dev).manual_seed(args.seed * 1000 + rank + seed_off)
        noise = torch.randn(warm + steps, nn, A, device=dev, generator=g, dtype=env.dtype) * SIGMA
        pol = make_policy(env)[0] if regime == "policy" else None
        if regime == "trained":      # the actor of a finished training run (tests/golden): a walking gait, 400-step episodes
            from learninghumanoidwalking_b200.rl.policies import install_reference_aliases
            install_reference_aliases()
            pol = torch.load(TRAINED_ACTOR, map_location="cpu", weights_only=False).to(dev).eval()
            noise = noise * (0.05 / SIGMA)
        obs = env.obs

        def action(k):
            if regime == "zero":
                return torch.zeros(nn, A, device=dev, dtype=env.dtype)
            if regime == "noise":
                return noise[k]
            with torch.no_grad():
                return (pol(obs.float()).to(env.dtype) + noise[k]).contiguous()
        for k in range(warm):
            obs = env.step(action(k))[0]
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        t0 = time.perf_counter()
        for k in range(steps):
            a = action(warm + k)
            if do_flush:
                flush.fill_(k & 0xFF)
            ev[k][0].record()
            obs = env.step(a)[0]
            ev[k][1].record()
        barrier()
        return [a.elapsed_time(b) for a, b in ev], time.perf_counter() - t0, noise[warm:]

    env = BatchedHumanoidEnv(n, model=wl["model"], precision=args.precision, seed=args.seed, first_env_id=rank * n,
                             device=local_rank)
    env.reset()
    A = env.act_dim
    launches0 = _lib.lib().lhw_launch_count()
    # ---- value: device resident, per-step CUDA events (L2 flushed before every step, flush not timed)
    step_ms, wall, acts = timed_steps(env, args.actions, PREROLL + W, K)
    total_ms = sum(step_ms)
    launches = K          # one lhw_sim_step launch per timed step (lhw_launch_count also counts the warm-up)
    assert _lib.lib().lhw_launch_count() - launches0 == K + W + PREROLL
    # env.step returns its own output buffers: until the next step they hold what the last timed step computed
    last_outputs = {name: t.cpu().numpy() for name, t in zip(("obs", "reward", "done", "ended"),
                                                            (env.obs, env.reward, env.done, env.ended))} if args.dump_outputs else None
    # ---- e2e: pinned host actions in, pinned host obs/reward/done out, every step
    h_acts = torch.empty(K, n, A, dtype=env.dtype).pin_memory()
    h_acts.copy_(acts.cpu())     # the policy regime's e2e leg plays the same exploration noise open loop (the host owns the actions)
    if args.actions == "zero":
        h_acts.zero_()
    h_obs = torch.empty(n, env.obs_dim, dtype=env.dtype).pin_memory()
    h_rew = torch.empty(n, dtype=env.dtype).pin_memory()
    h_done = torch.empty(n, dtype=torch.int32).pin_memory()
    d_act = torch.empty(n, A, dtype=env.dtype, device=dev)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(K):
        d_act.copy_(h_acts[k], non_blocking=True)
        obs, rew, done, _ = env.step(d_act)
        h_obs.copy_(obs, non_blocking=True)
        h_rew.copy_(rew, non_blocking=True)
        h_done.copy_(done, non_blocking=True)
        torch.cuda.current_stream().synchronize()   # the host consumer needs this step's result before the next action
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    iters = env.solver_iterations().float().mean().item()
    # ---- extras (not the headline): the other action regimes, the fp32 build of the same kernel, the full rollout loop with
    # the policy / critic MLPs (cuBLAS) and buffer writes in the loop (DeviceRolloutWorker.sample)
    extras = {}
    if not args.no_extras:
        Kx = max(20, min(K, 100))
        for regime in ("noise", "zero", "policy"):
            if regime == args.actions:
                extras[f"regime_{regime}_env_steps_per_s_per_gpu"] = n * K / (total_ms * 1e-3)
                continue
            ms, _, _ = timed_steps(env, regime, 30 if regime != "zero" else 60, Kx, seed_off=17)
            extras[f"regime_{regime}_env_steps_per_s_per_gpu"] = n * Kx / (sum(ms) * 1e-3)
        extras["regime_note"] = (f"device-resident, same kernel, {Kx} timed steps each (the headline regime: {K}); zero = standing with 8 "
                                 "contacts, policy = freshly initialised actor in the loop (its MLP is outside the event pair)")
        if wl["model"] == "jvrc_walk" and os.path.exists(TRAINED_ACTOR):
            ms, _, _ = timed_steps(env, "trained", 200, Kx, seed_off=23)
            extras["regime_trained_env_steps_per_s_per_gpu"] = n * Kx / (sum(ms) * 1e-3)
            extras["regime_trained_note"] = ("closed loop through tests/golden/trained_actor_jvrc_walk.pt (40 iterations of run_experiment.py "
                                             "train) + N(0, 0.05^2): the walking gait a training run converges to, after a 200-step warm-up")
        env32 = BatchedHumanoidEnv(n, model=wl["model"], precision=32, seed=args.seed, first_env_id=rank * n, device=local_rank)
        env32.reset()
        ms32, _, _ = timed_steps(env32, args.actions, 30, Kx, do_flush=False)
        extras["fp32_kernel_env_steps_per_s_per_gpu"] = n * Kx / (sum(ms32) * 1e-3)
        if n < 32768:      # the upper end of the north-star's batch range on this GPU (same fp64 kernel, 13.8 resident waves)
            big = BatchedHumanoidEnv(32768, model=wl["model"], precision=args.precision, seed=args.seed, first_env_id=rank * 32768,
                                     device=local_rank)
            big.reset()
            msb, _, _ = timed_steps(big, args.actions, 60, 30, do_flush=False)
            extras["envs_32768_env_steps_per_s_per_gpu"] = 32768 * 30 / (sum(msb) * 1e-3)
            big.close()
        # how long the fp32 kernel tracks the fp64 kernel (both product code, same seeds, a = 0): control steps until the
        # relative difference of qpos / qvel leaves 1e-4 (the parity bar applies to fp64; this is what fp32 costs)
        e64 = BatchedHumanoidEnv(64, model=wl["model"], precision=64, seed=args.seed + 1, device=local_rank)
        e32 = BatchedHumanoidEnv(64, model=wl["model"], precision=32, seed=args.seed + 1, device=local_rank)
        e64.reset(); e32.reset()
        inside = 200
        for k in range(200):
            e64.step(torch.zeros(64, A, device=dev, dtype=torch.float64))
            e32.step(torch.zeros(64, A, device=dev, dtype=torch.float32))
            d = max((e32.qpos.double() - e64.qpos).abs().max().item() / max(1.0, e64.qpos.abs().max().item()),
                    (e32.qvel.double() - e64.qvel).abs().max().item() / max(1.0, e64.qvel.abs().max().item()))
            if d > 1e-4:
                inside = k
                break
        extras["fp32_control_steps_inside_1e-4_of_fp64"] = inside
        e64.close(); e32.close(); env32.close()
        pol, cri = make_policy(env)
        worker = DeviceRolloutWorker(env, pol, cri, seed=args.seed)
        T = 32
        worker.sample(0.99, 0.95, T, 400)   # warm-up with the same horizon: captures the per-step CUDA graph
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        worker.sample(0.99, 0.95, T, 400)
        f1.record()
        barrier()
        extras["rollout_with_policy_env_steps_per_s_per_gpu"] = n * T / (f0.elapsed_time(f1) * 1e-3)
        extras["rollout_note"] = (f"DeviceRolloutWorker.sample: {T} control steps incl. actor+critic forward, sampling, buffer writes, GAE; batches of "
                                  ">= 1024 envs advance as two halves on two streams (one half's launch tail overlaps the other half's work), so "
                                  "this can exceed the isolated step-launch rate of `value`")
    env.close()
    # ---- train_iter: the PPO iteration as the reference defines fps, gradient exchange included, at every N
    train_iter = None
    if not args.no_train_iter:
        train_iter = bench_train_iter(args, wl, rank, world, local_rank, barrier)
    esz = 8 if args.precision == 64 else 4
    # max over ranks
    t = torch.tensor([total_ms, e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms = t.tolist()
    if rank == 0:
        value = n * world * K / (total_ms * 1e-3)
        e2e = n * world * K / (e2e_ms * 1e-3)
        peak, peak_src = peaks()
        kernel_ms = statistics.mean(step_ms)   # one launch per step: the event pair brackets exactly the step kernel
        # algorithmic bytes per env-step: state record read + written, actions in, obs / reward / flags out (DESIGN.md)
        state_reals = {"jvrc_walk": 119, "jvrc_step": 204, "jvrc_walk_terrain": 204, "h1": 188}[args.workload]
        obs_dim = {"jvrc_walk": 37, "jvrc_step": 39, "jvrc_walk_terrain": 37, "h1": 35}[args.workload]
        alg_bytes = ALG_BYTES[args.precision] if args.workload == "jvrc_walk" else \
            (2 * state_reals + A + obs_dim + 2) * esz + 2 * 8 * 4 + 2 * 4
        achieved = n * alg_bytes / (kernel_ms * 1e-3) / 1e9
        # secondary, honest bound: warp-instruction issue rate (instructions per env-step from the ncu capture of this
        # workload / precision) against 148 SMs x 4 schedulers x 1 warp-instruction per clock at the sampled SM clock
        cap, cap_src = ncu_counters(args.workload, args.precision)
        traffic, issue = None, {"unavailable": cap_src}
        if cap is not None:
            traffic = cap[0] * n / 4096.0
            inst_per_env_step = cap[1] / 4096.0
            sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
            issue_peak = 148 * 4 * sm_mhz * 1e6
            issue_ach = n * inst_per_env_step / (kernel_ms * 1e-3)
            issue = {"bound": "warp-issue", "achieved": issue_ach / 1e9, "peak": issue_peak / 1e9, "unit": "Gwarp-inst/s",
                     "frac": issue_ach / issue_peak, "warp_inst_per_env_step": inst_per_env_step, "source": cap_src}
        out = {"metric": metric, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
               "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "f64" if args.precision == 64 else "f32", "data": "synthetic",
               "config": dict(config, l2="flushed (256 MiB write) before every timed step; CUDA events bracket the step only",
                              wall_s_incl_flush=wall, newton_iters_per_env_step=iters),
               "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": n * A * esz,
                       "d2h_bytes_per_step": n * (obs_dim * esz + esz + 4)},
               "gpu_launches": int(launches),
               "clocks": clocks,
               "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                            "traffic": traffic, "peak_source": peak_src,
                            "algorithmic_bytes_per_env_step": alg_bytes,
                            "note": "the step kernel is ALU/latency bound (25 substeps of O(nv^3) work per ~2 KB of state); "
                                    "traffic = dram bytes of one 4096-env launch in the committed ncu capture (state L2 resident "
                                    "under ncu, hence below the algorithmic bytes), scaled to this batch; `issue` is the bound that "
                                    "actually applies",
                            "issue": issue}}
        out["extras"] = extras
        out["train_iter"] = train_iter
        if not args.no_cpu_baseline and world == 1:
            sps, threads, dt, nst = cpu_reference(n, 10.0, 2, args.seed, model=wl["model"])
            out["cpu_baseline"] = {"value": sps, "unit": UNIT, "cores": threads, "kind": "port",
                                   "sample": f"{n} envs (the GPU arm's batch) x {nst} control steps ({dt:.1f} s) after 2 warm-up steps, same "
                                             "action distribution; oracle/ C port with OpenMP (reference Ray+MuJoCo path not installable here)"}
        if last_outputs is not None:
            dump_outputs(args.dump_outputs, last_outputs)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def bench_train_iter(args, wl, rank, world, local_rank, barrier):
    """Whole PPO iterations (sampling + optimisation, rl/algos/ppo.py:468-595) with run_experiment.py's default flags on
    args.envs environments per GPU, and the exchange step (all-reduce + clip + Adam) timed alone, fused vs NCCL."""
    import importlib.util
    from functools import partial
    from types import SimpleNamespace

    import torch
    import torch.distributed as dist
    from learninghumanoidwalking_b200.envs import BatchedHumanoidEnv
    from learninghumanoidwalking_b200.rl import PPO
    from learninghumanoidwalking_b200.rl.comm import PeerComm
    from learninghumanoidwalking_b200.rl.optim import FusedClipAdam
    from learninghumanoidwalking_b200.rl.symmetric import SymmetricEnv
    spec = importlib.util.spec_from_file_location("lhw_run_experiment", os.path.join(ROOT, "run_experiment.py"))
    rx = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(rx)
    flags = {f[2:].replace("-", "_"): (False if kw.get("action") == "store_true" else kw.get("default")) for f, kw in rx.TRAIN_FLAGS}
    os.environ.setdefault("LHW_TENSORBOARD", "0")
    logdir = tempfile.TemporaryDirectory(prefix="lhw_bench_train_")     # the trainer's run directory: never in the tree
    dev = torch.device("cuda", local_rank)
    n, T, iters = args.envs, 400, 2
    out = {"definition": "samples / (sampling + optimisation time) as rl/algos/ppo.py:587-595, whole job, max over ranks of the wall "
                         f"time of {iters} iterations between barriers after 1 warm-up iteration (graph capture); no evaluation pass inside "
                         "(the reference evaluates every 100th iteration)",
           "flags": "run_experiment.py defaults (lr 3e-4, 3 epochs, minibatch 64 scaled by --minibatch-scale auto, mirror loss 0.4)",
           "envs_per_gpu": n, "steps_per_env": T, "samples_per_iteration": n * T * world}
    for prec in (args.precision, 32) if args.precision != 32 else (32,):
        base = partial(BatchedHumanoidEnv, n, model=wl["model"], precision=prec, seed=args.seed, first_env_id=rank * n,
                       device=local_rank, max_traj_len=T)
        probe = base()
        r = probe.robot
        probe.close()
        env_fn = base if not hasattr(r, "mirrored_obs") else partial(SymmetricEnv, base, mirrored_obs=r.mirrored_obs,
                                                                     mirrored_act=r.mirrored_acts, clock_inds=r.clock_inds)
        a = SimpleNamespace(**flags)
        a.num_procs, a.logdir, a.seed, a.eval_freq, a.eval_at_start, a.steps_per_env = n, logdir.name, args.seed, 10 ** 9, False, T
        a.env, a.precision = wl["model"], prec
        ppo = PPO(env_fn, a, seed=args.seed)
        ppo.train(None, 1, verbose=False)
        barrier()
        t0 = time.perf_counter()
        log = ppo.train(None, iters, verbose=False)
        barrier()
        dt = torch.tensor([time.perf_counter() - t0, log[-1]["sample_time"], log[-1]["optimize_time"]], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dt = dt.tolist()
        nb = (n * T) // ppo.minibatch_size
        out[f"fp{prec}"] = {"fps": world * n * T * iters / dt[0], "iter_s": dt[0] / iters, "sample_s": dt[1], "optimize_s": dt[2],
                            "minibatch_per_gpu": ppo.minibatch_size, "updates_per_iteration": nb * ppo.epochs,
                            "update_graph": ppo._ug is not None, "fused_exchange": ppo._comm is not None}
        ppo.env.close()
        if ppo._comm is not None:
            ppo._comm.close()
        del ppo
    # ---- the exchange step alone on the trainer's parameter count: fused (3 launches) vs NCCL all-reduce + 2 x (sumsq, clip+Adam)
    npar, n_actor = 154381, 78604
    comm = PeerComm(npar, dev)
    g = torch.Generator(device=dev).manual_seed(1)
    p, m, v = torch.randn(npar, device=dev, generator=g), torch.zeros(npar, device=dev), torch.zeros(npar, device=dev)
    comm.grad.copy_(torch.randn(npar, device=dev, generator=g) * 1e-3)

    def timed(fn, reps=200):
        for _ in range(20):
            fn()
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(reps):
            fn()
        a1.record()
        barrier()
        t = torch.tensor([a0.elapsed_time(a1) * 1e3 / reps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()
    ex = {"fused_peer_memory": timed(lambda: comm.fused_step(p, m, v, n_actor, 3e-4, (0.9, 0.999), 1e-5, 0.5))}
    comm.status()
    grad2 = torch.randn(npar, device=dev, generator=g) * 1e-3
    from learninghumanoidwalking_b200 import _lib
    L = _lib.lib()
    norm, stepd = torch.zeros(2, device=dev), torch.zeros(2, dtype=torch.int32, device=dev)

    def nccl_path():
        if world > 1:
            dist.all_reduce(grad2, op=dist.ReduceOp.SUM)
        st = _lib.current_stream_ptr()
        for k, (lo, hi) in enumerate(((0, n_actor), (n_actor, npar))):
            L.lhw_grad_sumsq(grad2[lo:hi].data_ptr(), norm[k:].data_ptr(), hi - lo, 1.0 / world, st)
            L.lhw_clip_adam_dev(p[lo:hi].data_ptr(), grad2[lo:hi].data_ptr(), m[lo:hi].data_ptr(), v[lo:hi].data_ptr(), norm[k:].data_ptr(),
                                hi - lo, stepd[k:].data_ptr(), 3e-4, 0.9, 0.999, 1e-5, 0.5, 1.0 / world, st)
    ex["nccl_allreduce_plus_clip_adam"] = timed(nccl_path)
    ex["note"] = ("microseconds per exchange step (gradient all-reduce over the N GPUs + clip_grad_norm_ x2 + Adam x2 on 154 381 parameters), "
                  "200 back-to-back steps between barriers, max over ranks; fused = csrc/comm_kernels.cu (3 launches), baseline = "
                  "torch.distributed NCCL all_reduce + lhw_grad_sumsq / lhw_clip_adam_dev per network (7 launches)")
    out["exchange_us"] = ex
    comm.close()
    logdir.cleanup()
    return out


if __name__ == "__main__":
    main()
